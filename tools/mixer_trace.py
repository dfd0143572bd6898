"""Per-CTA timeline (globaltimer stamps) of the last RepMixer depthwise launch of a forward (stage 2 at 1024 px)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import ml_fastvlm_b200 as pkg
from oracle import fixture as fx

NAMES = ["entry", "staged", "pdl_ok", "x_landed", "ph1_done(t0)", "ph1_sync", "ph2_done(t0)", "ph2_done(tN)"]


def main():
    R = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    dev = torch.device("cuda:0")
    pk = pkg.pack_tower(fx.tower_state_dict())
    pk.update(pkg.pack_projector(fx.projector_state_dict(896)))
    eng = pkg.Engine(R, 896, 2, 1).load(pk, dev)
    x = fx.synthetic_images(1, R).to(dev).to(torch.bfloat16)
    for _ in range(3):
        eng.forward(x, False, True)
    # one more forward with tracing on, launched step by step: a second engine, created under FVHD_NO_GRAPH=1 (switches are read
    # when a handle is created); the buffer keeps the stamps of the last mixer launch
    os.environ["FVHD_NO_GRAPH"] = "1"
    try:
        direct = pkg.Engine(R, 896, 2, 1).load(pk, dev)
    finally:
        os.environ.pop("FVHD_NO_GRAPH", None)
    direct.forward(x, False, True)
    n = 4096
    buf = torch.zeros(n * 8, dtype=torch.int64, device=dev)
    eng.lib.fvhd_debug_mixer_trace(buf.data_ptr())
    last = [i for i, s in enumerate(eng.steps(1)) if s["kernel"].startswith("repmixer")][-1]
    direct.forward(x, False, True)
    torch.cuda.synchronize()
    eng.lib.fvhd_debug_mixer_trace(None)
    t = buf.cpu().numpy().reshape(n, 8).astype(np.float64)
    t = t[t[:, 0] > 0]
    t0 = t[:, 0].min()
    rel = (t - t0) / 1e3
    print(f"last mixer launch (step {last}): {t.shape[0]} CTAs; us since first CTA entry")
    for q, name in [(50, "median"), (100, "max")]:
        print(f"  {name:7s} " + " ".join(f"{n_}={np.percentile(rel[:, i], q):.2f}" for i, n_ in enumerate(NAMES)))
    dur = t[:, 7] - t[:, 0]
    print(f"  per-CTA lifetime us: median {np.median(dur) / 1e3:.2f}  max {dur.max() / 1e3:.2f};  kernel span {rel[:, 6:8].max():.2f}")
    d = (t[:, 1:] - t[:, :-1]) / 1e3
    print("  median phase lengths: " + " ".join(f"{NAMES[i]}->{NAMES[i + 1]}={np.median(d[:, i]):.2f}" for i in range(7)))


if __name__ == "__main__":
    main()
