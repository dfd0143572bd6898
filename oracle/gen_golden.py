"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/* by executing the UNMODIFIED reference.

Run in the build container (needs /root/reference):   python -m oracle.gen_golden

What it pins (the reference ships no tests / golden vectors of its own, SURVEY.md section 4):
  * keys.json            -- name/shape/dtype of MobileCLIPVisionTower.state_dict() and of the
                            mlp2x_gelu projector, from the live reference modules.
  * ref_256.npz          -- reference outputs for the seeded fixture at R=256, fp32 CPU:
                            tokens [1,16,3072], projected [1,16,896], and for every unit on the
                            path (forward hooks on the reference modules) mean/std/absmax plus
                            256 values at seeded flat indices.
  * ref_1024_tokens_sample.npz -- fingerprint of the reference tower tokens [1,256,3072] at R=1024
                            (fp32): shape, mean/std/absmax and 65536 values at seeded flat indices
                            (the full tensor is 3 MB).
  * ref_b2_256.npz       -- batch-2 tokens at R=256 through the reference's list-input branch
                            (mobileclip_encoder.py:78-83) and tensor branch.
The oracle restatement must reproduce all of them (tests/test_oracle.py).
"""
import json
import os
import sys

import numpy as np
import torch

from . import fixture as fx
from . import ref_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
N_SAMPLES = 256
N_SAMPLES_1024 = 65536
PROJ_HIDDEN = 896  # Qwen2-0.5B hidden size


def sample_indices(numel, name, n=N_SAMPLES):
    seed = int.from_bytes(name.encode()[:8].ljust(8, b"\0"), "little") % (2 ** 31)
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, numel, size=n)


def fingerprint(name, t, n=N_SAMPLES):
    flat = t.detach().float().reshape(-1)
    idx = sample_indices(flat.numel(), name, n)
    return {
        "shape": np.array(t.shape, dtype=np.int64),
        "stats": np.array([flat.mean().item(), flat.std().item(), flat.abs().max().item()], dtype=np.float64),
        "samples": flat[torch.from_numpy(idx)].numpy().astype(np.float32),
    }


def main():
    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    os.makedirs(OUT, exist_ok=True)
    sd = fx.tower_state_dict()
    psd = fx.projector_state_dict(PROJ_HIDDEN)

    tower = ref_loader.reference_tower(256)
    ref_sd = tower.state_dict()
    proj = ref_loader.reference_projector(PROJ_HIDDEN)
    keys = {
        "reference": "apple/ml-fastvlm @ 592b4add, executed under oracle/timm_stub.py",
        "torch": torch.__version__,
        "tower": [[k, list(v.shape), str(v.dtype)] for k, v in ref_sd.items()],
        "projector": [[k, list(v.shape), str(v.dtype)] for k, v in proj.state_dict().items()],
    }
    assert [k for k, _, _ in keys["tower"]] == list(sd.keys()), "fixture key order differs from reference"
    with open(os.path.join(OUT, "keys.json"), "w") as f:
        json.dump(keys, f, indent=0)

    tower.load_state_dict(sd, strict=True)
    proj.load_state_dict(psd, strict=True)

    # ---- R=256, per-unit fingerprints through forward hooks on the reference modules
    fv = tower.vision_tower.model
    units = {"stem": fv.patch_embed, "conv_exp": fv.conv_exp}
    for idx, kind, i in fx.network_layout():
        units[f"network.{idx}"] = fv.network[idx]
        if kind == "stage":
            for b in range(fx.LAYERS[i]):
                units[f"network.{idx}.{b}"] = fv.network[idx][b]
    captured = {}
    hooks = [m.register_forward_hook(lambda mod, inp, out, n=n: captured.__setitem__(n, out)) for n, m in units.items()]
    x = fx.synthetic_images(1, 256)
    tokens = tower(x)
    for h in hooks:
        h.remove()
    projected = proj(tokens)
    blob = {"tokens": tokens.numpy(), "projected": projected.numpy()}
    for n, t in captured.items():
        fp = fingerprint(n, t)
        for k, v in fp.items():
            blob[f"unit/{n}/{k}"] = v
    np.savez_compressed(os.path.join(OUT, "ref_256.npz"), **blob)
    print("R=256 tokens", tuple(tokens.shape), "std %.3f absmax %.2f" % (tokens.std(), tokens.abs().max()))
    for n in ["stem"] + [f"network.{i}" for i in range(11)] + ["conv_exp"]:
        s = blob[f"unit/{n}/stats"]
        print(f"  {n:12s} shape {tuple(blob[f'unit/{n}/shape'])} std {s[1]:.3f} absmax {s[2]:.2f}")

    # ---- batch 2: list branch and tensor branch of forward_images
    x2 = fx.synthetic_images(2, 256, seed=7)
    t_tensor = tower(x2)
    t_list = tower([x2[0], x2[1]])
    assert isinstance(t_list, list) and t_list[0].shape == (1, 16, 3072)
    np.savez_compressed(os.path.join(OUT, "ref_b2_256.npz"), tokens=t_tensor.numpy(),
                        list0=t_list[0].numpy(), list1=t_list[1].numpy())

    # ---- R=1024 tokens (shape pin [1,256,3072]: app/FastVLM/FastVLM.swift:303)
    tower1024 = ref_loader.reference_tower(1024, sd)
    t1024 = tower1024(fx.synthetic_images(1, 1024))
    assert tuple(t1024.shape) == (1, 256, 3072)
    np.savez_compressed(os.path.join(OUT, "ref_1024_tokens_sample.npz"), **fingerprint("tokens_1024", t1024, N_SAMPLES_1024))
    print("R=1024 tokens std %.3f absmax %.2f" % (t1024.std(), t1024.abs().max()))

    # ---- fixture sensitivity (SURVEY finding 3): default layer-scale/BN init hides the branches
    sd0 = fx.default_init_like_reference(sd)
    tower.load_state_dict(sd0, strict=True)
    t0 = tower(x)
    rel = ((tokens - t0).norm() / tokens.norm()).item()
    print("rel-L2 change when layer scales -> 1e-5 and BN -> identity: %.3f" % rel)
    with open(os.path.join(OUT, "sensitivity.json"), "w") as f:
        json.dump({"rel_l2_default_vs_fixture": rel}, f)


if __name__ == "__main__":
    sys.exit(main())
