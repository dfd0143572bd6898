#!/usr/bin/env python
"""RepMixerBlock = [mixer ; ConvFFN] as the forward runs it (same stream, PDL launches), per mixer mode:
time of N back-to-back pairs vs N mixers + N ConvFFNs run separately -- shows what the pairing costs or hides.
    python tools/pair_bench.py [modes=tz] [batch=32]"""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch

import ml_fastvlm_b200 as pkg

modes = (sys.argv[1] if len(sys.argv) > 1 else "t,z").split(",")      # e.g. t,z,z:nopdl,z:skip4  (skip = FVHD_TZ_SKIP mask)
B = int(sys.argv[2]) if len(sys.argv) > 2 else 32
dev = torch.device("cuda:0")
SHAPES = [(256, 256, 96, 2), (128, 128, 192, 12), (64, 64, 384, 24)]
N = 8


def engine(mode):
    """Engine created under the switches `mode` names (they are read when a handle is created)."""
    opts = mode.split(":")
    os.environ["FVHD_MIXER"] = opts[0]
    os.environ.pop("FVHD_NO_PDL", None)
    os.environ["FVHD_TZ_SKIP"] = "0"
    os.environ.pop("FVHD_TZ_PDL", None)
    os.environ.pop("FVHD_TZ_PAIR", None)
    for o in opts[1:]:
        if o.startswith("cs"):                  # sibling-cluster size of the Toeplitz mixer (default 2)
            os.environ["FVHD_TZ_PAIR"] = o[2:]
        if o.startswith("pdl"):
            os.environ["FVHD_TZ_PDL"] = o[3:]
        if o == "nopdl":
            os.environ["FVHD_NO_PDL"] = "1"
        elif o.startswith("skip"):
            os.environ["FVHD_TZ_SKIP"] = o[4:]
    try:
        eng = pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_MIXER", None)
    return eng


def timed(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return min(ts)


for mode in modes:
    eng = engine(mode)
    tot_pair = tot_sep = 0.0
    for (H, W, C, nblk) in SHAPES:
        g = torch.Generator().manual_seed(H + C)
        x = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16).to(dev)
        w3 = (torch.randn(9, C, generator=g) / 3).to(dev)
        b3 = (torch.randn(C, generator=g) * 0.1).to(dev)
        w7 = (torch.randn(49, C, generator=g) / 7).to(dev)
        b7 = (torch.randn(C, generator=g) * 0.1).to(dev)
        w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
        w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.float16).to(dev)
        b1 = torch.randn(4 * C, generator=g).to(dev)
        b2 = torch.randn(C, generator=g).to(dev)
        M = B * H * W
        y, z = eng.mixer(x, w3, b3, w7, b7)

        def pairs():
            for _ in range(N):
                yy, zz = eng.mixer(x, w3, b3, w7, b7)
                eng.convffn2(zz.view(M, C), w1, b1, w2, b2, yy.view(M, C))

        def mixers():
            for _ in range(N):
                eng.mixer(x, w3, b3, w7, b7)

        def ffns():
            for _ in range(N):
                eng.convffn2(z.view(M, C), w1, b1, w2, b2, y.view(M, C))

        tp, tm, tf = timed(pairs) / N, timed(mixers) / N, timed(ffns) / N
        tot_pair += tp * nblk / B
        tot_sep += (tm + tf) * nblk / B
        print(json.dumps({"mode": mode, "B": B, "C": C, "pair_us": round(tp, 1), "mixer_us": round(tm, 1), "convffn_us": round(tf, 1),
                          "pair_minus_sum_us": round(tp - tm - tf, 1)}), flush=True)
    print(json.dumps({"mode": mode, "B": B, "blocks_us_per_image_paired": round(tot_pair, 1), "separate": round(tot_sep, 1)}), flush=True)
