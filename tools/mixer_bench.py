#!/usr/bin/env python
"""Time the RepMixer depthwise pair alone (fvhd_mixer test entry) for the three stage shapes at 1024 px, per mixer mode.
    python tools/mixer_bench.py [modes=tz] [batches=1,8,32]
Prints one JSON line per (mode, stage, batch): us per launch, us per image, algorithmic GB/s (3 * px * C * 2 B), useful TFLOP/s."""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
import torch.nn.functional as F

modes = sys.argv[1] if len(sys.argv) > 1 else "tz"
batches = [int(b) for b in (sys.argv[2].split(",") if len(sys.argv) > 2 else ["1", "8", "32"])]
skips = [int(b) for b in (sys.argv[3].split(",") if len(sys.argv) > 3 else ["0"])]     # FVHD_TZ_SKIP experiment masks (mixer_tz.cuh)
import ml_fastvlm_b200 as pkg

dev = torch.device("cuda:0")
SHAPES = [(256, 256, 96, 2), (128, 128, 192, 12), (64, 64, 384, 24)]       # H, W, C, blocks per forward


def engine(mode, skip):
    """Engine whose fvhd_mixer runs `mode` with the FVHD_TZ_SKIP mask `skip` (switches are read when a handle is created)."""
    os.environ["FVHD_MIXER"] = mode
    os.environ["FVHD_TZ_SKIP"] = str(skip)
    try:
        return pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_MIXER", None)
        os.environ.pop("FVHD_TZ_SKIP", None)


flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for mode in modes:
    for B, skip in [(b, k) for b in batches for k in skips]:
        eng = engine(mode, skip)
        tot_us = 0.0
        for (H, W, C, nblk) in SHAPES:
            g = torch.Generator().manual_seed(H + C + B)
            x = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16).to(dev)
            w3 = (torch.randn(9, C, generator=g) / 3).to(dev)
            b3 = (torch.randn(C, generator=g) * 0.1).to(dev)
            w7 = (torch.randn(49, C, generator=g) / 7).to(dev)
            b7 = (torch.randn(C, generator=g) * 0.1).to(dev)
            y, z = eng.mixer(x, w3, b3, w7, b7)
            torch.cuda.synchronize()
            # check against torch on the GPU (fp32 conv, y rounded to bf16 between the convs)
            xf = x.float().permute(0, 3, 1, 2)
            yr = F.conv2d(xf, w3.t().reshape(C, 1, 3, 3), b3, padding=1, groups=C)
            zr = F.conv2d(yr.to(torch.bfloat16).float(), w7.t().reshape(C, 1, 7, 7), b7, padding=3, groups=C)
            ey = ((y.float() - yr.permute(0, 2, 3, 1)).norm() / yr.norm()).item()
            ez = ((z.float() - zr.permute(0, 2, 3, 1)).norm() / zr.norm()).item()
            del xf, yr, zr
            reps = 5 if B >= 8 else 20
            for _ in range(2):
                eng.mixer(x, w3, b3, w7, b7)
            ts = []
            for _ in range(reps):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.mixer(x, w3, b3, w7, b7)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e3)
            ts.sort()
            us = ts[len(ts) // 2]
            px = B * H * W
            tot_us += us * nblk / B
            print(json.dumps({"mode": mode, "skip": skip, "B": B, "H": H, "W": W, "C": C, "us": round(us, 2), "us_min": round(ts[0], 2), "us_per_img": round(us / B, 2),
                              "gbs": round(3 * px * C * 2 / us / 1e3, 1), "tflops": round(2 * px * C * 58 / us / 1e6, 2),
                              "err_y": float(f"{ey:.2e}"), "err_z": float(f"{ez:.2e}")}), flush=True)
        print(json.dumps({"mode": mode, "skip": skip, "B": B, "mixer_us_per_image_38_blocks": round(tot_us, 1)}), flush=True)
