#!/usr/bin/env python
"""bench.py -- FastViTHD images/sec @1024 px + FastVLM TTFT (BASELINE.json metric), one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            # B200-native arm (this repo)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's projected tokens as DIR/projected.npy
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference algorithm on host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1)

Headline (`value`, `e2e`, `roofline`): BASELINE.json configs[1] -- one pass of the hot path (`encode_images`: FastViTHD tower +
mlp2x_gelu projector, H=896 as in FastVLM-0.5B) over ONE synthetic 1024x1024 image per GPU, random-init fixture weights, bf16.
Multi-GPU: images shard by batch, one process per GPU (weak scaling for the headline, SURVEY 8e).

  value      images/s, inputs already resident in HBM, CUDA events per step, max over ranks, L2 flushed (256 MiB write) between
             timed steps.
  e2e        same metric through the host-buffer C-ABI entry (fvhd_encode_images_host): pinned fp16 host images -> H2D -> forward
             -> D2H of the projected tokens, all inside the timed region.
  roofline   dominant kernels (all tcgen05 kernels: GEMM + fused ConvFFN kernels): algorithmic FLOPs of their launches in one
             step / their summed live CUDA-event durations, against the measured bf16 peak (MEASURED_PEAKS.json).
  cpu_baseline   oracle port (fp32 torch CPU restatement of the reference) timed on the host cores, N=1 only.
  gpu_eager_baseline   "the reference on this box" (BASELINE.md 2, second bar): the same reference modules (oracle port) in PyTorch
             eager bf16 channels-last on the B200 (cuDNN/cuBLAS), batch 1 and batch 32, N=1 only.
  config4    BASELINE.json configs[3]: global batch 256 sharded over the N ranks (rank r takes [r*256/N, (r+1)*256/N)), images/s
             (strong scaling) without any collective, with the all-gather FUSED into the projector epilogue (peer stores over
             NVLink into symmetric memory) and with a separate NCCL all-gather pass; tcgen05 roofline fraction at that batch.
  ttft       BASELINE.json configs[2] (and configs[4] with --ttft7b / at N=8): p50 time to first token, uint8 host image ->
             GPU preprocessing -> encode_images (splice store) -> Qwen2 prefill on the library (row f3) -> first token, with the
             stock-HF prefill timed next to it; every rank runs its own replica (a single image is not sharded: flat in N by design).
  sustained  >= 2 s of back-to-back forwards with the clock sampler running (the 50-step timed region is ~0.1 s).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RES = 1024
HIDDEN = 896            # Qwen2-0.5B hidden size (FastVLM-0.5B projector output)
METRIC = "fastvithd_images_per_sec_1024px"
UNIT = "images/s"
CONFIG4_BATCH = 256     # BASELINE.json configs[3]
CONFIG4_PASS = 32       # images per library pass (workspace 113 MB per image)
DUMP_BYTES = 64 * 1024 * 1024     # --dump-outputs writes at most this much (all ranks together)
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}    # /opt/skills/guides/B200_PROFILING.md fallback
TC_KERNELS = ("gemm_bf16_tcgen05_kernel", "convffn_tcgen05_kernel", "mlp_cluster_tcgen05_kernel", "mlp_fused_tcgen05_kernel",
              "attention_umma_kernel", "repmixer_umma_kernel")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return dict(FALLBACK_PEAKS), "fallback"


def make_config(world, batch):
    """The workload description BOTH arms print (same dict -> the driver's same_config check)."""
    return {"workload": f"encode_images: FastViTHD tower + mlp2x_gelu projector (H={HIDDEN}), batch {batch} per GPU, {RES}x{RES}",
            "resolution": RES, "batch_per_gpu": batch, "global_batch": batch * world, "weights": "seeded random fixture",
            "parallelism": f"batch-sharded x{world}, no data-path collective", "l2": "flushed (256 MiB write) between timed steps",
            "input": "bf16 NCHW resident in HBM (value); pinned fp16 host (e2e)"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=50):
        self.gpu = gpu_index
        self.period = period_ms
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            time.sleep(0.12)          # first sample lands before the timed region starts
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def cpu_reference_time(steps, warmup):
    """The reference algorithm (oracle port: same ATen fp32 ops as the reference's torch.nn modules) on the host cores.
    oneDNN does not scale monotonically with threads on many-core hosts (128 threads measured 10x slower than 8),
    so the thread count is calibrated first on a 512-px image over {8,16,32,64,all} and the fastest is used
    -- the reference gets its best configuration; `cores` reports the threads actually used."""
    import torch
    from oracle import fastvithd_oracle as orc
    from oracle import fixture as fx
    cores = _host_cores()
    sd = fx.tower_state_dict()
    psd = fx.projector_state_dict(HIDDEN)
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    best, best_t = cands[0], None
    xs = fx.synthetic_images(1, 512)
    with torch.inference_mode():
        for c in cands:
            torch.set_num_threads(c)
            orc.encode_images(xs, sd, psd)
            t0 = time.perf_counter()
            orc.encode_images(xs, sd, psd)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best, best_t = c, dt
        torch.set_num_threads(best)
        x = fx.synthetic_images(1, RES)
        for _ in range(warmup):
            orc.encode_images(x, sd, psd)
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            orc.encode_images(x, sd, psd)
            times.append(time.perf_counter() - t0)
    return times, best


def cpu_config1(threads):
    """BASELINE.json configs[0]: the predict.py flow (predict.py:18-72) on the CPU in fp32 -- one 256x256 image, tower
    `mobileclip_l_256` (16 visual tokens), mlp2x_gelu projector, random-init Qwen2-0.5B-shaped LLM, first token.
    Encoder = oracle port (the reference modules); LLM = stock HF.  Returns a dict (bounded: 1 warm-up + 3 runs)."""
    import torch
    from transformers import Qwen2Config, Qwen2ForCausalLM
    from oracle import fastvithd_oracle as orc
    from oracle import fixture as fx
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    cfg = Qwen2Config(hidden_size=896, num_hidden_layers=24, num_attention_heads=14, num_key_value_heads=2, intermediate_size=4864,
                      vocab_size=151936, max_position_embeddings=32768, tie_word_embeddings=True)
    llm = Qwen2ForCausalLM(cfg).eval()
    sd, psd = fx.tower_state_dict(), fx.projector_state_dict(HIDDEN)
    x = fx.synthetic_images(1, 256)
    n_pre, n_post = 14, 17
    ids = torch.randint(0, 150000, (1, n_pre + n_post))
    enc, tot = [], []
    with torch.inference_mode():
        for i in range(4):
            t0 = time.perf_counter()
            vis = orc.encode_images(x, sd, psd)
            t1 = time.perf_counter()
            txt = llm.get_input_embeddings()(ids)
            emb = torch.cat([txt[:, :n_pre], vis.to(txt.dtype), txt[:, n_pre:]], 1)
            llm(inputs_embeds=emb, use_cache=True).logits[:, -1].argmax(-1).item()
            t2 = time.perf_counter()
            if i:
                enc.append((t1 - t0) * 1e3)
                tot.append((t2 - t0) * 1e3)
    return {"workload": "predict.py flow, one 256x256 image, tower mobileclip_l_256 (16 tokens), Qwen2-0.5B-shaped random-init LLM, CPU fp32",
            "ttft_ms_median": statistics.median(tot), "encode_ms_median": statistics.median(enc), "threads": threads, "runs": 3,
            "sequence": n_pre + 16 + n_post}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = args.steps, max(0, args.warmup)
    times, cores = cpu_reference_time(steps, warmup)
    ms = 1e3 * sum(times) / len(times)
    val = 1e3 / ms
    sample = (f"{steps} steps x 1 image {RES}x{RES} fp32 (+{warmup} warm-up), oracle port of the reference modules, torch CPU, {cores} threads "
              "(calibrated best of 8/16/32/64/all)")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args.gpus, args.batch),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "min_ms": 1e3 * min(times), "median_ms": 1e3 * statistics.median(times)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_config1:
        try:
            line["config1"] = cpu_config1(cores)
        except Exception as e:  # noqa: BLE001
            line["config1"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def kernel_table(eng, images, flush, reps=5):
    """Live CUDA-event time of every launch of one forward -> per-kernel-class table + the tcgen05 roofline numerators."""
    B = images.shape[0]
    eng.profile_steps(images)
    acc = None
    for _ in range(reps):
        flush.fill_(1)
        ms = eng.profile_steps(images)
        acc = ms if acc is None else [a + b for a, b in zip(acc, ms)]
    ms = [a / reps for a in acc]
    kernels = {}
    for st, m in zip(eng.steps(B), ms):
        k = kernels.setdefault(st["kernel"], {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        k["launches"] += 1
        k["ms"] += m
        k["flops"] += st["flops"]
        k["bytes"] += st["bytes"]
    tot = sum(ms)
    ktab = [{"kernel": n, "launches": k["launches"], "ms": round(k["ms"], 4), "share": round(k["ms"] / tot, 4),
             "tflops": round(k["flops"] / k["ms"] / 1e9, 1) if k["ms"] > 0 else None,
             "gbs": round(k["bytes"] / k["ms"] / 1e6, 1) if k["ms"] > 0 else None}
            for n, k in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])]
    tc = [n for n in TC_KERNELS if n in kernels]
    gk = {"launches": sum(kernels[n]["launches"] for n in tc), "ms": sum(kernels[n]["ms"] for n in tc),
          "flops": sum(kernels[n]["flops"] for n in tc), "names": tc, "sum_ms": tot}
    return ktab, gk


CONV_KERNELS = ("repmixer_tz_kernel", "repmixer_tc_kernel", "repmixer_dw_kernel", "stem2_kernel", "stem_kernel", "dwconv_kernel")


def conv_roofline(ktab, peaks, peak_src):
    """north_star (i): the conv-stage kernels (stem, RepMixer depthwise pair, PatchEmbed / RepCPE depthwise convs) against the HBM roof:
    algorithmic bytes (inputs read once + outputs written once, `fvhd_step_info`) / live CUDA-event time."""
    rows = [k for k in ktab if k["kernel"].startswith(CONV_KERNELS) and k["ms"] > 0 and k["gbs"]]
    if not rows:
        return None
    ms = sum(k["ms"] for k in rows)
    gb = sum(k["gbs"] * k["ms"] for k in rows) / 1e3          # GB/s * ms = MB
    peak = float(peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"]))
    return {"bound": "hbm", "kernels": sorted({k["kernel"] for k in rows}), "achieved": round(gb * 1e3 / ms, 1), "peak": peak, "unit": "GB/s",
            "frac": round(gb * 1e3 / ms / peak, 4), "peak_source": f"{peak_src} (copy bandwidth)", "ms": round(ms, 4),
            "per_kernel_frac": {k["kernel"]: round(k["gbs"] / peak, 4) for k in rows}}


def roofline_obj(gk, peaks, peak_src, traffic=None, traffic_src=None):
    ach = gk["flops"] / gk["ms"] / 1e9
    peak = float(peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"]))
    return {"bound": "tensor", "kernel": " + ".join(gk["names"]), "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s",
            "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"{peak_src} (burst bf16 GEMM)",
            "launches_per_step": gk["launches"], "avg_launch_us": round(1e3 * gk["ms"] / gk["launches"], 2),
            "algorithmic_flops_per_step": gk["flops"], "share_of_step": round(gk["ms"] / gk["sum_ms"], 4)}


def timed_steps(fn, steps, flush, barrier):
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.fill_(i & 0xFF)                               # L2 flush, outside the timed bracket
        ev[i][0].record()
        fn()
        ev[i][1].record()
    barrier()
    return [a.elapsed_time(b) for a, b in ev]


def dump_outputs(out_dir, outputs, max_bytes):
    """Write each [B, ...] output as <out_dir>/<name>.npy in float32.  An output larger than `max_bytes` keeps a fixed, seeded
    subset of its images, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        keep = max(1, max_bytes // len(outputs) // (t[0].numel() * 4))
        if t.shape[0] > keep:
            idx = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def gpu_eager_baseline(dev, batches=(1, 32)):
    """Reference modules (oracle port) in torch eager bf16 channels-last on this GPU: cuDNN / cuBLAS, no code of this repo."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import eager_gpu
    out = {}
    for b in batches:
        r = eager_gpu.eager_time(b, res=RES, hidden=HIDDEN, steps=8 if b > 1 else 20, warmup=3, dev=str(dev))
        out[f"batch{b}"] = {"images_per_s": round(r["images_per_s"], 2), "ms_median": round(r["ms_median"], 3)}
    out["impl"] = "oracle port of the reference modules, torch eager bf16 channels_last (cuDNN/cuBLAS), same fixture weights and synthetic input"
    return out


def ttft_run(dev, res, hidden, llm_shape, runs, warmup, pkg, fx):
    """p50 TTFT of one replica on `dev` (see tools/ttft.py for the definition; FastVLMModel.swift:114-138, predict.py:51-65):
    uint8 host image -> H2D -> GPU preprocessing -> encode_images (projector epilogue stores at the <image> position of the LLM's input
    sequence) -> text embeddings -> LLM prefill -> first token on the host.  The prefill runs on the library (row f3, LlmPrefill: tcgen05
    GEMMs + llm.cuh, one CUDA graph); the same flow with the stock Hugging Face prefill is timed next to it (`hf_prefill`)."""
    import numpy as np
    import torch
    from transformers import Qwen2Config, Qwen2ForCausalLM
    torch.manual_seed(0)
    cfg = Qwen2Config(max_position_embeddings=32768, **llm_shape)
    with torch.device(dev):
        llm = Qwen2ForCausalLM(cfg)
    llm = llm.to(dtype=torch.bfloat16).eval()
    packed = pkg.pack_tower(fx.tower_state_dict())
    packed.update(pkg.pack_projector(fx.projector_state_dict(hidden)))
    eng = pkg.Engine(res, hidden, 2, 1).load(packed, dev)
    ntok = eng.num_tokens
    host_u8 = torch.from_numpy(np.random.default_rng(0).integers(0, 256, (res, res, 3), dtype=np.uint8)).pin_memory()
    img = torch.empty(1, 3, res, res, dtype=torch.float16, device=dev)
    n_pre, n_post = 14, 17                       # qwen_2 template around "<image>\nDescribe the image." (predict.py:34-42,80)
    seq = n_pre + ntok + n_post
    ids = torch.randint(0, 150000, (1, n_pre + n_post), device=dev)
    embed = llm.get_input_embeddings()
    prefill = pkg.LlmPrefill.from_hf(llm, max_seq=seq, device=dev)
    xin = prefill.input(seq).view(1, seq, hidden)

    def one_native():
        t0 = time.perf_counter()
        pkg.preprocess_into(eng, host_u8, img[0])     # uint8 H2D + resize/crop/scale on the GPU (row f1)
        eng.forward_into(img, xin, n_pre)             # projector epilogue stores at the <image> position of the LLM input (row f2)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        txt = embed(ids)
        xin[:, :n_pre] = txt[:, :n_pre]
        xin[:, n_pre + ntok:] = txt[:, n_pre:]
        tok, _ = prefill.prefill(seq)                 # row f3; returns after the token reached the host
        t2 = time.perf_counter()
        return (t2 - t0) * 1e3, (t1 - t0) * 1e3, (t2 - t1) * 1e3, tok

    def one_hf():
        t0 = time.perf_counter()
        pkg.preprocess_into(eng, host_u8, img[0])
        x = torch.empty(1, seq, hidden, dtype=torch.bfloat16, device=dev)
        eng.forward_into(img, x, n_pre)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        txt = embed(ids)
        x[:, :n_pre] = txt[:, :n_pre]
        x[:, n_pre + ntok:] = txt[:, n_pre:]
        tok = llm(inputs_embeds=x, use_cache=True).logits[:, -1].argmax(-1).item()      # first token on the host
        t2 = time.perf_counter()
        return (t2 - t0) * 1e3, (t1 - t0) * 1e3, (t2 - t1) * 1e3, tok

    with torch.inference_mode():
        for _ in range(warmup):
            one_native()
        rs = [one_native() for _ in range(runs)]
        hf_runs = max(10, runs // 3)
        for _ in range(3):
            one_hf()
        hs = [one_hf() for _ in range(hf_runs)]
        # same weights, same input: logits of the two prefills (random-init logits are nearly flat, so compare the vectors, not only argmax)
        _, lg = prefill.prefill(seq, want_logits=True)
        lh = llm(inputs_embeds=xin.clone(), use_cache=False).logits[0, -1].float()
        logit_err = ((lg.float() - lh).norm() / lh.norm()).item()
    launches = prefill.launches(seq)
    del llm, eng, prefill
    torch.cuda.empty_cache()
    tt = sorted(r[0] for r in rs)
    return {"ttft_ms_p50": statistics.median(tt), "encode_ms_p50": statistics.median(r[1] for r in rs),
            "prefill_first_token_ms_p50": statistics.median(r[2] for r in rs), "ttft_ms_min": tt[0], "ttft_ms_p90": tt[int(0.9 * (len(tt) - 1))],
            "runs": runs, "warmup": warmup, "sequence": seq, "resolution": res, "visual_tokens": ntok,
            "prefill": "library (row f3): tcgen05 GEMMs + RMSNorm / RoPE / causal GQA attention / SwiGLU / argmax kernels, one CUDA graph",
            "prefill_launches": launches,
            "hf_prefill": {"ttft_ms_p50": statistics.median(r[0] for r in hs), "prefill_first_token_ms_p50": statistics.median(r[2] for r in hs),
                           "runs": hf_runs, "impl": "stock transformers Qwen2ForCausalLM.forward (eager), same weights and input"},
            "first_token_equal_to_hf": bool(rs[-1][3] == hs[-1][3]), "last_logits_rel_l2_vs_hf_bf16": logit_err}


QWEN2_05B = dict(hidden_size=896, num_hidden_layers=24, num_attention_heads=14, num_key_value_heads=2, intermediate_size=4864,
                 vocab_size=151936, tie_word_embeddings=True)
QWEN2_7B = dict(hidden_size=3584, num_hidden_layers=28, num_attention_heads=28, num_key_value_heads=4, intermediate_size=18944,
                vocab_size=152064, tie_word_embeddings=False)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu_arm(args):
    import torch
    import ml_fastvlm_b200 as pkg
    from oracle import fixture as fx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"WORLD_SIZE {world} != --gpus {args.gpus}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch N>1 with torch.distributed.run (one process per GPU)")
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    steps, warmup = args.steps, max(3, args.warmup)
    packed = pkg.pack_tower(fx.tower_state_dict())
    packed.update(pkg.pack_projector(fx.projector_state_dict(HIDDEN)))
    eng = pkg.Engine(RES, HIDDEN, 2, B).load(packed, dev)

    host_img = fx.synthetic_images(B, RES, seed=100 + rank).half().pin_memory()
    dev_img = host_img.to(dev).to(torch.bfloat16)            # resident input for `value`
    host_out = torch.empty(B, eng.num_tokens, HIDDEN, dtype=torch.bfloat16).pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        if dist is None:
            return list(vals)
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    # ---- headline: device-resident timing
    for _ in range(warmup):
        eng.forward(dev_img, want_tokens=False, want_projected=True)
    barrier()
    sampler = ClockSampler(local_rank).start()
    last = {}

    def fwd():
        last["projected"] = eng.forward(dev_img, want_tokens=False, want_projected=True)[1]

    step_ms = timed_steps(fwd, steps, flush, barrier)
    total_ms = sum(step_ms)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"projected" if world == 1 else f"projected_rank{rank}": last["projected"]}, DUMP_BYTES // world)

    # ---- end to end through the host-buffer entry (H2D + forward + D2H inside the timed region)
    for _ in range(2):
        eng.encode_images_host(host_img, host_out)
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.encode_images_host(host_img, host_out)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)

    # ---- sustained: >= 2 s of back-to-back forwards, clocks sampled throughout
    barrier()
    n_sus, t_sus0 = 0, time.perf_counter()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record()
    while time.perf_counter() - t_sus0 < args.sustain_s:
        for _ in range(20):
            eng.forward(dev_img, want_tokens=False, want_projected=True)
        n_sus += 20
        torch.cuda.synchronize()
    es1.record()
    torch.cuda.synchronize()
    sus_ms = es0.elapsed_time(es1)
    clocks = sampler.stop()
    total_ms, e2e_ms, sus_ms = allmax([total_ms, e2e_ms, sus_ms])

    # ---- config 4: global batch 256 sharded over the ranks (strong scaling), with / without the all-gather
    cfg4 = None
    if not args.no_config4:
        from ml_fastvlm_b200 import parallel as par
        a4, b4 = par.shard_bounds(CONFIG4_BATCH, rank, world)
        nb4 = b4 - a4
        eng4 = pkg.Engine(RES, HIDDEN, 2, min(CONFIG4_PASS, nb4)).load(packed, dev)
        g = torch.Generator(device=dev).manual_seed(1000 + rank)
        shard = torch.empty(nb4, 3, RES, RES, dtype=torch.bfloat16, device=dev)
        for i in range(0, nb4, 8):
            shard[i:i + 8] = torch.rand((min(8, nb4 - i), 3, RES, RES), device=dev, generator=g).to(torch.bfloat16)
        out4 = torch.empty(nb4, eng4.num_tokens, HIDDEN, dtype=torch.bfloat16, device=dev)
        st4, wu4 = args.config4_steps, 1

        def fwd4():
            eng4.forward_into(shard, out4, 0)

        for _ in range(wu4):
            fwd4()
        barrier()
        s4 = ClockSampler(local_rank).start()
        ms_nog = sum(timed_steps(fwd4, st4, flush, barrier))
        ms_fused = ms_nccl = None
        gather_err = None
        if world > 1:
            try:
                ge = par.GatheredEncoder(eng4, CONFIG4_BATCH)
                for _ in range(wu4):
                    ge.encode(shard)
                barrier()
                ms_fused = sum(timed_steps(lambda: ge.encode(shard), st4, flush, barrier))
                # correctness of the fused gather against the NCCL collective (same bits expected)
                ref = par.all_gather_tokens(out4, CONFIG4_BATCH)
                torch.cuda.synchronize()
                gather_ok = bool(torch.equal(ref, ge.buf))
            except Exception as e:  # noqa: BLE001
                gather_err, gather_ok = repr(e)[:300], None
            barrier()

            def fwd_nccl():
                fwd4()
                par.all_gather_tokens(out4, CONFIG4_BATCH)

            fwd_nccl()
            barrier()
            ms_nccl = sum(timed_steps(fwd_nccl, st4, flush, barrier))
        c4clk = s4.stop()
        mx = allmax([ms_nog, ms_fused or 0.0, ms_nccl or 0.0])
        cfg4 = {"workload": f"encode_images, global batch {CONFIG4_BATCH} at {RES}x{RES}, batch-sharded over {world} GPU(s): rank r takes "
                            f"[r*{CONFIG4_BATCH}/N, (r+1)*{CONFIG4_BATCH}/N), {min(CONFIG4_PASS, nb4)} images per library pass",
                "global_batch": CONFIG4_BATCH, "images_per_rank": nb4, "steps": st4, "warmup": wu4, "scaling": "strong",
                "images_per_s_no_gather": CONFIG4_BATCH * st4 / (mx[0] / 1e3),
                "images_per_s_fused_gather": CONFIG4_BATCH * st4 / (mx[1] / 1e3) if ms_fused else None,
                "images_per_s_nccl_allgather": CONFIG4_BATCH * st4 / (mx[2] / 1e3) if ms_nccl else None,
                "ms_per_step_no_gather": mx[0] / st4, "clocks": c4clk,
                "gather": ("none needed (1 GPU)" if world == 1 else
                           "fused: projector epilogue stores into every rank's symmetric-memory buffer (fvhd_forward_gather); "
                           "nccl: all_gather_into_tensor after the forward")}
        if world > 1:
            cfg4["fused_gather_equals_nccl"] = gather_ok
            if gather_err:
                cfg4["fused_gather_error"] = gather_err
        if rank == 0:
            peaks, peak_src = load_peaks()
            bp = min(CONFIG4_PASS, nb4)
            ktab4, gk4 = kernel_table(eng4, shard[:bp], flush, reps=2)
            cfg4["roofline"] = roofline_obj(gk4, peaks, peak_src)
            cfg4["conv_roofline"] = conv_roofline(ktab4, peaks, peak_src)
            cfg4["kernels"] = ktab4
        del eng4, shard, out4
        torch.cuda.empty_cache()

    # ---- TTFT (every rank its own replica; p50 per rank, max over ranks reported)
    ttft = None
    if not args.no_ttft:
        try:
            t3 = ttft_run(dev, RES, HIDDEN, QWEN2_05B, args.ttft_runs, 5, pkg, fx)
            t3["ttft_ms_p50_max_over_ranks"] = allmax([t3["ttft_ms_p50"]])[0]
            t3["llm"] = "random-init Qwen2ForCausalLM (Qwen2-0.5B shape), bf16 weights"
            ttft = {"config3": t3}
            if args.ttft7b or world == 8:
                t5 = ttft_run(dev, 1536, 3584, QWEN2_7B, max(10, args.ttft_runs // 2), 3, pkg, fx)
                t5["ttft_ms_p50_max_over_ranks"] = allmax([t5["ttft_ms_p50"]])[0]
                t5["llm"] = "random-init Qwen2ForCausalLM (Qwen2-7B shape), bf16 weights"
                ttft["config5"] = t5
            ttft["note"] = ("one replica per GPU: a single image is not sharded, so TTFT is flat in N by design; "
                            "TTFT = uint8 host image -> H2D -> GPU preprocessing -> encode_images (splice store) -> LLM prefill -> first token")
        except Exception as e:  # noqa: BLE001
            ttft = {"unavailable": repr(e)[:300]}

    line = None
    if rank == 0:
        peaks, peak_src = load_peaks()
        ktab, gk = kernel_table(eng, dev_img, flush)
        traffic, tsrc = None, None      # dram__bytes_read+write per tcgen05 launch from this round's committed ncu pass of this command
        tpath = os.path.join(ROOT, "profiles", "r02_tc_dram_traffic.json")
        if B == 1 and os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic, tsrc = tj.get("bytes_per_launch"), tj.get("source")
        roofline = roofline_obj(gk, peaks, peak_src, traffic, tsrc)
        peak = roofline["peak"]
        F = sum(u["flops"] for u in eng.units()) * B
        step_ms_mean = total_ms / steps
        whole = {"tflops": round(F / step_ms_mean / 1e9, 1), "frac_of_bf16_peak": round(F / step_ms_mean / 1e9 / peak, 4),
                 "t_tensor_roof_ms": round(F / peak / 1e9, 4), "sum_kernel_ms": round(gk["sum_ms"], 4)}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            times, cores = cpu_reference_time(args.cpu_steps, 1)
            cms = 1e3 * sum(times) / len(times)
            cpu = {"value": 1e3 / cms, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{args.cpu_steps} images {RES}x{RES} fp32 (+1 warm-up) through the oracle port (torch CPU, {cores} threads = calibrated best of 8/16/32/64/all)",
                   "ms_per_image": cms}
        eager = None
        if world == 1 and not args.no_eager_baseline:
            try:
                del eng
                torch.cuda.empty_cache()
                eager = gpu_eager_baseline(dev)
            except Exception as e:  # noqa: BLE001
                eager = {"unavailable": repr(e)[:300]}
        line = {
            "metric": METRIC, "value": world * B * steps / (total_ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": make_config(world, B),
            "clocks": dict(clocks, window="timed steps + e2e loop + sustained loop"),
            "e2e": {"value": world * B * steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": host_img.numel() * 2,
                    "d2h_bytes_per_step": host_out.numel() * 2, "ms_per_step": e2e_ms / steps,
                    "api": "fvhd_encode_images_host (C ABI) via Engine.encode_images_host"},
            "roofline": roofline, "conv_roofline": conv_roofline(ktab, peaks, peak_src), "whole_step": whole, "kernels": ktab,
            "step_ms_min": min(step_ms), "step_ms_median": statistics.median(step_ms),
            "sustained": {"seconds": sus_ms / 1e3, "forwards": n_sus, "images_per_s": world * B * n_sus / (sus_ms / 1e3),
                          "note": "back-to-back forwards, no L2 flush, no host sync between launches of a group of 20"},
        }
        line["gpu_launches"] = int(sum(k["launches"] for k in ktab) + 1) * steps      # plan's launch list + set_io_kernel, per timed step
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if eager is not None:
            line["gpu_eager_baseline"] = eager
        if cfg4 is not None:
            line["config4"] = cfg4
        if ttft is not None:
            line["ttft"] = ttft
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 50; 8 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="images per GPU per step (BASELINE configs[1]: 1)")
    ap.add_argument("--cpu-steps", type=int, default=5, help="images timed for cpu_baseline (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--config4-steps", type=int, default=3)
    ap.add_argument("--no-ttft", action="store_true")
    ap.add_argument("--ttft-runs", type=int, default=50)
    ap.add_argument("--ttft7b", action="store_true", help="also run configs[4] (FastVLM-7B shape, 1536 px); default only at N=8")
    ap.add_argument("--no-config1", action="store_true", help="reference arm: skip the configs[0] predict.py-flow record")
    ap.add_argument("--sustain-s", type=float, default=2.0)
    ap.add_argument("--quick", action="store_true", help="headline only: no cpu/eager baselines, config4, ttft")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the projected tokens of the last one as "
                    "DIR/projected.npy (float32; per rank: projected_rank<r>.npy; at most 64 MB, a seeded subset of images beyond that)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.quick:
        args.no_cpu_baseline = args.no_eager_baseline = args.no_config4 = args.no_ttft = True
        args.sustain_s = 0.0
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 8
        return run_reference_arm(args)
    if args.steps is None:
        args.steps = 50
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
