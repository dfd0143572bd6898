"""GPU parity tests added in round 2 (-m gpu), all through the C ABI:

  * every unit in isolation at the BENCH size (R=1024) with the plan a large batch selects (batch 3: the stage-2 ConvFFN
    runs as the large-batch kernels, multi-wave GEMMs, 32 M-tiles per image), fed the oracle's own inputs ... rel-L2 <= 8e-3
  * encode_images at 1024 px, batch 5 through max_batch 3 (two passes): tower tokens AND projector vs the oracle
  * repeated-launch stress of the multi-tile cluster ConvFFN kernel and of CUDA-graph replays under PDL (determinism)
  * fused all-gather (fvhd_forward_gather) on 2 GPUs == NCCL all-gather of the per-rank results (skipped with < 2 GPUs)
"""
import os
import socket

import pytest
import torch

import ml_fastvlm_b200 as pkg
from oracle import fastvithd_oracle as orc
from oracle import fixture as fx

pytestmark = pytest.mark.gpu

UNIT_TOL_1024 = 8e-3
E2E_TOL = 5e-2


def rel_l2(a, b):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def packed(tower_sd, proj_sd):
    pk = pkg.pack_tower(tower_sd)
    pk.update(pkg.pack_projector(proj_sd))
    return pk


def _nhwc(t, dev):
    return t.permute(0, 2, 3, 1).contiguous().reshape(t.shape[0], -1).to(torch.bfloat16).to(dev)


@pytest.fixture(scope="module")
def oracle1024_b3(tower_sd, proj_sd):
    torch.set_num_threads(min(32, os.cpu_count() or 8))
    x = fx.synthetic_images(3, 1024, seed=21)
    col = {}
    ref = orc.encode_images(x, tower_sd, proj_sd, col)
    return x, ref, col


def test_every_unit_isolated_1024_large_batch_plan(packed, oracle1024_b3, dev):
    """Config 4's plan (BASELINE configs[3]): batch >= 3 at 1024 px.  Each unit is fed the ORACLE's input, so an error cannot hide
    behind the chain's amplification; tolerance is 8e-3 (bf16 storage of inputs/weights/outputs gives ~3-5e-3)."""
    x, ref, col = oracle1024_b3
    B = x.shape[0]
    eng = pkg.Engine(1024, 896, 2, B).load(packed, dev)
    kernels = {s["kernel"] for s in eng.steps(B)}
    assert "mlp_cluster_tcgen05_kernel" not in kernels, "batch 3 must select the large-batch stage-2 plan"
    prev, worst = None, {}
    for u in eng.units():
        name = u["name"]
        if name == "stem":
            xin, want = x.to(dev), col["stem"].permute(0, 2, 3, 1)
        elif name == "conv_exp":
            xin, want = _nhwc(prev, dev), col["tokens"]
        elif name == "projector":
            xin, want = col["tokens"].reshape(B, -1).to(torch.bfloat16).to(dev), ref
        else:
            xin, want = _nhwc(prev, dev), col[name].permute(0, 2, 3, 1)
        got = eng.run_units(u["index"], u["index"], xin, B)
        assert got.shape == (B, u["out_elems"])
        assert torch.isfinite(got.float()).all(), name
        worst[name] = rel_l2(got.float().reshape(-1), want.reshape(-1))
        prev = col.get(name)
    bad = {k: v for k, v in worst.items() if v > UNIT_TOL_1024}
    assert not bad, bad
    print("worst unit at 1024/B3:", max(worst.items(), key=lambda kv: kv[1]))


def test_encode_images_1024_multi_pass_vs_oracle(packed, oracle1024_b3, tower_sd, proj_sd, dev):
    """batch 5 with max_batch 3 -> passes of 3 + 2 images; tokens and PROJECTED tokens at 1024 px vs the oracle."""
    x3, ref3, col3 = oracle1024_b3
    x2 = fx.synthetic_images(2, 1024, seed=22)
    col2 = {}
    ref2 = orc.encode_images(x2, tower_sd, proj_sd, col2)
    eng = pkg.Engine(1024, 896, 2, 3).load(packed, dev)
    x = torch.cat([x3, x2], 0).to(dev)
    tokens, proj = eng.forward(x, True, True)
    assert tuple(tokens.shape) == (5, 256, 3072) and tuple(proj.shape) == (5, 256, 896)
    want_t = torch.cat([col3["tokens"], col2["tokens"]], 0)
    want_p = torch.cat([ref3, ref2], 0)
    for i in range(5):                                             # per image: one bad image must not average out
        assert rel_l2(tokens[i].float(), want_t[i]) < E2E_TOL, i
        assert rel_l2(proj[i].float(), want_p[i]) < E2E_TOL, i
    # the same images one at a time (batch-1 plan)
    eng1 = pkg.Engine(1024, 896, 2, 1).load(packed, dev)
    for i in (0, 4):
        _, p1 = eng1.forward(x[i:i + 1], False, True)
        # batch 1 selects other kernels for stage 2 (cluster ConvFFN, f16 partial sums): same result up to the chain's amplification of
        # rounding differences (measured 2e-2 through the 51 units; each path is within E2E_TOL of the oracle on its own)
        assert rel_l2(p1[0].float(), proj[i].float()) < E2E_TOL
        assert rel_l2(p1[0].float(), want_p[i]) < E2E_TOL


def test_cluster_convffn_multi_tile_stress(dev):
    """500 launches of the multi-tile 4-CTA-cluster ConvFFN kernel (M = 2 x resident clusters x 128 rows + a ragged tail) back to
    back under PDL: every launch must give the same bits (cross-CTA mbarrier protocol, DSMEM staging reuse across tiles)."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(3)
    C, M = 384, 9000
    z = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.bfloat16).to(dev)
    b1 = torch.randn(4 * C, generator=g).to(dev)
    b2 = torch.randn(C, generator=g).to(dev)
    r = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    first = eng.convffn(z, w1, b1, w2, b2, r)
    torch.cuda.synchronize()
    ref = r.float() + torch.nn.functional.gelu(z.float() @ w1.float().t() + b1) @ w2.float().t() + b2
    assert rel_l2(first.float(), ref) < 6e-3
    for i in range(500):
        out = eng.convffn(z, w1, b1, w2, b2, r)
        if i % 50 == 49:
            assert torch.equal(out, first), i
    torch.cuda.synchronize()
    assert torch.equal(out, first)


def test_graph_replay_determinism_1024(packed, dev):
    """200 CUDA-graph replays of the batch-2 forward at 1024 px (137 PDL-chained kernels each): identical bits every time."""
    eng = pkg.Engine(1024, 896, 2, 2).load(packed, dev)
    x = fx.synthetic_images(2, 1024, seed=31).to(dev)
    _, p0 = eng.forward(x, False, True)
    p0 = p0.clone()
    for i in range(200):
        _, p = eng.forward(x, False, True)
        if i % 40 == 39:
            assert torch.equal(p, p0), i
    torch.cuda.synchronize()


def test_engine_rejects_malformed_buffers(packed, dev):
    eng = pkg.Engine(256, 896, 2, 2).load(packed, dev)
    x = fx.synthetic_images(1, 256).to(dev)
    with pytest.raises(pkg.FvhdError):
        eng.forward(x[:, :, :128], True, True)                       # wrong spatial size
    with pytest.raises(pkg.FvhdError):
        eng.forward(x.cpu(), True, True)                             # wrong device
    emb = torch.zeros(1, 40, 896, dtype=torch.bfloat16, device=dev)
    with pytest.raises(pkg.FvhdError):
        eng.forward_into(x[:, :, :128], emb, 0)                      # forward_into validates images too
    with pytest.raises(pkg.FvhdError):
        eng.encode_images_host(x, None)                              # device tensor passed as host buffer
    with pytest.raises(pkg.FvhdError):
        eng.encode_images_host(x.cpu(), torch.empty(1, 16, 896))     # host_out not bf16
    host = eng.encode_images_host(fx.synthetic_images(5, 256).half().pin_memory())      # batch > max_batch: runs in passes
    assert tuple(host.shape) == (5, 16, 896) and torch.isfinite(host.float()).all()


# ------------------------------------------------------------------ fused all-gather on 2 GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from ml_fastvlm_b200 import parallel as par
        pk = pkg.pack_tower(fx.tower_state_dict())
        pk.update(pkg.pack_projector(fx.projector_state_dict(896)))
        batch = 5                                                     # ragged: 3 + 2, max_batch 2 -> two passes on rank 0
        eng = pkg.Engine(256, 896, 2, 2).load(pk, dev)
        images = fx.synthetic_images(batch, 256, seed=41).to(dev)
        a, b = par.shard_bounds(batch, rank, world)
        ge = par.GatheredEncoder(eng, batch)
        gathered = ge.encode(images[a:b]).clone()
        _, local = eng.forward(images[a:b], False, True)
        ref = par.all_gather_tokens(local, batch)                     # NCCL collective of the per-rank results
        _, full = eng.forward(images, False, True)                    # everything on one GPU
        torch.cuda.synchronize()
        ok = bool(torch.equal(gathered, ref)) and bool(torch.equal(gathered, full))
        gathered2 = ge.encode(images[a:b])                            # buffer reuse
        torch.cuda.synchronize()
        ok = ok and bool(torch.equal(gathered2, full))
        torch.save({"ok": ok}, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (run with gpurun --gpus 2)")
def test_fused_all_gather_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_gather_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert torch.load(os.path.join(str(tmp_path), f"r{r}.pt"))["ok"], f"rank {r}"


# ------------------------------------------------------------------ tcgen05 depthwise mixer (mixer_umma.cuh)
def _mixer_ref(x_nhwc, w3, b3, w7, b7, round_weights):
    """torch fp32 reference of the RepMixer depthwise pair; y is rounded to bf16 between the convs (as the kernel stores it)."""
    import torch.nn.functional as F
    C = x_nhwc.shape[-1]
    x = x_nhwc.float().permute(0, 3, 1, 2)
    if round_weights:
        w3, w7 = w3.to(torch.bfloat16).float(), w7.to(torch.bfloat16).float()
    k3 = w3.t().reshape(C, 1, 3, 3)
    k7 = w7.t().reshape(C, 1, 7, 7)
    y = F.conv2d(x, k3, b3, padding=1, groups=C)
    yb = y.to(torch.bfloat16).float()
    z = F.conv2d(yb, k7, b7, padding=3, groups=C)
    return y.permute(0, 2, 3, 1), z.permute(0, 2, 3, 1)


@pytest.mark.parametrize("B,H,W,C", [
    (1, 64, 64, 384),      # stage 2 at 1024 px
    (2, 128, 128, 192),    # stage 1, batch 2
    (1, 256, 256, 96),     # stage 0
    (1, 16, 16, 384),      # stage 2 at 256 px: map smaller than the 16 x 32 tile
    (3, 40, 24, 32),       # ragged in both directions, 2 channel groups, batch 3
    (1, 96, 96, 48),       # 1536-px geometry (3 tiles across), 3 groups
])
@pytest.mark.parametrize("mode", ["z", "u", "2"])
def test_umma_mixer_vs_torch(dev, B, H, W, C, mode):
    """mode z: Toeplitz tcgen05 kernel (mixer_tz.cuh, bf16 planes and taps); mode u: tcgen05 diagonal-tap kernel (mixer_umma.cuh, bf16
    taps); mode 2: both convs on mma.sync (mixer_tc2.cuh, f16 taps)."""
    os.environ["FVHD_MIXER"] = mode                      # read when the handle is created
    try:
        eng = pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_MIXER", None)
    g = torch.Generator().manual_seed(B * 1000 + H * 10 + C)
    x = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16)
    w3 = torch.randn(9, C, generator=g) / 3.0
    b3 = torch.randn(C, generator=g) * 0.1
    w7 = torch.randn(49, C, generator=g) / 7.0
    b7 = torch.randn(C, generator=g) * 0.1
    y, z = eng.mixer(x.to(dev), w3.to(dev), b3.to(dev), w7.to(dev), b7.to(dev))
    torch.cuda.synchronize()
    yr, zr = _mixer_ref(x, w3, b3, w7, b7, round_weights=(mode == "u"))   # mode u rounds the taps to bf16; mode 2 to f16 (~exact)
    if mode == "z":                                     # mode z: fp32 3x3 taps (FMA pipes), bf16 7x7 taps (Toeplitz tiles)
        yr, zr = _mixer_ref(x, w3, b3, w7.to(torch.bfloat16).float(), b7, round_weights=False)
    ye, ze = _mixer_ref(x, w3, b3, w7, b7, round_weights=False)      # exact fp32 taps (what the oracle computes)
    ey, ez = rel_l2(y.float(), yr), rel_l2(z.float(), zr)
    print(f"mixer[{mode}] {B}x{H}x{W}x{C}: y {ey:.2e} z {ez:.2e} | vs fp32 taps: y {rel_l2(y.float(), ye):.2e} z {rel_l2(z.float(), ze):.2e}")
    assert torch.isfinite(y.float()).all() and torch.isfinite(z.float()).all()
    assert ey < 3e-3 and ez < 4e-3, (ey, ez)                           # bf16 output rounding (y also feeds z)
    assert rel_l2(y.float(), ye) < 5e-3 and rel_l2(z.float(), ze) < 6e-3


@pytest.mark.parametrize("mode", ["z", "u", "2"])
def test_umma_mixer_identity_taps(dev, mode):
    """Centre taps = 1, everything else 0: y == x + b3, z == y + b7 exactly (bf16 in, fp32 accumulate, bf16 out)."""
    os.environ["FVHD_MIXER"] = mode
    try:
        eng = pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_MIXER", None)
    g = torch.Generator().manual_seed(1)
    B, H, W, C = 1, 48, 80, 32
    x = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16)
    w3 = torch.zeros(9, C); w3[4] = 1.0
    w7 = torch.zeros(49, C); w7[24] = 1.0
    zb = torch.zeros(C)
    y, z = eng.mixer(x.to(dev), w3.to(dev), zb.to(dev), w7.to(dev), zb.to(dev))
    if mode in ("u", "z"):
        assert torch.equal(y.cpu(), x) and torch.equal(z.cpu(), x)
    else:       # f16 planes: bf16 values below 2^-14 land on the f16 subnormal grid (quantum 2^-24); everything else is exact
        assert (y.float().cpu() - x.float()).abs().max().item() <= 2 ** -24 and (z.float().cpu() - x.float()).abs().max().item() <= 2 ** -23
        big = x.float().abs() >= 2 ** -14
        assert torch.equal(y.cpu()[big], x[big])


# ------------------------------------------------------------------ second-generation fused ConvFFN (convffn.cuh)
@pytest.mark.parametrize("C,M", [(96, 434), (96, 70000), (192, 9000), (192, 128), (384, 4096), (384, 9000)])
def test_convffn2_vs_torch(dev, C, M):
    """One CTA per 128-row tile, 16 epilogue warps, packed-half GELU, f16 hidden x f16 W2."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(C + M)
    z = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.bfloat16).to(dev)
    b1 = torch.randn(4 * C, generator=g).to(dev)
    b2 = torch.randn(C, generator=g).to(dev)
    r = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w2h = w2.to(torch.float16)                  # the packer's `fc2.wh`
    out = eng.convffn2(z, w1, b1, w2h, b2, r)
    torch.cuda.synchronize()
    ref = r.float() + torch.nn.functional.gelu(z.float() @ w1.float().t() + b1) @ w2h.float().t() + b2
    err = rel_l2(out.float(), ref)
    print(f"convffn2 C={C} M={M}: rel-L2 {err:.2e}")
    assert torch.isfinite(out.float()).all()
    assert err < 4e-3, err                       # bf16 output rounding (2^-9) dominates; H is f16
    out2 = eng.convffn2(z, w1, b1, w2h, b2, r)
    assert torch.equal(out, out2)


def test_convffn2_large_preactivations(dev):
    """Pre-activations far outside the f16-exact range of the packed GELU (|x| up to ~400: x^2 overflows f16 and is clamped)."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(11)
    C, M = 192, 1000
    z = (torch.randn(M, C, generator=g) * 8).to(torch.bfloat16).to(dev)
    w1 = torch.randn(4 * C, C, generator=g).to(torch.bfloat16).to(dev)          # pre-activations ~ N(0, 110^2)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5 / 50).to(torch.float16).to(dev)
    b1 = torch.zeros(4 * C).to(dev)
    b2 = torch.zeros(C).to(dev)
    r = torch.zeros(M, C).to(torch.bfloat16).to(dev)
    out = eng.convffn2(z, w1, b1, w2, b2, r)
    pre = z.float() @ w1.float().t()
    ref = torch.nn.functional.gelu(pre) @ w2.float().t()
    assert pre.abs().max().item() > 300
    assert torch.isfinite(out.float()).all()
    assert rel_l2(out.float(), ref) < 5e-3


@pytest.mark.skipif(os.environ.get("FVHD_PROBE_MIXED") != "1", reason="poisons the CUDA context when unsupported: run alone with FVHD_PROBE_MIXED=1")
def test_convffn2_mixed_format_probe(dev):
    """Probe: f16 hidden x bf16 W2 in one tcgen05.mma (kind::f16 with different A / B formats).  Recorded result in DESIGN.md."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(2)
    C, M = 192, 512
    z = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.bfloat16).to(dev)
    b1 = torch.randn(4 * C, generator=g).to(dev)
    b2 = torch.randn(C, generator=g).to(dev)
    r = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    out = eng.convffn2(z, w1, b1, w2, b2, r)          # bf16 w2 -> mixed-format MMA2
    torch.cuda.synchronize()
    ref = r.float() + torch.nn.functional.gelu(z.float() @ w1.float().t() + b1) @ w2.float().t() + b2
    print("mixed-format probe rel-L2", rel_l2(out.float(), ref))
    assert rel_l2(out.float(), ref) < 4e-3


# ------------------------------------------------------------------ MHSA core: tcgen05 / TMEM kernel (attention_umma.cuh) vs mma.sync kernel vs torch
@pytest.mark.parametrize("mode", ["u", "m"])
@pytest.mark.parametrize("B,N,C", [(1, 1024, 768), (2, 256, 1536), (1, 64, 768), (3, 16, 1536), (1, 2304, 768), (2, 300, 64)])
def test_attention_core_vs_torch(dev, B, N, C, mode):
    """softmax((q 32^-1/2) k^T) v per head of 32 (mci.py:675-679).  N = 1024 / 256: stages 3 / 4 at 1024 px; 64 / 16: at 256 px (one partly
    filled key tile); 2304: 1536 px (18 key tiles, 9 query pairs); 300: ragged tail in keys AND queries."""
    os.environ["FVHD_ATTN"] = mode
    try:
        eng = pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_ATTN", None)
    g = torch.Generator().manual_seed(N + C + B)
    qkv = (torch.randn(B * N, 3 * C, generator=g) * 1.5).to(torch.bfloat16)
    out = eng.attention(qkv.to(dev), B, N)
    torch.cuda.synchronize()
    h = C // 32
    t = qkv.float().reshape(B, N, 3, h, 32).permute(2, 0, 3, 1, 4)
    q, k, v = t[0], t[1], t[2]
    ref = ((q * 32 ** -0.5) @ k.transpose(-2, -1)).softmax(-1) @ v
    ref = ref.transpose(1, 2).reshape(B * N, C)
    err = rel_l2(out.float(), ref)
    print(f"attention[{mode}] B={B} N={N} C={C}: rel-L2 {err:.2e}")
    assert torch.isfinite(out.float()).all()
    assert err < 6e-3, err                       # bf16 P and bf16 output


# ------------------------------------------------------------------ second fixture: the survey's layer-scale range U(0.5, 1.5)
def test_second_fixture_survey_layer_scales(dev):
    """oracle/fixture.py variant "b" (every layer_scale* ~ U(0.5, 1.5), SURVEY 8d): every unit in isolation <= 8e-3, and the whole
    encode_images within 5e-2 AND within 1.25x of the reference algorithm's own bf16 error on this fixture."""
    sd = fx.tower_state_dict(variant="b")
    psd = fx.projector_state_dict(896)
    pk = pkg.pack_tower(sd)
    pk.update(pkg.pack_projector(psd))
    eng = pkg.Engine(256, 896, 2, 1).load(pk, dev)
    x = fx.synthetic_images(1, 256, seed=9)
    col = {}
    ref = orc.encode_images(x, sd, psd, col)
    prev, worst = None, {}
    for u in eng.units():
        name = u["name"]
        if name == "stem":
            xin, want = x.to(dev), col["stem"].permute(0, 2, 3, 1)
        elif name == "conv_exp":
            xin, want = _nhwc(prev, dev), col["tokens"]
        elif name == "projector":
            xin, want = col["tokens"].reshape(1, -1).to(torch.bfloat16).to(dev), ref
        else:
            xin, want = _nhwc(prev, dev), col[name].permute(0, 2, 3, 1)
        got = eng.run_units(u["index"], u["index"], xin, 1)
        worst[name] = rel_l2(got.float().reshape(-1), want.reshape(-1))
        prev = col.get(name)
    bad = {k: v for k, v in worst.items() if v > 8e-3}
    assert not bad, bad
    _, proj = eng.forward(x.to(dev), False, True)
    sdb = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v) for k, v in sd.items()}
    psdb = {k: v.to(torch.bfloat16) for k, v in psd.items()}
    with torch.no_grad():
        prj_b = orc.mm_projector(orc.feature_select(orc.fastvit_forward(x.to(torch.bfloat16), sdb)), psdb)
    e, eb = rel_l2(proj.float(), ref), rel_l2(prj_b.float(), ref)
    print(f"fixture b: encode_images rel-L2 {e:.3e} (reference's own bf16 run: {eb:.3e}); worst unit {max(worst.values()):.2e}")
    assert e < E2E_TOL and e <= 1.25 * eb


def test_repmixer_block_large_activations(packed, tower_sd, dev):
    """The f16 paths inside a RepMixer block (y planes of the mma.sync mixer, packed-half GELU / f16 hidden of the fused ConvFFN,
    f16 partials of the cluster ConvFFN) keep their accuracy for activations three orders of magnitude above the fixture's
    (|x| ~ 4e3, well inside the f16 range the reference itself runs in -- predict.py:58 `.half()`), and SATURATE to finite
    values (cvt.satfinite) instead of producing inf / NaN when an activation leaves the f16 range."""
    eng = pkg.Engine(256, 896, 2, 1).load(packed, dev)
    units = {u["name"]: u for u in eng.units()}
    g = torch.Generator().manual_seed(17)
    for name, c, hw in (("network.2.3", 192, 32), ("network.4.5", 384, 16)):       # a stage-1 block (fused kernel) and a stage-2 block (cluster kernel)
        u = units[name]
        p = fx.TOWER_PREFIX + name
        for scale, check in ((1e3, True), (1e5, False)):
            x = (torch.randn(1, c, hw, hw, generator=g) * scale).to(torch.bfloat16)
            want = orc.repmixer_block(x.float(), tower_sd, p).permute(0, 2, 3, 1).reshape(-1)
            got = eng.run_units(u["index"], u["index"], _nhwc(x.float(), dev), 1).float().reshape(-1)
            assert torch.isfinite(got).all(), (name, scale)
            if check:
                err = rel_l2(got, want)
                print(f"{name} x{scale:g}: rel-L2 {err:.2e}")
                assert err < 8e-3, (name, scale, err)


# ------------------------------------------------------------------ plan variants: Toeplitz tcgen05 mixer, stem generations
def _engine_env(R, packed, dev, env, batch=1, max_batch=None):
    """Engine created, and its first plan (`batch` images) built, under the given FVHD_* switches (the library reads them once per
    handle, when the handle is created); the mixer / stem switches the caller does not name are unset meanwhile."""
    keys = {"FVHD_MIX_TILE", "FVHD_MIXER", "FVHD_STEM", *env}
    old = {k: os.environ.pop(k, None) for k in keys}
    os.environ.update(env)
    try:
        eng = pkg.Engine(R, 896, 2, max_batch or batch).load(packed, dev)
        eng.forward(fx.synthetic_images(batch, R).to(dev), False, True)
    finally:
        for k in keys:
            os.environ.pop(k, None)
            if old[k] is not None:
                os.environ[k] = old[k]
    return eng


def test_tz_mixer_units_vs_oracle_1024(packed, oracle1024_b3, dev):
    """Every RepMixer block through the Toeplitz tcgen05 mixer (mixer_tz.cuh, FVHD_MIXER=z) at 1024 px, batch 3, fed the oracle's inputs."""
    x, ref, col = oracle1024_b3
    B = x.shape[0]
    eng = _engine_env(1024, packed, dev, {"FVHD_MIXER": "z"}, batch=B)
    steps = eng.steps(B)
    assert any(s["kernel"] == "repmixer_tz_kernel" for s in steps)
    prev, worst, n = None, 0.0, 0
    for u in eng.units():
        name = u["name"]
        if prev is not None and any(s["unit"] == u["index"] and s["kernel"] == "repmixer_tz_kernel" for s in steps):
            got = eng.run_units(u["index"], u["index"], _nhwc(prev, dev), B)
            assert torch.isfinite(got.float()).all(), name
            worst = max(worst, rel_l2(got.float().reshape(-1), col[name].permute(0, 2, 3, 1).reshape(-1)))
            n += 1
        prev = col.get(name)
    print(f"tz mixer blocks: {n}, worst unit error {worst:.2e}")
    assert n == 38 and worst < UNIT_TOL_1024, (n, worst)


def test_tz_mixer_end_to_end_256_and_ragged(packed, tower_sd, proj_sd, dev):
    """encode_images with FVHD_MIXER=z at 256 px (maps smaller than the 64 x 32 tile in stage 2) vs the oracle, and == itself on a rerun."""
    x = fx.synthetic_images(2, 256, seed=7)
    ref = orc.encode_images(x, tower_sd, proj_sd)
    eng = _engine_env(256, packed, dev, {"FVHD_MIXER": "z"}, batch=2)
    _, p1 = eng.forward(x.to(dev), False, True)
    _, p2 = eng.forward(x.to(dev), False, True)
    torch.cuda.synchronize()
    assert torch.equal(p1, p2)
    assert rel_l2(p1.float(), ref) < E2E_TOL


@pytest.mark.parametrize("R,B", [(256, 2), (1024, 1)])
def test_stem_generations_agree(packed, tower_sd, proj_sd, dev, R, B):
    """stem2_kernel (default: persistent, packed-half GELUs) and the first-generation stem_kernel (FVHD_STEM=1) against the oracle's stem."""
    x = fx.synthetic_images(B, R, seed=11)
    col = {}
    want = orc.convolutional_stem(x, tower_sd).permute(0, 2, 3, 1).reshape(-1)
    outs = {}
    for gen in ("2", "1"):
        eng = _engine_env(R, packed, dev, {"FVHD_STEM": gen}, batch=B)
        names = {s["kernel"] for s in eng.steps(B)}
        assert ("stem2_kernel" in names) == (gen == "2") and ("stem_kernel" in names) == (gen == "1")
        u = eng.units()[0]
        assert u["name"] == "stem"
        for dt in (torch.bfloat16, torch.float16, torch.float32):
            got = eng.run_units(0, 0, x.to(dev).to(dt), B)
            e = rel_l2(got.float().reshape(-1), want)
            assert torch.isfinite(got.float()).all() and e < UNIT_TOL_1024, (gen, dt, e)
        outs[gen] = eng.run_units(0, 0, x.to(dev).to(torch.bfloat16), B)
    d = rel_l2(outs["2"].float(), outs["1"].float())
    print(f"stem R={R}: gen2 vs gen1 {d:.2e}")
    assert d < 6e-3


# ------------------------------------------------------------------ fused ConvFFN, 2-CTA clusters sharing the weight stream
@pytest.mark.parametrize("C,M", [(96, 70000), (192, 9000), (192, 128), (384, 4096), (384, 9000), (384, 40000)])
def test_convffn2_weight_sharing_clusters_bit_identical(dev, C, M):
    """convffn_tcgen05_kernel<C, 2> (TMA-multicast weight ring shared by two CTAs; odd tile counts leave rank 1 one dummy tile) must
    reproduce the single-CTA kernel bit for bit: same MMAs in the same order, only the origin of the weight bytes differs."""
    g = torch.Generator().manual_seed(3 * C + M)
    z = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
    w2h = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.float16).to(dev)
    b1 = torch.randn(4 * C, generator=g).to(dev)
    b2 = torch.randn(C, generator=g).to(dev)
    r = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    outs = {}
    for cs in ("1", "2"):
        os.environ["FVHD_CONVFFN_CS"] = cs                # read when the handle is created: one engine per cluster size
        try:
            eng = pkg.Engine(64, 0, 2, 1)
        finally:
            os.environ.pop("FVHD_CONVFFN_CS", None)
        outs[cs] = [eng.convffn2(z, w1, b1, w2h, b2, r) for _ in range(3)]
        torch.cuda.synchronize()
    ref = r.float() + torch.nn.functional.gelu(z.float() @ w1.float().t() + b1) .to(torch.float16).float() @ w2h.float().t() + b2
    assert rel_l2(outs["1"][0].float(), ref) < 6e-3
    for o in outs["2"]:
        assert torch.equal(o, outs["1"][0])


def test_default_plan_picks_mixer_per_launch(packed, dev):
    """Default plan at 1024 px: the Toeplitz tcgen05 mixer where a launch has at least one 64 x 32 x 8 item per SM (stages 0-1 at batch 1,
    every stage at batch 4), the finer-grained mma.sync mixer below that (stage 2 of a single image: 96 items)."""
    eng = _engine_env(1024, packed, dev, {}, batch=4)
    k1 = [s["kernel"] for s in eng.steps(1)]
    k4 = [s["kernel"] for s in eng.steps(4)]
    assert k1.count("repmixer_tz_kernel") == 14 and k1.count("repmixer_tc_kernel") == 24, (k1.count("repmixer_tz_kernel"), k1.count("repmixer_tc_kernel"))
    assert k4.count("repmixer_tz_kernel") == 38 and "repmixer_tc_kernel" not in k4


def test_handles_keep_their_own_switches(packed, dev):
    """Kernel-selection switches are read once per handle, when it is created: a handle created later without them changes
    neither the plans nor the single-kernel entries of an earlier one, and is not affected by it either."""
    a = _engine_env(256, packed, dev, {"FVHD_MIXER": "u"}, batch=1, max_batch=2)
    b = _engine_env(256, packed, dev, {})
    assert "repmixer_umma_kernel" in {s["kernel"] for s in a.steps(2)}          # A's batch-2 plan is built after B exists
    g = torch.Generator().manual_seed(6)
    x = torch.randn(1, 32, 32, 96, generator=g).to(torch.bfloat16).to(dev)
    w3, b3 = (torch.randn(9, 96, generator=g) / 3).to(dev), (torch.randn(96, generator=g) * 0.1).to(dev)
    w7, b7 = (torch.randn(49, 96, generator=g) / 7).to(dev), (torch.randn(96, generator=g) * 0.1).to(dev)
    os.environ["FVHD_MIXER"] = "u"
    try:
        fresh_u = pkg.Engine(64, 0, 2, 1)
    finally:
        os.environ.pop("FVHD_MIXER", None)
    ya, za = a.mixer(x, w3, b3, w7, b7)
    yu, zu = fresh_u.mixer(x, w3, b3, w7, b7)
    assert torch.equal(ya, yu) and torch.equal(za, zu)
    fresh = _engine_env(256, packed, dev, {})
    assert b.steps(1) == fresh.steps(1)
    assert "repmixer_umma_kernel" not in {s["kernel"] for s in b.steps(1)}


@pytest.mark.parametrize("env", [{}, {"FVHD_CONVFFN": "1"}, {"FVHD_NO_FUSED_MLP": "1"}])
@pytest.mark.parametrize("R", [256, 1024])
def test_launches_per_forward_is_the_plan(packed, dev, R, env):
    """fvhd_launches_per_forward == the plan's kernels + set_io_kernel for every batch up to max_batch (at 1024 px the stage-2
    ConvFFN kernel depends on the batch), and the sum over the passes above it."""
    mb = 4
    eng = _engine_env(R, packed, dev, env, batch=1, max_batch=mb)
    per_pass = {b: len(eng.steps(b)) + 1 for b in range(1, mb + 1)}
    for b, n in per_pass.items():
        assert eng.launches_per_forward(b) == n, (b, n)
    assert eng.launches_per_forward(2 * mb + 3) == 2 * per_pass[mb] + per_pass[3]


# ------------------------------------------------------------------ row f4 on the GPU: released-layout checkpoint -> drop-in modules
def test_released_layout_checkpoint_runs_on_gpu(tmp_path, tower_sd, proj_sd, dev):
    """A released-style folder (sharded safetensors with `model.vision_tower.*` / `model.mm_projector.*` keys among LLM tensors,
    config.json) -> `load_pretrained` -> the drop-in tower + projector on the GPU: `encode_images` (the reference's two calls,
    llava_arch.py:141-144) matches the oracle run on the same state dicts."""
    import json
    from safetensors.torch import save_file
    full = {("model.vision_tower." + k): v.contiguous() for k, v in tower_sd.items()}
    full.update({("model.mm_projector." + k): v.contiguous() for k, v in proj_sd.items()})
    full["model.embed_tokens.weight"] = torch.zeros(8, 896)
    keys = list(full.keys())
    half = len(keys) // 2
    save_file({k: full[k] for k in keys[:half]}, str(tmp_path / "model-00001-of-00002.safetensors"))
    save_file({k: full[k] for k in keys[half:]}, str(tmp_path / "model-00002-of-00002.safetensors"))
    json.dump({"mm_vision_tower": "mobileclip_l_256", "hidden_size": 896, "mm_hidden_size": 3072, "mm_projector_type": "mlp2x_gelu"},
              open(tmp_path / "config.json", "w"))
    tower, proj, cfg = pkg.load_pretrained(str(tmp_path), device=dev, dtype=torch.float16)
    x = fx.synthetic_images(2, 256, seed=5)
    ref = orc.encode_images(x, tower_sd, proj_sd)
    with torch.no_grad():
        feats = proj(tower(x.to(dev).half()))                       # the reference's encode_images body, module by module
        fused = tower.encode_with_projector(x.to(dev).half(), proj)  # the one-call path encode_images takes (glue.py)
    assert feats.dtype == torch.float16 and tuple(feats.shape) == (2, 16, 896)
    assert rel_l2(feats.float(), ref) < E2E_TOL and rel_l2(fused.float(), ref) < E2E_TOL
