"""GPU parity tests (-m gpu): the CUDA path through the C ABI vs the oracle, the golden vectors of the
unmodified reference, and size-independent properties at the bench size.

Tolerances (bf16 activations + bf16 GEMM weights, fp32 accumulation, vs the fp32 oracle):
  * a single unit fed the oracle's own input ........ rel-L2 <= 8e-3 (measured 2.3e-3 .. 4.5e-3)
  * whole tower / encode_images (51 units chained) .. rel-L2 <= 5e-2 AND <= 1.25 x the error of the
    reference algorithm's own bf16 run (PyTorch bf16, same fixture: 3.8e-2 at R=256; bf16 weight
    rounding alone gives ~7e-3; measured CUDA path: 3.3e-2)
  * token count / shapes ............................ exact.
"""
import os

import numpy as np
import pytest
import torch

import ml_fastvlm_b200 as pkg
from oracle import fastvithd_oracle as orc
from oracle import fixture as fx
from oracle.gen_golden import N_SAMPLES_1024, sample_indices

pytestmark = pytest.mark.gpu

UNIT_TOL = 8e-3
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


@pytest.fixture(scope="module")
def eng256(packed, dev):
    return pkg.Engine(256, 896, 2, 2).load(packed, dev)


@pytest.fixture(scope="module")
def oracle256(tower_sd, proj_sd):
    col = {}
    out = orc.encode_images(fx.synthetic_images(1, 256), tower_sd, proj_sd, col)
    return out, col


# ------------------------------------------------------------------ tcgen05 GEMM
@pytest.mark.parametrize("M,N,K,act,use_bias,use_res", [
    (128, 128, 64, 0, False, False),       # one tile, one k-block
    (128, 128, 512, 0, False, False),      # ring wraps (8 k-blocks, 3 stages)
    (1000, 96, 96, 1, True, False),        # ragged M, BN=96, K not a multiple of 64 (TMA zero fill)
    (65536, 96, 96, 1, True, False),       # stem 1x1 at R=1024
    (4096, 1536, 384, 1, True, False),     # stage-2 fc1
    (4096, 384, 1536, 0, True, True),      # stage-2 fc2 + residual
    (16, 896, 3072, 1, True, False),       # projector layer 0 at R=256 (M << tile)
    (300, 2304, 768, 0, False, False),     # qkv, no bias
    (512, 200, 256, 0, True, False),       # N % 32 != 0 (column tail)
    (1, 3584, 3584, 0, True, False),       # single row
])
def test_gemm_against_fp32(dev, M, N, K, act, use_bias, use_res):
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, generator=g).to(torch.bfloat16).to(dev)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(torch.bfloat16).to(dev)
    b = torch.randn(N, generator=g).to(dev) if use_bias else None
    r = torch.randn(M, N, generator=g).to(torch.bfloat16).to(dev) if use_res else None
    D = eng.gemm(A, W, b, r, act)
    ref = A.float() @ W.float().t()
    if b is not None:
        ref = ref + b
    if act:
        ref = torch.nn.functional.gelu(ref)
    if r is not None:
        ref = ref + r.float()
    assert D.shape == (M, N) and D.dtype == torch.bfloat16
    assert rel_l2(D.float(), ref) < 4e-3            # bf16 output rounding only (2^-9 relative)
    assert (D.float() - ref).abs().max().item() < 0.05 * max(1.0, ref.abs().max().item())


def test_gemm_gelu_epilogue_wide_range(dev):
    """The epilogue GELU (1-MUFU tanh form fitted to erf) must hold for pre-activations far outside +-8."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(9)
    M, N, K = 512, 256, 128
    A = (torch.randn(M, K, generator=g) * 8).to(torch.bfloat16).to(dev)
    W = (torch.randn(N, K, generator=g)).to(torch.bfloat16).to(dev)       # pre-activations ~ N(0, 90^2)
    D = eng.gemm(A, W, None, None, 1)
    pre = A.float() @ W.float().t()
    ref = torch.nn.functional.gelu(pre)
    assert pre.abs().max().item() > 200
    assert rel_l2(D.float(), ref) < 4e-3
    small = pre.abs() < 6                                                  # the non-saturated region, absolute check
    assert (D.float() - ref)[small].abs().max().item() < 0.03


def test_gemm_linearity_large(dev):
    """Size-independent property at a bench-size problem: D(A1 + A2) == D(A1) + D(A2) (no bias)."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(5)
    M, N, K = 65536, 384, 96
    A1 = torch.randn(M, K, generator=g).to(torch.bfloat16).to(dev)
    A2 = (torch.randn(M, K, generator=g) * 2 ** -9).to(torch.bfloat16).to(dev)   # keeps A1 + A2 exact in bf16? no: compare in fp32
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(torch.bfloat16).to(dev)
    d1 = eng.gemm(A1, W).float()
    d2 = eng.gemm(A2, W).float()
    d12 = eng.gemm((A1.float() + A2.float()).to(torch.bfloat16), W).float()
    ref12 = (A1.float() + A2.float()).to(torch.bfloat16).float() @ W.float().t()
    assert rel_l2(d12, ref12) < 4e-3
    assert rel_l2(d1 + d2, A1.float() @ W.float().t() + A2.float() @ W.float().t()) < 4e-3


# ------------------------------------------------------------------ units, isolated
def _nhwc(t, dev):
    return t.permute(0, 2, 3, 1).contiguous().reshape(t.shape[0], -1).to(torch.bfloat16).to(dev)


def test_every_unit_isolated_256(eng256, oracle256, dev):
    ref, col = oracle256
    x = fx.synthetic_images(1, 256)
    prev = None
    worst = {}
    for u in eng256.units():
        name = u["name"]
        if name == "stem":
            xin, want = x.to(dev), col["stem"].permute(0, 2, 3, 1)
        elif name == "conv_exp":
            xin, want = _nhwc(prev, dev), col["tokens"]
        elif name == "projector":
            xin, want = col["tokens"].reshape(1, -1).to(torch.bfloat16).to(dev), ref
        else:
            xin, want = _nhwc(prev, dev), col[name].permute(0, 2, 3, 1)
        got = eng256.run_units(u["index"], u["index"], xin, 1)
        assert got.shape == (1, u["out_elems"])
        assert torch.isfinite(got.float()).all(), name
        worst[name] = rel_l2(got.float().reshape(-1), want.reshape(-1))
        prev = col.get(name)
    bad = {k: v for k, v in worst.items() if v > UNIT_TOL}
    assert not bad, bad


def _engine_with_env(R, packed, dev, env, batch=1):
    """Engine created, and its first plan built, under the given environment switches (the library reads them once per handle,
    when the handle is created); the mixer / ConvFFN switches the caller does not name are unset meanwhile."""
    keys = {"FVHD_MIX_TILE", "FVHD_MIXER", "FVHD_NO_FUSED_MLP", "FVHD_NO_CLUSTER_MLP", "FVHD_CONVFFN", *env}
    old = {k: os.environ.pop(k, None) for k in keys}
    os.environ.update(env)
    try:
        eng = pkg.Engine(R, 896, 2, batch).load(packed, dev)
        eng.forward(fx.synthetic_images(batch, R).to(dev), False, True)
    finally:
        for k in keys:
            os.environ.pop(k, None)
            if old[k] is not None:
                os.environ[k] = old[k]
    return eng


def test_mixer_variants_agree(packed, oracle256, dev):
    """RepMixer depthwise pair: tcgen05 diagonal-tap mixer (mixer_umma.cuh, FVHD_MIXER=u) vs the mma.sync-7x7 kernel (FVHD_MIXER=t) vs the Toeplitz tcgen05 kernel (default) vs the FMA-pipe
    kernel (FVHD_MIX_TILE=a): same oracle inputs, each block in isolation, including ragged maps smaller than a tile."""
    ref, col = oracle256
    um, tc, fma, tz = (_engine_with_env(256, packed, dev, e) for e in ({"FVHD_MIXER": "u"}, {"FVHD_MIXER": "t"}, {"FVHD_MIX_TILE": "a"}, {"FVHD_MIXER": "z"}))
    kern = lambda e: {s["kernel"] for s in e.steps(1)}
    assert "repmixer_umma_kernel" in kern(um) and "repmixer_tc_kernel" in kern(tc) and "repmixer_dw_kernel" in kern(fma)
    assert "repmixer_tz_kernel" in kern(tz)               # Toeplitz tcgen05 mixer (mixer_tz.cuh): the default wherever a launch has >= 1 item per SM
    prev, worst = None, 0.0
    for u in um.units():
        name = u["name"]
        if prev is not None and any(s["unit"] == u["index"] and s["kernel"] == "repmixer_umma_kernel" for s in um.steps(1)):
            xin = _nhwc(prev, dev)
            outs = [e.run_units(u["index"], u["index"], xin, 1) for e in (um, tc, fma, tz)]
            want = col[name].permute(0, 2, 3, 1).reshape(-1)
            for o in outs:
                assert rel_l2(o.float().reshape(-1), want) < UNIT_TOL, name
            worst = max(worst, rel_l2(outs[0], outs[1]), rel_l2(outs[0], outs[2]), rel_l2(outs[0], outs[3]))
        prev = col.get(name)
    assert 0.0 < worst < 8e-3, worst          # different rounding inside the block (bf16 taps / f16 y / bf16 y), nothing more
    # ragged tiles: at 128 px stage 1 is 16x16, stage 2 is 8x8 -- smaller than any tile; random activations
    outs = {}
    for key, env in (("u", {"FVHD_MIXER": "u"}), ("a", {"FVHD_MIX_TILE": "a"})):
        eng = _engine_with_env(128, packed, dev, env)
        units = [u for u in eng.units() if u["name"].startswith("network.4.") or u["name"].startswith("network.2.")]
        g = torch.Generator().manual_seed(5)
        res = []
        for u in (units[0], units[-1]):
            xin = torch.randn(1, u["in_elems"], generator=g).to(torch.bfloat16).to(dev)
            res.append(eng.run_units(u["index"], u["index"], xin, 1))
        outs[key] = res
    for a, b in zip(outs["u"], outs["a"]):
        assert torch.isfinite(a.float()).all() and rel_l2(a, b) < 8e-3


# ------------------------------------------------------------------ end to end
def test_encode_images_256_vs_oracle_and_reference_golden(eng256, oracle256, golden_dir, dev):
    ref, col = oracle256
    tokens, proj = eng256.forward(fx.synthetic_images(1, 256).to(dev), True, True)
    assert tuple(tokens.shape) == (1, 16, 3072) and tuple(proj.shape) == (1, 16, 896)       # bit-exact shapes
    assert rel_l2(tokens.float(), col["tokens"]) < E2E_TOL
    assert rel_l2(proj.float(), ref) < E2E_TOL
    g = np.load(os.path.join(golden_dir, "ref_256.npz"))                                      # unmodified reference
    assert rel_l2(tokens.float(), g["tokens"]) < E2E_TOL
    assert rel_l2(proj.float(), g["projected"]) < E2E_TOL


def test_not_worse_than_reference_bf16(eng256, oracle256, tower_sd, proj_sd, dev):
    """Anchor: run the reference algorithm itself in bf16 (torch CPU) and require the CUDA path to be
    within 1.25x of that error against the fp32 oracle."""
    ref, col = oracle256
    x = fx.synthetic_images(1, 256)
    sdb = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v) for k, v in tower_sd.items()}
    psdb = {k: v.to(torch.bfloat16) for k, v in proj_sd.items()}
    with torch.no_grad():
        tok_b = orc.feature_select(orc.fastvit_forward(x.to(torch.bfloat16), sdb))
        prj_b = orc.mm_projector(tok_b, psdb)
    tokens, proj = eng256.forward(x.to(dev), True, True)
    assert rel_l2(tokens.float(), col["tokens"]) <= 1.25 * rel_l2(tok_b.float(), col["tokens"])
    assert rel_l2(proj.float(), ref) <= 1.25 * rel_l2(prj_b.float(), ref)


def test_tokens_1024_vs_reference_golden(packed, tower_sd, golden_dir, dev):
    eng = pkg.Engine(1024, 0, 2, 1).load({k: v for k, v in packed.items() if not k.startswith("projector")}, dev)
    x = fx.synthetic_images(1, 1024)
    tokens, _ = eng.forward(x.to(dev), True, False)
    assert tuple(tokens.shape) == (1, 256, 3072)                                              # FastVLM.swift:303
    g = np.load(os.path.join(golden_dir, "ref_1024_tokens_sample.npz"))                      # unmodified reference, seeded sample
    flat = tokens.float().reshape(-1).cpu()
    assert rel_l2(flat[torch.from_numpy(sample_indices(flat.numel(), "tokens_1024", N_SAMPLES_1024))], g["samples"]) < E2E_TOL
    assert rel_l2(tokens.float(), orc.tower_forward(x, tower_sd)) < E2E_TOL                   # whole tensor vs the oracle


def test_encode_images_1536_7b_shape_vs_oracle(tower_sd, dev):
    """BASELINE configs[4] geometry: R=1536 -> 576 tokens, projector H=3584 (Qwen2-7B).  Maps of 384/192/96/48/24 px: partial
    16x16 tiles, TMA zero-filled halos past the edge, 2304-key attention."""
    psd = fx.projector_state_dict(3584)
    pk = pkg.pack_tower(tower_sd)
    pk.update(pkg.pack_projector(psd))
    eng = pkg.Engine(1536, 3584, 2, 1).load(pk, dev)
    x = fx.synthetic_images(1, 1536, seed=2)
    tokens, proj = eng.forward(x.to(dev), True, True)
    assert tuple(tokens.shape) == (1, 576, 3072) and tuple(proj.shape) == (1, 576, 3584)
    col = {}
    ref = orc.encode_images(x, tower_sd, psd, col)
    assert rel_l2(tokens.float(), col["tokens"]) < E2E_TOL
    assert rel_l2(proj.float(), ref) < E2E_TOL


def test_input_dtypes_and_batch_chunking(eng256, dev):
    """fp32 / fp16 / bf16 images; B=5 with max_batch=2 (3 passes) == per-image results, bit-exact.
    The random-weight fixture amplifies an input perturbation ~70x (fp16 rounding of the pixels, 5e-4, moves the
    tokens by ~3.5e-2), so cross-dtype agreement is only checked loosely; same-dtype results must be identical."""
    x = fx.synthetic_images(5, 256, seed=11)
    t32, p32 = eng256.forward(x.to(dev), True, True)
    t16, _ = eng256.forward(x.half().to(dev), True, False)
    tbf, _ = eng256.forward(x.bfloat16().to(dev), True, False)
    assert rel_l2(t16.float(), t32.float()) < 0.1 and rel_l2(tbf.float(), t32.float()) < 0.5
    t16b, _ = eng256.forward(x.half().float().to(dev), True, False)        # same values, other container dtype
    assert torch.equal(t16, t16b)
    for i in range(5):
        ti, pi = eng256.forward(x[i:i + 1].to(dev), True, True)
        assert torch.equal(ti[0], t32[i]) and torch.equal(pi[0], p32[i])                      # images are independent
    with pytest.raises(pkg.FvhdError):
        eng256.forward(torch.rand(1, 3, 128, 128, device=dev))                                # wrong R


def test_host_entry_matches_device_entry(eng256, dev):
    x = fx.synthetic_images(2, 256, seed=3)
    host_in = x.half().pin_memory()
    host_out = eng256.encode_images_host(host_in)
    _, proj16 = eng256.forward(x.half().to(dev), False, True)
    assert host_out.dtype == torch.bfloat16 and tuple(host_out.shape) == (2, 16, 896)
    assert torch.equal(host_out, proj16.cpu())                                                # same bits as the device entry


def test_missing_weights_and_workspace_fail_loudly(packed, dev):
    eng = pkg.Engine(256, 896, 2, 1)
    with pytest.raises(pkg.FvhdError):
        eng.load({k: v for k, v in packed.items() if k != "network.4.7.fc1.w"}, dev)
    with pytest.raises(pkg.FvhdError):
        pkg.Engine(256, 0, 2, 1).forward(torch.rand(1, 3, 256, 256, device=dev))            # load() not called


def test_fused_convffn_is_bit_identical_to_two_gemms(packed, dev):
    """mlp_fused_tcgen05_kernel keeps the fc2 accumulation order of the unfused path (hidden chunk j == k-block j), so the
    whole forward must agree BIT FOR BIT with FVHD_NO_FUSED_MLP=1 (each variant on its own engine, created under its switches)."""
    x = fx.synthetic_images(2, 512, seed=4).to(dev)

    def run(env):
        eng = _engine_with_env(512, packed, dev, env, batch=2)
        t, p = eng.forward(x, True, True)
        return {"t": t.cpu(), "p": p.cpu(), "launches": eng.launches_per_forward(2)}

    outs = [run({"FVHD_NO_FUSED_MLP": v, "FVHD_NO_CLUSTER_MLP": "1", "FVHD_CONVFFN": "1"}) for v in ("0", "1")]     # first-generation fused kernel
    assert outs[0]["launches"] == outs[1]["launches"] - 14            # 2 + 12 RepMixer blocks lose one launch each
    assert torch.isfinite(outs[0]["p"].float()).all()
    assert torch.equal(outs[0]["t"], outs[1]["t"]) and torch.equal(outs[0]["p"], outs[1]["p"])
    # stage 2 (C = 384): the 4-CTA-cluster kernel sums four partial accumulators (hidden split across the cluster; the three
    # remote ones travel as f16) instead of one 24-k-block chain, so it is NOT bit-identical: single-ulp bf16 differences
    # per block, which this random-weight fixture amplifies ~70x through the remaining depth (tests/golden/sensitivity.json;
    # the reference's own bf16 run sits 3.8e-2 from its fp32 run).  Bound: two valid bf16 pipelines must agree to that
    # level; parity of the cluster path itself is checked unit by unit and end to end against the oracle above.
    clus = run({"FVHD_NO_FUSED_MLP": "0", "FVHD_NO_CLUSTER_MLP": "0", "FVHD_CONVFFN": "1"})
    assert clus["launches"] == outs[0]["launches"] - 24               # 24 stage-2 blocks lose one launch each
    assert torch.isfinite(clus["p"].float()).all()
    dt, dp = rel_l2(clus["t"], outs[0]["t"]), rel_l2(clus["p"], outs[0]["p"])
    assert dt < 4e-2 and dp < 4e-2, (dt, dp)
    # the default plan (second-generation fused kernel, f16 hidden + packed-half GELU, convffn.cuh): same launch count as the
    # fully fused first-generation plan, and -- a different but equally valid rounding of the hidden -- within the same bound
    gen2 = run({})
    assert gen2["launches"] == clus["launches"]
    dt, dp = rel_l2(gen2["t"], outs[1]["t"]), rel_l2(gen2["p"], outs[1]["p"])
    assert torch.isfinite(gen2["p"].float()).all() and dt < 4e-2 and dp < 4e-2, (dt, dp)


@pytest.mark.parametrize("C,M", [(96, 128 * 150 + 40), (192, 128 * 9), (384, 4096), (384, 128 * 80 + 128)])
def test_convffn_kernels_standalone(C, M, dev):
    """Fused ConvFFN kernels on random operands vs torch (fp32 math on the same bf16 operands, hidden rounded to bf16 as the
    kernels do): single-CTA kernel for C = 96 / 192 (ragged last tile, several tiles per CTA), 4-CTA-cluster kernel for
    C = 384 (one tile per cluster, and 81 tiles over <= 37 clusters: the multi-tile path re-uses the DSMEM receive buffer)."""
    eng = pkg.Engine(64, 0, 2, 1)
    g = torch.Generator().manual_seed(C + M)
    z = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    resid = torch.randn(M, C, generator=g).to(torch.bfloat16).to(dev)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(dev)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.bfloat16).to(dev)
    b1 = torch.randn(4 * C, generator=g).to(dev)
    b2 = torch.randn(C, generator=g).to(dev)
    out = eng.convffn(z, w1, b1, w2, b2, resid)
    hid = torch.nn.functional.gelu(z.float() @ w1.float().t() + b1).to(torch.bfloat16).float()
    ref = hid @ w2.float().t() + b2 + resid.float()
    assert torch.isfinite(out.float()).all()
    assert rel_l2(out, ref) < 4e-3                                   # bf16 output rounding (2^-9) + GELU approximation
    assert (out.float() - ref).abs().max().item() < 0.08
    again = eng.convffn(z, w1, b1, w2, b2, resid)
    assert torch.equal(out, again)                                   # deterministic (fixed reduction order)


# ------------------------------------------------------------------ drop-in modules
class _Args:
    mm_vision_tower = "mobileclip_l_256"
    unfreeze_mm_vision_tower = False
    mm_projector_type = "mlp2x_gelu"
    mm_hidden_size = 3072
    hidden_size = 896


def test_tower_and_projector_modules(tower_sd, proj_sd, oracle256, golden_dir, dev):
    ref, col = oracle256
    tower = pkg.build_vision_tower(_Args())
    tower.load_state_dict(tower_sd, strict=True)
    proj = pkg.build_vision_projector(_Args())
    proj.load_state_dict(proj_sd, strict=True)
    tower.to(device=dev, dtype=torch.bfloat16)          # llava/model/builder.py:173 does .to(device, dtype)
    proj.to(device=dev, dtype=torch.bfloat16)
    x = fx.synthetic_images(2, 256, seed=7)
    g = np.load(os.path.join(golden_dir, "ref_b2_256.npz"))
    feats = tower(x.to(dev))                            # fp32 images -> features come back in images.dtype
    assert feats.dtype == torch.float32 and tuple(feats.shape) == (2, 16, 3072)
    assert rel_l2(feats, g["tokens"]) < E2E_TOL
    lst = tower([x[0].to(dev), x[1].to(dev)])           # list branch (mobileclip_encoder.py:78-83)
    assert isinstance(lst, list) and tuple(lst[0].shape) == (1, 16, 3072)
    assert rel_l2(lst[1], g["list1"]) < E2E_TOL

    class Model:                                        # the two accessors encode_images uses (llava_arch.py:141-144)
        def __init__(self):
            self.mm_projector = proj
        def get_model(self):
            return self
        def get_vision_tower(self):
            return tower
    m = Model()
    with pytest.raises(NotImplementedError):            # nn.Linear parameters require grad by default: training is refused loudly
        proj(feats.to(dev))
    with torch.inference_mode():                        # predict.py:60 / HF generate run the path without grad
        fused = pkg.encode_images(m, fx.synthetic_images(1, 256).to(dev))
        split = proj(tower(fx.synthetic_images(1, 256).to(dev)))
    assert tuple(fused.shape) == (1, 16, 896)
    assert rel_l2(fused, ref) < E2E_TOL and rel_l2(split, ref) < E2E_TOL
    assert rel_l2(fused, split) < 5e-3                  # same kernels; split path rounds tokens through fp32->bf16 once more


def test_splice_into_embedding_buffer(eng256, dev):
    """Row f2: projected tokens written straight into a [B, L, H] LLM embedding buffer at the <image> position."""
    x = fx.synthetic_images(3, 256, seed=13).to(dev)          # max_batch = 2 -> two passes, strided destination
    _, proj = eng256.forward(x, False, True)
    L, pos = 16 + 9, 4
    emb = torch.full((3, L, 896), 7.0, dtype=torch.bfloat16, device=dev)
    out = eng256.forward_into(x, emb, pos)
    assert out.data_ptr() == emb.data_ptr()
    assert torch.equal(emb[:, pos:pos + 16], proj)                                  # same bits as the dense call
    assert (emb[:, :pos] == 7).all() and (emb[:, pos + 16:] == 7).all()             # text positions untouched
    with pytest.raises(pkg.FvhdError):
        eng256.forward_into(x, emb, L - 3)                                          # does not fit


# ------------------------------------------------------------------ bench-size properties (R=1024)
def test_batch_independence_and_determinism_1024(packed, dev):
    eng = pkg.Engine(1024, 896, 2, 2).load(packed, dev)
    x = fx.synthetic_images(2, 1024, seed=5).to(dev)
    t, p = eng.forward(x, True, True)
    t2, p2 = eng.forward(x, True, True)
    assert torch.equal(t, t2) and torch.equal(p, p2)                          # deterministic (no atomics on the path)
    ts, ps = eng.forward(x.flip(0), True, True)
    assert torch.equal(ts.flip(0), t) and torch.equal(ps.flip(0), p)          # image i's tokens do not depend on its batch slot
    assert torch.isfinite(p.float()).all()
