"""CPU tests: pin oracle/fastvithd_oracle.py to the outputs of the unmodified reference
(tests/golden/*, produced by oracle/gen_golden.py) and check the fixture itself."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import fastvithd_oracle as orc
from oracle import fixture as fx
from oracle.gen_golden import N_SAMPLES_1024, sample_indices

# fp32 CPU vs fp32 CPU of the same ATen ops; oneDNN may pick other kernels on another host.
RTOL = 2e-4


def rel_l2(a, b):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def test_fixture_keys_match_reference(tower_sd, proj_sd, golden_dir):
    keys = json.load(open(os.path.join(golden_dir, "keys.json")))
    assert [k for k, _, _ in keys["tower"]] == list(tower_sd.keys())
    for k, shape, dtype in keys["tower"]:
        assert list(tower_sd[k].shape) == shape and str(tower_sd[k].dtype) == dtype, k
    assert [k for k, _, _ in keys["projector"]] == list(proj_sd.keys())
    for k, shape, dtype in keys["projector"]:
        assert list(proj_sd[k].shape) == shape, k
    assert len(tower_sd) == 629
    n_on_path = sum(v.numel() for k, v in tower_sd.items() if "head.proj" not in k and "num_batches" not in k)
    assert abs(n_on_path / 1e6 - 122.7) < 0.5  # 125.07 M total - 2.36 M head.proj (SURVEY 2.2)


@pytest.fixture(scope="module")
def run256(tower_sd, proj_sd):
    col = {}
    out = orc.encode_images(fx.synthetic_images(1, 256), tower_sd, proj_sd, col)
    return out, col


def test_tokens_and_projection_match_reference_256(run256, golden_dir):
    out, col = run256
    g = np.load(os.path.join(golden_dir, "ref_256.npz"))
    assert tuple(col["tokens"].shape) == (1, 16, 3072)          # (R/64)^2 tokens x 3072
    assert rel_l2(col["tokens"], g["tokens"]) < RTOL
    assert tuple(out.shape) == (1, 16, 896)
    assert rel_l2(out, g["projected"]) < RTOL


def test_every_unit_matches_reference_256(run256, golden_dir):
    _, col = run256
    g = np.load(os.path.join(golden_dir, "ref_256.npz"))
    names = sorted({k.split("/")[1] for k in g.files if k.startswith("unit/")})
    assert len(names) == 2 + 11 + sum(fx.LAYERS)
    for n in names:
        t = col[n]
        assert list(t.shape) == list(g[f"unit/{n}/shape"]), n
        flat = t.reshape(-1)
        idx = sample_indices(flat.numel(), n)
        got = flat[torch.from_numpy(idx)].numpy()
        ref = g[f"unit/{n}/samples"]
        scale = g[f"unit/{n}/stats"][2]
        assert np.abs(got - ref).max() <= RTOL * scale, n
        assert abs(flat.std().item() - g[f"unit/{n}/stats"][1]) <= RTOL * scale, n


def test_batch2_tensor_and_list_branches(tower_sd, golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_b2_256.npz"))
    x2 = fx.synthetic_images(2, 256, seed=7)
    t = orc.tower_forward(x2, tower_sd)
    assert rel_l2(t, g["tokens"]) < RTOL
    # list input == per-image calls (mobileclip_encoder.py:78-83)
    assert rel_l2(t[0:1], g["list0"]) < RTOL and rel_l2(t[1:2], g["list1"]) < RTOL


def test_tokens_match_reference_1024(tower_sd, golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_1024_tokens_sample.npz"))
    t = orc.tower_forward(fx.synthetic_images(1, 1024), tower_sd)
    assert tuple(t.shape) == (1, 256, 3072) == tuple(g["shape"])   # app/FastVLM/FastVLM.swift:303
    flat = t.reshape(-1)
    got = flat[torch.from_numpy(sample_indices(flat.numel(), "tokens_1024", N_SAMPLES_1024))]
    assert rel_l2(got, g["samples"]) < RTOL
    mean, std, absmax = g["stats"]
    assert abs(flat.mean().item() - mean) <= RTOL * absmax and abs(flat.std().item() - std) <= RTOL * absmax
    assert abs(flat.abs().max().item() - absmax) <= RTOL * absmax


def test_fixture_is_not_blind(run256, tower_sd, golden_dir):
    """With the reference's default layer-scale/BN init ~98 % of the MACs are invisible
    (SURVEY finding 3); the fixture must not regress to that."""
    _, col = run256
    sd0 = fx.default_init_like_reference(tower_sd)
    t0 = orc.tower_forward(fx.synthetic_images(1, 256), sd0)
    change = rel_l2(t0, col["tokens"])
    assert change > 0.5
    ref = json.load(open(os.path.join(golden_dir, "sensitivity.json")))["rel_l2_default_vs_fixture"]
    assert abs(change - ref) < 1e-2


def test_shape_contracts():
    assert orc.num_tokens(256) == 16 and orc.num_tokens(1024) == 256 and orc.num_tokens(1536) == 576
    assert abs(orc.gmacs_per_image(1024) - 243.35) < 0.01       # SURVEY 8(a) probe value
    assert abs(orc.gmacs_per_image(256) - 14.81) < 0.01
    assert abs(orc.gmacs_per_image(1536) - 566.80) < 0.01
