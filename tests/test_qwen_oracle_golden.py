"""Pin oracle/qwen_oracle.py to the goldens that tests/golden/make_golden_qwen.py produced by executing the REFERENCE's
Qwen2-VL FlashMemory (CPU-only tests; /root/reference is not needed here)."""
from __future__ import annotations

import os

import numpy as np
import pytest
import torch

from oracle import qwen_oracle as QO
from tests import qwen_inputs as QI

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# relative tolerance of one rounding in the output dtype (the oracle's fp32 summation order differs from ATen's)
RTOL = {"bf16": 2.0 ** -7, "f16": 2.0 ** -10, "f32": 2e-5}


def _load(name):
    return np.load(os.path.join(G, name))


def _members(g, name):
    cnt, flat = g[name + "_members"], g[name + "_members_flat"]
    out, p = [], 0
    for c in cnt:
        out.append(flat[p:p + c].tolist())
        p += c
    return out


def assert_close_dtype(got: torch.Tensor, want: torch.Tensor, dt: str, frac_1ulp=0.02):
    g, w = got.float().numpy(), want.float().numpy()
    assert g.shape == w.shape
    scale = np.maximum(np.abs(w), np.abs(w).max() * 1e-3)
    err = np.abs(g - w) / scale
    assert err.max() <= 2.5 * RTOL[dt], f"max rel err {err.max():.3e}"
    if dt != "f32":   # almost all elements must be bit-identical after the final rounding
        assert (g != w).mean() <= frac_1ulp, f"{(g != w).mean():.4f} of elements differ by one rounding step"


@pytest.mark.parametrize("case", QI.POOL_CASES, ids=[c[0] for c in QI.POOL_CASES])
def test_temporal_pool_matches_reference(case):
    name, t, h, w, dt, seed = case
    g = _load("qwen_pool.npz")
    x = QI.pool_input(t, h, w, dt, seed)
    assert (QI.checksum(x) == g[name + "_chk"]).all(), "seeded input drifted"
    y, thw = QO.temporal_pool(x, [t, h, w])
    assert list(thw) == g[name + "_thw"].tolist()
    assert np.array_equal(QI.to_bits(y), g[name + "_y"])          # bit-exact: 4-term fp32 sums are exact


def test_temporal_pool_odd_half_grid_raises():
    with pytest.raises(NotImplementedError):
        QO.temporal_pool(torch.zeros(1 * 6 * 4, 1176, dtype=torch.bfloat16), [1, 6, 4])


@pytest.mark.parametrize("name", list(QI.KMEANS_CASES))
def test_kmeans_ordered_matches_reference(name):
    c = QI.KMEANS_CASES[name]
    g = _load("qwen_kmeans.npz")
    x, w = QI.kmeans_input(c)
    assert (QI.checksum(x) == g[name + "_chk"]).all(), "seeded input drifted"
    feat, weights, ts, idx = QO.weighted_kmeans_ordered_feature(x, c["K"], w, init_idx=g[name + "_init"],
                                                                refill_idx=g[name + "_refill"])
    assert idx == _members(g, name)
    assert np.array_equal(ts.numpy(), g[name + "_ts"])
    np.testing.assert_allclose(weights.numpy(), g[name + "_weights"], rtol=1e-5)
    assert feat.dtype == QI.DT[c["dtype"]]
    assert_close_dtype(feat, QI.from_bits(g[name + "_feat"], feat.dtype), c["dtype"])


def test_kmeans_ordered_pass_through():
    x = torch.randn(4, 2, 512).bfloat16()
    out = QO.weighted_kmeans_ordered_feature(x, 6)
    assert len(out) == 3 and out[0].dtype == torch.float32 and out[2] == [[[0], [1], [2], [3]]]


def test_unique_rows_order_matches_torch_unique():
    g = torch.Generator().manual_seed(5)
    base = torch.randn(5, 64, generator=g)
    X = base[torch.randint(0, 5, (17,), generator=g)]
    order = QO.unique_rows_order(X.numpy())
    assert torch.equal(X[torch.from_numpy(order).long()], torch.unique(X, dim=0))


@pytest.mark.parametrize("name", list(QI.MEMORY_CASES))
def test_flash_memory_forward_matches_reference(name):
    c = QI.MEMORY_CASES[name]
    g = _load("qwen_memory.npz")
    x, small, thw, small_thw, pos, vis = QI.memory_input(c)
    assert (QI.checksum(x) == g[name + "_chk"]).all(), "seeded input drifted"
    fm = QO.FlashMemoryOracle(c["temporal_length"], c["spatial_length"])
    order = g[name + "_sort1"] if int(g[name + "_n_sorts"][0]) >= 2 else None
    new_x, new_pos, aux = fm.forward_one(x, thw[0], small, small_thw[0], pos[:, 0], vis[0], init_idx=g[name + "_init"],
                                         refill_idx=g[name + "_refill"], order=order)
    assert np.array_equal(aux["spa_positions"].numpy(), g[name + "_spa_pos"])
    assert np.array_equal(aux["tem_timestamps"].numpy(), g[name + "_tem_ts"])
    np.testing.assert_allclose(aux["tem_weights"].numpy(), g[name + "_tem_w"], rtol=1e-5)
    assert np.array_equal(new_pos.numpy(), g[name + "_new_pos"][:, 0])
    assert_close_dtype(new_x, QI.from_bits(g[name + "_new_x"], new_x.dtype), c["dtype"])


@pytest.mark.parametrize("name", list(QI.COS_CASES))
def test_klarge_retrieve_cos_matches_reference(name):
    """§8f-4 spatial_method='klarge_retrieve_cos' (vstream_qwen2vl_model.py:208-215): the oracle selects the frames the
    reference's spatial_enhance selected (goldens of tests/golden/make_golden_qwen_cos.py) and its similarities sit within
    one rounding of the reference expression's (the fp32 accumulation order of the CPU GEMM / norm differs)."""
    c = QI.COS_CASES[name]
    g = _load("qwen_klarge_cos.npz")
    x, small, thw, small_thw, pos, vis = QI.memory_input(c)
    assert (QI.checksum(x) == g[name + "_chk"]).all(), "seeded input drifted"
    dt = QI.DT[c["dtype"]]
    fm = QO.FlashMemoryOracle(c["temporal_length"], c["spatial_length"], flash_memory_spatial_method="klarge_retrieve_cos")
    tem_x = QI.from_bits(g[name + "_tem_x"], dt)
    tem_thw = [int(v) for v in g[name + "_tem_thw"]]
    order = g[name + "_sort1"]
    spa_x, spa_thw, spa_pos = fm.spatial_enhance(x, small, thw[0], tem_x, tem_thw, torch.from_numpy(g[name + "_tem_w"]), None,
                                                 order=order)
    assert np.array_equal(spa_pos.numpy(), g[name + "_spa_pos"])
    assert torch.equal(spa_x.reshape(-1, x.shape[-1]), QI.from_bits(g[name + "_spa_x"], dt).reshape(-1, x.shape[-1]))
    cent = tem_x.reshape(tem_thw[0], -1)[torch.from_numpy(order[: fm.spatial_length].copy())]
    sim = QO.klarge_cosine(cent, small.reshape(c["t"], -1))
    # similarities are O(0.01..1): one rounding step of the 16-bit dtype at |sim| <= 1, plus one for the norm rounding
    np.testing.assert_allclose(sim, g[name + "_sim"], rtol=0, atol=2.0 * RTOL[c["dtype"]])


def test_klarge_cosine_zero_row_is_nan_and_wins():
    g = torch.Generator().manual_seed(3)
    bank = torch.randn(6, 2048, generator=g).bfloat16()
    bank[4] = 0
    sim = QO.klarge_cosine(bank[[1, 2]], bank)
    assert np.isnan(sim[:, 4]).all() and not np.isnan(np.delete(sim, 4, axis=1)).any()
    assert QO.argmin_first_nan(sim, axis=1).tolist() == [4, 4]          # torch.argmin returns the NaN
    assert torch.argmin(torch.from_numpy(sim), dim=1).tolist() == [4, 4]


def test_reference_fast_variant_is_the_same_arithmetic():
    """§8f-4: `fast_weighted_kmeans_ordered_feature` (compress_functions.py:301) — executed by tests/golden/make_golden_seams.py
    from the reference, same seeds — returns exactly what `weighted_kmeans_ordered_feature` (:181) returns, which is why the
    mirror serves both from the same kernels (flash_vstream_b200/qwen/compress_functions.py); the oracle reproduces it from
    the draws the fast variant consumed."""
    g = _load("seams.npz")
    c = QI.KMEANS_CASES["ko_scene_bf16"]
    x, w = QI.kmeans_input(c)
    assert (QI.checksum(x) == g["fast_chk"]).all(), "seeded input drifted"
    for k in ("feat", "weights", "ts", "members", "members_flat", "init", "refill"):
        assert np.array_equal(g["slow_" + k], g["fast_" + k]), k
    feat, weights, ts, idx = QO.weighted_kmeans_ordered_feature(x, c["K"], w, init_idx=g["fast_init"],
                                                                refill_idx=g["fast_refill"])
    assert idx == _members(g, "fast")
    assert np.array_equal(ts.numpy(), g["fast_ts"])
    np.testing.assert_allclose(weights.numpy(), g["fast_weights"], rtol=1e-5)
    assert_close_dtype(feat, QI.from_bits(g["fast_feat"], feat.dtype), c["dtype"])
