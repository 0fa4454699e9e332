"""CPU tests that PIN the oracle (run everywhere, no GPU):

1. against a pure-Python transliteration of the reference CPU loops on small inputs
   (spconv/csrc/sparse/indices.py:1640-1778) -- catches C-port bugs, pins pair ORDER;
2. against torch dense conv3d outputs/gradients on a seeded case (tests.util.dense_conv_case; the
   reference's own correctness criterion, test/test_conv.py:247-357) and against the committed,
   independently computed facts of the reference LiDAR fixture (BASELINE.md section 2).
"""
import json
import os

import numpy as np
import pytest

from tests.util import dense_conv_case

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _py_subm(indices, dims, ksize, dilation):
    n, nd = indices.shape[0], len(dims)
    kv = int(np.prod(ksize))
    pad = [(k // 2) * d for k, d in zip(ksize, dilation)]
    table = {}
    for i, c in enumerate(indices):
        table.setdefault(tuple(c), i)           # unordered_map::insert: first wins
    pairs = np.full((2, kv, n), -1, np.int32)
    num = np.zeros(kv, np.int32)
    for k in range(kv // 2 + 1):
        r, kk = [0] * nd, k
        for a in range(nd - 1, -1, -1):
            r[a] = kk % ksize[a]
            kk //= ksize[a]
        if k == kv // 2:
            pairs[0, k, :] = np.arange(n)
            pairs[1, k, :] = np.arange(n)
            continue
        for i, c in enumerate(indices):
            o = [c[0]] + [c[a + 1] + pad[a] - r[a] * dilation[a] for a in range(nd)]
            if any(o[a + 1] < 0 or o[a + 1] >= dims[a] for a in range(nd)):
                continue
            j = table.get(tuple(o))
            if j is None:
                continue
            q = num[k]
            num[k] += 1
            pairs[0, k, q], pairs[1, k, q] = i, j
            pairs[0, kv - 1 - k, q], pairs[1, kv - 1 - k, q] = j, i
    return pairs, num


def _py_conv(indices, out_dims, ksize, stride, padding, dilation, transposed=False):
    n, nd = indices.shape[0], len(out_dims)
    kv = int(np.prod(ksize))
    table, outs = {}, []
    pairs = np.full((2, kv, n), -1, np.int32)
    num = np.zeros(kv, np.int32)
    for k in range(kv):
        r, kk = [0] * nd, k
        for a in range(nd - 1, -1, -1):
            r[a] = kk % ksize[a]
            kk //= ksize[a]
        for i, c in enumerate(indices):
            o, ok = [int(c[0])], True
            for a in range(nd):
                if transposed:
                    v = int(c[a + 1]) * stride[a] - padding[a] + r[a] * dilation[a]
                else:
                    h = int(c[a + 1]) + padding[a] - r[a] * dilation[a]
                    v = int(h / stride[a])                    # C truncation
                    ok = ok and (h - v * stride[a] == 0)
                ok = ok and 0 <= v < out_dims[a]
                o.append(v)
            if not ok:
                continue
            key = tuple(o)
            if key not in table:
                table[key] = len(outs)
                outs.append(o)
            q = num[k]
            num[k] += 1
            pairs[0, k, q], pairs[1, k, q] = i, table[key]
    return np.array(outs, np.int32).reshape(-1, nd + 1), pairs, num


@pytest.mark.parametrize("nd", [2, 3])
def test_subm_matches_python_transliteration(oracle, nd):
    rng = np.random.default_rng(3)
    dims = [9, 8, 7][:nd]
    _, inds = oracle.generate_sparse_data(dims, [60, 50], 1, rng)
    for ksize, dil in (([3] * nd, [1] * nd), ([3] * nd, [2] * nd), ([5] + [3] * (nd - 1), [1] * nd)):
        out, pairs, num = oracle.get_indice_pairs(inds, 2, dims, ksize, [1] * nd, [0] * nd, dil,
                                                  [0] * nd, True)
        rp, rn = _py_subm(inds, dims, ksize, dil)
        assert np.array_equal(num, rn)
        assert np.array_equal(pairs, rp)
        assert out is not None and np.array_equal(out, inds)


@pytest.mark.parametrize("cfg", [([3] * 3, [2] * 3, [1] * 3, [1] * 3, False),
                                 ([2] * 3, [2] * 3, [0] * 3, [1] * 3, False),
                                 ([3] * 3, [1] * 3, [0] * 3, [2] * 3, False),
                                 ([3] * 3, [3] * 3, [2] * 3, [1] * 3, False),
                                 ([3] * 3, [2] * 3, [1] * 3, [1] * 3, True)])
def test_conv_matches_python_transliteration(oracle, cfg):
    ksize, stride, padding, dilation, transposed = cfg
    rng = np.random.default_rng(4)
    dims = [9, 8, 7]
    _, inds = oracle.generate_sparse_data(dims, [80], 1, rng)
    out, pairs, num = oracle.get_indice_pairs(inds, 1, dims, ksize, stride, padding, dilation,
                                              [0] * 3, False, transposed)
    if transposed:
        odims = oracle.get_deconv_output_size(dims, ksize, stride, padding, dilation, [0] * 3)
    else:
        odims = oracle.get_conv_output_size(dims, ksize, stride, padding, dilation)
    ro, rp, rn = _py_conv(inds, odims, ksize, stride, padding, dilation, transposed)
    assert np.array_equal(out, ro)
    assert np.array_equal(num, rn)
    assert np.array_equal(pairs, rp)


def test_duplicate_coordinates_first_wins(oracle):
    inds = np.array([[0, 1, 1, 1], [0, 1, 1, 2], [0, 1, 1, 1], [0, 1, 1, 3]], np.int32)
    _, pairs, num = oracle.get_indice_pairs(inds, 1, [4, 4, 4], [3] * 3, [1] * 3, [1] * 3, [1] * 3,
                                            [0] * 3, True)
    rp, rn = _py_subm(inds, [4, 4, 4], [3] * 3, [1] * 3)
    assert np.array_equal(pairs, rp) and np.array_equal(num, rn)


def test_fixture_facts(oracle):
    """Reference LiDAR fixture: pair counts equal an independent numpy computation."""
    facts = json.load(open(os.path.join(GOLD, "fixture_facts.json")))
    data = np.load(os.path.join(GOLD, "fixture_coords.npz"))
    coors, shape = data["coors"], [int(s) for s in data["shape"]]
    assert coors.shape[0] == facts["num_voxels"] == 125562
    _, pairs, num = oracle.get_indice_pairs(coors, 1, shape, [3] * 3, [1] * 3, [1] * 3, [1] * 3,
                                            [0] * 3, True)
    per_offset = facts["subm_k3_pairs_per_offset"]
    kv = 27
    for k in range(kv // 2):
        assert num[k] == per_offset[k] == per_offset[kv - 1 - k]
    assert per_offset[kv // 2] == coors.shape[0]
    assert 2 * int(num.sum()) + coors.shape[0] == facts["subm_k3_pairs_total"] == 788888
    out, pairs, num = oracle.get_indice_pairs(coors, 1, shape, [3] * 3, [2] * 3, [1] * 3, [1] * 3,
                                              [0] * 3, False)
    assert int(num.sum()) == facts["conv_k3s2p1_pairs"] == 422946
    assert out.shape[0] == facts["conv_k3s2p1_outputs"] == 136998


@pytest.mark.parametrize("tag,k,s,p,d", [("k3s2p1d1", 3, 2, 1, 1), ("k3s1p1d1", 3, 1, 1, 1),
                                         ("k2s2p0d1", 2, 2, 0, 1)])
def test_dense_conv_golden(oracle, tag, k, s, p, d):
    """SparseConv3d(...).dense() == nn.Conv3d on the densified input, forward and both gradients
    (test/test_conv.py:323-357, atol 1e-4 on O(1) values)."""
    g = dense_conv_case()
    inds, feats, shape = g["inds"], g["feats"], [int(v) for v in g["shape"]]
    w, y, dy, dw, dx = (g[f"{tag}_{n}"] for n in ("w", "y", "dy", "dw", "dx"))
    out_inds, pairs, num = oracle.get_indice_pairs(inds, 2, shape, [k] * 3, [s] * 3, [p] * 3,
                                                   [d] * 3, [0] * 3, False)
    out = oracle.indice_conv(feats, w, pairs, num, out_inds.shape[0], False, False)
    oshape = oracle.get_conv_output_size(shape, [k] * 3, [s] * 3, [p] * 3, [d] * 3)
    got = oracle.dense_from_sparse(out, out_inds, oshape, 2)
    assert np.abs(got - y).max() < 1e-4
    dout = dy[out_inds[:, 0], :, out_inds[:, 1], out_inds[:, 2], out_inds[:, 3]]
    din, dwe = oracle.indice_conv_backward(feats, w, dout, pairs, num, False, False)
    # expected gradients: torch dense conv3d backward with dy masked to the active outputs
    assert np.abs(dwe - dw).max() < 1e-3
    assert np.abs(din - dx).max() < 1e-4
    # every non-active output cell of the dense conv is exactly zero
    active = np.zeros_like(y)
    active[out_inds[:, 0], :, out_inds[:, 1], out_inds[:, 2], out_inds[:, 3]] = 1
    assert np.abs(y * (1 - active)).max() == 0.0


def test_subm_dense_equivalence(oracle):
    """SubM == dense conv restricted to the input's active set (any seed, computed live)."""
    import torch
    rng = np.random.default_rng(11)
    shape = [12, 11, 10]
    feats, inds = oracle.generate_sparse_data(shape, [400, 300], 8, rng)
    w = rng.uniform(-1, 1, size=(12, 3, 3, 3, 8)).astype(np.float32)
    for dil in (1, 2):
        _, pairs, num = oracle.get_indice_pairs(inds, 2, shape, [3] * 3, [1] * 3, [0] * 3, [dil] * 3,
                                                [0] * 3, True)
        out = oracle.indice_conv(feats, w, pairs, num, inds.shape[0], False, True)
        dense = torch.from_numpy(oracle.dense_from_sparse(feats, inds, shape, 2))
        ref = torch.nn.functional.conv3d(dense, torch.from_numpy(w).permute(0, 4, 1, 2, 3).contiguous(),
                                         padding=dil, dilation=dil).numpy()
        ref_rows = ref[inds[:, 0], :, inds[:, 1], inds[:, 2], inds[:, 3]]
        assert np.abs(out - ref_rows).max() < 1e-4


def test_implicit_gemm_tables_consistency(oracle):
    rng = np.random.default_rng(5)
    shape = [10, 10, 10]
    _, inds = oracle.generate_sparse_data(shape, [300], 1, rng)
    out, pairs, num = oracle.get_indice_pairs(inds, 1, shape, [3] * 3, [2] * 3, [1] * 3, [1] * 3,
                                              [0] * 3, False)
    t = oracle.implicit_gemm_tables(pairs, num, inds.shape[0], out.shape[0], False)
    kv = 27
    for k in range(kv):
        n = num[k]
        assert np.array_equal(t["pair_fwd"][k][pairs[1, k, :n]], pairs[0, k, :n])
        assert np.array_equal(t["pair_bwd"][k][pairs[0, k, :n]], pairs[1, k, :n])
        assert (t["pair_fwd"][k] >= 0).sum() == n
    assert np.all(np.diff(t["mask_fwd"][:, 0].astype(np.int64)) >= 0)
    assert np.array_equal(t["mask_fwd"], t["mask_fwd_unsorted"][t["argsort_fwd"]])


def test_int8_formula(oracle):
    """clip(round(acc*scale + bias + add*add_scale)) with round-half-even (test_all_algo.py:272-287)."""
    rng = np.random.default_rng(6)
    shape = [8, 8, 8]
    _, inds = oracle.generate_sparse_data(shape, [200], 1, rng)
    x = rng.integers(-3, 3, size=(200, 32)).astype(np.int8)
    w = rng.integers(-3, 3, size=(32, 3, 3, 3, 32)).astype(np.int8)
    _, pairs, num = oracle.get_indice_pairs(inds, 1, shape, [3] * 3, [1] * 3, [1] * 3, [1] * 3, [0] * 3, True)
    scales = np.full(32, 0.5, np.float32)
    bias = np.zeros(32, np.float32)
    q = oracle.int8_conv_forward(x, w, pairs, num, 200, True, scales, bias)
    acc = oracle.indice_conv(x.astype(np.float32), w.astype(np.float32), pairs, num, 200, False, True)
    assert np.array_equal(q, np.clip(np.round(acc * 0.5), -128, 127).astype(np.int8))
    assert (np.abs(acc * 0.5 % 1 - 0.5) < 1e-6).any()      # ties are exercised
