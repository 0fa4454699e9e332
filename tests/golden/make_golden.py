"""Regenerates tests/golden/*.  Needs the reference source tree (``SPCONV_REFERENCE_ROOT``, see
oracle/make_ref.py); the tests themselves only read the files written here.

* ``reference_cpu.json``  -- what the reference's own CPU code (oracle/_ref) returns on every input of
  tests/test_oracle_ref.py and tests/test_pointops_gpu.py: rulebooks, gather / scatter-add, max-pool
  forward / backward / global rearrange, voxel generator.  Arrays are SHA-256 digests
  (``tests.util.digest``); per-offset pair counts are stored as numbers.
* ``fixture_coords.npz``  -- voxel coordinates of the reference's own LiDAR fixture
  (test/data/test_spconv.pkl: 125 562 voxels, shape [80, 1600, 1600]); data, not source.
* ``fixture_facts.json``  -- rulebook facts of that fixture computed with an implementation that
  shares nothing with oracle/ (sorted linear keys + np.searchsorted): per-offset SubM pair counts,
  pair / output counts of SparseConv3d(k3, s2, p1).  BASELINE.md section 2 quotes the same totals.
"""
import json
import os
import pickle
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def linear(c, shape):
    k = c[:, 0].astype(np.int64)
    for a, d in enumerate(shape):
        k = k * d + c[:, a + 1]
    return k


def reference_records():
    """Runs the reference's own CPU code (oracle/_ref) on the inputs of the reference-parity tests."""
    from oracle import oracle as orc
    from tests import test_oracle_ref as t
    from tests import test_pointops_gpu as tp
    from tests.util import digest
    assert orc.have_ref(), "oracle/_ref is not built: the reference source tree is needed"
    rec = {"rulebook": {}}
    rb = rec["rulebook"]

    def ref_rulebook(key, inds, *args):
        rb[key] = t.rulebook_record(inds, t.rulebook(orc, inds, *args, impl="ref"))

    for case in t.CASES:
        shape, pts, ksize, stride, padding, dilation, subm, transpose = case
        for seed in t.SEEDS:
            ref_rulebook(f"{t.case_id(case)}/{seed}", t.rulebook_case_input(case, seed), len(pts), shape, ksize,
                         stride, padding, dilation, subm, transpose)
    inds = t.duplicates_input()
    ref_rulebook("duplicates/subm", inds, 1, [16] * 3, [3] * 3, [1] * 3, [1] * 3, [1] * 3, True, False)
    ref_rulebook("duplicates/conv", inds, 1, [16] * 3, [3] * 3, [2] * 3, [1] * 3, [1] * 3, False, False)
    inds, shape = t.lidar_fixture_input()
    ref_rulebook("lidar/subm", inds, 1, shape, [3] * 3, [1] * 3, [1] * 3, [1] * 3, True, False)
    ref_rulebook("lidar/conv", inds, 1, shape, [3] * 3, [2] * 3, [1] * 3, [1] * 3, False, False)
    inds = t.kitti_surface_input()
    ref_rulebook("kitti_surface/subm", inds, 2, [41, 1600, 1408], [3] * 3, [1] * 3, [1] * 3, [1] * 3, True, False)
    ref_rulebook("kitti_surface/conv", inds, 2, [41, 1600, 1408], [3] * 3, [2] * 3, [1] * 3, [1] * 3, False, False)

    src, inds, dst = t.gather_input()
    r = orc.ref_lib()
    buf = np.empty((3000, 24), np.float32)
    rec_g = {"inputs": [digest(src), digest(inds), digest(dst)]}
    r.ref_gather_f32(orc._ptr(buf), orc._ptr(src), orc._ptr(inds), 3000, 24, 5000)
    r.ref_scatter_add_f32(orc._ptr(dst), orc._ptr(buf), orc._ptr(inds), 3000, 24, 5000)
    rec_g.update(gather=digest(buf), scatter_add=digest(dst))
    rec["gather_scatter"] = rec_g

    _, inds = t.random_cloud(np.random.default_rng(0), [8, 8, 8], [50], 1)
    try:
        orc.get_indice_pairs(inds, 1, [8] * 3, [2] * 3, [1] * 3, [0] * 3, [1] * 3, [0] * 3, True, impl="ref")
    except RuntimeError as e:
        rec["subm_even_ksize_error"] = str(e)
    assert "subm_even_ksize_error" in rec, "the reference accepted an even SubM kernel size"

    rng, feats, inds = t.pooling_input()
    ref_rulebook("pooling", inds, 2, [18, 20, 22], [3] * 3, [2] * 3, [1] * 3, [1] * 3, False, False)
    o, pairs, num = t.rulebook(orc, inds, 2, [18, 20, 22], [3] * 3, [2] * 3, [1] * 3, [1] * 3, False, False,
                               impl="ref")
    fwd = orc.indice_maxpool(feats, pairs, num, o.shape[0])                      # the reference's loop
    tabs = orc.implicit_gemm_tables(pairs, num, inds.shape[0], o.shape[0], False)
    dense = orc.maxpool_implicit_gemm(feats, tabs["pair_fwd"], -3e38)
    g = rng.standard_normal(fwd.shape).astype(np.float32)
    bwd = orc.indice_maxpool_backward(feats, dense, g, pairs, num)               # the reference's loop
    oi, cnt = orc.global_pool_rearrange(inds, 2)
    rec["pooling"] = {"forward": digest(fwd), "grad_inputs": digest(g), "backward": digest(bwd),
                      "rearrange": digest(oi), "rearrange_counts": digest(cnt)}

    pts = t.point2voxel_input()
    p2v = {"inputs": digest(pts)}
    for max_voxels, max_points in t.P2V_LIMITS:
        p2v[f"{max_voxels}x{max_points}"] = [digest(a) for a in orc.point2voxel_ref(pts, t.P2V_VS, t.P2V_CR,
                                                                                      max_voxels, max_points)]
    _, grid, stride, _ = orc.point2voxel_meta(t.P2V_VS, t.P2V_CR)
    p2v["meta"] = {"grid": grid.tolist(), "stride": stride.tolist()}
    rec["point2voxel"] = p2v
    rec["point2voxel_gpu_cases"] = {}
    for n, max_voxels, max_points in tp.P2V_CASES:
        pts = tp._points(n, n)
        out = orc.point2voxel_ref(pts, tp.VS, tp.CR, max_voxels, max_points)
        rec["point2voxel_gpu_cases"][f"{n}/{max_voxels}x{max_points}"] = {
            "inputs": digest(pts), "outputs": [digest(a) for a in out]}
    return rec


def main():
    from oracle import make_ref
    rec = reference_records()
    with open(os.path.join(HERE, "reference_cpu.json"), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    voxels, coors, shape = pickle.load(open(os.path.join(make_ref.REF_ROOT, "test", "data", "test_spconv.pkl"), "rb"))
    coors = np.ascontiguousarray(coors.astype(np.int32))
    np.savez_compressed(os.path.join(HERE, "fixture_coords.npz"), coors=coors,
                        shape=np.array(shape, np.int32))
    keys = linear(coors, shape)
    order = np.argsort(keys)
    skeys = keys[order]
    counts = []
    for kz in range(3):
        for ky in range(3):
            for kx in range(3):
                nb = coors.astype(np.int64).copy()
                nb[:, 1] += 1 - kz
                nb[:, 2] += 1 - ky
                nb[:, 3] += 1 - kx
                ok = np.all((nb[:, 1:] >= 0) & (nb[:, 1:] < np.array(shape)), axis=1)
                nk = linear(nb[ok], shape)
                pos = np.searchsorted(skeys, nk)
                pos[pos >= len(skeys)] = 0
                counts.append(int((skeys[pos] == nk).sum()))
    # strided conv k3 s2 p1
    oshape = [(s + 2 - 2 - 1) // 2 + 1 for s in shape]
    pairs = 0
    outs = set()
    for kz in range(3):
        for ky in range(3):
            for kx in range(3):
                h = coors[:, 1:].astype(np.int64) + 1 - np.array([kz, ky, kx])
                ok = np.all((h % 2 == 0) & (h >= 0) & (h // 2 < np.array(oshape)), axis=1)
                o = h[ok] // 2
                pairs += int(ok.sum())
                ok_keys = (o[:, 0] * oshape[1] + o[:, 1]) * oshape[2] + o[:, 2]
                outs.update(np.unique(ok_keys).tolist())
    facts = {"num_voxels": int(coors.shape[0]), "shape": [int(s) for s in shape],
             "subm_k3_pairs_per_offset": counts, "subm_k3_pairs_total": int(sum(counts)),
             "conv_k3s2p1_pairs": pairs, "conv_k3s2p1_outputs": len(outs),
             "conv_k3s2p1_out_shape": oshape}
    json.dump(facts, open(os.path.join(HERE, "fixture_facts.json"), "w"), indent=1)
    print(facts["subm_k3_pairs_total"], pairs, len(outs))


if __name__ == "__main__":
    main()
