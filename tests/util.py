"""Shared helpers for the parity tests (inputs are seeded numpy -> identical for CUDA and oracle)."""
import functools
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def random_cloud(rng, shape, num_per_batch, channels, dtype=np.float32):
    """Unique uniform-random coordinates per sample (spconv/test_utils.py:142-195 semantics)."""
    total = int(np.prod(shape))
    inds = []
    for b, n in enumerate(num_per_batch):
        flat = rng.permutation(total)[:n]
        coords = np.stack(np.unravel_index(flat, shape), axis=-1).astype(np.int32)
        inds.append(np.concatenate([np.full((n, 1), b, np.int32), coords], axis=1))
    indices = np.concatenate(inds, 0)
    feats = rng.uniform(-1, 1, size=(indices.shape[0], channels)).astype(dtype)
    return feats, indices


from bench_utils import surface_cloud  # noqa: E402,F401  (clustered LiDAR-like clouds)


@functools.lru_cache(maxsize=None)
def dense_conv_case() -> dict:
    """One seeded dense-equivalence case of the reference's test/test_conv.py:247-357 (its seeds, a small
    grid): inputs plus torch.nn.functional.conv3d outputs / input-grad / weight-grad per ``<tag>_*``."""
    import torch
    from oracle import oracle as orc
    rs = np.random.RandomState(484)
    shape, bs, npts, C, K = [19, 18, 17], 2, 1500, 16, 16
    total = int(np.prod(shape))
    inds = []
    for b in range(bs):
        flat = rs.permutation(total)[:npts]
        cc = np.stack(np.unravel_index(flat, shape), -1).astype(np.int32)
        inds.append(np.concatenate([np.full((npts, 1), b, np.int32), cc], 1))
    inds = np.concatenate(inds, 0)
    feats = rs.uniform(-1, 1, size=(inds.shape[0], C)).astype(np.float32)
    case = {"inds": inds, "feats": feats, "shape": np.array(shape)}
    for tag, (k, s, p, d) in {"k3s2p1d1": (3, 2, 1, 1), "k3s1p1d1": (3, 1, 1, 1),
                              "k2s2p0d1": (2, 2, 0, 1)}.items():
        w = rs.uniform(-1, 1, size=(K, k, k, k, C)).astype(np.float32)
        dense = torch.zeros((bs, C, *shape))
        dense[inds[:, 0], :, inds[:, 1], inds[:, 2], inds[:, 3]] = torch.from_numpy(feats)
        dense.requires_grad_(True)
        wt = torch.from_numpy(w).permute(0, 4, 1, 2, 3).contiguous().requires_grad_(True)
        y = torch.nn.functional.conv3d(dense, wt, stride=s, padding=p, dilation=d)
        dy = torch.from_numpy(rs.uniform(-0.2, 0.2, size=tuple(y.shape)).astype(np.float32))
        # the sparse op only defines gradients through its ACTIVE outputs: mask dy to them
        oi, _, _ = orc.get_indice_pairs(inds, bs, shape, [k] * 3, [s] * 3, [p] * 3, [d] * 3, [0] * 3, False)
        act = torch.zeros_like(y)
        act[oi[:, 0], :, oi[:, 1], oi[:, 2], oi[:, 3]] = 1
        y.backward(dy * act)
        case[f"{tag}_w"] = w
        case[f"{tag}_y"] = y.detach().numpy()
        case[f"{tag}_dy"] = dy.numpy()
        case[f"{tag}_dw"] = wt.grad.permute(0, 2, 3, 4, 1).contiguous().numpy()      # back to KRSC
        case[f"{tag}_dx"] = dense.grad[inds[:, 0], :, inds[:, 1], inds[:, 2], inds[:, 3]].numpy()
    return case


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and bytes: equal digests <=> bit-identical arrays.  The golden
    records of the reference's outputs (tests/golden/reference_cpu.json) are kept in this form."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def describe_mismatch(got, ref, name="", max_rows=5):
    """Human-readable summary of where two matrices differ (used in assertion messages so one
    GPU run tells as much as possible)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref)
    bad = err > (1e-2 + 1e-2 * np.abs(ref))
    rows = np.unique(np.nonzero(bad)[0])
    cols = np.unique(np.nonzero(bad)[1]) if bad.ndim > 1 else []
    msg = (f"{name}: shape {got.shape} max_abs_err {err.max():.4g} rel_l2 {rel_l2(got, ref):.4g} "
           f"bad {bad.sum()}/{bad.size} bad_rows {len(rows)} (first {rows[:max_rows].tolist()}) "
           f"bad_cols {len(cols)} (first {list(cols[:16])}) nan {np.isnan(got).sum()}")
    if len(rows):
        r = rows[0]
        msg += f"\n  row {r} got {np.round(got[r][:8], 3).tolist()} ref {np.round(ref[r][:8], 3).tolist()}"
    return msg
