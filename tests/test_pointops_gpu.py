"""Point cloud -> voxel front end (SURVEY 8 f2): the CUDA generator against the REFERENCE's CPU
generator (``Point2VoxelCPU::point_to_voxel_static``, ``spconv/csrc/sparse/pointops.py:589-695``)
-- bit-exact: voxel order, kept points, counts, per-point ids.  The comparison runs against the numpy
restatement, which must first reproduce the reference's recorded outputs (tests/golden/reference_cpu.json)."""
import json
import os

import numpy as np
import pytest
import torch

from tests.util import digest

pytestmark = pytest.mark.gpu

VS, CR = [0.4, 0.4, 0.5], [0, -40, -3, 70.4, 40, 1]          # a KITTI-like range, 8 x 200 x 176 grid
P2V_CASES = [(20000, 3000, 5), (20000, 50000, 5), (60000, 40000, 3), (500, 100, 8)]
GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_cpu.json")


def _points(seed, n):
    rng = np.random.default_rng(seed)
    return rng.uniform([-1, -41, -4, 0], [71, 41, 2, 1], size=(n, 4)).astype(np.float32)   # some out of range


@pytest.mark.parametrize("n,max_voxels,max_points", P2V_CASES)
def test_point_to_voxel_equals_reference_cpu(n, max_voxels, max_points, oracle, cuda_dev):
    from spconv_b200.pytorch.utils import PointToVoxel, gather_features_by_pc_voxel_id
    pts = _points(n, n)
    want = json.load(open(GOLD))["point2voxel_gpu_cases"][f"{n}/{max_voxels}x{max_points}"]
    assert digest(pts) == want["inputs"]
    gen = PointToVoxel(VS, CR, 4, max_voxels, max_points, cuda_dev)
    assert gen.grid_size == [8, 200, 176]
    vox, ind, num, ids = gen.generate_voxel_with_id(torch.from_numpy(pts).to(cuda_dev))
    r_vox, r_ind, r_num, r_ids = oracle.point2voxel(pts, VS, CR, max_voxels, max_points)
    assert [digest(a) for a in (r_vox, r_ind, r_num, r_ids)] == want["outputs"]   # restatement == reference
    assert vox.shape[0] == r_vox.shape[0]
    assert np.array_equal(ind.cpu().numpy(), r_ind)
    assert np.array_equal(num.cpu().numpy(), r_num)
    assert np.array_equal(ids.cpu().numpy(), r_ids)
    assert np.array_equal(vox.cpu().numpy(), r_vox)
    # second call on the same object: buffers are reused, result unchanged
    vox2, ind2, num2 = gen(torch.from_numpy(pts).to(cuda_dev))
    assert torch.equal(vox2, vox) and torch.equal(ind2, ind) and torch.equal(num2, num)
    # per-point gather of per-voxel results
    seg = torch.arange(vox.shape[0], device=cuda_dev, dtype=torch.float32).view(-1, 1) + 1
    back = gather_features_by_pc_voxel_id(seg, ids)
    want = np.where(r_ids >= 0, r_ids + 1, 0).astype(np.float32)
    assert np.array_equal(back.cpu().numpy()[:, 0], want)


def test_point_to_voxel_empty_mean_and_feeds_the_conv_path(oracle, cuda_dev):
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch.utils import PointToVoxel
    pts = _points(3, 30000)
    gen = PointToVoxel(VS, CR, 4, 20000, 4, cuda_dev)
    vox, ind, num = gen(torch.from_numpy(pts).to(cuda_dev), empty_mean=True)
    r_vox, r_ind, r_num, _ = oracle.point2voxel(pts, VS, CR, 20000, 4, empty_mean=True)
    assert np.array_equal(ind.cpu().numpy(), r_ind) and np.array_equal(num.cpu().numpy(), r_num)
    assert np.abs(vox.cpu().numpy() - r_vox).max() < 1e-5
    # voxel features (first point of every voxel) -> SparseConvTensor -> SubMConv3d
    feats = vox[:, 0, :]
    coords = torch.cat([torch.zeros((ind.shape[0], 1), dtype=torch.int32, device=cuda_dev), ind], 1)
    x = spconv.SparseConvTensor(feats.contiguous(), coords, gen.grid_size, 1)
    y = spconv.SubMConv3d(4, 16, 3, padding=1).to(cuda_dev)(x)
    assert y.features.shape == (ind.shape[0], 16) and torch.isfinite(y.features).all()
