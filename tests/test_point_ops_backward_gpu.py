"""SURVEY.md 8f rank 4: backward passes of the five differentiable point/voxel operators, through torch.autograd on the
library's Functions, against the reference's OWN backward kernels (vox.cu:86-110, trilinear_devox.cu:119-162,
grouping.cu:58-77, neighbor_interpolate.cu:145-170, sampling.cu:52-66) fed with the same saved indices, whose outputs on
these inputs are stored in tests/golden/ref_point_ops_backward.npz (tests/golden/make_golden_ref_kernels.py).
Gather-type gradients are bit-identical; scatter-adds (fp32 atomics on both sides) agree to 1e-6."""
import pytest
import torch

from tests.util import RefGolden, gen

pytestmark = pytest.mark.gpu
REF = RefGolden("ref_point_ops_backward")


def _F():
    from lion_b200.third_party.pvcnn import functional as F
    return F


def key(test, *params):
    return test + "/" + "_".join(str(p) for p in params)


# Inputs of every case; make_golden_ref_kernels.py runs the reference's backward kernels on exactly these.
AVG_VOXELIZE_CASES = [(2, 16, 2048, 32), (3, 7, 300, 8), (32, 64, 2048, 32)]
DEVOX_CASES = [(2, 32, 2048, 32), (2, 5, 100, 4), (32, 64, 1024, 16)]
GROUPING_CASES = [(2, 35, 2048, 1024, 32), (3, 9, 64, 16, 32)]
THREE_NN_CASES = [(2, 192, 256, 64), (2, 17, 2048, 1024)]


def avg_voxelize_inputs(B, C, N, r):
    feats = gen(1, B, C, N)
    vox = torch.randint(0, r, (B, 3, N), generator=torch.Generator().manual_seed(2), dtype=torch.int32)
    vox[0, :, : N // 2] = 1                                   # many points in one voxel
    return feats, vox, gen(3, B, C, r, r, r)


def devox_inputs(B, C, N, r):
    coords = torch.rand(B, 3, N, generator=torch.Generator().manual_seed(5)) * (r - 1)
    return gen(4, B, C, r, r, r), coords, gen(6, B, C, N)


def grouping_inputs(B, C, N, M, U):
    idx = torch.randint(0, N, (B, M, U), generator=torch.Generator().manual_seed(8), dtype=torch.int32)
    idx1 = torch.randint(0, N, (B, M), generator=torch.Generator().manual_seed(11), dtype=torch.int32)
    return gen(7, B, C, N), idx, gen(9, B, C, M, U), gen(10, B, C, N), idx1, gen(12, B, C, M)


def three_nn_inputs(B, C, N, M):
    pts = gen(13, B, 3, N, scale=0.5)
    return pts, pts[:, :, :M].contiguous(), gen(14, B, C, M), gen(15, B, C, N)


@pytest.mark.parametrize("B,C,N,r", AVG_VOXELIZE_CASES)
def test_avg_voxelize_backward(B, C, N, r):
    F = _F()
    feats, vox, gy = (t.cuda() for t in avg_voxelize_inputs(B, C, N, r))
    feats.requires_grad_(True)
    out = F.avg_voxelize(feats, vox, r)
    out.backward(gy)
    REF.exact(key("avg_voxelize", B, C, N, r) + "/grad", feats.grad,
              "avg_voxelize backward is a pure gather: must be bit-identical to the reference kernel")


@pytest.mark.parametrize("B,C,N,r", DEVOX_CASES)
def test_trilinear_devoxelize_backward(B, C, N, r):
    F = _F()
    grid, coords, gy = (t.cuda() for t in devox_inputs(B, C, N, r))
    grid.requires_grad_(True)
    out = F.trilinear_devoxelize(grid, coords, r, True)
    out.backward(gy)
    REF.close(key("devox", B, C, N, r) + "/grad", grid.grad.view(B, C, -1), 1e-6,
              "trilinear_devoxelize backward vs reference kernel")


@pytest.mark.parametrize("B,C,N,M,U", GROUPING_CASES)
def test_grouping_and_gather_backward(B, C, N, M, U):
    F = _F()
    feats, idx, gy, feats2, idx1, gy1 = (t.cuda() for t in grouping_inputs(B, C, N, M, U))
    feats.requires_grad_(True)
    g = F.grouping(feats, idx)
    g.backward(gy)
    k = key("grouping", B, C, N, M, U)
    REF.close(k + "/grad", feats.grad, 1e-6, "grouping backward vs reference kernel")
    feats2.requires_grad_(True)
    o = F.gather(feats2, idx1)
    o.backward(gy1)
    REF.close(k + "/gather_grad", feats2.grad, 1e-6, "gather backward vs reference kernel")


@pytest.mark.parametrize("B,C,N,M", THREE_NN_CASES)
def test_nearest_neighbor_interpolate_backward(B, C, N, M):
    F = _F()
    pts, ctr, cf, gy = (t.cuda() for t in three_nn_inputs(B, C, N, M))
    cf.requires_grad_(True)
    out = F.nearest_neighbor_interpolate(pts, ctr, cf)
    out.backward(gy)
    REF.close(key("three_nn", B, C, N, M) + "/grad", cf.grad, 1e-6, "3-NN interpolate backward vs reference kernel")


def test_no_grad_path_is_unchanged():
    """The sampling path (no_grad) keeps the plain forward calls: no autograd graph, same values."""
    F = _F()
    feats = gen(16, 2, 8, 512).cuda().requires_grad_(True)
    idx = torch.randint(0, 512, (2, 64, 32), generator=torch.Generator().manual_seed(17), dtype=torch.int32).cuda()
    with torch.no_grad():
        a = F.grouping(feats, idx)
    b = F.grouping(feats, idx)
    assert not a.requires_grad and b.requires_grad and torch.equal(a, b.detach())
