"""The seven point/voxel operators through the C ABI, against (a) the CPU oracle and (b) the outputs of the
reference's own CUDA kernels on the same inputs, stored in tests/golden/ref_point_ops.npz by
tests/golden/make_golden_ref_kernels.py (bit-exact for every index output)."""
import numpy as np
import pytest
import torch

from oracle import point_ops as P
from tests.util import RefGolden, assert_close, gen

pytestmark = pytest.mark.gpu
REF = RefGolden("ref_point_ops")


def _F():
    from lion_b200.third_party.pvcnn import functional as F
    return F


def key(test, *params):
    return test + "/" + "_".join(str(p) for p in params)


def cloud(seed, B, N, spread=0.5):
    return gen(seed, B, 3, N, scale=spread)


# Inputs of every case that is compared with the reference kernels; make_golden_ref_kernels.py runs the reference on
# exactly these.
VOXELIZE_CASES = [(2, 2048, 32), (3, 1024, 16), (2, 256, 8), (1, 64, 8)]
DEVOX_CASES = [(2, 32, 2048, 32), (2, 64, 1024, 16), (1, 130, 64, 8)]
FPS_CASES = [(3, 2048, 1024), (2, 1024, 256), (2, 256, 64), (4, 64, 16), (1, 700, 33)]
BALL_QUERY_CASES = [(2, 2048, 1024, 0.1), (2, 1024, 256, 0.2), (2, 256, 64, 0.4), (2, 64, 16, 0.8)]
THREE_NN_CASES = [(2, 192, 64, 16), (2, 192, 256, 64), (2, 64, 1024, 256), (2, 17, 2048, 1024)]


def voxelize_inputs(B, N, r):
    return cloud(1, B, N), gen(2, B, 7, N)


def devox_inputs(B, C, N, r):
    grid = gen(4, B, C, r, r, r)
    coords = torch.rand(B, 3, N, generator=torch.Generator().manual_seed(5)) * (r - 1)
    coords[:, :, :8] = torch.floor(coords[:, :, :8])       # exact lattice points: hi offset must be 0
    coords[:, :, 8] = r - 1                                 # upper corner of the grid
    coords[:, :, 9] = 0
    return grid, coords


def fps_inputs(B, N, M):
    coords = cloud(6, B, N)
    if N >= 256:
        coords[0, :, 100:140] = coords[0, :, 7:8]          # duplicates => exact ties in the distances
    return coords


def ball_query_inputs(B, N, M, radius):
    pts = cloud(7, B, N, spread=0.3)
    ctr = pts[:, :, :M].clone()
    ctr[0, :, 0] = 50.0                                     # a centre with no neighbour: all zeros
    return pts, ctr


def three_nn_inputs(B, C, N, M):
    pts = cloud(9, B, N)
    ctr = pts[:, :, :M].clone()                            # centres coincide with points: d = 0 -> clamp 1e-10
    return pts, ctr, gen(10, B, C, M)


def fused_inputs():
    return cloud(29, 32, 2048, spread=0.41), gen(30, 32, 8, 2048)


@pytest.mark.parametrize("B,N,r", VOXELIZE_CASES)
def test_voxel_coords_and_avg_voxelize(B, N, r):
    F = _F()
    coords, feats = voxelize_inputs(B, N, r)
    nc_cpu, _ = P.voxel_coords(coords, r)                    # torch-CPU summation order: values agree to rounding
    nc, vox = F.voxel_coords(coords.cuda(), r)
    assert_close(nc, nc_cpu, 2e-6, "norm_coords")
    # bit-exact voxel index assignment: the oracle's restatement of the reference ON CUDA (the mean's summation
    # order is torch-CUDA's, oracle/point_ops.py::cuda_mean_lastdim) gives identical coordinates and indices
    nc_o, vox_o = P.voxel_coords_cuda_order(coords, r)
    assert torch.equal(nc.cpu(), nc_o)
    assert torch.equal(vox.cpu(), vox_o)
    out = F.avg_voxelize(feats.cuda(), vox, r)
    out_o, ind_o, cnt_o = P.avg_voxelize(feats, vox.cpu(), r)
    assert_close(out, out_o, 1e-5, "avg_voxelize")
    k = key("voxelize", B, N, r)
    REF.exact(k + "/ind", ind_o, "avg_voxelize indices: oracle vs reference kernel")
    REF.exact(k + "/cnt", cnt_o, "avg_voxelize counts: oracle vs reference kernel")
    REF.close(k + "/out", out.view(B, 7, -1), 1e-5, "avg_voxelize vs reference kernel")


def test_avg_voxelize_collisions_and_single_point():
    F = _F()
    B, C, N, r = 2, 5, 33, 4
    feats = gen(3, B, C, N)
    vox = torch.zeros(B, 3, N, dtype=torch.int32)          # every point in voxel 0
    vox[1, :, 1:] = r - 1                                   # batch 1: one point alone, rest in the last voxel
    out = F.avg_voxelize(feats.cuda(), vox.cuda(), r)
    out_o, _, _ = P.avg_voxelize(feats, vox, r)
    assert_close(out, out_o, 1e-5, "avg_voxelize collisions")


@pytest.mark.parametrize("B,C,N,r", DEVOX_CASES)
def test_trilinear_devoxelize(B, C, N, r):
    F = _F()
    grid, coords = devox_inputs(B, C, N, r)
    out = F.trilinear_devoxelize(grid.cuda(), coords.cuda(), r, False)
    assert_close(out, P.trilinear_devoxelize(grid, coords, r), 2e-6, "trilinear_devoxelize")
    k = key("devox", B, C, N, r)
    REF.close(k + "/out", out, 1e-6, "devox vs reference kernel")
    idx_o, w_o = P.trilinear_corners(coords, r)
    REF.exact(k + "/inds", idx_o, "devox corner indices: oracle vs reference kernel")
    REF.exact(k + "/wgts", w_o, "devox corner weights: oracle vs reference kernel")


@pytest.mark.parametrize("B,N,M", FPS_CASES)
def test_furthest_point_sampling(B, N, M):
    from lion_b200.third_party.pvcnn.functional import furthest_point_sample_indices
    F = _F()
    coords = fps_inputs(B, N, M)
    idx = furthest_point_sample_indices(coords.cuda(), M)
    REF.exact(key("fps", B, N, M) + "/idx", idx, "FPS indices")
    idx_o = P.furthest_point_sample_idx(coords, M)
    assert torch.equal(idx.cpu(), idx_o), "FPS differs from the oracle"
    centers = F.furthest_point_sample(coords.cuda(), M)
    assert torch.equal(centers.cpu(), P.gather(coords, idx_o))


@pytest.mark.parametrize("B,N,M,radius", BALL_QUERY_CASES)
def test_ball_query_and_grouping(B, N, M, radius):
    F = _F()
    pts, ctr = ball_query_inputs(B, N, M, radius)
    idx = F.ball_query(ctr.cuda(), pts.cuda(), radius, 32)
    REF.exact(key("ball_query", B, N, M, radius) + "/idx", idx, "ball query indices")
    idx_o = P.ball_query(ctr, pts, radius, 32)
    assert torch.equal(idx.cpu(), idx_o), "ball query differs from the oracle"
    assert (idx[0, 0] == 0).all()
    feats = gen(8, B, 9, N)
    g = F.grouping(feats.cuda(), idx)
    assert torch.equal(g.cpu(), P.grouping(feats, idx_o))


@pytest.mark.parametrize("B,C,N,M", THREE_NN_CASES)
def test_nearest_neighbor_interpolate(B, C, N, M):
    F = _F()
    pts, ctr, cf = three_nn_inputs(B, C, N, M)
    out = F.nearest_neighbor_interpolate(pts.cuda(), ctr.cuda(), cf.cuda())
    out_o = P.nearest_neighbor_interpolate(pts, ctr, cf)
    assert_close(out, out_o, 2e-6, "3-NN interpolate")
    k = key("three_nn", B, C, N, M)
    idx_o, w_o = P.three_nn(pts, ctr)
    REF.exact(k + "/idx", idx_o, "3-NN indices: oracle vs reference kernel")
    REF.close(k + "/out", out, 1e-6, "3-NN interpolate vs reference kernel")


def test_gather():
    F = _F()
    feats = gen(11, 3, 5, 100)
    idx = torch.randint(0, 100, (3, 40), generator=torch.Generator().manual_seed(1), dtype=torch.int32)
    assert torch.equal(F.gather(feats.cuda(), idx.cuda()).cpu(), P.gather(feats, idx))


# ---- a5: bit-exact voxel index assignment against torch ON CUDA (the reference's Voxelization.forward) ----
def _voxelization_torch(coords, r):
    """Voxelization.forward's coordinate part evaluated by torch on whatever device `coords` lives on
    (models/pvcnn2_ada.py:173-188, normalize=True, eps=0)."""
    nc = coords - coords.mean(2, keepdim=True)
    nc = nc / (nc.norm(dim=1, keepdim=True).max(dim=2, keepdim=True).values * 2.0 + 0.0) + 0.5
    nc = torch.clamp(nc * r, 0, r - 1)
    return nc, torch.round(nc).to(torch.int32)


@pytest.mark.parametrize("B,N", [(32, 2048), (32, 1024), (32, 256), (32, 64), (1, 2048), (2, 1024), (3, 256), (4, 64), (5, 4096),
                                 (2, 700), (3, 33), (16, 130), (7, 128), (1, 5)])
def test_cuda_mean_emulation_matches_torch(B, N):
    """oracle/point_ops.py::cuda_mean_lastdim restates the summation ORDER of torch's CUDA reduction kernel
    (third-party arithmetic, not in /root/reference): pinned here against torch itself, bit for bit."""
    x = cloud(21, B, N)
    want = x.cuda().mean(2).cpu()
    got = torch.from_numpy(P.cuda_mean_lastdim(x.numpy()))
    assert torch.equal(got, want), "emulated torch-CUDA mean differs on %d of %d values" % ((got != want).sum().item(), got.numel())


@pytest.mark.parametrize("B", [32, 2, 1])
@pytest.mark.parametrize("N,r", [(2048, 32), (1024, 16), (256, 8), (64, 8)])
def test_voxel_indices_bit_exact_vs_torch_cuda(B, N, r):
    """north_star: 'bit-exact voxel index assignment'.  lion_voxel_coords (same device code as the fused path's
    k_vox_prep) against the reference's Voxelization.forward evaluated by torch on CUDA: normalised coordinates
    and voxel indices identical, at the network's four (N, r) levels and at B = 32 (BASELINE configs[1])."""
    F = _F()
    coords = cloud(22 + N, B, N, spread=0.37)
    nc, vox = F.voxel_coords(coords.cuda(), r)
    nc_t, vox_t = _voxelization_torch(coords.cuda(), r)
    assert torch.equal(vox, vox_t), "%d voxel indices differ from torch-CUDA" % (vox != vox_t).sum().item()
    assert torch.equal(nc, nc_t)
    # and the CPU oracle's CUDA-order restatement agrees with both
    nc_o, vox_o = P.voxel_coords_cuda_order(coords, r)
    assert torch.equal(vox.cpu(), vox_o) and torch.equal(nc.cpu(), nc_o)


def test_fused_path_voxel_indices_bit_exact_b32():
    """The fused network path (k_vox_prep inside lion_pvconv_fwd) uses the same statistics code: a PVConv's
    scatter/gather indices at B = 32 are those of torch-CUDA.  Checked through avg_voxelize on the indices of
    lion_voxel_coords against the reference's own kernel fed with torch-CUDA indices."""
    F = _F()
    B, N, r = 32, 2048, 32
    coords, feats = fused_inputs()
    _, vox = F.voxel_coords(coords.cuda(), r)
    out = F.avg_voxelize(feats.cuda(), vox, r)
    REF.close("fused_b32/out", out.view(B, 8, -1), 1e-5, "avg_voxelize at B=32 on torch-CUDA voxel indices")
