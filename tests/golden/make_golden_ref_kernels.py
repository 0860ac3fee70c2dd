"""Generate tests/golden/ref_{point_ops,point_ops_backward,metrics,fullsize}.npz: the outputs of the reference's own
CUDA kernels on the inputs of the GPU tests that compare with them.

    python oracle/build_ref.py                                  # the reference's extensions -> oracle/_ref/
    python tests/golden/make_golden_ref_kernels.py [OUT_DIR]    # needs a GPU; OUT_DIR defaults to tests/golden

The kernels are the reference's pvcnn point ops (_pvcnn_backend.so), its chamfer_3D and PyTorchEMD extensions, all
compiled unmodified by oracle/build_ref.py; the full-size step runs oracle/net.py on CUDA with those point kernels
(oracle/ref_cuda_ops.py), the reference's eager path.  Inputs come from the test modules themselves, so the stored
vectors cannot drift from what the tests feed their own kernels.  Each output is kept by tests/util.py::record:
shape, SHA-256 (bit-exact checks), max-abs / rms, and a fixed seeded sample of values (tolerance checks).
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import torch  # noqa: E402

from oracle import build_ref  # noqa: E402
from oracle import point_ops as P  # noqa: E402
from tests import test_fullsize_gpu as TF  # noqa: E402
from tests import test_metrics_gpu as TM  # noqa: E402
from tests import test_point_ops_backward_gpu as TB  # noqa: E402
from tests import test_point_ops_gpu as TP  # noqa: E402
from tests.util import record, save_golden  # noqa: E402

EXACT, CLOSE, FULLSIZE = 32, 512, 4096      # stored sample sizes: bit-exact checks use the digest, the sample is for messages


def loaded(mod, what):
    assert mod is not None, "oracle/_ref/%s is missing: run `python oracle/build_ref.py` first" % what
    return mod


def point_ops(ref):
    out = {}
    for B, N, r in TP.VOXELIZE_CASES:
        coords, feats = TP.voxelize_inputs(B, N, r)
        _, vox = P.voxel_coords_cuda_order(coords, r)          # the tests pin lion_voxel_coords to these indices
        o, ind, cnt = ref.avg_voxelize_forward(feats.cuda(), vox.to(torch.int32).cuda().contiguous(), r)
        k = TP.key("voxelize", B, N, r)
        record(out, k + "/out", o, CLOSE)
        record(out, k + "/ind", ind, EXACT)
        record(out, k + "/cnt", cnt, EXACT)
    for B, C, N, r in TP.DEVOX_CASES:
        grid, coords = TP.devox_inputs(B, C, N, r)
        o, inds, wgts = ref.trilinear_devoxelize_forward(r, True, coords.cuda(), grid.view(B, C, -1).cuda())
        k = TP.key("devox", B, C, N, r)
        record(out, k + "/out", o, CLOSE)
        record(out, k + "/inds", inds, EXACT)
        record(out, k + "/wgts", wgts, EXACT)
    for B, N, M in TP.FPS_CASES:
        record(out, TP.key("fps", B, N, M) + "/idx", ref.furthest_point_sampling(TP.fps_inputs(B, N, M).cuda(), M), EXACT)
    for B, N, M, radius in TP.BALL_QUERY_CASES:
        pts, ctr = TP.ball_query_inputs(B, N, M, radius)
        record(out, TP.key("ball_query", B, N, M, radius) + "/idx", ref.ball_query(ctr.cuda(), pts.cuda(), radius, 32), EXACT)
    for B, C, N, M in TP.THREE_NN_CASES:
        pts, ctr, cf = TP.three_nn_inputs(B, C, N, M)
        o, idx, _ = ref.three_nearest_neighbors_interpolate_forward(pts.cuda(), ctr.cuda(), cf.cuda())
        k = TP.key("three_nn", B, C, N, M)
        record(out, k + "/out", o, CLOSE)
        record(out, k + "/idx", idx, EXACT)
    coords, feats = TP.fused_inputs()
    _, vox_t = TP._voxelization_torch(coords.cuda(), 32)      # the reference's Voxelization.forward, torch on CUDA
    record(out, "fused_b32/out", ref.avg_voxelize_forward(feats.cuda(), vox_t.contiguous(), 32)[0], CLOSE)
    return out


def point_ops_backward(ref):
    out = {}
    for B, C, N, r in TB.AVG_VOXELIZE_CASES:
        feats, vox, gy = (t.cuda() for t in TB.avg_voxelize_inputs(B, C, N, r))
        _, ind, cnt = ref.avg_voxelize_forward(feats, vox, r)
        record(out, TB.key("avg_voxelize", B, C, N, r) + "/grad", ref.avg_voxelize_backward(gy.view(B, C, -1).contiguous(), ind, cnt), EXACT)
    for B, C, N, r in TB.DEVOX_CASES:
        grid, coords, gy = (t.cuda() for t in TB.devox_inputs(B, C, N, r))
        _, inds, wgts = ref.trilinear_devoxelize_forward(r, True, coords, grid.view(B, C, -1))
        record(out, TB.key("devox", B, C, N, r) + "/grad", ref.trilinear_devoxelize_backward(gy, inds, wgts, r), CLOSE)
    for B, C, N, M, U in TB.GROUPING_CASES:
        _, idx, gy, _, idx1, gy1 = (t.cuda() for t in TB.grouping_inputs(B, C, N, M, U))
        k = TB.key("grouping", B, C, N, M, U)
        record(out, k + "/grad", ref.grouping_backward(gy, idx, N), CLOSE)
        record(out, k + "/gather_grad", ref.gather_features_backward(gy1, idx1, N), CLOSE)
    for B, C, N, M in TB.THREE_NN_CASES:
        pts, ctr, cf, gy = (t.cuda() for t in TB.three_nn_inputs(B, C, N, M))
        _, idx, wgt = ref.three_nearest_neighbors_interpolate_forward(pts, ctr, cf)
        record(out, TB.key("three_nn", B, C, N, M) + "/grad", ref.three_nearest_neighbors_interpolate_backward(gy, idx, wgt, M), CLOSE)
    return out


def metrics(chamfer, emd):
    out = {}
    for B, N, M in TM.CHAMFER_CASES:
        a, b = (t.cuda() for t in TM.chamfer_inputs(B, N, M))
        d1, d2 = torch.zeros(B, N, device="cuda"), torch.zeros(B, M, device="cuda")
        i1, i2 = torch.zeros(B, N, dtype=torch.int32, device="cuda"), torch.zeros(B, M, dtype=torch.int32, device="cuda")
        chamfer.forward(a, b, d1, d2, i1, i2)
        k = TM.key("chamfer", B, N, M)
        for name, t in (("dist1", d1), ("dist2", d2), ("idx1", i1), ("idx2", i2)):
            record(out, k + "/" + name, t, EXACT)
    for B, N, M in TM.EMD_CASES:
        a, b = (t.cuda() for t in TM.emd_inputs(B, N, M))
        cost = emd.matchcost_forward(a, b, emd.approxmatch_forward(a, b)) / float(N)
        record(out, TM.key("emd", B, N, M) + "/cost", cost, CLOSE)
    return out


def fullsize():
    from oracle import net as ON
    from oracle import point_ops as cpu_point_ops
    from oracle import ref_cuda_ops
    dev = torch.device("cuda")
    x, style, t, sd_l, sd_g = TF.inputs()
    ON.set_point_ops(ref_cuda_ops)
    try:
        with torch.no_grad():
            eps = ON.prior_forward({k: v.to(dev) for k, v in sd_l.items()}, ON.prior_spec(), x.to(dev), t.to(dev), style.to(dev))
            eg = ON.global_prior_forward({k: v.to(dev) for k, v in sd_g.items()}, style.to(dev), t.to(dev))
    finally:
        ON.set_point_ops(cpu_point_ops)
    out = {}
    record(out, "pvcnn2prior", eps, FULLSIZE)
    record(out, "global_prior", eg, FULLSIZE)
    return out


def main():
    dst = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(dst, exist_ok=True)
    assert torch.cuda.is_available(), "the reference's kernels need a GPU"
    pv = loaded(build_ref.load_ref(), "_pvcnn_backend.so")
    for name, out in (("ref_point_ops", point_ops(pv)), ("ref_point_ops_backward", point_ops_backward(pv)),
                      ("ref_metrics", metrics(loaded(build_ref.load_chamfer(), "chamfer_3D.so"), loaded(build_ref.load_emd(), "emd_ext.so"))),
                      ("ref_fullsize", fullsize())):
        path = os.path.join(dst, name + ".npz")
        save_golden(path, out)
        print(name, len(out), "outputs,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
