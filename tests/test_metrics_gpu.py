"""SURVEY 8f rank 2 (Chamfer part): lion_chamfer_forward / lion_chamfer_pairwise through the
reference-facing wrappers, against the CPU oracle and the outputs of the reference's own chamfer_3D and
PyTorchEMD extensions on the same inputs, stored in tests/golden/ref_metrics.npz by
tests/golden/make_golden_ref_kernels.py: distances bit-exact, indices exact."""
import numpy as np
import pytest
import torch

from oracle import metrics as OM
from tests.util import RefGolden, assert_close, gen

pytestmark = pytest.mark.gpu
REF = RefGolden("ref_metrics")

# Inputs of every case; make_golden_ref_kernels.py runs the reference's kernels on exactly these.
CHAMFER_CASES = [(3, 2048, 2048), (2, 1000, 777), (1, 5, 3000), (4, 1, 1), (2, 4100, 513)]
EMD_CASES = [(3, 2048, 2048), (2, 512, 512), (2, 1024, 256), (2, 300, 1200), (1, 7, 5)]


def case_id(params):
    return "_".join(str(p) for p in params)


def key(test, *params):
    return test + "/" + case_id(params)


def chamfer_inputs(B, N, M):
    a, b = gen(81, B, N, 3), gen(82, B, M, 3)
    if N > 4 and M > 4:
        b[:, 3] = b[:, 1]                      # duplicated candidates: exact ties, lowest index must win
        a[:, 2] = a[:, 0]
    return a, b


def emd_inputs(B, N, M):
    return gen(91, B, N, 3) * 0.4, gen(92, B, M, 3) * 0.4 + 0.1


@pytest.mark.parametrize("B,N,M", CHAMFER_CASES)
def test_chamfer_forward_matches_oracle_and_reference_kernel(B, N, M):
    from lion_b200.third_party.ChamferDistancePytorch.chamfer3D.dist_chamfer_3D import chamfer_3DDist_nograd
    a, b = chamfer_inputs(B, N, M)
    d1, d2, i1, i2 = chamfer_3DDist_nograd()(a.cuda(), b.cuda())
    assert i1.dtype == torch.int32 and d1.shape == (B, N) and i2.shape == (B, M)
    o1, o2, j1, j2 = OM.chamfer_forward(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), j1) and np.array_equal(i2.cpu().numpy(), j2)
    assert np.array_equal(d1.cpu().numpy(), o1) and np.array_equal(d2.cpu().numpy(), o2)
    k = key("chamfer", B, N, M)
    REF.exact(k + "/idx1", i1, "indices (a -> b) vs the reference kernel")
    REF.exact(k + "/idx2", i2, "indices (b -> a) vs the reference kernel")
    REF.exact(k + "/dist1", d1, "distances (a -> b) vs the reference kernel")
    REF.exact(k + "/dist2", d2, "distances (b -> a) vs the reference kernel")


def _stored_cases(test):
    return {name.split("/")[1] for name in REF.keys() if name.startswith(test + "/")}


def test_reference_chamfer_vectors_cover_every_case():
    """Every Chamfer case above is compared with the reference kernel's stored outputs; none of them can silently
    lose that leg."""
    assert _stored_cases("chamfer") == {case_id(c) for c in CHAMFER_CASES}


def test_pairwise_cd_matrix():
    from lion_b200.utils.evaluation_metrics_fast import _pairwise_EMD_CD_, distChamferCUDAnograd
    s, r = gen(83, 5, 2048, 3), gen(84, 7, 2048, 3) * 1.1
    cd, cd2 = _pairwise_EMD_CD_('CD', s.cuda(), r.cuda(), batch_size=3, require_grad=False)
    assert cd.shape == (5, 7) and cd2 is cd
    assert_close(cd, torch.from_numpy(OM.pairwise_cd(s.numpy(), r.numpy())), 1e-5, "pairwise CD vs oracle")
    # the reference's composition: one sample expanded against the reference batch, dl.mean(1) + dr.mean(1)
    for i in (0, 4):
        dl, dr = distChamferCUDAnograd(s[i:i + 1].expand(7, -1, -1).contiguous().cuda(), r.cuda())
        assert_close(cd[i], dl.mean(1) + dr.mean(1), 1e-5, "pairwise CD vs drop-in composition")
    again, _ = _pairwise_EMD_CD_('CD', s.cuda(), r.cuda(), batch_size=3)
    assert torch.equal(again, cd), "pairwise CD is not bit-reproducible"
    # ragged sizes
    s2, r2 = gen(85, 2, 300, 3), gen(86, 3, 1111, 3)
    cd3, _ = _pairwise_EMD_CD_('CD', s2.cuda(), r2.cuda(), batch_size=8)
    assert_close(cd3, torch.from_numpy(OM.pairwise_cd(s2.numpy(), r2.numpy())), 1e-5, "ragged pairwise CD")
    with pytest.raises(NotImplementedError):
        _pairwise_EMD_CD_('JSD', s.cuda(), r.cuda(), batch_size=3)


@pytest.mark.parametrize("B,N,M", EMD_CASES)
def test_emd_approx_matches_reference_kernels_and_oracle(B, N, M):
    """lion_emd_approx (fused approxmatch + matchcost, no match matrix) against the reference's own
    kernels (stored outputs) -- the annealing iterates follow the same arithmetic, only the final
    sum is ordered differently: 2e-5 -- and against the float64 restatement (exact exp vs __expf: 2e-3)."""
    from lion_b200.third_party.PyTorchEMD.emd_nograd import earth_mover_distance_nograd
    a, b = emd_inputs(B, N, M)
    cost = earth_mover_distance_nograd(a.cuda(), b.cuda(), transpose=False)
    assert cost.shape == (B,) and torch.isfinite(cost).all()
    assert torch.equal(cost, earth_mover_distance_nograd(a.cuda(), b.cuda(), transpose=False)), "EMD is not bit-reproducible"
    assert_close(earth_mover_distance_nograd(a.transpose(1, 2).cuda(), b.transpose(1, 2).cuda()), cost, 0, "transpose=True path")
    REF.close(key("emd", B, N, M) + "/cost", cost, 2e-5, "EMD vs the reference kernels")
    if N * M <= 1024 * 1024:
        assert_close(cost, torch.from_numpy(OM.emd_approx(a.numpy(), b.numpy()) / N), 2e-3, "EMD vs float64 restatement")


def test_reference_emd_vectors_cover_every_case():
    assert _stored_cases("emd") == {case_id(c) for c in EMD_CASES}


def test_pairwise_emd_matrix():
    from lion_b200.utils.evaluation_metrics_fast import _pairwise_EMD_CD_, emd_approx
    s, r = gen(93, 3, 1024, 3) * 0.4, gen(94, 4, 1024, 3) * 0.5
    emd, emd2 = _pairwise_EMD_CD_('EMD', s.cuda(), r.cuda(), batch_size=2, require_grad=False)
    assert emd.shape == (3, 4) and emd2 is emd
    for i in range(3):
        row = emd_approx(s[i:i + 1].expand(4, -1, -1).contiguous().cuda(), r.cuda(), require_grad=False)
        assert torch.equal(emd[i], row), "pairwise EMD differs from the per-pair op"
