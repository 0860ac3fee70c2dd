"""Full-size parity (B = 32, BASELINE.json configs[1] shapes) of one denoising step of both priors against
a GPU evaluation of the oracle: oracle/net.py on CUDA tensors with the REFERENCE's own point kernels
(oracle/ref_cuda_ops.py) and torch's cuDNN / cuBLAS layers, i.e. the reference's eager path.  Its outputs on
these inputs are stored in tests/golden/ref_fullsize.npz (tests/golden/make_golden_ref_kernels.py): the
global prior's whole output and a fixed sample of the PVCNN2Prior's, with max-abs and rms of the whole.
The CPU oracle needs ~10 s per shape for this, the GPU one a fraction of a second."""
import json
import os

import pytest
import torch

from tests.synth import synth_state_dict
from tests.util import RefGolden

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
KEYS = json.load(open(os.path.join(G, "keys.json")))
REF = RefGolden("ref_fullsize")


def inputs():
    """x, style, t and the two priors' state dicts of the B = 32 step"""
    B = 32
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, 8192, 1, 1, generator=g)
    style = torch.randn(B, 128, 1, 1, generator=g)
    t = torch.randint(1, 1001, (B,), generator=g).float()
    return x, style, t, synth_state_dict(KEYS["prior"], 11), synth_state_dict(KEYS["global"], 14)


def test_prior_step_b32_matches_reference_eager_path_on_gpu():
    from lion_b200.config import default_prior_cfg
    from lion_b200.models.latent_points_ada_localprior import PVCNN2Prior
    from lion_b200.models.score_sde.resnet import PriorSEDrop
    x, style, t, sd_l, sd_g = inputs()
    cfg = default_prior_cfg()
    lp = PVCNN2Prior(cfg.sde, 1, cfg)
    lp.load_state_dict(sd_l)
    gp = PriorSEDrop(cfg.sde, 128, cfg)
    gp.load_state_dict(sd_g)
    lp, gp = lp.cuda().eval(), gp.cuda().eval()
    eps = lp(x=x.cuda(), t=t.cuda(), condition_input=style.cuda())
    eg = gp(x=style.cuda(), t=t.cuda(), condition_input=None)
    REF.close("global_prior", eg, 2e-3, "global prior, B=32")
    # both sides run TF32 convolutions (cuDNN vs tcgen05) on identical voxel / FPS / ball-query indices
    assert REF.rms("pvcnn2prior", eps) < 4e-3
    REF.close("pvcnn2prior", eps, 1e-2, "PVCNN2Prior step, B=32")
