"""User models with Uniform / Gamma / GaussianMixture proposals and theta_dim up to 8 (csrc/user_model.cu): CPU checks.
The proposal kinds are compiled into the NVRTC module, so every kind in each slot of the GlobalMCMC, GLMCMC (iSIR) and
GLMALA kernels must compile for sm_100a; the distribution code NVRTC compiles is the text of csrc/dist_device.cuh,
embedded in the library at build time."""
import ctypes as C
import os

import pytest
import torch

from helpers import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = (abi.DIST_DIAG_GAUSSIAN, abi.DIST_UNIFORM, abi.DIST_GAMMA, abi.DIST_GAUSSIAN_MIXTURE)

# theta in R^D, y = theta + params[0] * noise, Gaussian prior N(params[1], 1) per coordinate, Euclidean discrepancy to
# y_obs = params[2..]: its ABC posterior is Gaussian in closed form (tests/test_user_model_proposals_gpu.py)
GAUSS_SRC = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* p, float* y)
{
    for (int k = 0; k < D; ++k) y[k] = theta[k] + p[0] * noise[k];
}
__device__ float glabc_user_prior_log_prob(const float* theta, const float* p)
{
    float s = 0.f;
    for (int k = 0; k < D; ++k) s += (theta[k] - p[1]) * (theta[k] - p[1]);
    return -0.5f * s;
}
__device__ float glabc_user_discrepancy(const float* y, const float* p)
{
    float s = 0.f;
    for (int k = 0; k < D; ++k) s += (y[k] - p[2 + k]) * (y[k] - p[2 + k]);
    return sqrtf(s);
}
"""


def _model(d):
    import glabc_b200 as g
    return g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=0.3, params=[0.3, 1.5] + [2.0] * d)


def _check(um, local_kind, far_kind):
    log = C.create_string_buffer(8192)
    pod = um.user_pod()
    st = abi.load().glabc_user_model_check_proposals(C.byref(pod), local_kind, far_kind, 100, log, len(log))
    return st, log.value.decode(errors="replace")


# (local kind, far kind): every kind in each slot, and a DiagGaussian beside a non-Gaussian slot in either order
PAIRS = [(KINDS[0], KINDS[0]), (KINDS[1], KINDS[2]), (KINDS[2], KINDS[3]), (KINDS[3], KINDS[1]),
         (KINDS[0], KINDS[1]), (KINDS[2], KINDS[0])]


@pytest.mark.parametrize("d", [2, 8])
def test_every_proposal_kind_compiles_in_every_slot(d):
    """one module holds the three kernels: the far kind is the Global_Proposal of glabc_k_global_user and the
    Importance_Proposal of glabc_k_isir_user / glabc_k_mala_user, the local kind their Local_Proposal"""
    um = _model(d)
    for lk, fk in PAIRS:
        st, log = _check(um, lk, fk)
        assert st == abi.OK, (lk, fk, log)


def test_glmala_width_compiles_with_every_importance_kind():
    um = _model(5)   # the widest model glabc_run_mala_user runs (its gradient lives in the aux slots)
    for fk in KINDS:
        st, log = _check(um, abi.DIST_DIAG_GAUSSIAN, fk)
        assert st == abi.OK, (fk, log)


def test_check_names_proposals_and_refuses_unknown_kinds():
    import glabc_b200 as g
    um = _model(3)
    box = g.Uniform(3, torch.zeros(3), torch.full((3,), 4.0))
    gam = g.Gamma(torch.full((3,), 8.0), torch.full((3,), 4.0))
    mix = g.GaussianMixture(2, 3, loc=[[1.5] * 3, [2.5] * 3], scale=[[0.7] * 3] * 2, weights=[0.5, 0.5])
    assert um.check() and um.check(proposals=(box, gam)) and um.check(proposals=(None, mix))
    for bad in ((0, abi.DIST_UNIFORM), (abi.DIST_UNIFORM, 5)):
        assert _check(um, *bad)[0] == abi.ERR_INVALID
    broken = g.UserModel(GAUSS_SRC.replace("sqrtf(s)", "sqrtf(s) +* 1"), 3, 3, 3, 0.3, [0.3, 1.5, 2.0, 2.0, 2.0])
    with pytest.raises(ValueError, match="does not compile"):
        broken.check(proposals=(gam, box))


def test_library_embeds_the_distribution_header():
    """NVRTC compiles the header's text as built into libglabc.so, not a copy and not a file read at run time"""
    text = open(os.path.join(ROOT, "gl-abc-mcmc_b200", "csrc", "dist_device.cuh"), "rb").read()
    lib = open(abi.load()._name, "rb").read()
    assert text in lib
    assert b'#include "dist_device.cuh"' in lib
