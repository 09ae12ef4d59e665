"""Block iSIR for run-time compiled user models (GLMCMC-NFs and pooled AGLMCMC, csrc/user_model.cu): CPU checks.
The two block kernels (glabc_k_block_isir_user, glabc_k_block_weights_user) are part of the same NVRTC module as the other
user kernels, with the Local_Proposal's kind compiled in, so they must compile for sm_100a at every theta_dim, at the widest
y_dim, without and with the most simulator noise, and for every local kind."""
import ctypes as C
import os

import pytest

from helpers import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = (abi.DIST_DIAG_GAUSSIAN, abi.DIST_UNIFORM, abi.DIST_GAMMA, abi.DIST_GAUSSIAN_MIXTURE)

# y_dim outputs from D parameters and NN noise draws (NN may be 0)
WIDE_SRC = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* p, float* y)
{
    for (int k = 0; k < YD; ++k) y[k] = theta[k % D] + (NN > 0 ? p[0] * noise[k % (NN > 0 ? NN : 1)] : 0.f);
}
__device__ float glabc_user_prior_log_prob(const float* theta, const float* p)
{
    float s = 0.f;
    for (int k = 0; k < D; ++k) s += theta[k] * theta[k];
    return -0.5f * s;
}
__device__ float glabc_user_discrepancy(const float* y, const float* p)
{
    float s = 0.f;
    for (int k = 0; k < YD; ++k) s += (y[k] - p[1]) * (y[k] - p[1]);
    return sqrtf(s);
}
"""


@pytest.mark.parametrize("d", [1, 2, 4, 8])
@pytest.mark.parametrize("n_noise", [0, 32])
def test_block_kernels_compile_for_every_local_kind(d, n_noise):
    import glabc_b200 as g
    um = g.UserModel(WIDE_SRC, theta_dim=d, y_dim=16, n_noise=n_noise, epsilon=0.3, params=[0.3, 1.0])
    pod = um.user_pod()
    for lk in KINDS:
        log = C.create_string_buffer(8192)
        st = abi.load().glabc_user_model_check_proposals(C.byref(pod), lk, abi.DIST_DIAG_GAUSSIAN, 100, log, len(log))
        assert st == abi.OK, (d, n_noise, lk, log.value.decode(errors="replace"))


def test_block_kernels_are_in_the_module_source():
    """the compiled module is the embedded kernel text: both block kernels are in it, with their slot range"""
    lib = open(abi.load()._name, "rb").read()
    for name in (b"glabc_k_block_isir_user", b"glabc_k_block_weights_user", b"#define GLABC_SLOT_BLOCK 0xA0000000u"):
        assert name in lib


def test_block_entries_are_exported_and_mirrored():
    lib = abi.load()
    assert abi._SIGNATURES["glabc_run_block_isir_user"] == (
        C.c_int, [C.c_void_p, C.POINTER(abi.RunPOD), C.POINTER(abi.BlockIsirPOD), C.POINTER(abi.UserModelPOD)])
    assert abi._SIGNATURES["glabc_block_weights_user"] == (
        C.c_int, [C.c_void_p, C.POINTER(abi.RunPOD), C.POINTER(abi.BlockIsirPOD), C.c_uint32, C.POINTER(abi.UserModelPOD)])
    for name in ("glabc_run_block_isir_user", "glabc_block_weights_user"):
        assert hasattr(lib, name)
    header = open(os.path.join(ROOT, "include", "glabc.h")).read()
    assert "GLABC_API int glabc_run_block_isir_user(" in header and "GLABC_API int glabc_block_weights_user(" in header
    # a null context is refused before anything else, without a GPU
    assert lib.glabc_run_block_isir_user(None, None, None, None) == abi.ERR_INVALID
    assert lib.glabc_block_weights_user(None, None, None, 0, None) == abi.ERR_INVALID
