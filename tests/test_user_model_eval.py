"""User models as plugin objects, CPU checks: the NVRTC module with the evaluation kernel glabc_k_eval_user compiles for
sm_100a at the extremes of theta_dim, y_dim and n_noise; glabc_user_simulate / glabc_user_evaluate load with their
signatures and refuse bad calls without a context; the plugin methods refuse to run without a GPU; the checkpoint
fingerprint of a model follows what its kernels compute with."""
import ctypes as C

import pytest
import torch

from helpers import abi

# generic in D, YD and NN: every output coordinate reads the parameters and, when there is noise, one noise draw
GENERIC_SRC = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* p, float* y)
{
    for (int k = 0; k < YD; ++k) {
        float v = theta[k % D] * p[0];
#if NN > 0
        v += noise[k % NN];
#endif
        y[k] = v;
    }
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


def _model(d, yd, nn, **kw):
    import glabc_b200 as g
    args = dict(source=GENERIC_SRC, theta_dim=d, y_dim=yd, n_noise=nn, epsilon=0.1, params=[0.5, 1.0])
    args.update(kw)
    return g.UserModel(**args)


@pytest.mark.parametrize("d", [1, 8])
@pytest.mark.parametrize("nn", [0, 1, 32])
def test_module_with_the_eval_kernel_compiles(d, nn):
    """one module: the three step kernels and glabc_k_eval_user; NN = 0 and odd NN leave the SIMULATE noise array well
    formed, y_dim 16 is the widest output row"""
    assert _model(d, 16, nn).check()


def test_new_symbols_load_with_their_signatures():
    lib = abi.load()
    for name in ("glabc_user_simulate", "glabc_user_evaluate"):
        res, args = abi._SIGNATURES[name]
        fn = getattr(lib, name)
        assert fn.restype is res and list(fn.argtypes) == args
    assert (abi.USER_SIMULATE, abi.USER_PRIOR, abi.USER_DISCREPANCY, abi.USER_LOG_KERNEL) == (0, 1, 2, 3)


def test_entries_refuse_a_null_context():
    lib = abi.load()
    pod = _model(2, 2, 2).user_pod()
    assert lib.glabc_user_simulate(None, C.byref(pod), None, 0, 1, 0, None, None) == abi.ERR_INVALID
    assert lib.glabc_user_evaluate(None, C.byref(pod), abi.USER_PRIOR, None, 0, None, None) == abi.ERR_INVALID


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_plugin_methods_have_no_cpu_fallback():
    um = _model(2, 2, 2)
    for call in (lambda: um.generate_samples(torch.zeros(2)), lambda: um.prior_log_prob(torch.zeros(3, 2)),
                 lambda: um.discrepancy(torch.zeros(3, 2)), lambda: um.calculate_log_kernel(torch.zeros(3, 2)),
                 lambda: um.calculate_log_kernel_dis(torch.zeros(3))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_checkpoint_fingerprint_follows_the_model():
    base = _model(2, 2, 2)
    fp = base.fingerprint()
    assert fp == _model(2, 2, 2).fingerprint() and len(fp) == 64
    others = [_model(2, 2, 2, source=GENERIC_SRC + "\n"), _model(2, 2, 2, params=[0.5, 1.25]), _model(2, 2, 2, params=[0.5, 1.0, 0.0]),
              _model(2, 2, 2, epsilon=0.2), _model(3, 2, 2), _model(2, 3, 2), _model(2, 2, 3)]
    fps = [m.fingerprint() for m in others]
    assert fp not in fps and len(set(fps)) == len(fps)


def test_user_model_has_no_y_obs():
    """the fused-family lowering keeps refusing a UserModel (AGLMCMC and GLMCMC-NFs take the built-in family only)"""
    from glabc_b200.models import fused_model
    um = _model(2, 2, 2)
    assert not hasattr(um, "y_obs")
    with pytest.raises(NotImplementedError, match="y_obs"):
        fused_model(um)
