"""User models as plugin objects on the GPU (glabc_k_eval_user, glabc_user_simulate / glabc_user_evaluate, the user-model
driver): the simulator's device draws, the prior / discrepancy / log kernel against the built-in family's torch formulas,
simulated initial y in all three user samplers, checkpoint / resume, and the C-ABI refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# y = noise: the simulator's raw N(0,1) draws, five per row
NOISE_SRC = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* p, float* y)
{
    for (int k = 0; k < 5; ++k) y[k] = noise[k];
}
__device__ float glabc_user_prior_log_prob(const float* theta, const float* p) { return 0.f; }
__device__ float glabc_user_discrepancy(const float* y, const float* p) { return 0.f; }
"""

BOX_SRC = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* p, float* y)
{
    y[0] = theta[0] + noise[0];
    y[1] = theta[1] + noise[1];
}
__device__ float glabc_user_prior_log_prob(const float* theta, const float* p)
{
    const bool in = theta[0] > 0.f && theta[0] < 2.f && theta[1] > 0.f && theta[1] < 2.f;
    return in ? -1.3862944f : -INFINITY;
}
__device__ float glabc_user_discrepancy(const float* y, const float* p) { return fabsf(y[0]) + fabsf(y[1]); }
"""


def _g():
    import glabc_b200 as g
    return g


def _noise_model():
    return _g().UserModel(NOISE_SRC, theta_dim=1, y_dim=5, n_noise=5, epsilon=1.0)


def _readme_model():
    from glabc_b200.models import mixture_user_model
    return mixture_user_model(0.05)


def _props():
    g = _g()
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    gp = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    return lp, gp


def _corr(a, b):
    a, b = a.double() - a.double().mean(), b.double() - b.double().mean()
    return float((a * b).sum() / (a.norm() * b.norm()))


def test_simulate_noise_only():
    from scipy import stats as sst
    um = _noise_model()
    n = 400_003
    th = torch.zeros(n, 1)
    y = um.generate_samples(th, seed=11)
    assert y.shape == (n, 5) and y.dtype == torch.float32 and y.is_cuda
    yc = y.cpu()
    for k in range(5):
        assert sst.kstest(yc[:, k].numpy().astype(np.float64), "norm").statistic < 0.005, k
    cc = np.corrcoef(yc.double().numpy().T)
    assert np.abs(cc - np.eye(5)).max() < 0.01                        # coordinates (both halves of a Box-Muller pair)
    for k in range(5):
        assert abs(_corr(yc[:-1, k], yc[1:, k])) < 0.01               # neighbouring rows
    rep = um.generate_samples(torch.zeros(50_000, 1), num_samples=4, seed=11).cpu()
    assert rep.shape == (50_000, 4, 5)
    assert torch.equal(rep.reshape(-1, 5), yc[:200_000])             # row i * m + j = repeat j of theta row i
    for j in range(1, 4):
        assert abs(_corr(rep[:, 0, 0], rep[:, j, 0])) < 0.02          # repeats of one theta are independent draws
    # deterministic per (seed, row); row_base shifts the rows; another seed gives other draws
    assert torch.equal(um.generate_samples(th, seed=11).cpu(), yc)
    k = 1234
    assert torch.equal(um.generate_samples(th[:1000], seed=11, row_base=k).cpu(), yc[k:k + 1000])
    other = um.generate_samples(th[:1000], seed=12).cpu()
    assert not torch.equal(other, yc[:1000]) and abs(_corr(other[:, 0], yc[:1000, 0])) < 0.15
    # shapes of AbsNormalModel.generate_samples
    assert um.generate_samples(torch.zeros(1), 7, seed=1).shape == (7, 5)
    assert um.generate_samples(torch.zeros(1, 1), 7, seed=1).shape == (7, 5)
    assert um.generate_samples(torch.zeros(3, 1), seed=1).shape == (3, 5)


def test_simulate_readme_model_is_abs_theta_plus_scaled_noise():
    um, noise = _readme_model(), _noise_model()
    n = 100_001
    th = torch.randn(n, 2, generator=torch.Generator().manual_seed(3))
    got = um.generate_samples(th, seed=5, row_base=77).cpu()
    z = noise.generate_samples(torch.zeros(n, 1), seed=5, row_base=77).cpu()[:, :2]
    s = torch.tensor(um.params[2], dtype=torch.float32)
    def within_one_ulp(got, th, z):
        want = (th.abs().double() + s.double() * z.double()).float()     # |theta| + s * noise, rounded once
        ulp = torch.nextafter(want.abs(), torch.tensor(float("inf"))) - want.abs()
        return bool(((got - want).abs() <= ulp).all())
    assert within_one_ulp(got, th, z)
    one = um.generate_samples(th[5], 3, seed=5, row_base=77).cpu()    # theta [d], 3 repeats: rows 77, 78, 79
    assert one.shape == (3, 2) and within_one_ulp(one, th[5].expand(3, 2), z[:3])


def test_prior_discrepancy_log_kernel_agree_with_the_builtin_family():
    g = _g()
    um, ref = _readme_model(), g.Mixture_set(0.05)
    gen = torch.Generator().manual_seed(8)
    th = torch.randn(200_001, 2, generator=gen) * 2.0
    y = 1.5 + torch.randn(200_001, 2, generator=gen) * 0.4
    got_p, want_p = um.prior_log_prob(th), ref.prior_log_prob(th).float()
    assert got_p.is_cuda and got_p.dtype == torch.float32 and got_p.shape == (200_001,)
    assert float(((got_p.cpu() - want_p).abs() / want_p.abs()).max()) < 1e-6
    got_d, want_d = um.discrepancy(y).cpu(), ref.discrepancy(y).float()
    assert float(((got_d - want_d).abs() / want_d.abs()).max()) < 1e-6
    got_k, want_k = um.calculate_log_kernel(y).cpu().double(), ref.calculate_log_kernel(y).double().reshape(-1)
    eps = 0.05
    terms = torch.maximum(torch.full_like(want_k, abs(-0.5 * np.log(2 * np.pi) - np.log(eps))), want_d.double() ** 2 / (2 * eps ** 2))
    assert float(((got_k - want_k).abs() / terms).max()) < 1e-6
    # another epsilon: the torch formula, as AbsNormalModel's
    got_e = um.calculate_log_kernel(y[:1000], epsilon=0.2).cpu()
    assert torch.allclose(got_e, ref.calculate_log_kernel(y[:1000], epsilon=0.2).reshape(-1).float(), rtol=1e-6, atol=1e-6)
    dis = torch.rand(100) * 0.3
    assert torch.allclose(um.calculate_log_kernel_dis(dis).cpu(), ref.calculate_log_kernel_dis(dis).cpu(), rtol=1e-6, atol=1e-6)
    # -inf passes through a box prior
    box = g.UserModel(BOX_SRC, theta_dim=2, y_dim=2, n_noise=2, epsilon=0.1)
    pts = torch.tensor([[1.0, 1.0], [2.5, 1.0], [-0.1, 0.3], [0.5, 1.9]])
    lp = box.prior_log_prob(pts).cpu()
    inside = torch.tensor(-1.3862944).item()
    assert lp[0].item() == lp[3].item() == inside and bool(torch.isneginf(lp[1:3]).all())


def _run(sampler, um, T, theta0, y0, **kw):
    g = _g()
    lp, gp = _props()
    if sampler == "global":
        return g.GlobalMCMC(um, T, theta0, y0, gp, None, 0.5, lp, **kw)
    if sampler == "isir":
        return g.GLMCMC(um, T, theta0, y0, lp, None, 0.8, gp, 4, **kw)
    return g.GLMALA(um, T, theta0, y0, 0.3, 40, None, 0.7, gp, 4, **kw)


SAMPLERS = ["global", "isir", "mala"]


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_initial_y_none_is_the_simulator_draw_and_shards(sampler):
    um = _readme_model()
    Cn, T, s = 1000, 120, 21
    th0 = torch.randn(Cn, 2, generator=torch.Generator().manual_seed(4))
    kw = dict(num_chains=Cn, seed=s, trace="chain", return_stats=True)
    a, sa = _run(sampler, um, T, th0, None, **kw)
    b, sb = _run(sampler, um, T, th0, um.generate_samples(th0, seed=s), **kw)
    assert torch.equal(a, b) and torch.equal(sa.raw, sb.raw)
    h = Cn // 2
    lo, slo = _run(sampler, um, T, th0[:h], None, **dict(kw, num_chains=h))
    hi, shi = _run(sampler, um, T, th0[h:], None, chain_id_base=h, **dict(kw, num_chains=Cn - h))
    assert torch.equal(torch.cat([lo, hi]), a) and torch.equal(torch.cat([slo.raw, shi.raw]), sa.raw)


def test_initial_y_none_readme_posterior_and_sweep():
    from scipy import stats as sst
    g = _g()
    from glabc_b200.sweeps import esjd_sweep
    um = _readme_model()
    lp, gp = _props()
    Cn, T = 16384, 6001
    out = g.GlobalMCMC(um, T, torch.zeros(2), None, gp, None, 0.5, lp, num_chains=Cn, seed=3, trace="time")
    a = out[-1].abs().cpu().numpy().astype(np.float64)
    for i in range(2):   # SURVEY.md App. D: |theta_i| ~ N(1.42518, 0.049881)
        assert sst.kstest(a[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.02
    best, table = esjd_sweep(lambda gf, **kw: g.GlobalMCMC(um, 201, torch.zeros(2), None, gp, None, gf, lp, **kw),
                             grid=[0.2, 0.8], num_chains=2048)
    assert best in (0.2, 0.8) and bool(torch.isfinite(table).all()) and bool((table[:, 1] > 0).all())


def _ck(path):
    return torch.load(path, map_location="cpu", weights_only=True)


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_checkpoint_resume_continues_bit_identically(sampler, tmp_path):
    um = _readme_model()
    Cn, s = 700, 5
    th0 = torch.randn(Cn, 2, generator=torch.Generator().manual_seed(6))
    kw = dict(num_chains=Cn, seed=s, trace="chain", return_stats=True)
    full, st_full = _run(sampler, um, 301, th0, None, checkpoint=str(tmp_path / "full.pt"), **kw)
    first, _ = _run(sampler, um, 151, th0, None, checkpoint=str(tmp_path / "cut.pt"), **kw)
    rest, st_rest = _run(sampler, um, 301, None, None, resume=str(tmp_path / "cut.pt"), checkpoint=str(tmp_path / "end.pt"), **kw)
    assert first.shape == (Cn, 151, 2) and rest.shape == (Cn, 150, 2)
    assert torch.equal(torch.cat([first, rest], dim=1), full)
    a, b = _ck(tmp_path / "full.pt"), _ck(tmp_path / "end.pt")
    assert a["sampler"] == b["sampler"] == sampler + "_user" and a["model"] == um.fingerprint() and a["step_base"] == 300
    for key in ("theta", "y", "aux"):
        assert (a[key] is None and b[key] is None) or torch.equal(a[key], b[key]), key
    # a launch sums its own steps before adding them to the accumulators, so the float sums are re-associated at the cut;
    # the counts are exact, and two resumes from one checkpoint agree bit for bit
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4]) and torch.allclose(st_rest.raw, st_full.raw, rtol=1e-4, atol=1e-3)
    _, st_again = _run(sampler, um, 301, None, None, resume=str(tmp_path / "cut.pt"), **kw)
    assert torch.equal(st_again.raw, st_rest.raw)
    # nothing left to do: no trace, the state stays
    none, st_none = _run(sampler, um, 301, None, None, resume=str(tmp_path / "end.pt"), **kw)
    assert none is None and torch.equal(st_none.raw, st_rest.raw)
    with pytest.raises(ValueError, match="already at iteration"):
        _run(sampler, um, 200, None, None, resume=str(tmp_path / "end.pt"), **kw)


def test_resume_refuses_other_models_and_samplers(tmp_path):
    g = _g()
    um = _readme_model()
    lp, gp = _props()
    kw = dict(num_chains=64, seed=2, trace="none")
    _run("global", um, 51, torch.zeros(2), None, checkpoint=str(tmp_path / "user.pt"), **kw)
    g.GlobalMCMC(g.Mixture_set(0.05), 51, torch.zeros(2), None, gp, None, 0.5, lp, checkpoint=str(tmp_path / "builtin.pt"), **kw)
    from glabc_b200.models import mixture_user_model
    for other in (mixture_user_model(0.06), g.UserModel(um.source + "\n", 2, 2, 2, 0.05, um.params),
                  g.UserModel(um.source, 2, 2, 2, 0.05, [1.5, 1.4, um.params[2]])):
        with pytest.raises(ValueError, match="another user model"):
            _run("global", other, 101, None, None, resume=str(tmp_path / "user.pt"), **kw)
    with pytest.raises(ValueError, match="sampler"):
        _run("global", um, 101, None, None, resume=str(tmp_path / "builtin.pt"), **kw)
    with pytest.raises(ValueError, match="sampler"):
        _run("isir", um, 101, None, None, resume=str(tmp_path / "user.pt"), **kw)
    with pytest.raises(ValueError, match="sampler"):
        g.GlobalMCMC(g.Mixture_set(0.05), 101, None, None, gp, None, 0.5, lp, resume=str(tmp_path / "user.pt"), **kw)


def test_abi_refusals_launch_nothing():
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    eng = get_engine()
    lib, h = eng.lib, eng.ctx.handle
    um = _readme_model()
    pod = um.user_pod()
    n = 257
    th = torch.randn(n, 2, device="cuda")
    y = torch.full((n, 2), 7.25, device="cuda")
    out = torch.full((n,), 7.25, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.glabc_user_simulate(h, C.byref(pod), p(th), -1, 1, 0, p(y), stream) == abi.ERR_INVALID
    assert lib.glabc_user_simulate(h, C.byref(pod), p(th), n, 1, 0, None, stream) == abi.ERR_INVALID
    assert lib.glabc_user_simulate(h, C.byref(pod), None, n, 1, 0, p(y), stream) == abi.ERR_INVALID
    for op in (abi.USER_SIMULATE, 4, -1):
        assert lib.glabc_user_evaluate(h, C.byref(pod), op, p(th), n, p(out), stream) == abi.ERR_INVALID
    assert lib.glabc_user_evaluate(h, C.byref(pod), abi.USER_PRIOR, p(th), -3, p(out), stream) == abi.ERR_INVALID
    assert lib.glabc_user_evaluate(h, C.byref(pod), abi.USER_PRIOR, p(th), n, None, stream) == abi.ERR_INVALID
    for bad in (dict(theta_dim=0), dict(y_dim=17), dict(n_noise=33), dict(epsilon=0.0)):
        bp = um.user_pod()
        for k, v in bad.items():
            setattr(bp, k, v)
        assert lib.glabc_user_simulate(h, C.byref(bp), p(th), n, 1, 0, p(y), stream) == abi.ERR_INVALID, bad
        assert lib.glabc_user_evaluate(h, C.byref(bp), abi.USER_PRIOR, p(th), n, p(out), stream) == abi.ERR_INVALID, bad
    broken = _g().UserModel(um.source.replace("sqrtf", "sqrtf +*"), 2, 2, 2, 0.05, um.params).user_pod()
    assert lib.glabc_user_evaluate(h, C.byref(broken), abi.USER_PRIOR, p(th), n, p(out), stream) == abi.ERR_INVALID
    assert b"does not compile" in lib.glabc_last_error(h)
    assert lib.glabc_user_simulate(h, C.byref(pod), None, 0, 1, 0, None, stream) == abi.OK   # n == 0: nothing to do
    torch.cuda.synchronize()
    assert bool((y == 7.25).all()) and bool((out == 7.25).all())
