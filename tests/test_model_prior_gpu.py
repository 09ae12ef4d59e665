"""GPU tests of a Uniform / Gamma / GaussianMixture model prior (glabc_model_prior_set) in every sampler.

With the identity link the Gaussian ABC kernel of width eps on ||y - y_obs|| makes the ABC likelihood exactly
prod_i N(theta_i; m_i, s_i^2), m_i = y_obs_i - noise_loc_i, s_i^2 = sigma_i^2 + eps^2 (the algebra behind the README's
N(1.42518, 0.049881)), so the exact posterior marginals are a truncated normal (Uniform box), Gamma x Normal (Gamma) and a
Gaussian mixture (GaussianMixture).  Each case is chosen so that ignoring the prior (the model's N(0, I)) would fail."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from scipy import integrate
from scipy import stats as sst

from helpers import abi, fresh_mala_state

pytestmark = pytest.mark.gpu

M, S2 = 1.5, 0.05 + float(np.float32(0.05)) ** 2      # likelihood N(theta_i; M, S2) per coordinate
LO, HI = 1.4, 3.0                                      # Uniform box, both coordinates
GA, GB = 20.0, 10.0                                    # Gamma(shape, rate), both coordinates
MIX_LOC, MIX_SD, MIX_W = np.array([[0.8, 0.8], [2.2, 2.2]]), 0.3, np.array([3.0, 1.0])
SENTINEL = -7.25


def priors():
    import glabc_b200 as g
    return dict(uniform=g.Uniform(2, torch.tensor([LO, LO]), torch.tensor([HI, HI])),
                gamma=g.Gamma(torch.tensor([GA, GA]), torch.tensor([GB, GB])),
                mix=g.GaussianMixture(2, 2, loc=MIX_LOC, scale=[[MIX_SD, MIX_SD]] * 2, weights=MIX_W))


def exact_cdf(name):
    """CDF of one coordinate's exact posterior marginal (both coordinates have the same one)"""
    s = math.sqrt(S2)
    if name == "uniform":
        return sst.truncnorm((LO - M) / s, (HI - M) / s, loc=M, scale=s).cdf
    if name == "gamma":
        f = lambda x: x ** (GA - 1) * math.exp(-GB * x) * math.exp(-0.5 * (x - M) ** 2 / S2)   # noqa: E731
        grid = np.linspace(0.0, 4.0, 801)
        cum = np.concatenate([[0.0], np.cumsum([integrate.quad(f, a, b)[0] for a, b in zip(grid[:-1], grid[1:])])])
        cum /= cum[-1] + integrate.quad(f, 4.0, np.inf)[0]
        return lambda x: np.interp(x, grid, cum, left=0.0, right=1.0)
    v = MIX_SD ** 2
    logw = np.log(MIX_W / MIX_W.sum()) + sst.norm(MIX_LOC, math.sqrt(v + S2)).logpdf(M).sum(axis=1)
    pi = np.exp(logw - logw.max())
    pi /= pi.sum()
    mu, sd = (MIX_LOC[:, 0] / v + M / S2) / (1 / v + 1 / S2), math.sqrt(1 / (1 / v + 1 / S2))
    return lambda x: sum(p * sst.norm(u, sd).cdf(x) for p, u in zip(pi, mu))


def ignored_cdf():
    """the posterior marginal the model's own N(0, 1) prior would give"""
    return sst.norm(M / (1 + S2), math.sqrt(S2 / (1 + S2))).cdf


def setup(eng=None, prior=None):
    import glabc_b200 as g
    model = g.AbsNormalModel(0.05, y_obs=(M, M), noise_var=0.05, link="identity", prior=prior)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.2, 0.2])))
    gp = g.DiagGaussian(2, torch.tensor([M, M]), torch.log(torch.tensor([0.5, 0.5])))
    if eng is not None:
        eng.bind_model(model)
        eng.bind_proposal(abi.SLOT_LOCAL, lp)
        eng.bind_proposal(abi.SLOT_GLOBAL, gp)
        eng.bind_proposal(abi.SLOT_IMPORTANCE, gp)
    return g, model, lp, gp


@pytest.fixture(scope="module")
def eng():
    from glabc_b200.engine import get_engine
    return get_engine()


def check_support(name, trace):
    if name == "uniform":
        assert bool(((trace >= LO) & (trace <= HI)).all())
    elif name == "gamma":
        assert bool((trace > 0).all())


def check_coverage(name, trace, band):
    cdf = exact_cdf(name)
    grid = np.linspace(-1.0, 4.0, 5001)
    assert np.abs(cdf(grid) - ignored_cdf()(grid)).max() >= 3 * band   # the test would fail if the prior were ignored
    a = trace[-1].cpu().numpy().astype(np.float64)    # independent chains: the last rows are an i.i.d. posterior sample
    for i in range(2):
        ks = sst.kstest(a[:, i], cdf).statistic
        assert ks < band, (name, i, ks)


RUNS = {
    "global": lambda g, model, lp, gp, n, th0, **kw: g.GlobalMCMC(model, n, th0, None, gp, None, 0.5, lp, **kw),
    "glmcmc": lambda g, model, lp, gp, n, th0, **kw: g.GLMCMC(model, n, th0, None, lp, None, 0.5, gp, 5, **kw),
    "glmala": lambda g, model, lp, gp, n, th0, **kw: g.GLMALA(model, n, th0, None, 0.15, 10, None, 0.5, gp, 5, **kw),
    "aglmcmc": lambda g, model, lp, gp, n, th0, **kw: g.AGLMCMC(model, n, th0, None, lp, gp, None, 0.9, 100, 5, 0.8, 0.2, **kw),
    "aglmcmc_pooled": lambda g, model, lp, gp, n, th0, **kw: g.AGLMCMC(model, n, th0, None, lp, gp, None, 0.9, 50, 5, 0.8, 0.2,
                                                                       pooled=True, kde_train=20000, **kw),
    "glmcmc_nf": lambda g, model, lp, gp, n, th0, **kw: g.GLMCMC_NF(model, n, th0, None, lp, None, 0.5, 50, 5, None, 0, **kw),
}
CASES = [(s, p) for s in ("global", "glmcmc", "glmala") for p in ("uniform", "gamma", "mix")] + \
        [(s, p) for s in ("aglmcmc", "aglmcmc_pooled") for p in ("uniform", "gamma")] + [("glmcmc_nf", "uniform")]


@pytest.mark.parametrize("sampler,name", CASES)
def test_posterior_and_support(eng, sampler, name):
    """KS of the final states against the exact marginal within the band of the sampler's existing tests, and every
    trace row (AGLMCMC: across ~25 adaptations) inside the prior's support"""
    g, model, lp, gp = setup(prior=priors()[name])
    band = 0.05 if sampler.startswith("aglmcmc") or sampler == "glmcmc_nf" else 0.03
    chains = 4096 if sampler.startswith("aglmcmc") else 8192
    # a start in the bulk of the posterior and 8,000 steps (16,000 for the bimodal mixture posterior): with the ABC kernel at
    # eps = 0.05 about 1 % of the proposals are accepted, and a chain holding a lucky simulation stays put for long
    grid = np.linspace(0.0, 4.0, 4001)
    start = float(grid[np.searchsorted(exact_cdf(name)(grid), 0.5)])
    steps = 16001 if name == "mix" else 8001
    trace = RUNS[sampler](g, model, lp, gp, steps, torch.tensor([start, start]), num_chains=chains, seed=11, trace="time")
    check_support(name, trace)
    check_coverage(name, trace, band)


@pytest.mark.parametrize("sampler", ["global", "glmcmc", "glmala", "aglmcmc"])
def test_chain_started_outside_the_box_stays_in_it(eng, sampler):
    g, model, lp, gp = setup(prior=priors()["uniform"])
    tr = RUNS[sampler](g, model, lp, gp, 801, torch.zeros(2), num_chains=1024, seed=5, trace="chain")
    inside = ((tr >= LO) & (tr <= HI)).all(dim=2)            # [C, rows]
    assert not bool(inside[:, 0].any())
    entered = inside.float().cummax(dim=1).values.bool()     # at or after the first accepted move
    assert bool(entered[:, -1].float().mean() > 0.99)
    assert torch.equal(inside, entered)


def dev_state(sampler, C, seed=1):
    theta = torch.full((C, 2), M, device="cuda")
    y = (torch.randn(C, 2, generator=torch.Generator().manual_seed(seed)) * 0.2236 + M).cuda()
    kw = dict(K=5)
    if sampler == "isir":
        aux = torch.zeros(C, abi.AUX_SLOTS, device="cuda")
        aux[:, abi.AUX_LOCAL] = 1.0
        kw["aux"] = aux
    elif sampler == "mala":
        aux, s64 = fresh_mala_state(C)
        kw.update(aux=torch.from_numpy(aux).cuda(), state64=torch.from_numpy(s64).cuda(), num_grad=10, tau=0.15)
    return theta, y, kw


def run_dev(eng, sampler, C, T, cut=None, seed=7):
    """chain-major trace of T steps, in one launch or two (the second continues at step_base = cut)"""
    theta, y, kw = dev_state(sampler, C)
    trace = torch.full((C, T + 1, 2), SENTINEL, device="cuda")
    if cut is None:
        eng.run(sampler, theta=theta, y=y, n_steps=T, gf=0.5, seed=seed, trace=trace, **kw)
    else:
        eng.run(sampler, theta=theta, y=y, n_steps=cut, gf=0.5, seed=seed, trace=trace, trace_rows=T + 1, **kw)
        eng.run(sampler, theta=theta, y=y, n_steps=T - cut, step_base=cut, gf=0.5, seed=seed, trace=trace, trace_rows=T + 1,
                write_row0=False, **kw)
    torch.cuda.synchronize()
    return trace, theta, y


def prior_set(eng, pod):
    return eng.lib.glabc_model_prior_set(eng.ctx.handle, None if pod is None else C.byref(pod), C.sizeof(abi.DistPOD))


@pytest.mark.parametrize("sampler", ["global", "isir", "mala"])
def test_gaussian_prior_set_and_model_reset_are_bit_identical(eng, sampler):
    """a DiagGaussian given to glabc_model_prior_set == the same prior in the model POD; glabc_model_set after a Uniform prior
    == a fresh context; NULL restores the model's DiagGaussian"""
    import glabc_b200 as g
    from glabc_b200.engine import Engine
    fresh = Engine()
    setup(fresh)
    want = run_dev(fresh, sampler, 512, 200)
    setup(eng)
    assert prior_set(eng, g.DiagGaussian(2, torch.zeros(2), torch.zeros(2)).lower()) == abi.OK
    assert all(torch.equal(a, b) for a, b in zip(run_dev(eng, sampler, 512, 200), want))
    setup(eng, prior=priors()["uniform"])
    assert not torch.equal(run_dev(eng, sampler, 512, 200)[0], want[0])
    setup(eng)
    assert all(torch.equal(a, b) for a, b in zip(run_dev(eng, sampler, 512, 200), want))
    setup(eng, prior=priors()["uniform"])
    assert prior_set(eng, None) == abi.OK
    assert all(torch.equal(a, b) for a, b in zip(run_dev(eng, sampler, 512, 200), want))
    # a DiagGaussian other than the POD's changes the run; NULL goes back to the POD's
    assert prior_set(eng, g.DiagGaussian(2, torch.tensor([1.0, 1.0]), torch.zeros(2)).lower()) == abi.OK
    assert not torch.equal(run_dev(eng, sampler, 512, 200)[0], want[0])
    assert prior_set(eng, None) == abi.OK
    assert all(torch.equal(a, b) for a, b in zip(run_dev(eng, sampler, 512, 200), want))


@pytest.mark.parametrize("sampler", ["global", "isir", "mala"])
def test_two_launches_equal_one(eng, sampler):
    setup(eng, prior=priors()["uniform"])
    one = run_dev(eng, sampler, 1000, 300)
    two = run_dev(eng, sampler, 1000, 300, cut=113)
    assert all(torch.equal(a, b) for a, b in zip(one, two))
    check_support("uniform", one[0])


@pytest.mark.parametrize("sampler", ["global", "isir"])
def test_host_entry_equals_device_entry(eng, sampler):
    """with a non-Gaussian prior the host entry takes the dense transport (the event writer lives in the tuned kernels)"""
    setup(eng, prior=priors()["uniform"])
    C, T = 512, 600
    want, th_d, y_d = run_dev(eng, sampler, C, T)
    theta, y, kw = dev_state(sampler, C)
    kw = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in kw.items()}
    host = torch.full((C, T + 1, 2), SENTINEL)
    hth, hy = theta.cpu(), y.cpu()
    eng.run_host(sampler, theta=hth, y=hy, n_steps=T, gf=0.5, seed=7, trace=host, trace_layout=abi.TRACE_CHAIN_MAJOR, **kw)
    assert torch.equal(host, want.cpu()) and torch.equal(hth, th_d.cpu()) and torch.equal(hy, y_d.cpu())


@pytest.mark.parametrize("which", ["global", "glmala"])
def test_checkpoint_resume_continues_bit_identically(tmp_path, which):
    g, model, lp, gp = setup(prior=priors()["gamma"])
    kw = dict(num_chains=300, seed=17, chain_id_base=5, trace="time")
    run = lambda n, **extra: RUNS[which](g, model, lp, gp, n, torch.tensor([M, M]), **kw, **extra)   # noqa: E731
    full = run(301)
    ck = str(tmp_path / "ck.pt")
    head = run(151, checkpoint=ck)
    tail = run(301, resume=ck)
    assert torch.equal(torch.cat([head, tail]), full)
    check_support("gamma", full)


def expect_refusal(eng, status, fn):
    with pytest.raises(abi.GlabcError) as e:
        fn()
    assert e.value.status == status


@pytest.mark.parametrize("sampler", ["global", "isir", "mala", "aglmcmc"])
def test_strict_replay_and_dumps_are_refused_before_any_launch(eng, sampler):
    setup(eng, prior=priors()["uniform"])
    Cn, T = 64, 20
    theta, y, kw = dev_state(sampler, Cn)
    theta.fill_(SENTINEL)
    y.fill_(SENTINEL)
    trace = torch.full((Cn, T + 1, 2), SENTINEL, device="cuda")
    tape = torch.zeros(T * 64 * Cn, device="cuda")
    tape64 = torch.zeros(T * 64 * Cn, dtype=torch.float64, device="cuda")
    if sampler == "aglmcmc":
        kw["ag"] = eng.aglmcmc_params(step_size=4, alpha=0.8, hat_eps_T=0.2)
    run = lambda **extra: eng.run(sampler, theta=theta, y=y, n_steps=T, gf=0.5, seed=1, trace=trace, **{**kw, **extra})  # noqa: E731
    cases = [dict(arith=abi.ARITH_STRICT), dict(rng_mode=abi.RNG_REPLAY, tape32=tape, tape64=tape64, tape_grad0=tape)]
    if sampler != "aglmcmc":
        cases.append(dict(tape_dump=tape, tape64_dump=tape64, tape_grad0_dump=tape))
    else:
        rec = torch.zeros(4, abi.AG_REC_SLOTS, Cn, device="cuda")
        cases.append(dict(ag=eng.aglmcmc_params(step_size=4, alpha=0.8, hat_eps_T=0.2, ad_rec=rec)))
    for extra in cases:
        expect_refusal(eng, abi.ERR_UNSUPPORTED, lambda: run(**extra))
    if sampler != "aglmcmc":
        host = torch.full((Cn, T + 1, 2), SENTINEL)
        hkw = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in kw.items()}
        ht, hy = torch.full((Cn, 2), SENTINEL), torch.full((Cn, 2), SENTINEL)
        expect_refusal(eng, abi.ERR_UNSUPPORTED, lambda: eng.run_host(sampler, theta=ht, y=hy, n_steps=T, gf=0.5, trace=host,
                                                                    trace_layout=abi.TRACE_CHAIN_MAJOR, arith=abi.ARITH_STRICT, **hkw))
        assert bool((host == SENTINEL).all() and (ht == SENTINEL).all() and (hy == SENTINEL).all())
    torch.cuda.synchronize()
    for t in (theta, y, trace):
        assert bool((t == SENTINEL).all())


def test_bad_priors_are_refused(eng):
    import glabc_b200 as g
    from glabc_b200.engine import Engine
    lone = Engine()   # a context without a model
    assert prior_set(lone, priors()["uniform"].lower()) == abi.ERR_INVALID
    setup(eng)
    assert prior_set(eng, g.Uniform(3, torch.zeros(3), torch.ones(3)).lower()) == abi.ERR_INVALID
    assert prior_set(eng, g.Uniform(2, torch.ones(2), torch.zeros(2)).lower()) == abi.ERR_INVALID
    assert prior_set(eng, g.Gamma(torch.tensor([0.0, 1.0]), torch.tensor([1.0, 1.0])).lower()) == abi.ERR_INVALID
    assert prior_set(eng, g.GaussianMixture(2, 2, loc=MIX_LOC, scale=[[0.3, -0.3]] * 2).lower()) == abi.ERR_INVALID
    # none of these bound a prior: the run is the model's own
    want = run_dev(eng, "global", 256, 50)
    setup(eng)
    assert all(torch.equal(a, b) for a, b in zip(run_dev(eng, "global", 256, 50), want))
