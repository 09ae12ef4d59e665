"""User models with Uniform / Gamma / GaussianMixture proposals and theta_dim up to 8 on the GPU (csrc/user_model.cu).
- posterior: an identity-link Gaussian user model, whose ABC posterior is Gaussian in closed form, is recovered with every
  non-Gaussian global / importance proposal in GlobalMCMC, GLMCMC and GLMALA, and with a centred Uniform local proposal;
- the README Mixture model written as a user model moves like the built-in general kernels on the same proposals;
- support, determinism, theta_dim 6, and the all-DiagGaussian user path against fingerprints taken before the proposal
  kinds became compile-time options."""
import hashlib

import numpy as np
import pytest
import torch

from test_user_model_proposals import GAUSS_SRC

pytestmark = pytest.mark.gpu

# GAUSS_SRC with sigma = 0.3, prior N(1.5, 1), y_obs = 2, epsilon = 0.3: per coordinate the ABC likelihood is
# N(2; theta, sigma^2 + epsilon^2), so the posterior is N(POST_MU, POST_SD^2) in every coordinate
SIG, PRIOR_MU, Y_OBS, EPS = 0.3, 1.5, 2.0, 0.3
_PREC = 1.0 + 1.0 / (SIG ** 2 + EPS ** 2)
POST_MU, POST_SD = (PRIOR_MU + Y_OBS / (SIG ** 2 + EPS ** 2)) / _PREC, _PREC ** -0.5


def _model(d):
    import glabc_b200 as g
    return g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=[SIG, PRIOR_MU] + [Y_OBS] * d)


def _dists(d):
    import glabc_b200 as g
    f = lambda v: torch.full((d,), float(v))  # noqa: E731
    return dict(
        gauss=g.DiagGaussian(d, f(POST_MU), torch.log(f(0.8))),
        uniform=g.Uniform(d, f(-1.0), f(5.0)),
        gamma=g.Gamma(f(8.0), f(4.0)),
        mix=g.GaussianMixture(2, d, loc=[[1.5] * d, [2.5] * d], scale=[[0.7] * d] * 2, weights=[0.4, 0.6]),
        local_gauss=g.DiagGaussian(d, torch.zeros(1, d), torch.log(f(0.3))),
        local_uniform=g.Uniform(d, f(-0.5), f(0.5)),
    )


def _start(cn, d, theta0=2.0, seed=1):
    th = torch.full((1, d), float(theta0))
    y = th + SIG * torch.randn(cn, d, generator=torch.Generator().manual_seed(seed))
    return th, y


def _ks(last, tol):
    from scipy import stats as sst
    a = last.double().cpu().numpy()
    assert np.isfinite(a).all()
    worst = max(sst.kstest(a[:, i], sst.norm(POST_MU, POST_SD).cdf).statistic for i in range(a.shape[1]))
    assert worst < tol, worst


def _last_state(sampler, um, far, local, T, cn, **kw):
    """(final states [C, d], time-major trace [T, C, d]) of C chains started at theta0 with their own simulator draws"""
    import glabc_b200 as g
    th, y = _start(cn, um.theta_dim, kw.pop("theta0", 2.0))
    gf, seed = kw.pop("gf", 0.5), kw.pop("seed", 3)
    if sampler == "global":
        out = g.GlobalMCMC(um, T, th, y, far, None, gf, local, num_chains=cn, seed=seed, trace="time")
    elif sampler == "isir":
        out = g.GLMCMC(um, T, th, y, local, None, gf, far, 5, num_chains=cn, seed=seed, trace="time")
    else:
        out = g.GLMALA(um, T, th, y, 0.3, 50, None, gf, far, 5, num_chains=cn, seed=seed, trace="time")
    return out[-1].clone(), out


POSTERIOR_CASES = [(s, far, "local_gauss") for s in ("global", "isir", "mala") for far in ("uniform", "mix", "gamma")] + \
                  [("global", "gauss", "local_uniform"), ("isir", "gauss", "local_uniform")]


@pytest.mark.parametrize("sampler,far,local", POSTERIOR_CASES)
def test_posterior_with_non_gaussian_proposals(sampler, far, local):
    um, ds = _model(2), _dists(2)
    T = {"global": 2001, "isir": 1001, "mala": 801}[sampler]
    last, out = _last_state(sampler, um, ds[far], ds[local], T, 32768)
    assert bool(torch.isfinite(out).all())
    _ks(last, 0.03 if sampler == "mala" else 0.015)   # GLMALA's noisy synthetic-likelihood gradient: test_user_model.py's band


# the README Mixture model as a user model against the built-in general kernels on the same non-Gaussian proposals;
# the Gamma local proposal gives the reference's biased chain (no q term for a local move) in both
AGREE_CASES = [("global", "uniform", "gamma"), ("isir", "mix", "gamma"), ("isir", "gamma", "uniform"), ("mala", "uniform", None),
               ("mala", "gamma", None)]


@pytest.mark.parametrize("sampler,far,local", AGREE_CASES)
def test_mixture_user_model_moves_like_the_builtin_kernels(sampler, far, local):
    import glabc_b200 as g
    from glabc_b200.models import mixture_user_model
    dists = dict(uniform=g.Uniform(2, torch.full((2,), -3.0), torch.full((2,), 3.0)),
                 gamma=g.Gamma(torch.full((2,), 2.0), torch.full((2,), 4.0)),
                 mix=g.GaussianMixture(2, 2, loc=[[1.4, 1.4], [-1.4, -1.4]], scale=[[0.5, 0.5]] * 2, weights=[0.5, 0.5]))
    loc_dists = dict(gamma=g.Gamma(torch.full((2,), 2.0), torch.full((2,), 10.0)),
                     uniform=g.Uniform(2, torch.full((2,), -0.6), torch.full((2,), 0.6)))
    Cn = 16384
    T = {"global": 3001, "isir": 2001, "mala": 1001}[sampler]
    y0 = torch.randn(Cn, 2, generator=torch.Generator().manual_seed(1)) * 0.2236
    th0 = torch.tensor([1.0, 1.0])
    gf = 0.5
    stats = []
    for model, seed in ((mixture_user_model(), 3), (g.Mixture_set(0.05), 4)):
        if sampler == "global":
            _, st = g.GlobalMCMC(model, T, th0, y0, dists[far], None, gf, loc_dists[local], num_chains=Cn, seed=seed, trace="none",
                                 return_stats=True)
        elif sampler == "isir":
            _, st = g.GLMCMC(model, T, th0, y0, loc_dists[local], None, gf, dists[far], 5, num_chains=Cn, seed=seed, trace="none",
                             return_stats=True)
        else:
            _, st = g.GLMALA(model, T, th0, y0, 0.3, 100, None, gf, dists[far], 5, num_chains=Cn, seed=seed, trace="none",
                             return_stats=True)
        stats.append(st)
    u, b = stats
    ratio = lambda x, y: float(x) / max(float(y), 1e-12)  # noqa: E731
    assert abs(float(u.global_steps.mean()) / (T - 1) - gf) < 0.005
    assert abs(ratio(u.accepted_global.mean(), b.accepted_global.mean()) - 1) < 0.06, (u.accepted_global.mean(), b.accepted_global.mean())
    assert abs(ratio(u.accepted_local.mean(), b.accepted_local.mean()) - 1) < 0.06, (u.accepted_local.mean(), b.accepted_local.mean())
    assert abs(ratio(u.esjd().mean(), b.esjd().mean()) - 1) < 0.1, (u.esjd().mean(), b.esjd().mean())


@pytest.mark.parametrize("sampler", ["isir", "mala"])
def test_state_outside_the_importance_box_waits_for_a_local_move(sampler):
    """log q(theta) = -inf outside a Uniform importance proposal: the current state's weight is +inf, so a global move
    selects nothing and the chain stays until a local (random-walk / MALA) move takes it inside"""
    import glabc_b200 as g
    um = _model(2)
    box = g.Uniform(2, torch.zeros(2), torch.full((2,), 4.0))
    lp = _dists(2)["local_gauss"]
    cn = 4096
    _, out = _last_state(sampler, um, box, lp, 60, cn, gf=1.0, theta0=-1.0)
    assert bool(torch.isfinite(out).all())
    assert bool((out == -1.0).all())                               # global moves only: nobody moves
    last, out = _last_state(sampler, um, box, lp, 1501, cn, gf=0.7, theta0=-1.0)
    assert bool(torch.isfinite(out).all())
    inside = ((last > 0) & (last < 4)).all(1).float().mean()
    assert float(inside) > 0.99
    _ks(last, 0.04)


def _fresh(um, sampler, cn):
    from glabc_b200 import _abi as abi
    d = um.theta_dim
    th, y = _start(cn, d)
    th = th.expand(cn, d).contiguous().cuda()
    y = y[:cn].cuda()
    aux = None
    if sampler != "global":
        aux = torch.zeros(cn, abi.AUX_SLOTS, device="cuda")
        aux[:, abi.AUX_LOCAL] = 1.0
    return th, y, aux


@pytest.mark.parametrize("sampler,far,local", [("global", "mix", "local_uniform"), ("global", "gamma", "gamma"),
                                               ("isir", "uniform", "gamma"), ("mala", "gamma", None)])
def test_chunks_and_shards_give_the_same_chains(sampler, far, local):
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    um, ds = _model(2), _dists(2)
    eng = get_engine()
    far_slot = abi.SLOT_GLOBAL if sampler == "global" else abi.SLOT_IMPORTANCE
    eng.bind_proposal(far_slot, ds[far])
    if local is not None:
        eng.bind_proposal(abi.SLOT_LOCAL, ds[local])
    kw = dict(gf=0.6, seed=9, sampler=sampler, trace_layout=abi.TRACE_TIME_MAJOR)
    if sampler != "global":
        kw["K"] = 4
    if sampler == "mala":
        kw.update(num_grad=33, tau=0.3)
    cn, n = 70, 150
    th, y, aux = _fresh(um, sampler, cn)
    full = eng.run_user(um, theta=th, y=y, aux=aux, n_steps=n, **kw)
    assert bool(torch.isfinite(full).all())
    th2, y2, aux2 = _fresh(um, sampler, cn)
    buf = torch.zeros(n + 1, cn, 2, device="cuda")
    eng.run_user(um, theta=th2, y=y2, aux=aux2, n_steps=60, trace=buf, trace_rows=n + 1, **kw)
    eng.run_user(um, theta=th2, y=y2, aux=aux2, n_steps=n - 60, step_base=60, trace=buf, trace_rows=n + 1, write_row0=False, **kw)
    assert torch.equal(buf, full) and torch.equal(th2, th) and torch.equal(y2, y)
    if aux is not None:
        assert torch.equal(aux2, aux)
    th3, y3, aux3 = _fresh(um, sampler, cn)
    th3, y3 = th3[37:].contiguous(), y3[37:].contiguous()
    aux3 = aux3[37:].contiguous() if aux3 is not None else None
    part = eng.run_user(um, theta=th3, y=y3, aux=aux3, n_steps=n, chain_id_base=37, **kw)
    assert torch.equal(part, full[:, 37:])


def gaussian_user_fingerprints():
    """sha256 of the state and trace of short all-DiagGaussian runs of the Mixture user model in the three user kernels"""
    import glabc_b200 as g
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    from glabc_b200.models import mixture_user_model
    eng = get_engine()
    um = mixture_user_model()
    eng.bind_proposal(abi.SLOT_LOCAL, g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35]))))
    eng.bind_proposal(abi.SLOT_GLOBAL, g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0])))
    eng.bind_proposal(abi.SLOT_IMPORTANCE, g.DiagGaussian(2, torch.tensor([0.5, 0.5]), torch.tensor([0.0, 0.0])))
    out = {}
    for sampler in ("global", "isir", "mala"):
        cn = 1000
        th = torch.zeros(cn, 2, device="cuda")
        y = (torch.randn(cn, 2, generator=torch.Generator().manual_seed(1)) * 0.2236).cuda()
        aux = torch.zeros(cn, abi.AUX_SLOTS, device="cuda")
        aux[:, abi.AUX_LOCAL] = 1.0
        stats = torch.zeros(cn, abi.nstats(2), device="cuda")
        kw = dict(gf=0.6, seed=11, sampler=sampler, trace_layout=abi.TRACE_TIME_MAJOR, stats=stats)
        if sampler != "global":
            kw.update(K=5, aux=aux)
        if sampler == "mala":
            kw.update(num_grad=40, tau=0.3)
        tr = eng.run_user(um, theta=th, y=y, n_steps=300, **kw)
        torch.cuda.synchronize()
        h = hashlib.sha256()
        for t in (tr, th, y, aux, stats):
            h.update(t.cpu().numpy().tobytes())
        out[sampler] = h.hexdigest()
    return out


# taken with the library before the proposal kinds became compile-time options, on an NVIDIA B200 (1000 W power limit)
GAUSSIAN_FINGERPRINTS = {
    "global": "844d5aef1f229659aaa2fcc59c5ff702cf089c1f7de69554ae82d7fe49ef163c",
    "isir": "56b0a91de9db0a53e759ab1ddc9c7841008f41b1b8e47b8a48b4a398804f454a",
    "mala": "2c857318a62ff8692aba9727f12857ffd673e00292c81ce5844fa6d1706b4fec",
}


def test_all_gaussian_user_runs_are_unchanged():
    assert gaussian_user_fingerprints() == GAUSSIAN_FINGERPRINTS


@pytest.mark.parametrize("sampler", ["global", "isir"])
@pytest.mark.parametrize("kind", ["gauss", "uniform"])
def test_theta_dim_6_recovers_its_marginals(sampler, kind):
    import glabc_b200 as g
    um = _model(6)
    if kind == "gauss":
        far = g.DiagGaussian(6, torch.full((6,), POST_MU), torch.log(torch.full((6,), 0.6)))
        local = _dists(6)["local_gauss"]
    else:
        far = g.Uniform(6, torch.full((6,), 0.0), torch.full((6,), 4.0))
        local = g.Uniform(6, torch.full((6,), -0.4), torch.full((6,), 0.4))
    last, out = _last_state(sampler, um, far, local, 2001, 32768)
    assert bool(torch.isfinite(out).all())
    _ks(last, 0.015)


def test_theta_dim_6_limits():
    """GLMALA keeps its theta_dim <= 5 limit; a dim-5 distribution is refused by the built-in paths before any launch and
    the context stays usable"""
    import ctypes as C
    import glabc_b200 as g
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    um, ds = _model(6), _dists(6)
    th, y = _start(64, 6)
    with pytest.raises(abi.GlabcError, match="theta_dim at most 5"):
        g.GLMALA(um, 11, th, y, 0.3, 20, None, 0.5, ds["uniform"], 5, num_chains=64, seed=1, trace="none")
    eng = get_engine()
    five = g.Uniform(5, torch.zeros(5), torch.ones(5))
    with pytest.raises(abi.GlabcError) as e:
        g.GlobalMCMC(g.Mixture_set(0.05), 11, torch.zeros(2), torch.zeros(1, 2), five, None, 0.5, five, num_chains=64, seed=1, trace="none")
    assert e.value.status == abi.ERR_INVALID
    eng.bind_proposal(abi.SLOT_LOCAL, five)
    with pytest.raises(abi.GlabcError, match="dim 1..4") as e:
        eng.dist_sample(abi.SLOT_LOCAL, 16, 5)
    assert e.value.status == abi.ERR_UNSUPPORTED
    with pytest.raises(abi.GlabcError, match="dim 1..4") as e:
        eng.dist_log_prob(abi.SLOT_LOCAL, torch.zeros(16, 5, device="cuda"))
    assert e.value.status == abi.ERR_UNSUPPORTED
    eng.bind_model(g.Mixture_set(0.05))
    pod = five.lower()
    assert eng.lib.glabc_model_prior_set(eng.ctx.handle, C.byref(pod), C.sizeof(pod)) == abi.ERR_UNSUPPORTED
    eng.bind_proposal(abi.SLOT_LOCAL, g.Uniform(2, torch.zeros(2), torch.ones(2)))
    z, lp = eng.dist_sample(abi.SLOT_LOCAL, 16, 2)
    torch.cuda.synchronize()
    assert bool(((z >= 0) & (z <= 1)).all()) and bool(torch.isfinite(lp).all())
