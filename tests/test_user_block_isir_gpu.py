"""Block iSIR for run-time compiled user models on the GPU: GLMCMC-NFs (one shared RealNVP) and pooled AGLMCMC (one shared
KernelDensity) with a `models.UserModel` (csrc/user_model.cu: glabc_k_block_isir_user, glabc_k_block_weights_user).
- the block weights equal the plugin methods' exp(prior + log K - log q), and the simulator's draws are N(0, 1), uncorrelated;
- the README model as a user model follows the closed-form ABC posterior and the move rates of the built-in kernels;
- training, pooled adaptation, a box prior, a Uniform local proposal, checkpoint / resume and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_user_model import QUANTILE_SRC
from test_user_model_proposals import GAUSS_SRC

pytestmark = pytest.mark.gpu

POST = (1.42518, np.sqrt(0.049881))    # SURVEY.md App. D: |theta_i| of the README model ~ N(1.42518, 0.049881)


def _objects():
    import glabc_b200 as g
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    from glabc_b200.models import mixture_user_model
    return g, mixture_user_model(0.05), lp, ip


def _ks_abs(last, tol):
    from scipy import stats as sst
    a = last.abs().double().cpu().numpy()
    for i in range(a.shape[1]):
        s = sst.kstest(a[:, i], sst.norm(*POST).cdf).statistic
        assert s < tol, (i, s)


def _rates(st):
    acc_g = float(st.accepted_global.sum() / st.global_steps.sum())
    acc_l = float(st.accepted_local.sum() / (st.steps - st.global_steps).sum())
    return acc_g, acc_l, float(st.esjd().mean())


# ---------------------------------------------------------------------------------------------
# 1. block weights
# ---------------------------------------------------------------------------------------------
def test_block_weights_match_the_plugin_methods():
    from scipy import stats as sst
    from glabc_b200 import _abi as abi
    from glabc_b200.block_isir import Block
    from glabc_b200.engine import get_engine
    g, um, lp, _ = _objects()
    eng = get_engine()
    eng.bind_proposal(abi.SLOT_LOCAL, lp)
    c, K, S = 512, 5, 40
    blk = Block(c, K, S, 2, 2, eng.device)
    gen = torch.Generator(device="cuda").manual_seed(0)
    sign = torch.where(torch.rand(c, K * S, 2, device="cuda", generator=gen) < 0.5, -1.0, 1.0)
    blk.theta.copy_(sign * (1.42 + 0.15 * torch.randn(c, K * S, 2, device="cuda", generator=gen)))
    lq = -1.8378771 - 0.5 * (blk.theta ** 2).sum(-1) + 0.3 * torch.randn(c, K * S, device="cuda", generator=gen)
    lq[::7, 3] = float("nan")
    blk.lq.copy_(lq)
    theta, y = torch.zeros(c, 2, device="cuda"), torch.zeros(c, 2, device="cuda")

    def weights(rnd):
        eng.run_user(um, sampler="block_weights", theta=theta, y=y, n_steps=0, gf=0.5, seed=11, K=K, blk=blk.pod, round=rnd,
                     trace_layout=abi.TRACE_NONE)
        torch.cuda.synchronize()
        return blk.w.clone(), blk.x.clone()

    w0, x0 = weights(0)
    th = blk.theta.reshape(-1, 2)
    ref = torch.exp(um.prior_log_prob(th) + um.calculate_log_kernel(x0.reshape(-1, 2)) - blk.lq.reshape(-1)).reshape(c, -1)
    nan = torch.isnan(blk.lq)
    assert bool((w0[nan] == 0).all()) and bool(torch.isfinite(w0).all())
    big = ~nan & (ref > 1e-30)
    rel = ((w0 - ref).abs() / ref)[big]
    assert float(rel.max()) <= 1e-6, float(rel.max())
    assert float(w0[~nan & ~big].abs().max()) < 1e-30
    assert int(big.sum()) > 0.8 * c * K * S              # most candidates are near the modes: a weight above 1e-30
    # the simulator's draws: y = |theta| + sqrt(0.05) N(0, 1), independent across candidates, chains and refill rounds
    e0 = (x0 - blk.theta.abs()) / 0.05 ** 0.5
    assert sst.kstest(e0.reshape(-1).double().cpu().numpy(), "norm").statistic < 0.01
    corr = lambda a, b: float(torch.corrcoef(torch.stack([a.reshape(-1), b.reshape(-1)]))[0, 1])  # noqa: E731
    w1, x1 = weights(1)
    e1 = (x1 - blk.theta.abs()) / 0.05 ** 0.5
    for a, b in ((e0[:, :-1], e0[:, 1:]), (e0[:-1], e0[1:]), (e0, e1), (e0[..., 0], e0[..., 1])):
        assert abs(corr(a, b)) < 0.01, corr(a, b)
    w2, x2 = weights(0)
    assert torch.equal(w2, w0) and torch.equal(x2, x0)


# ---------------------------------------------------------------------------------------------
# 2. - 4. GLMCMC-NFs: law, training, against the built-in family
# ---------------------------------------------------------------------------------------------
def test_user_glmcmc_nf_equals_glmcmc_semantics():
    """untrained flow (proposal N(0, I) exactly), no training: iSIR with pre-generated N(0, I) candidates, as for the built-in
    model (tests/test_flow_gpu.py::test_block_isir_equals_glmcmc_semantics)"""
    g, um, lp, _ = _objects()
    out, st = g.GLMCMC_NF(um, 3001, torch.zeros(2), None, lp, None, 0.9, 50, 5, None, 0, num_chains=8192, seed=3, trace="none",
                          return_stats=True)
    assert out is None and bool((st.steps == 3000).all())
    move, e = float(st.move_rate.mean()), float(st.esjd().mean())
    assert 0.0075 < move < 0.0110, move
    assert 0.024 < e < 0.035, e
    out2 = g.GLMCMC_NF(um, 2001, torch.zeros(2), None, lp, None, 0.9, 50, 5, None, 0, num_chains=8192, seed=4, trace="time")
    _ks_abs(out2[-1], 0.03)
    # chains pause / resume individually (lq refresh after local accepts): every row of every chain was written
    assert torch.isfinite(out2).all() and torch.equal(out2[0], torch.zeros(8192, 2, device=out2.device))


def test_user_glmcmc_nf_training_improves_the_proposal():
    g, um, lp, _ = _objects()
    torch.manual_seed(1234)
    res, st, flow, losses = g.GLMCMC_NF(um, 4001, torch.zeros(2), None, lp, None, 0.5, 25, 5, None, 50, num_chains=2048, seed=1,
                                        trace="time", return_stats=True, return_flow=True, lr=3e-3)
    assert len(losses) == 50 and np.mean(losses[-10:]) < np.mean(losses[:5]) - 0.3, losses
    th, _ = flow.fused_sample_from(torch.randn(50000, 2, device="cuda"))
    near_mode = ((th.abs() - 1.425).abs() < 0.7).all(1).float().mean()
    assert float(near_mode) > 0.25, float(near_mode)            # N(0, I) puts ~9 % there
    _ks_abs(res[-1], 0.05)
    assert float(st.move_rate.mean()) > 0.012                   # the untrained proposal moves 0.9 % of the time


def test_user_block_samplers_match_the_builtin_family():
    """same seeds, same initial state: the README model as CUDA source against the built-in Mixture_set kernels, in
    GLMCMC-NFs and pooled AGLMCMC.  The simulator draws differ (other Philox slots), so the runs agree in law only."""
    g, um, lp, ip = _objects()
    builtin = g.Mixture_set(0.05)
    y0 = torch.randn(8192, 2, generator=torch.Generator().manual_seed(1)) * 0.2236
    got = {}
    for name, model in (("user", um), ("builtin", builtin)):
        _, st = g.GLMCMC_NF(model, 2001, torch.zeros(2), y0, lp, None, 0.5, 50, 5, None, 0, num_chains=8192, seed=7,
                            trace="none", return_stats=True)
        _, st2 = g.AGLMCMC(model, 1001, torch.zeros(2), y0[:2048], lp, ip, None, 0.9, 50, 5, 0.8, 0.2, num_chains=2048, seed=7,
                           trace="none", return_stats=True, pooled=True, kde_train=20000)
        got[name] = (_rates(st), _rates(st2))
    print("\nuser / built-in (global accept, local accept, ESJD):", got)
    for (u, b) in zip(got["user"], got["builtin"]):
        assert abs(u[0] / b[0] - 1) < 0.06 and abs(u[1] / b[1] - 1) < 0.06, (u, b)
        assert abs(u[2] / b[2] - 1) < 0.10, (u, b)


# ---------------------------------------------------------------------------------------------
# 5. pooled AGLMCMC
# ---------------------------------------------------------------------------------------------
def test_user_aglmcmc_pooled_kde_posterior():
    g, um, lp, ip = _objects()
    Cn = 2048
    out, st, prop = g.AGLMCMC(um, 1501, torch.zeros(2), None, lp, ip, None, 0.9, 50, 5, 0.8, 0.2, num_chains=Cn, seed=3,
                              trace="none", return_stats=True, pooled=True, kde_train=20000, return_proposal=True)
    assert out is None and len(prop.history) >= 10
    eps_hist = [h[0] for h in prop.history]
    assert all(a >= b for a, b in zip(eps_hist, eps_hist[1:])) and eps_hist[-1] == pytest.approx(0.2)
    assert prop.history[-1][1] > 15000
    assert float(st.accepted_global.sum() / st.global_steps.sum()) > 0.03
    out2 = g.AGLMCMC(um, 1001, torch.zeros(2), None, lp, ip, None, 0.9, 50, 5, 0.8, 0.2, num_chains=Cn, seed=5, trace="time",
                     pooled=True, kde_train=20000)
    _ks_abs(out2[-1], 0.05)
    quad = ((out2[-1][:, 0] > 0).long() * 2 + (out2[-1][:, 1] > 0).long()).bincount(minlength=4).cpu().numpy() / Cn
    assert np.abs(quad - 0.25).max() < 0.05


def test_user_aglmcmc_pooled_box_prior():
    """a 3-parameter model outside the family with a Uniform-box prior (-inf outside): KDE candidates outside the box get
    log q = +inf (the prior floor of PooledKDEProposal.fill, evaluated by the model's compiled prior), so no chain leaves it"""
    import glabc_b200 as g
    lp = g.DiagGaussian(3, torch.zeros(1, 3), torch.log(torch.tensor([0.2, 0.2, 0.2])))
    ip = g.DiagGaussian(3, torch.tensor([3.0, 1.0, 2.0]), torch.log(torch.tensor([1.0, 0.5, 1.0])))
    obs = [3.0 + 1.0 * z for z in (-1.2, -0.5, 0.0, 0.6, 1.4)]
    qm = g.UserModel(QUANTILE_SRC, theta_dim=3, y_dim=5, n_noise=5, epsilon=0.5, params=obs)
    out, st, prop = g.AGLMCMC(qm, 801, torch.tensor([3.0, 1.0, 2.0]), torch.tensor(obs), lp, ip, None, 0.5, 20, 5, 0.8, 0.5,
                              num_chains=1024, seed=2, trace="time", return_stats=True, pooled=True, kde_train=5000,
                              return_proposal=True)
    assert out.shape == (801, 1024, 3) and bool(torch.isfinite(out).all())
    assert bool(((out > 0) & (out < 10)).all())
    assert len(prop.history) >= 2 and 0.01 < float(st.move_rate.mean()) < 0.9


# ---------------------------------------------------------------------------------------------
# 6. local proposals
# ---------------------------------------------------------------------------------------------
def test_uniform_local_proposal_in_the_block_step():
    """identity-link Gaussian user model (closed-form ABC posterior N(POST_MU, POST_SD^2) per coordinate), a centred Uniform
    Local_Proposal compiled into the block step"""
    from scipy import stats as sst
    import glabc_b200 as g
    sig, mu0, yo, eps = 0.3, 1.5, 2.0, 0.3
    prec = 1.0 + 1.0 / (sig ** 2 + eps ** 2)
    post_mu, post_sd = (mu0 + yo / (sig ** 2 + eps ** 2)) / prec, prec ** -0.5
    um = g.UserModel(GAUSS_SRC, theta_dim=2, y_dim=2, n_noise=2, epsilon=eps, params=[sig, mu0, yo, yo])
    lu = g.Uniform(2, torch.full((2,), -0.5), torch.full((2,), 0.5))
    out, st = g.GLMCMC_NF(um, 1501, torch.full((2,), 2.0), None, lu, None, 0.5, 50, 5, None, 0, num_chains=4096, seed=6,
                          trace="time", return_stats=True)
    a = out[-1].double().cpu().numpy()
    assert np.isfinite(a).all() and float(st.accepted_local.sum()) > 0
    for i in range(2):
        s = sst.kstest(a[:, i], sst.norm(post_mu, post_sd).cdf).statistic
        assert s < 0.03, (i, s)


# ---------------------------------------------------------------------------------------------
# 7. checkpoint / resume
# ---------------------------------------------------------------------------------------------
def test_user_glmcmc_nf_checkpoint_resume(tmp_path):
    g, um, lp, _ = _objects()
    C_, T, T1 = 512, 601, 257
    kw = dict(num_chains=C_, seed=5, trace="time", return_stats=True, return_flow=True, lr=2e-3)
    run = lambda n, gf, model=um, **k: g.GLMCMC_NF(model, n, torch.zeros(2), None, lp, None, gf, 20, 5, None, 50, **kw, **k)  # noqa: E731
    torch.manual_seed(3)
    full, st_full, flow_full, loss_full = run(T, 1.0)
    ck = tmp_path / "nf.pt"
    torch.manual_seed(3)
    first, _, _, loss_1 = run(T1, 1.0, checkpoint=str(ck))
    torch.manual_seed(99)
    rest, st_rest, flow_rest, loss_2 = run(T, 1.0, resume=str(ck))
    assert len(loss_1) >= 3 and len(loss_2) > len(loss_1)
    assert torch.equal(first, full[:T1]) and torch.equal(rest, full[T1:])
    assert loss_2 == loss_full
    assert torch.equal(flow_rest.flat_params(), flow_full.flat_params())
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4])
    ck2 = tmp_path / "nf2.pt"
    torch.manual_seed(3)
    run(T1, 0.6, checkpoint=str(ck2))
    a, st_a, flow_a, loss_a = run(T, 0.6, resume=str(ck2))
    torch.manual_seed(12345)
    b, st_b, flow_b, loss_b = run(T, 0.6, resume=str(ck2))
    assert torch.equal(a, b) and loss_a == loss_b and torch.equal(flow_a.flat_params(), flow_b.flat_params())
    assert torch.equal(st_a.raw, st_b.raw) and float(st_a.move_rate.mean()) > 0.005
    # refusals: another user model, a built-in checkpoint, and a user checkpoint resumed by a built-in run
    with pytest.raises(ValueError, match="another model"):
        run(T, 1.0, model=g.models.mixture_user_model(0.06), resume=str(ck))
    ck3 = tmp_path / "nf_builtin.pt"
    run(T1, 1.0, model=g.Mixture_set(0.05), checkpoint=str(ck3))
    with pytest.raises(ValueError, match="another model"):
        run(T, 1.0, resume=str(ck3))
    with pytest.raises(ValueError, match="another model"):
        run(T, 1.0, model=g.Mixture_set(0.05), resume=str(ck))


def test_user_pooled_checkpoint_resume(tmp_path):
    g, um, lp, ip = _objects()
    C_, T, T1 = 400, 301, 137
    run = lambda n, model=um, **kw: g.AGLMCMC(model, n, torch.zeros(2), None, lp, ip, None, 1.0, 20, 5, 0.8, 0.2, num_chains=C_,  # noqa: E731
                                              seed=4, trace="time", return_stats=True, return_proposal=True, pooled=True,
                                              kde_train=4000, **kw)
    full, st_full, prop_full = run(T)
    ck = tmp_path / "agp.pt"
    first, _, prop_1 = run(T1, checkpoint=str(ck))
    rest, st_rest, prop_rest = run(T, resume=str(ck))
    assert len(prop_1.history) >= 2 and len(prop_rest.history) > len(prop_1.history)
    assert torch.equal(first, full[:T1]) and torch.equal(rest, full[T1:])
    assert prop_rest.history == prop_full.history
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4])
    with pytest.raises(ValueError, match="another model"):
        run(T, model=g.Mixture_set(0.05), resume=str(ck))


# ---------------------------------------------------------------------------------------------
# 8. refusals
# ---------------------------------------------------------------------------------------------
def test_sampler_refusals():
    import glabc_b200 as g
    _, um, lp, ip = _objects()
    wide = g.UserModel(GAUSS_SRC, theta_dim=3, y_dim=3, n_noise=3, epsilon=0.3, params=[0.3, 1.5, 2.0, 2.0, 2.0])
    lp3 = g.DiagGaussian(3, torch.zeros(1, 3), torch.zeros(1, 3))
    with pytest.raises(NotImplementedError, match="theta_dim must be 2"):
        g.GLMCMC_NF(wide, 11, torch.zeros(3), None, lp3, None, 0.5, 5, 5, None, 0, num_chains=4)
    five = g.UserModel(GAUSS_SRC, theta_dim=5, y_dim=5, n_noise=5, epsilon=0.3, params=[0.3, 1.5] + [2.0] * 5)
    lp5 = g.DiagGaussian(5, torch.zeros(1, 5), torch.zeros(1, 5))
    with pytest.raises(NotImplementedError, match="theta_dim <= 4"):
        g.AGLMCMC(five, 11, torch.zeros(5), None, lp5, lp5, None, 0.5, 5, 5, 0.8, 0.2, num_chains=4, pooled=True)
    with pytest.raises(NotImplementedError, match="pooled=True"):
        g.AGLMCMC(um, 11, torch.zeros(2), None, lp, ip, None, 0.5, 5, 5, 0.8, 0.2, num_chains=4)


def test_abi_refusals_launch_nothing():
    from glabc_b200 import _abi as abi
    from glabc_b200.block_isir import Block
    from glabc_b200.engine import Engine
    g, um, lp, _ = _objects()
    eng = Engine(torch.device("cuda", torch.cuda.current_device()))   # a fresh context: no slot bound yet
    c, K, S = 64, 5, 4
    blk = Block(c, K, S, 2, 2, eng.device)
    for t in (blk.theta, blk.x, blk.w, blk.lq, blk.lq_cur):
        t.fill_(0.25)
    theta, y = torch.full((c, 2), 0.5, device="cuda"), torch.full((c, 2), 0.5, device="cuda")
    stats = torch.zeros(c, abi.nstats(2), device="cuda")
    watched = (theta, y, stats, blk.theta, blk.x, blk.w, blk.lq, blk.kk, blk.pending, blk.next_step, blk.lq_cur, blk.lq_valid)
    before = [t.clone() for t in watched]
    upod = um.user_pod()

    def call(weights, n_chains=c, k=K, arith=abi.ARITH_FAST, rng=abi.RNG_NATIVE, pod=None, model=upod):
        r = abi.RunPOD(n_chains=n_chains, n_steps=10, step_base=0, seed=1, global_frequency=0.5, rng_mode=rng, arith_mode=arith,
                       trace_layout=abi.TRACE_NONE, n_candidates=k, trace_chains=c, theta=theta.data_ptr(), y=y.data_ptr(),
                       stats=stats.data_ptr(), stream=eng._stream())
        pod = blk.pod if pod is None else pod
        if weights:
            return eng.lib.glabc_block_weights_user(eng.ctx.handle, C.byref(r), C.byref(pod), 0, C.byref(model))
        return eng.lib.glabc_run_block_isir_user(eng.ctx.handle, C.byref(r), C.byref(pod), C.byref(model))

    def pod_with(**kw):
        f = {name: getattr(blk.pod, name) for name, _ in abi.BlockIsirPOD._fields_}
        f.update(kw)
        return abi.BlockIsirPOD(**f)

    for weights in (False, True):
        assert call(weights) == abi.ERR_INVALID                                   # LOCAL slot unbound
    eng.bind_proposal(abi.SLOT_LOCAL, g.DiagGaussian(3, torch.zeros(1, 3), torch.zeros(1, 3)))
    for weights in (False, True):
        assert call(weights) == abi.ERR_INVALID                                   # LOCAL dim != theta_dim
    eng.bind_proposal(abi.SLOT_LOCAL, lp)
    bad_model = um.user_pod()
    bad_model.epsilon = 0.0
    for weights in (False, True):
        assert call(weights, pod=pod_with(blk_w=None)) == abi.ERR_INVALID         # null block buffer
        assert call(weights, pod=pod_with(block=K * S + 1)) == abi.ERR_INVALID    # block != K S
        assert call(weights, k=0) == abi.ERR_INVALID and call(weights, k=abi.MAX_K + 1) == abi.ERR_INVALID
        assert call(weights, model=bad_model) == abi.ERR_INVALID                  # invalid model
        assert call(weights, arith=abi.ARITH_STRICT) == abi.ERR_UNSUPPORTED
        assert call(weights, rng=abi.RNG_REPLAY) == abi.ERR_UNSUPPORTED
        assert call(weights, n_chains=0) == abi.OK                               # nothing to do
    torch.cuda.synchronize()
    for a, b in zip(watched, before):
        assert torch.equal(a, b)
    assert call(False) == abi.OK                                                 # the same call, valid, does run
    torch.cuda.synchronize()
    assert float(stats[:, abi.STAT_STEPS].sum()) > 0
