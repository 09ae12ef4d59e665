"""Batched user models on the GPU: many observed datasets in one run (UserModel with params [G, n_params],
chains_per_dataset=m, the -DGLABC_BATCHED kernels).  A batched run equals the G one-dataset runs bit for bit, every dataset
gets its own closed-form posterior, simulation-based calibration over 1024 datasets is uniform, checkpoint / resume, and
the Python and C-ABI refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_user_model_proposals import GAUSS_SRC

pytestmark = pytest.mark.gpu

P0, EPS = 0.3, 0.3      # simulator noise sd and ABC kernel width of the GAUSS_SRC models below


def _g():
    import glabc_b200 as g
    return g


def _table(G, d, seed):
    """params rows [p0, prior mean, y_obs (d)] of G datasets"""
    gen = torch.Generator().manual_seed(seed)
    mu = torch.randn(G, 1, generator=gen) * 0.5
    y_obs = torch.randn(G, d, generator=gen) * 1.5
    return torch.cat([torch.full((G, 1), P0), mu, y_obs], dim=1)


def _props(d):
    g = _g()
    lp = g.DiagGaussian(d, torch.zeros(1, d), torch.log(torch.full((d,), 0.4)))
    gp = g.DiagGaussian(d, torch.zeros(d), torch.log(torch.full((d,), 2.0)))
    return lp, gp


def _run(sampler, um, T, theta0, y0, d=2, **kw):
    g = _g()
    lp, gp = _props(d)
    if sampler == "global":
        return g.GlobalMCMC(um, T, theta0, y0, gp, None, 0.4, lp, **kw)
    if sampler == "isir":
        return g.GLMCMC(um, T, theta0, y0, lp, None, 0.5, gp, 4, **kw)
    return g.GLMALA(um, T, theta0, y0, 0.3, 8, None, 0.5, gp, 4, **kw)


def _ck(path):
    return torch.load(path, map_location="cpu", weights_only=True)


SAMPLERS = ["global", "isir", "mala"]


@pytest.mark.parametrize("sampler", SAMPLERS)
@pytest.mark.parametrize("m", [7, 33, 64])
def test_batched_run_equals_the_one_dataset_runs(sampler, m, tmp_path):
    """chain g of one batched launch = chain g of the launch of dataset g // m alone (same seed, same global ids), with
    Initial_y=None; m = 7 and 33 put several datasets in one warp (GLMALA serves each chain's gradient with its own row)"""
    g = _g()
    G, d, T, s = 8, 2, 60, 17
    um = g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=_table(G, d, 1))
    th0 = torch.randn(G, d, generator=torch.Generator().manual_seed(2))        # one row per dataset
    kw = dict(seed=s, trace="chain", return_stats=True)
    tr, st = _run(sampler, um, T, th0, None, chains_per_dataset=m, checkpoint=str(tmp_path / "b.pt"), **kw)
    assert tr.shape == (G * m, T, d)
    b = _ck(tmp_path / "b.pt")
    assert b["chains_per_dataset"] == m
    for gi in range(G):
        one = um.dataset(gi)
        t1, s1 = _run(sampler, one, T, th0[gi], None, num_chains=m, chain_id_base=gi * m, checkpoint=str(tmp_path / "u.pt"), **kw)
        u = _ck(tmp_path / "u.pt")
        rows = slice(gi * m, (gi + 1) * m)
        assert torch.equal(tr.view(G, m, T, d)[gi], t1), gi
        assert torch.equal(st.raw[rows], s1.raw), gi
        for key in ("theta", "y", "aux"):
            assert (b[key] is None and u[key] is None) or torch.equal(b[key][rows], u[key]), (gi, key)
    # two shards cut inside a dataset = the unsplit run
    cut = 3 * m + 2
    lo, slo = _run(sampler, um, T, th0, None, chains_per_dataset=m, num_chains=cut, **kw)
    hi, shi = _run(sampler, um, T, th0, None, chains_per_dataset=m, num_chains=G * m - cut, chain_id_base=cut, **kw)
    assert torch.equal(torch.cat([lo, hi]), tr) and torch.equal(torch.cat([slo.raw, shi.raw]), st.raw)


def test_posterior_of_every_dataset():
    """64 datasets x 256 chains of GAUSS_SRC at theta_dim 1: prior N(p1, 1), effective likelihood N(y_obs; theta, p0^2 + eps^2),
    so dataset g's ABC posterior is normal with variance v = 1 / (1 + 1 / s2) and mean v (p1 + y_obs / s2)"""
    g = _g()
    G, m, T, burn = 64, 256, 3001, 1000
    tab = _table(G, 1, 5)
    tab[:, 2] = torch.linspace(-2.5, 2.5, G)
    um = g.UserModel(GAUSS_SRC, theta_dim=1, y_dim=1, n_noise=1, epsilon=EPS, params=tab)
    tr = _run("global", um, T, torch.zeros(1), None, d=1, chains_per_dataset=m, seed=9, trace="chain")
    x = tr.view(G, m, T)[:, :, burn:].double().reshape(G, -1)
    s2 = P0 ** 2 + EPS ** 2
    v = 1.0 / (1.0 + 1.0 / s2)
    mean = v * (tab[:, 1].double() + tab[:, 2].double() / s2)
    got_mean, got_var = x.mean(1).cpu(), x.var(1).cpu()
    assert float((got_mean - mean).abs().max()) < 0.03
    assert float((got_var / v - 1).abs().max()) < 0.1


def test_simulation_based_calibration_is_uniform(tmp_path):
    """SBC end to end in one call: theta*_g ~ prior, y_obs_g = simulate(theta*_g) + eps xi (the Gaussian-kernel ABC posterior
    is then exact for y_obs_g); the rank of theta*_g among the final states of its 63 chains is uniform on 0..63"""
    from scipy import stats as sst
    g = _g()
    G, m = 1024, 63
    gen = torch.Generator().manual_seed(11)
    mu = torch.randn(G, generator=gen) * 0.5
    theta_star = mu + torch.randn(G, generator=gen)
    y_obs = theta_star + P0 * torch.randn(G, generator=gen) + EPS * torch.randn(G, generator=gen)
    um = g.UserModel(GAUSS_SRC, theta_dim=1, y_dim=1, n_noise=1, epsilon=EPS,
                     params=torch.stack([torch.full((G,), P0), mu, y_obs], dim=1))
    th0 = (mu.repeat_interleave(m) + torch.randn(G * m, generator=gen)).reshape(-1, 1)   # prior draws, one per chain
    _, rs = _run("global", um, 401, th0, None, d=1, chains_per_dataset=m, seed=12, trace="none", return_stats=True,
                 checkpoint=str(tmp_path / "sbc.pt"))
    final = _ck(tmp_path / "sbc.pt")["theta"].view(G, m)
    ranks = (final < theta_star.view(G, 1)).sum(1).numpy()
    counts = np.bincount(ranks // 8, minlength=8)
    assert sst.chisquare(counts).pvalue > 1e-3, counts
    assert float(rs.raw[:, 0].min()) == 400.0


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_checkpoint_resume_of_a_batched_run(sampler, tmp_path):
    g = _g()
    G, m, d, s = 8, 33, 2, 4
    um = g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=_table(G, d, 3))
    kw = dict(seed=s, trace="chain", return_stats=True, chains_per_dataset=m)
    full, st_full = _run(sampler, um, 201, torch.zeros(d), None, checkpoint=str(tmp_path / "full.pt"), **kw)
    first, _ = _run(sampler, um, 101, torch.zeros(d), None, checkpoint=str(tmp_path / "cut.pt"), **kw)
    rest, st_rest = _run(sampler, um, 201, None, None, resume=str(tmp_path / "cut.pt"), checkpoint=str(tmp_path / "end.pt"), **kw)
    assert torch.equal(torch.cat([first, rest], dim=1), full)
    a, b = _ck(tmp_path / "full.pt"), _ck(tmp_path / "end.pt")
    assert a["model"] == b["model"] == um.fingerprint() and a["chains_per_dataset"] == b["chains_per_dataset"] == m
    for key in ("theta", "y", "aux"):
        assert (a[key] is None and b[key] is None) or torch.equal(a[key], b[key]), key
    # the counts are exact; the float sums are re-associated at the cut, as in the one-dataset checkpoint tests
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4]) and torch.allclose(st_rest.raw, st_full.raw, rtol=1e-4, atol=1e-3)
    other = g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=_table(G, d, 4))
    with pytest.raises(ValueError, match="another user model"):
        _run(sampler, other, 201, None, None, resume=str(tmp_path / "cut.pt"), **kw)
    with pytest.raises(ValueError, match="chains_per_dataset"):
        _run(sampler, um, 201, None, None, resume=str(tmp_path / "cut.pt"), **dict(kw, chains_per_dataset=m + 1))
    with pytest.raises(ValueError, match="another user model"):
        _run(sampler, um.dataset(0), 201, None, None, resume=str(tmp_path / "cut.pt"), **dict(kw, chains_per_dataset=None))


def test_python_refusals(tmp_path):
    g = _g()
    G, d = 4, 2
    um = g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=_table(G, d, 6))
    one = um.dataset(1)
    lp, gp = _props(d)
    with pytest.raises(ValueError, match="needs chains_per_dataset"):
        _run("global", um, 11, torch.zeros(d), None)
    for model in (one, g.Mixture_set(0.05)):
        for sampler in SAMPLERS:
            with pytest.raises(ValueError, match="batched UserModel"):
                _run(sampler, model, 11, torch.zeros(d), None, num_chains=8, chains_per_dataset=2)
    with pytest.raises(ValueError, match="at least 1"):
        _run("global", um, 11, torch.zeros(d), None, chains_per_dataset=0)
    with pytest.raises(ValueError, match="reach beyond"):
        _run("global", um, 11, torch.zeros(d), None, chains_per_dataset=3, num_chains=13)
    with pytest.raises(ValueError, match="reach beyond"):
        _run("isir", um, 11, torch.zeros(d), None, chains_per_dataset=3, num_chains=4, chain_id_base=9)
    with pytest.raises(ValueError, match="one per dataset"):
        _run("mala", um, 11, torch.zeros(3, d), None, chains_per_dataset=3)
    with pytest.raises(ValueError, match="dataset"):
        um.generate_samples(torch.zeros(1, d))
    with pytest.raises(ValueError, match="GLMCMC_NF"):
        g.GLMCMC_NF(um, 11, torch.zeros(d), None, lp, None, 0.5, 4, 2, gp, 1, num_chains=8)
    with pytest.raises(ValueError, match="batched"):
        g.AGLMCMC(um, 11, torch.zeros(d), None, lp, gp, None, 0.5, 4, 2, 0.5, 0.1, num_chains=8, pooled=True)
    # the MCMCRunner entries pass chains_per_dataset through **kw
    runner = g.MCMCRunner(um, output_dir=str(tmp_path))
    tr = runner.run_global_mcmc(11, torch.zeros(d), None, 0.5, lp, gp, output_file=None, chains_per_dataset=2, seed=1)
    assert tr.shape == (G * 2, 11, d)


def test_abi_refusals_launch_nothing():
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    g = _g()
    eng = get_engine()
    lib, h = eng.lib, eng.ctx.handle
    G, m, d, n = 4, 8, 2, 32
    um = g.UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=EPS, params=_table(G, d, 7))
    lp, gp = _props(d)
    eng.bind_proposal(abi.SLOT_LOCAL, lp)
    eng.bind_proposal(abi.SLOT_GLOBAL, gp)
    eng.bind_proposal(abi.SLOT_IMPORTANCE, gp)
    theta, y = torch.full((n, d), 0.5, device="cuda"), torch.full((n, d), 0.5, device="cuda")
    stats = torch.zeros(n, abi.nstats(d), device="cuda")
    aux = torch.zeros(n, abi.AUX_SLOTS, device="cuda")
    out = torch.full((n,), 7.25, device="cuda")
    watched = (theta, y, stats, aux, out)
    before = [t.clone() for t in watched]
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = eng._stream()

    def run(fn, pod, n_chains=n, base=0):
        r = abi.RunPOD(n_chains=n_chains, n_steps=10, step_base=0, chain_id_base=base, seed=1, global_frequency=0.5,
                       rng_mode=abi.RNG_NATIVE, arith_mode=abi.ARITH_FAST, trace_layout=abi.TRACE_NONE, n_candidates=4,
                       trace_chains=n_chains, theta=p(theta), y=p(y), aux=p(aux), stats=p(stats), num_grad=8, tau=0.3,
                       stream=stream)
        return fn(h, C.byref(r), C.byref(pod))

    def pod_with(**kw):
        pod = um.user_pod(eng.device, m)
        for k, v in kw.items():
            setattr(pod, k, v)
        return pod

    entries = (lib.glabc_run_global_user, lib.glabc_run_isir_user, lib.glabc_run_mala_user)
    bad = [pod_with(dataset_params=None), pod_with(chains_per_dataset=0), pod_with(chains_per_dataset=-2),
           pod_with(n_datasets=-1), pod_with(n_datasets=0), pod_with(n_datasets=2 ** 62, chains_per_dataset=4)]
    for fn in entries:
        for pod in bad:
            assert run(fn, pod) == abi.ERR_INVALID
        assert run(fn, pod_with(), n_chains=n, base=G * m - n + 1) == abi.ERR_INVALID     # the last id is G m
        assert run(fn, pod_with(), n_chains=n, base=-1) == abi.ERR_INVALID
    one = um.dataset(0).user_pod()
    one.chains_per_dataset = 2                                                             # m without a table
    assert run(lib.glabc_run_global_user, one) == abi.ERR_INVALID
    for pod in bad[:2]:
        assert lib.glabc_user_simulate(h, C.byref(pod), p(theta), n, 1, 0, p(y), stream) == abi.ERR_INVALID
        assert lib.glabc_user_evaluate(h, C.byref(pod), abi.USER_PRIOR, p(theta), n, p(out), stream) == abi.ERR_INVALID
    assert lib.glabc_user_simulate(h, C.byref(pod_with()), p(theta), n, 1, G * m - n + 1, p(y), stream) == abi.ERR_INVALID
    assert lib.glabc_user_evaluate(h, C.byref(pod_with(chains_per_dataset=7)), abi.USER_PRIOR, p(theta), n, p(out),
                                   stream) == abi.ERR_INVALID                              # 4 x 7 rows < 32
    from glabc_b200.block_isir import Block
    blk = Block(n, 4, 2, d, d, eng.device)
    r = abi.RunPOD(n_chains=n, n_steps=10, seed=1, global_frequency=0.5, rng_mode=abi.RNG_NATIVE, arith_mode=abi.ARITH_FAST,
                   trace_layout=abi.TRACE_NONE, n_candidates=4, trace_chains=n, theta=p(theta), y=p(y), stats=p(stats),
                   stream=stream)
    assert lib.glabc_run_block_isir_user(h, C.byref(r), C.byref(blk.pod), C.byref(pod_with())) == abi.ERR_UNSUPPORTED
    assert lib.glabc_block_weights_user(h, C.byref(r), C.byref(blk.pod), 0, C.byref(pod_with())) == abi.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    for t, b in zip(watched, before):
        assert torch.equal(t, b)
    # the same launch with a valid table runs
    assert run(lib.glabc_run_global_user, pod_with()) == abi.OK
    torch.cuda.synchronize()
    assert not torch.equal(stats, before[2])
