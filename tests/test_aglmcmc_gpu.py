"""GPU parity tests of K5 (KernelDensity) and K6 (AGLMCMC) through the C-ABI."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, abi, check_aglmcmc, gauss_pod, load_cases, model_pod, rel_max
from oracle import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from glabc_b200.engine import Engine
    return Engine()


def bind(eng, model, lp, ip):
    eng.ctx.check(eng.lib.glabc_model_set(eng.ctx.handle, C.byref(model), C.sizeof(model)))
    eng.ctx.check(eng.lib.glabc_dist_set(eng.ctx.handle, abi.SLOT_LOCAL, C.byref(lp), C.sizeof(lp)))
    eng.ctx.check(eng.lib.glabc_dist_set(eng.ctx.handle, abi.SLOT_IMPORTANCE, C.byref(ip), C.sizeof(ip)))


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------------------------------------
# KernelDensity
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", [abi.ARITH_STRICT, abi.ARITH_FAST])
def test_kde_golden(eng, arith):
    """kernel_density.py fit / log_prob against the reference's own outputs: weighted / unweighted, Silverman / Scott,
    d = 1..3, and queries 40 sigma away (every kernel underflows without the max shift)"""
    z = np.load(os.path.join(GOLDEN, "kde.npz"))
    for i in range(int(z["n_cases"])):
        X, x, w = dev(z[f"kde{i}/X"]), dev(z[f"kde{i}/x"]), z[f"kde{i}/w"]
        weights, bw = eng.kde_fit(X, dev(w) if w.size else None, rule=int(z[f"kde{i}/rule"]))
        assert rel_max(weights.cpu().numpy(), z[f"kde{i}/weights"]) < 1e-6
        assert rel_max(bw.cpu().numpy(), z[f"kde{i}/bw"]) < 1e-6
        lp = eng.kde_log_prob(X, weights, bw, x, arith=arith).cpu().numpy()
        assert np.isfinite(lp).all()
        assert rel_max(lp, z[f"kde{i}/log_prob"], 1.0) < (1e-5 if arith == abi.ARITH_STRICT else 3e-5), i


@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_kde_matches_oracle_batched(eng, d):
    """ragged batched sets (the AGLMCMC shape) and one larger set, against the oracle"""
    rng = np.random.default_rng(d)
    sets, cap, m = 7, 700, 333
    n = rng.integers(5, cap + 1, sets).astype(np.int32)
    n[0] = cap
    X = (rng.standard_normal((sets, cap, d)) * (0.5 + rng.random((sets, 1, d)))).astype(np.float32)
    w = (rng.random((sets, cap)) ** 4).astype(np.float32)
    x = (rng.standard_normal((sets, m, d)) * 1.5).astype(np.float32)
    weights, bw = eng.kde_fit(dev(X), dev(w), n=dev(n))
    lp_s = eng.kde_log_prob(dev(X), weights, bw, dev(x), n=dev(n), arith=abi.ARITH_STRICT).cpu().numpy()
    lp_f = eng.kde_log_prob(dev(X), weights, bw, dev(x), n=dev(n), arith=abi.ARITH_FAST).cpu().numpy()
    for s in range(sets):
        wo, bo = oracle.kde_fit(X[s, :n[s]].copy(), w[s, :n[s]].copy())
        assert rel_max(weights[s, :n[s]].cpu().numpy(), wo) < 1e-6 and rel_max(bw[s].cpu().numpy(), bo) < 2e-6
        want = oracle.kde_log_prob(X[s, :n[s]].copy(), wo, bo, x[s].copy())
        assert rel_max(lp_s[s], want, 1.0) < 1e-5 and rel_max(lp_f[s], want, 1.0) < 5e-5
    # one big set through the two-queries-per-thread path
    nb, mb = 6000, 2500
    Xb, xb = rng.standard_normal((nb, d)).astype(np.float32), (rng.standard_normal((mb, d)) * 2).astype(np.float32)
    wb, bb = eng.kde_fit(dev(Xb), None, rule=abi.BW_SCOTT)
    got = eng.kde_log_prob(dev(Xb), wb, bb, dev(xb)).cpu().numpy()
    wo, bo = oracle.kde_fit(Xb, None, abi.BW_SCOTT)
    assert rel_max(got, oracle.kde_log_prob(Xb, wo, bo, xb), 1.0) < 5e-5


def test_kde_sample(eng):
    """replay: X[idx] + noise * bw exactly (kernel_density.py:148-149); native: the categorical draw follows the weights"""
    rng = np.random.default_rng(3)
    n, m, d = 500, 4096, 2
    X = rng.standard_normal((n, d)).astype(np.float32)
    w = (rng.random(n) ** 3).astype(np.float32)
    weights, bw = eng.kde_fit(dev(X), dev(w))
    idx = rng.integers(0, n, m).astype(np.int32)
    noise = rng.standard_normal((m, d)).astype(np.float32)
    got = eng.kde_sample(dev(X), weights, bw, m, idx_tape=dev(idx), noise_tape=dev(noise)).cpu().numpy()
    want = X[idx] + noise * bw.cpu().numpy()[None, :]
    assert np.array_equal(got, want)
    big = eng.kde_sample(dev(X), weights, bw, 400000, seed=5).cpu().numpy().astype(np.float64)
    wn = weights.cpu().numpy().astype(np.float64)
    mean = (wn[:, None] * X).sum(0)
    var = (wn[:, None] * (X - mean) ** 2).sum(0) + bw.cpu().numpy().astype(np.float64) ** 2
    assert np.abs(big.mean(0) - mean).max() < 0.01 and np.abs(big.var(0) / var - 1).max() < 0.02
    assert not np.array_equal(big[:1000], eng.kde_sample(dev(X), weights, bw, 1000, seed=6).cpu().numpy())


def test_kernel_density_class(eng):
    """the reference-shaped class: fit / log_prob / sample / forward, str and numeric bandwidths"""
    import glabc_b200 as g
    z = np.load(os.path.join(GOLDEN, "kde.npz"))
    kde = g.KernelDensity(bandwidth="silverman").fit(torch.from_numpy(z["kde0/X"]), torch.from_numpy(z["kde0/w"]))
    assert kde.n_samples == 300 and kde.dim == 2
    lp = kde.log_prob(torch.from_numpy(z["kde0/x"]))
    assert rel_max(lp.cpu().numpy(), z["kde0/log_prob"], 1.0) < 3e-5
    s, lps = kde.forward(64)
    assert s.shape == (64, 2) and torch.allclose(lps, kde.log_prob(s))
    fixed = g.KernelDensity(bandwidth=0.3).fit(torch.from_numpy(z["kde0/X"]))
    ref = torch.logsumexp(torch.distributions.Normal(torch.from_numpy(z["kde0/X"])[None], 0.3).log_prob(
        torch.from_numpy(z["kde0/x"])[:, None]).sum(-1) + np.log(1 / 300 + 1e-10), dim=1)
    assert torch.allclose(fixed.log_prob(torch.from_numpy(z["kde0/x"])).cpu(), ref, rtol=1e-4, atol=1e-4)
    with pytest.raises(RuntimeError):
        g.KernelDensity().log_prob(torch.zeros(1, 2))


# ---------------------------------------------------------------------------------------------
# AGLMCMC
# ---------------------------------------------------------------------------------------------
def run_golden(eng, case, arith):
    T, Cn, K, S = int(case["T"]), case["theta0"].shape[0], int(case["K"]), int(case["S"])
    d = case["theta0"].shape[1]
    B, R = K * S, case["ad_idx"].shape[0]
    bind(eng, model_pod(case), gauss_pod(case, "lp"), gauss_pod(case, "ip"))
    theta, y = dev(case["theta0"]), dev(case["y0"])
    dbg = torch.zeros(T - 1, abi.DEBUG_SLOTS, Cn, device="cuda")
    ad_rec = torch.zeros(R, abi.AG_REC_SLOTS, Cn, device="cuda")
    ad_blk = torch.zeros(R, B, d + 3, Cn, device="cuda")
    init_w = torch.zeros(B, Cn, device="cuda")
    tapes = dict(init_p=dev(case["init_p"]), init_s=dev(case["init_s"]), ad_idx=dev(case["ad_idx"]), ad_noise=dev(case["ad_noise"]),
                 ad_sim=dev(case["ad_sim"]))
    ag = eng.aglmcmc_params(step_size=S, alpha=float(case["alpha"]), hat_eps_T=float(case["hat_eps_T"]), ad_rec=ad_rec,
                            ad_blk=ad_blk, init_w=init_w, **tapes)
    tr = eng.run("aglmcmc", theta=theta, y=y, n_steps=T - 1, gf=float(case["gf"]), rng_mode=abi.RNG_REPLAY, arith=arith,
                 trace_layout=abi.TRACE_TIME_MAJOR, tape32=dev(case["tape32"]), tape64=dev(case["tape64"]), debug=dbg, K=K, ag=ag)
    torch.cuda.synchronize()
    return tr.cpu().numpy(), dbg.cpu().numpy(), ad_rec.cpu().numpy(), ad_blk.cpu().numpy(), init_w.cpu().numpy()


@pytest.mark.parametrize("ci", range(3))
def test_aglmcmc_replay_golden(eng, ci):
    """the reference's own draws, incl. its torch.multinomial indices, through 16-18 adaptations per chain: every
    branch / move / resample index bit-exact; eps-hat, KDE bandwidth, block log-densities and weights to 1e-5"""
    case = load_cases("aglmcmc.npz")[ci]
    tr, dbg, ad_rec, ad_blk, init_w = run_golden(eng, case, abi.ARITH_STRICT)
    check_aglmcmc(case, tr, dbg, ad_rec, ad_blk, init_w)
    # FAST arithmetic (MUFU exp, fixed-shift KDE log-sum-exp): same decisions except at rounding-level ties
    tr_f, dbg_f, rec_f, _, _ = run_golden(eng, case, abi.ARITH_FAST)
    same = dbg_f[:, 0].astype(np.int64) == case["rec"][:, 0].astype(np.int64)
    assert same.mean() > 0.999
    n = int(case["n_adapt"].min())
    if same.all():
        assert rel_max(rec_f[:n, 0], case["ad_rec"][:n, 0]) < 1e-4


def readme_setup(eng, family=abi.MODEL_ABS_NORMAL):
    case = load_cases("aglmcmc.npz")[0]
    bind(eng, model_pod(case, family), gauss_pod(case, "lp"), gauss_pod(case, "ip"))
    return case


def check_native_matches_oracle(eng, family):
    case = readme_setup(eng, family)
    Cn, T, d, K, S = 64, 300, 2, 4, 20
    theta0 = np.zeros((Cn, d), np.float32)
    y0 = (np.random.default_rng(1).standard_normal((Cn, d)) * 0.2236).astype(np.float32)
    theta, y = dev(theta0), dev(y0)
    st = torch.zeros(Cn, abi.nstats(d), device="cuda")
    ag = eng.aglmcmc_params(step_size=S, alpha=0.8, hat_eps_T=0.2)
    got = eng.run("aglmcmc", theta=theta, y=y, n_steps=T, gf=0.8, seed=9, chain_id_base=5, arith=abi.ARITH_STRICT,
                  trace_layout=abi.TRACE_TIME_MAJOR, K=K, ag=ag, stats=st).cpu().numpy()
    th_o, y_o = theta0.copy(), y0.copy()
    st_o = np.zeros((Cn, abi.nstats(d)), np.float32)
    want = oracle.run("aglmcmc", model_pod(case, family), gauss_pod(case, "lp"), gauss_pod(case, "ip"), theta=th_o, y=y_o, n_steps=T,
                      gf=0.8, seed=9, chain_id_base=5, K=K, stats=st_o, ag=oracle.aglmcmc_params(S=S, alpha=0.8, hat_eps_T=0.2))
    assert np.array_equal(st.cpu().numpy()[:, abi.STAT_GLOBAL_STEPS], st_o[:, abi.STAT_GLOBAL_STEPS])   # same branch coins
    close = np.isclose(got, want, rtol=1e-4, atol=1e-4).all(-1)
    assert close[:40].mean() > 0.99          # identical until approximate-vs-libm normals flip a decision somewhere
    assert close.mean() > 0.7


def test_aglmcmc_native_matches_oracle(eng):
    """native Philox mode, strict arithmetic, gf < 1 (chains pause at different iterations): the kernels and the
    oracle draw the same streams; decisions agree except where MUFU-vs-libm normals differ in the last bits"""
    check_native_matches_oracle(eng, abi.MODEL_ABS_NORMAL)


def test_aglmcmc_native_matches_oracle_identity_link(eng):
    """the same with the identity link, which the AGLMCMC kernels choose at run time (model_simulate)"""
    check_native_matches_oracle(eng, abi.MODEL_ID_NORMAL)


def test_aglmcmc_invariances(eng):
    """sharding by chain_id_base and both trace layouts give bit-identical chains; a run continued with init = 0
    (workspace kept in the context) equals the uninterrupted one"""
    readme_setup(eng)
    Cn, T, d, K, S = 96, 260, 2, 5, 12
    theta0 = torch.zeros(Cn, d, device="cuda")
    y0 = (torch.randn(Cn, d, generator=torch.Generator().manual_seed(3)) * 0.2236).cuda()

    def run(lo, hi, layout, **kw):
        t, yv = theta0[lo:hi].clone(), y0[lo:hi].clone()
        ag = eng.aglmcmc_params(step_size=S, alpha=0.8, hat_eps_T=0.2)
        return eng.run("aglmcmc", theta=t, y=yv, n_steps=T - 1, gf=0.75, seed=7, chain_id_base=lo, K=K, ag=ag,
                       trace_layout=layout, **kw)

    full = run(0, Cn, abi.TRACE_TIME_MAJOR)
    assert torch.equal(run(0, Cn, abi.TRACE_CHAIN_MAJOR).permute(1, 0, 2), full)
    assert torch.equal(torch.cat([run(0, 40, abi.TRACE_TIME_MAJOR), run(40, Cn, abi.TRACE_TIME_MAJOR)], dim=1), full)
    t, yv = theta0.clone(), y0.clone()
    buf = torch.zeros(T, Cn, d, device="cuda")
    base = 0
    for n in (50, 101, T - 1 - 151):
        ag = eng.aglmcmc_params(step_size=S, alpha=0.8, hat_eps_T=0.2, init=(base == 0))
        eng.run("aglmcmc", theta=t, y=yv, n_steps=n, step_base=base, gf=0.75, seed=7, K=K, ag=ag, trace=buf, trace_rows=T,
                trace_layout=abi.TRACE_TIME_MAJOR, write_row0=(base == 0))
        base += n
    assert torch.equal(buf, full)


def test_aglmcmc_posterior(eng):
    """README model with the example's settings (Mixture.py:74: gf = 1, K = 5, step 200, alpha 0.8, eps-hat_T 0.2):
    closed-form ABC posterior (SURVEY.md App. D)"""
    from scipy import stats as sst
    readme_setup(eng)
    Cn, T, d = 4096, 3000, 2
    theta = torch.zeros(Cn, d, device="cuda")
    y = torch.randn(Cn, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)) * 0.2236
    st = torch.zeros(Cn, abi.nstats(d), device="cuda")
    ag = eng.aglmcmc_params(step_size=200, alpha=0.8, hat_eps_T=0.2)
    eng.run("aglmcmc", theta=theta, y=y, n_steps=T, gf=1.0, seed=11, K=5, ag=ag, trace_layout=abi.TRACE_NONE, stats=st)
    torch.cuda.synchronize()
    a = theta.abs().cpu().numpy().astype(np.float64)
    for i in range(d):
        assert sst.kstest(a[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.04
    quad = ((theta[:, 0] > 0).long() * 2 + (theta[:, 1] > 0).long()).bincount(minlength=4).cpu().numpy() / Cn
    assert np.abs(quad - 0.25).max() < 0.04
    from glabc_b200.engine import RunStats
    assert 0.005 < float(RunStats(st, d).move_rate.mean()) < 0.2


def test_public_api_aglmcmc(eng, tmp_path):
    """examples/Mixture.py:74-75: run_aglmcmc(num_ite, theta0, y0, 1, lp, ip, 5, 200, 0.8, 0.2)"""
    import glabc_b200 as g
    torch.manual_seed(0)
    model = g.Mixture_set(epsilon=0.05)
    theta0 = torch.tensor([0.0, 0.0])
    y0 = model.generate_samples(theta0)
    lp = g.DiagGaussian(2, loc=torch.zeros(1, 2), log_scale=torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    runner = g.MCMCRunner(model, output_dir=str(tmp_path))
    chain = runner.run_aglmcmc(1000, theta0, y0, 1, lp, ip, 5, 200, 0.8, 0.2, output_file="aglmcmc_results.csv", verbose=False)
    assert chain.shape == (1000, 2) and chain.dtype == torch.float32 and torch.equal(chain[0], theta0)
    assert (tmp_path / "aglmcmc_results.csv").exists()
    out = runner.run_aglmcmc(12000, theta0, None, 1, lp, ip, 5, 200, 0.8, 0.2, output_file=None, num_chains=32, seed=4)
    assert out.shape == (32, 12000, 2)   # the reference stops at 10,000 rows (SURVEY.md B-10)


def test_aglmcmc_pooled_kde_posterior(eng):
    """pooled=True: ONE KernelDensity over the pooled weighted draws of all chains (BASELINE config 5) — the sampler must
    still target the ABC posterior (closed form, SURVEY.md App. D) and the tolerance must anneal down to eps-hat_T"""
    from scipy import stats as sst
    import glabc_b200 as g
    model = g.Mixture_set(epsilon=0.05)
    lp = g.DiagGaussian(2, loc=torch.zeros(1, 2), log_scale=torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    Cn = 2048
    out, st, prop = g.AGLMCMC(model, 1501, torch.zeros(2), None, lp, ip, None, 0.9, 50, 5, 0.8, 0.2, num_chains=Cn, seed=3,
                              trace="none", return_stats=True, pooled=True, kde_train=20000, return_proposal=True)
    assert out is None and len(prop.history) >= 10
    eps_hist = [h[0] for h in prop.history]
    assert all(a >= b for a, b in zip(eps_hist, eps_hist[1:])) and eps_hist[-1] == pytest.approx(0.2)
    assert prop.history[-1][1] > 15000                    # the pooled training set is (almost) kde_train draws
    # the adapted proposal concentrates on the four posterior modes: the global acceptance beats the N(0, I) start
    assert float(st.accepted_global.sum() / st.global_steps.sum()) > 0.03
    out2 = g.AGLMCMC(model, 1001, torch.zeros(2), None, lp, ip, None, 0.9, 50, 5, 0.8, 0.2, num_chains=Cn, seed=5, trace="time",
                     pooled=True, kde_train=20000)
    th = out2[-1].abs().cpu().numpy().astype(np.float64)
    for i in range(2):
        assert sst.kstest(th[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.05
    quad = ((out2[-1][:, 0] > 0).long() * 2 + (out2[-1][:, 1] > 0).long()).bincount(minlength=4).cpu().numpy() / Cn
    assert np.abs(quad - 0.25).max() < 0.05


def test_kde_logprob_large_batch_paths(eng):
    """the 1-, 2- and 4-queries-per-thread instantiations of the packed (FFMA2) pair loop agree with the strict kernel,
    odd point counts included"""
    g = torch.Generator(device="cuda").manual_seed(2)
    for n, m in ((999, 700), (1025, 128 * 8 * 148 * 2 + 5), (513, 128 * 8 * 148 * 4 + 3)):
        X = torch.randn(n, 2, device="cuda", generator=g)
        w = torch.rand(n, device="cuda", generator=g)
        wn, bw = eng.kde_fit(X, w)
        x = torch.randn(m, 2, device="cuda", generator=g) * 1.5
        fast = eng.kde_log_prob(X, wn, bw, x, arith=abi.ARITH_FAST)
        strict = eng.kde_log_prob(X, wn, bw, x, arith=abi.ARITH_STRICT)
        assert float((fast - strict).abs().max()) < 2e-4


def test_checkpoint_resume_and_host_entry_are_bit_identical(tmp_path):
    """SURVEY.md 8(f) n4 for AGLMCMC: the end-of-run state incl. every chain's candidate block, KernelDensity, counters and
    eps-hat (glabc_aglmcmc_state) — a run cut in two continues bit-identically through further adaptations; and the
    host-buffer entry glabc_run_aglmcmc_host (time chunks, the workspace carried from chunk to chunk) delivers the same chains."""
    import glabc_b200 as g
    from glabc_b200.engine import get_engine
    model = g.Mixture_set(0.05)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    C, T, T1, S, K = 300, 401, 173, 20, 5
    run = lambda n, **kw: g.AGLMCMC(model, n, torch.zeros(2), None, lp, ip, None, 0.8, S, K, 0.8, 0.2, num_chains=C, seed=9,   # noqa: E731
                                    trace="time", return_stats=True, **kw)
    full, st_full = run(T)
    ck = tmp_path / "ag.pt"
    first, _ = run(T1, checkpoint=str(ck))
    rest, st_rest = run(T, resume=str(ck))
    assert torch.equal(first, full[:T1]) and torch.equal(rest, full[T1:])
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4]) and torch.allclose(st_rest.raw, st_full.raw, rtol=1e-4, atol=1e-3)
    assert float(st_full.move_rate.mean()) > 0.01
    # host entry: pinned host buffers, 64-row chunks
    eng = get_engine()
    eng.bind_model(model)
    eng.bind_proposal(abi.SLOT_LOCAL, lp)
    eng.bind_proposal(abi.SLOT_IMPORTANCE, ip)
    from glabc_b200.samplers import initial_state
    th0, y0, _ = initial_state(eng, eng.bind_model(model), torch.zeros(2), None, C, 9)
    h_th, h_y = th0.cpu().contiguous(), y0.cpu().contiguous()
    h_stats = torch.zeros(C, abi.nstats(2))
    h_trace = torch.zeros(T, C, 2).pin_memory()
    ag = eng.aglmcmc_params(step_size=S, alpha=0.8, hat_eps_T=0.2)
    eng.run_host("aglmcmc", theta=h_th, y=h_y, n_steps=T - 1, gf=0.8, seed=9, trace=h_trace, trace_layout=abi.TRACE_TIME_MAJOR,
                 stats=h_stats, K=K, ag=ag, chunk_steps=64)
    assert torch.equal(h_trace, full.cpu())
    assert torch.equal(h_stats[:, :4], st_full.raw.cpu()[:, :4]) and torch.allclose(h_stats, st_full.raw.cpu(), rtol=1e-4, atol=1e-3)


def test_pooled_checkpoint_resume_is_bit_identical(tmp_path):
    """the pooled-KDE mode (one KernelDensity shared by all chains): blocks, the KDE, eps-hat and the generators travel in the
    checkpoint; a run cut in two continues bit-identically through further pooled adaptations"""
    import glabc_b200 as g
    model = g.Mixture_set(0.05)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    C, T, T1 = 400, 301, 137
    run = lambda n, **kw: g.AGLMCMC(model, n, torch.zeros(2), None, lp, ip, None, 1.0, 20, 5, 0.8, 0.2, num_chains=C, seed=4,   # noqa: E731
                                    trace="time", return_stats=True, return_proposal=True, pooled=True, kde_train=4000, **kw)
    full, st_full, prop_full = run(T)
    ck = tmp_path / "agp.pt"
    first, _, prop_1 = run(T1, checkpoint=str(ck))
    rest, st_rest, prop_rest = run(T, resume=str(ck))
    assert len(prop_1.history) >= 2 and len(prop_rest.history) > len(prop_1.history)
    assert torch.equal(first, full[:T1]) and torch.equal(rest, full[T1:])
    assert prop_rest.history == prop_full.history
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4])
