"""GPU parity tests of K2 (GLMCMC / iSIR step kernel) through the C-ABI."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import abi, gauss_pod, load_cases, model_pod, rel_err
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


def fresh_aux(c, device=None):
    a = np.zeros((c, abi.AUX_SLOTS), np.float32)
    a[:, abi.AUX_LOCAL] = 1.0
    return a if device is None else dev(a)


@pytest.mark.parametrize("arith", [abi.ARITH_STRICT, abi.ARITH_FAST])
@pytest.mark.parametrize("ci", range(4))
def test_replay_golden(eng, ci, arith):
    """the reference's own draws (K = 5, 3, 8, 12): branch, move and resample index bit-exact, incl. the
    `None` steps where every weight underflows (SURVEY.md B-1); log-weights within 1e-5"""
    case = load_cases("glmcmc.npz")[ci]
    T, Cn, K = int(case["T"]), case["theta0"].shape[0], int(case["K"])
    bind(eng, model_pod(case), gauss_pod(case, "lp"), gauss_pod(case, "ip"))
    theta, y, aux = dev(case["theta0"]), dev(case["y0"]), fresh_aux(Cn, "cuda")
    debug = torch.zeros(T - 1, abi.DEBUG_SLOTS, Cn, device="cuda")
    trace = eng.run("isir", theta=theta, y=y, aux=aux, n_steps=T - 1, gf=float(case["gf"]), rng_mode=abi.RNG_REPLAY,
                    arith=arith, trace_layout=abi.TRACE_TIME_MAJOR, tape32=dev(case["tape32"]), tape64=dev(case["tape64"]),
                    debug=debug, K=K)
    torch.cuda.synchronize()
    dbg, rec = debug.cpu().numpy(), case["rec"]
    flags_ok = dbg[:, 0].astype(np.int32) == rec[:, 0].astype(np.int32)
    if arith == abi.ARITH_STRICT:
        assert flags_ok.all()
        assert np.array_equal(trace.cpu().numpy(), case["trace"])
    else:
        # FAST evaluates the resampling compare as u*S < cumsum(w) in float64 (no float32 quotients) and uses
        # MUFU.EX2: same decisions except when u64 lands within ~1e-7 of a bin edge
        assert flags_ok.mean() > 0.9995
        if flags_ok.all():
            assert np.allclose(trace.cpu().numpy(), case["trace"], rtol=2e-6, atol=1e-6)
    n = rec.shape[1]
    glob = (rec[:, 0].astype(np.int32) & 1) == 1
    for k in range(1, n):
        a, b = dbg[:, k], rec[:, k]
        if k == 1:   # log-weight of the current state: -inf-free, may be hugely negative
            m = np.isfinite(b)
        elif k in (2, 3):  # S and the normalised weight: ratios of exps of O(100) numbers -> compare where S > 0
            m = glob & (rec[:, 2] > 0) if arith == abi.ARITH_STRICT else np.zeros_like(glob)
        else:
            m = np.isfinite(b)
        m = m & flags_ok
        if m.any():
            # log-weights are sums of O(100..1000) terms that may cancel to O(1): absolute floor = 1e-5 x O(few)
            tol = 1e-5 if k != 2 and k != 3 else 2e-5
            assert np.allclose(a[m], b[m], rtol=tol, atol=3e-6 if arith == abi.ARITH_STRICT else 3e-5), k


def synthetic_case(d, Cn, T, K, seed):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)  # noqa: E731
    case = dict(y_obs=(1.0 + 0.5 * rng.random(d)).astype(np.float32), noise_loc=0.05 * f(d),
                noise_scale=(0.2 + 0.2 * rng.random(d)).astype(np.float32), prior_loc=0.1 * f(d),
                prior_log_scale=0.2 * f(d), eps_log_scale=np.float32(np.log(0.4)), lp_loc=0.01 * f(d),
                lp_log_scale=np.log(0.2 + 0.3 * rng.random(d)).astype(np.float32), ip_loc=0.2 * f(d),
                ip_log_scale=0.3 * f(d))
    case["prior_scale"] = np.exp(case["prior_log_scale"])
    case["eps_scale"] = np.exp(case["eps_log_scale"])
    case["lp_scale"], case["ip_scale"] = np.exp(case["lp_log_scale"]), np.exp(case["ip_log_scale"])
    slots = 2 + 2 * K * d
    tape = f(T, slots, Cn)
    tape[:, 0] = rng.random((T, Cn), dtype=np.float32)
    tape[:, slots - 1] = rng.random((T, Cn), dtype=np.float32)
    tape64 = rng.random((T, Cn))
    return case, tape, tape64, f(Cn, d), 1.0 + 0.3 * f(Cn, d)


@pytest.mark.parametrize("d,K", [(1, 1), (2, 5), (3, 7), (4, 16), (2, 15)])
@pytest.mark.parametrize("layout", [abi.TRACE_TIME_MAJOR, abi.TRACE_CHAIN_MAJOR])
def test_replay_matches_oracle(eng, d, K, layout):
    Cn, T = 500 + 13, 120
    family = abi.MODEL_ABS_NORMAL if d % 2 == 0 else abi.MODEL_ID_NORMAL
    case, tape, tape64, theta0, y0 = synthetic_case(d, Cn, T, K, seed=10 * d + K)
    m, lp, ip = model_pod(case, family), gauss_pod(case, "lp"), gauss_pod(case, "ip")
    th_o, y_o, aux_o = theta0.copy(), y0.copy(), fresh_aux(Cn)
    st_o = np.zeros((Cn, abi.nstats(d)), np.float32)
    want = oracle.run("isir", m, lp, ip, theta=th_o, y=y_o, aux=aux_o, n_steps=T, gf=0.7, rng_mode=abi.RNG_REPLAY,
                      tape32=tape, tape64=tape64, trace_layout=layout, stats=st_o, K=K)
    bind(eng, m, lp, ip)
    theta, y, aux = dev(theta0), dev(y0), fresh_aux(Cn, "cuda")
    stats = torch.zeros(Cn, abi.nstats(d), device="cuda")
    got = eng.run("isir", theta=theta, y=y, aux=aux, n_steps=T, gf=0.7, rng_mode=abi.RNG_REPLAY, arith=abi.ARITH_STRICT,
                  trace_layout=layout, tape32=dev(tape), tape64=dev(tape64), stats=stats, K=K, block_threads=96)
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(theta.cpu().numpy(), th_o) and np.array_equal(y.cpu().numpy(), y_o)
    assert np.array_equal(aux.cpu().numpy()[:, :2], aux_o[:, :2])
    st = stats.cpu().numpy()
    assert np.array_equal(st[:, :4], st_o[:, :4])
    assert np.allclose(st[:, 4:], st_o[:, 4:], rtol=1e-4, atol=1e-4)


def readme_pods():
    case = load_cases("glmcmc.npz")[0]
    return case, model_pod(case), gauss_pod(case, "lp"), gauss_pod(case, "ip")


def test_native_draws_replayed_by_oracle(eng):
    case, m, lp, ip = readme_pods()
    Cn, T, d, K = 333, 300, 2, 5
    bind(eng, m, lp, ip)
    theta0 = np.zeros((Cn, d), np.float32)
    y0 = (np.random.default_rng(1).standard_normal((Cn, d)) * 0.2236).astype(np.float32)
    theta, y, aux = dev(theta0), dev(y0), fresh_aux(Cn, "cuda")
    slots = abi.tape_isir_slots(d, d, K)
    dump = torch.zeros(T, slots, Cn, device="cuda")
    dump64 = torch.zeros(T, Cn, device="cuda", dtype=torch.float64)
    got = eng.run("isir", theta=theta, y=y, aux=aux, n_steps=T, gf=0.9, seed=21, chain_id_base=3, arith=abi.ARITH_STRICT,
                  trace_layout=abi.TRACE_TIME_MAJOR, tape_dump=dump, tape64_dump=dump64, K=K)
    torch.cuda.synchronize()
    th_o, y_o, aux_o = theta0.copy(), y0.copy(), fresh_aux(Cn)
    want = oracle.run("isir", m, lp, ip, theta=th_o, y=y_o, aux=aux_o, n_steps=T, gf=0.9, rng_mode=abi.RNG_REPLAY,
                      tape32=dump.cpu().numpy(), tape64=dump64.cpu().numpy(), K=K)
    assert np.array_equal(got.cpu().numpy(), want)
    # the oracle's native mode draws the same Philox streams: identical uniforms (U_b, U64), normals to MUFU accuracy
    th_n, y_n, aux_n = theta0.copy(), y0.copy(), fresh_aux(Cn)
    st_n = np.zeros((Cn, abi.nstats(d)), np.float32)
    nat = oracle.run("isir", m, lp, ip, theta=th_n, y=y_n, aux=aux_n, n_steps=T, gf=0.9, seed=21, chain_id_base=3, K=K, stats=st_n)
    moved_k = (want[1:] != want[:-1]).any(-1)
    moved_n = (nat[1:] != nat[:-1]).any(-1)
    assert (moved_k == moved_n).mean() > 0.999
    assert np.array_equal(st_n[:, abi.STAT_GLOBAL_STEPS], ((dump.cpu().numpy()[:, 0] < 0.9).sum(0)).astype(np.float32))


def test_native_invariances_and_host_entry(eng):
    case, m, lp, ip = readme_pods()
    Cn, T, d, K = 200, 161, 2, 5
    bind(eng, m, lp, ip)
    theta0 = torch.zeros(Cn, d, device="cuda")
    y0 = (torch.randn(Cn, d, generator=torch.Generator().manual_seed(3)) * 0.2236).cuda()
    run = lambda **kw: eng.run("isir", gf=0.9, seed=7, K=K, **kw)  # noqa: E731
    th, yy, ax = theta0.clone(), y0.clone(), fresh_aux(Cn, "cuda")
    full = run(theta=th, y=yy, aux=ax, n_steps=T - 1, trace_layout=abi.TRACE_TIME_MAJOR)
    th2, yy2, ax2 = theta0.clone(), y0.clone(), fresh_aux(Cn, "cuda")
    buf = torch.zeros(Cn, T, d, device="cuda")
    base = 0
    for n in (33, 64, T - 1 - 97):
        run(theta=th2, y=yy2, aux=ax2, n_steps=n, step_base=base, trace=buf, trace_rows=T, trace_layout=abi.TRACE_CHAIN_MAJOR,
            write_row0=(base == 0))
        base += n
    assert torch.equal(buf.permute(1, 0, 2), full) and torch.equal(th2, th) and torch.equal(ax2[:, :2], ax[:, :2])
    parts = []
    for lo, hi in ((0, 64), (64, Cn)):
        t, yv, a = theta0[lo:hi].clone(), y0[lo:hi].clone(), fresh_aux(hi - lo, "cuda")
        parts.append(run(theta=t, y=yv, aux=a, n_steps=T - 1, chain_id_base=lo, trace_layout=abi.TRACE_TIME_MAJOR))
    assert torch.equal(torch.cat(parts, dim=1), full)
    host = torch.zeros(T, Cn, d).pin_memory()
    hth, hy, hax = theta0.cpu().clone(), y0.cpu().clone(), torch.from_numpy(fresh_aux(Cn))
    eng.run_host("isir", theta=hth, y=hy, aux=hax, n_steps=T - 1, gf=0.9, seed=7, K=K, trace=host,
                 trace_layout=abi.TRACE_TIME_MAJOR, chunk_steps=32)
    assert torch.equal(host, full.cpu()) and torch.equal(hth, th.cpu())


def test_native_posterior_and_reference_bands(eng):
    """README model via run_glmcmc settings (gf=0.9, K=5): closed-form posterior (SURVEY.md App. D) and the
    reference's measured move rate 0.92 % +- 0.04 and ESJD 0.0295 +- 0.0011 (BASELINE.md section 2)."""
    from scipy import stats as sst
    case, m, lp, ip = readme_pods()
    Cn, T, d, K = 16384, 4000, 2, 5
    bind(eng, m, lp, ip)
    theta = torch.zeros(Cn, d, device="cuda")
    y = torch.randn(Cn, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)) * 0.2236
    aux = fresh_aux(Cn, "cuda")
    eng.run("isir", theta=theta, y=y, aux=aux, n_steps=T, gf=0.9, seed=11, K=K, trace_layout=abi.TRACE_NONE)
    st = torch.zeros(Cn, abi.nstats(d), device="cuda")
    eng.run("isir", theta=theta, y=y, aux=aux, n_steps=T, step_base=T, gf=0.9, seed=11, K=K, trace_layout=abi.TRACE_NONE, stats=st)
    torch.cuda.synchronize()
    a = theta.abs().cpu().numpy().astype(np.float64)
    for i in range(d):
        assert sst.kstest(a[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.02
    quad = ((theta[:, 0] > 0).long() * 2 + (theta[:, 1] > 0).long()).bincount(minlength=4).cpu().numpy() / Cn
    assert np.abs(quad - 0.25).max() < 0.02
    from glabc_b200.engine import RunStats
    rs = RunStats(st, d)
    move = float(rs.move_rate.mean())
    assert 0.0080 < move < 0.0104, move
    e = float(rs.esjd().mean())
    assert 0.026 < e < 0.033, e


def test_public_api_glmcmc(eng, tmp_path):
    """examples/Mixture.py:61-76: seed 0, 1,000 its of run_glmcmc(gf=0.9, K=5), esjd printed"""
    import glabc_b200 as g
    torch.manual_seed(0)
    model = g.Mixture_set(epsilon=0.05)
    theta0 = torch.tensor([0.0, 0.0])
    y0 = model.generate_samples(theta0)
    lp = g.DiagGaussian(2, loc=torch.zeros(1, 2), log_scale=torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    runner = g.MCMCRunner(model, output_dir=str(tmp_path))
    chain = runner.run_glmcmc(1000, theta0, y0, 0.9, lp, ip, 5, output_file="glmcmc_results.csv", verbose=False)
    assert chain.shape == (1000, 2) and chain.dtype == torch.float32 and torch.equal(chain[0], theta0)
    assert (tmp_path / "glmcmc_results.csv").exists()
    assert g.esjd(chain).shape == ()
    out, st = runner.run_glmcmc(300, theta0, None, 0.9, lp, ip, 5, output_file=None, num_chains=128, seed=4, return_stats=True)
    assert out.shape == (128, 300, 2)
    assert np.allclose(g.esjd(out), st.esjd().cpu().numpy(), rtol=1e-4, atol=1e-7)


def test_esjd_sweep(eng, tmp_path):
    """examples/Mixture_hyper.py:23-41: ESJD / time over a global_frequency grid; for the README model the global (iSIR)
    move dominates the score, so the best grid point is at the high end (the reference's own sweep picks gf >= 0.8)"""
    import glabc_b200 as g
    from glabc_b200.sweeps import esjd_sweep
    model = g.Mixture_set(epsilon=0.05)
    lp = g.DiagGaussian(2, loc=torch.zeros(1, 2), log_scale=torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    runner = g.MCMCRunner(model, output_dir=str(tmp_path))
    best, table = esjd_sweep(lambda gf, **kw: runner.run_glmcmc(1000, torch.zeros(2), None, gf, lp, ip, 5, output_file=None, **kw),
                             grid=[0.0, 0.5, 0.9, 1.0], num_chains=4096)
    assert table.shape == (4, 4) and best >= 0.5
    assert table[0, 1] < table[2, 1]          # esjd(gf = 0) < esjd(gf = 0.9): 0.0007 vs 0.03 in the reference


def test_pipelined_fast_loop_equals_plain_loop(eng):
    """K = 5 in FAST native mode runs the software-pipelined loop (candidates of step i+1 generated while step i
    resolves); with a tape dump attached the plain loop runs.  Same Philox streams, same arithmetic: same chains."""
    case, m, lp, ip = readme_pods()
    Cn, d, K = 777, 2, 5
    bind(eng, m, lp, ip)
    y0 = (torch.randn(Cn, d, generator=torch.Generator().manual_seed(9)) * 0.2236).cuda()
    for T in (1, 2, 97, 400):
        th, yy, ax = torch.zeros(Cn, d, device="cuda"), y0.clone(), fresh_aux(Cn, "cuda")
        st = torch.zeros(Cn, abi.nstats(d), device="cuda")
        piped = eng.run("isir", theta=th, y=yy, aux=ax, n_steps=T, gf=0.9, seed=5, K=K, trace_layout=abi.TRACE_TIME_MAJOR, stats=st)
        th2, yy2, ax2 = torch.zeros(Cn, d, device="cuda"), y0.clone(), fresh_aux(Cn, "cuda")
        st2 = torch.zeros(Cn, abi.nstats(d), device="cuda")
        dump = torch.zeros(T, abi.tape_isir_slots(d, d, K), Cn, device="cuda")
        plain = eng.run("isir", theta=th2, y=yy2, aux=ax2, n_steps=T, gf=0.9, seed=5, K=K, trace_layout=abi.TRACE_TIME_MAJOR,
                        stats=st2, tape_dump=dump)
        torch.cuda.synchronize()
        same = (piped == plain).all(-1).all(0)                       # per chain
        assert float(same.float().mean()) > 0.995                    # an FMA contracted differently may flip a rare decision
        assert torch.equal(st[:, abi.STAT_GLOBAL_STEPS], st2[:, abi.STAT_GLOBAL_STEPS])
        assert torch.allclose(ax[same][:, :2], ax2[same][:, :2], rtol=1e-5, atol=1e-6)


def test_host_entry_event_transport_isir(eng, monkeypatch):
    """glabc_run_isir_host with a chain-major host trace (event transport, tests/test_global_gpu.py): equals the device trace"""
    case, m, lp, ip = readme_pods()
    Cn, T, d, K = 700, 1200, 2, 5
    bind(eng, m, lp, ip)
    y0 = (torch.randn(Cn, d, generator=torch.Generator().manual_seed(3)) * 0.2236)
    for frac in ("1.0", "0.5"):
        monkeypatch.setenv("GLABC_HOST_EVENT_FRACTION", frac)
        th, yy, ax = torch.zeros(Cn, d, device="cuda"), y0.cuda(), fresh_aux(Cn, "cuda")
        want = eng.run("isir", theta=th, y=yy, aux=ax, n_steps=T - 1, gf=0.9, seed=7, K=K, trace_layout=abi.TRACE_CHAIN_MAJOR)
        torch.cuda.synchronize()
        host = torch.full((Cn, T, d), float("nan")).pin_memory()
        hth, hy, hax = torch.zeros(Cn, d), y0.clone(), torch.from_numpy(fresh_aux(Cn))
        eng.run_host("isir", theta=hth, y=hy, aux=hax, n_steps=T - 1, gf=0.9, seed=7, K=K, trace=host, trace_layout=abi.TRACE_CHAIN_MAJOR)
        assert torch.equal(host, want.cpu()) and torch.equal(hth, th.cpu()) and torch.equal(hax[:, :2], ax.cpu()[:, :2])
