"""GPU tests of K4 (RealNVP flow, tcgen05 tensor cores).  normflows is not installable here (SURVEY.md 8(c)): parity is
UNPINNED against the package; the kernel is pinned against the fp32 torch restatement of Appendix C and by invariants."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def flow_weights():
    from glabc_b200.flows import RealNVP
    torch.manual_seed(0)
    f = RealNVP(device="cuda")
    with torch.no_grad():       # a "trained" flow: small random last layers so the map is far from the identity
        f.w3.copy_(0.05 * torch.randn_like(f.w3))
        f.b3.copy_(0.02 * torch.randn_like(f.b3))
        f.loc.copy_(torch.tensor([[0.1, -0.2]]))
        f.log_scale.copy_(torch.tensor([[0.05, -0.1]]))
    return f


@pytest.fixture
def flow(flow_weights):
    """bound into the (shared) engine context for this test, single-FP16 mode unless the test asks otherwise"""
    flow_weights.bind().flow_precision("fast")
    return flow_weights


def test_precise_mode_meets_1e5_against_float64(flow):
    """GLABC_FLOW_PRECISE (FP16 hi + lo split, three MMAs, FP32 accumulate; the samplers' default): log q of sample() and
    log_prob() agree with a FLOAT64 evaluation of the same float32 weights (flows.RealNVP in double — the reference's
    normflows network is float32, GLMCMC_NFs.py:56-61) to <= 1e-5 relative at the 99.9th percentile over 1e6 samples —
    the tolerance north_star states for log-densities.  The single-FP16 mode on the same inputs misses it by > 20x."""
    import copy
    n = 1_000_000
    eps = torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(11))
    f64 = copy.deepcopy(flow).double()
    with torch.no_grad():
        th_r, lq_r = f64.sample_from(eps.double())
    try:
        th, lq = flow.fused_sample_from(eps, precision="precise")
        e_q = ((lq.double() - lq_r).abs() / lq_r.abs().clamp_min(1.0))
        e_t = ((th.double() - th_r).abs() / th_r.abs().clamp_min(1.0)).max(1).values
        assert float(e_q.quantile(0.999)) <= 1e-5, float(e_q.quantile(0.999))
        assert float(e_t.quantile(0.999)) <= 1e-5, float(e_t.quantile(0.999))
        assert float(e_q.max()) < 1e-3 and float(e_t.max()) < 1e-3, (float(e_q.max()), float(e_t.max()))
        # log_prob at the flow's own float64 samples (+ a jitter): the inverse pass
        x = (th_r + 0.05 * torch.randn(n, 2, device="cuda", dtype=torch.float64, generator=torch.Generator(device="cuda").manual_seed(12))).float()
        with torch.no_grad():
            lp_r = f64.log_prob(x.double())
        lp = flow.fused_log_prob(x)
        ok = torch.isfinite(lp_r)
        assert ok.float().mean() > 0.999 and torch.equal(torch.isfinite(lp), ok)
        e_p = (lp.double()[ok] - lp_r[ok]).abs() / lp_r[ok].abs().clamp_min(1.0)
        assert float(e_p.quantile(0.999)) <= 1e-5, float(e_p.quantile(0.999))
        # and the fp32 torch module itself is no closer to float64 than the kernel is (it is the reference's own arithmetic)
        with torch.no_grad():
            _, lq_32 = flow.sample_from(eps[:100000])
        e_32 = (lq_32.double() - lq_r[:100000]).abs() / lq_r[:100000].abs().clamp_min(1.0)
        print(f"precise: log q p99.9 {float(e_q.quantile(0.999)):.2e} median {float(e_q.median()):.2e}; theta p99.9 "
              f"{float(e_t.quantile(0.999)):.2e}; log_prob p99.9 {float(e_p.quantile(0.999)):.2e}; torch fp32 log q p99.9 {float(e_32.quantile(0.999)):.2e}")
        _, lq_f = flow.fused_sample_from(eps[:100000], precision="fast")
        e_f = (lq_f.double() - lq_r[:100000]).abs() / lq_r[:100000].abs().clamp_min(1.0)
        assert float(e_f.quantile(0.999)) > 2e-4
    finally:
        flow.bind().flow_precision("fast")


def test_precise_mode_invariants():
    """identity at init, ragged sizes and sample / log_prob consistency in the split-precision mode"""
    from glabc_b200.flows import RealNVP
    f = RealNVP(device="cuda")
    eng = f.bind()
    eng.flow_precision("precise")
    try:
        eps = torch.randn(5000, 2, device="cuda")
        th, lq = f.fused_sample_from(eps)
        assert torch.equal(th, eps)
        torch.manual_seed(1)
        with torch.no_grad():
            f.w3.copy_(0.05 * torch.randn_like(f.w3))
        f.bind()
        for n in (1, 127, 129, 4097):
            e = torch.randn(n, 2, device="cuda")
            th, lq = f.fused_sample_from(e)
            with torch.no_grad():
                th_r, lq_r = f.sample_from(e)
            assert torch.allclose(th, th_r, rtol=2e-5, atol=2e-5) and torch.allclose(lq, lq_r, rtol=2e-5, atol=2e-5)
            lp = f.fused_log_prob(th)
            assert torch.allclose(lp, lq, rtol=1e-4, atol=1e-4)
    finally:
        eng.flow_precision("fast")


def test_native_base_normals(flow):
    """glabc_flow_sample_native: q0's normals are drawn inside the kernel (Philox keyed by (seed, sample index)).  Through the
    identity flow they come out as theta: standard normal (KS), different per seed, the same per (seed, index) whatever n;
    and the trained flow fed those normals through the eps entry gives the identical samples."""
    from scipy import stats as sst
    from glabc_b200.flows import RealNVP
    ident = RealNVP(device="cuda")
    eng = ident.bind()
    eps, lq = ident.fused_sample(200000, seed=7, eng=eng, precision="fast")
    e = eps.cpu().numpy().astype(np.float64)
    for i in range(2):
        assert sst.kstest(e[:, i], "norm").statistic < 0.005
    assert abs(np.corrcoef(e[:, 0], e[:, 1])[0, 1]) < 0.01
    assert torch.allclose(lq, -np.log(2 * np.pi) - 0.5 * (eps ** 2).sum(1), rtol=0, atol=2e-6)
    again, _ = ident.fused_sample(1000, seed=7, eng=eng)
    other, _ = ident.fused_sample(1000, seed=8, eng=eng)
    assert torch.equal(again, eps[:1000]) and not torch.equal(other, eps[:1000])
    flow.bind().flow_precision("fast")
    th_n, lq_n = flow.fused_sample(200000, seed=7)
    th_e, lq_e = flow.fused_sample_from(eps)
    assert torch.equal(th_n, th_e) and torch.equal(lq_n, lq_e)


def test_identity_at_init():
    """init_zeros=True: the untrained flow is the identity, so sample == base draw and log_prob == base density exactly"""
    from glabc_b200.flows import RealNVP
    f = RealNVP(device="cuda")
    f.bind()
    eps = torch.randn(5000, 2, device="cuda")
    th, lq = f.fused_sample_from(eps)
    assert torch.equal(th, eps)
    want = -np.log(2 * np.pi) - 0.5 * (eps ** 2).sum(1)
    assert torch.allclose(lq, want, rtol=0, atol=2e-6)
    assert torch.allclose(f.fused_log_prob(eps), want, rtol=0, atol=2e-6)


@pytest.mark.parametrize("n", [1, 127, 128, 1024, 1025, 50000])
def test_matches_fp32_torch(flow, n):
    """sample / log_prob against the fp32 autograd path; tolerance = 11-bit operand rounding (FP16 activations, W2, and the
    FP16-staged w1 / b1 / W3 vectors) through 32 blocks: tight in the bulk, amplified by exp(s) in the tails"""
    eps = torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n))
    th, lq = flow.fused_sample_from(eps)
    with torch.no_grad():
        th_r, lq_r = flow.sample_from(eps)
        e_th = ((th - th_r).abs() / (1 + th_r.abs())).max(1).values
        assert float(e_th.median()) < 1.5e-3 and float(e_th.quantile(0.99)) < 1e-2 and float(e_th.max()) < 0.1, float(e_th.max())
        assert torch.allclose(lq, lq_r, rtol=0, atol=2e-2), float((lq - lq_r).abs().max())
        # queries around the flow's own samples (far outside its support exp(-s) overflows in fp32 for both paths)
        x = th_r + 0.1 * torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n + 1))
        lp, lp_r = flow.fused_log_prob(x), flow.log_prob(x)
        ok = torch.isfinite(lp_r)
        assert ok.float().mean() > 0.99 and torch.equal(torch.isfinite(lp), ok)
        err = (lp[ok] - lp_r[ok]).abs() / (1 + 0.01 * lp_r[ok].abs())
        # FP16 operand rounding (2^-11 relative) through 32 blocks: tight in the bulk, amplified by exp(-s) in the tails
        assert float(err.median()) < 3e-3 and float(err.quantile(0.99)) < 5e-2 and float(err.max()) < 5.0, float(err.max())
        if n >= 1024:
            assert float(err.quantile(0.999)) < 0.3


def test_fast_pipeline_many_chunks_per_cta(flow):
    """more chunks than SMs (the pipelined kernel's persistent loop, double-buffered operands and barrier phases run on
    across chunk boundaries) and a ragged last tile: every row's result is independent of where its tile sits, so rows of
    the big launch equal the same rows run as a small batch bit for bit; and the big launch agrees with PRECISE"""
    n = 148 * 32 * 128 + 148 * 8 * 128 + 77
    eps = torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(11))
    th, lq = flow.fused_sample_from(eps)
    pick = torch.cat([torch.arange(0, 300), torch.arange(606_000, 606_600), torch.arange(n - 300, n)]).cuda()
    th_s, lq_s = flow.fused_sample_from(eps[pick].contiguous())
    assert torch.equal(th[pick], th_s) and torch.equal(lq[pick], lq_s)
    lp = flow.fused_log_prob(th)
    lp_s = flow.fused_log_prob(th[pick].contiguous())
    assert torch.equal(lp[pick], lp_s)
    th_p, lq_p = flow.fused_sample_from(eps, precision="precise")
    flow.bind().flow_precision("fast")
    e_th = ((th - th_p).abs() / (1 + th_p.abs())).max(1).values
    assert float(e_th.median()) < 1.5e-3 and float(e_th.quantile(0.99)) < 1e-2, (float(e_th.median()), float(e_th.quantile(0.99)))
    assert float((lq - lq_p).abs().median()) < 2e-3


@pytest.mark.parametrize("n_blocks", [1, 2, 3, 5])
def test_pipeline_kernels_with_few_coupling_blocks(n_blocks):
    """the pipelined kernels prefetch the next coupling block's operands into a double buffer and carry their barrier
    phases across blocks and chunks: 1, 2, 3 and 5 blocks (odd and even, fewer than the buffer depth) over one and over
    several chunks per CTA, both precisions, against the fp32 torch module"""
    from glabc_b200.flows import RealNVP
    torch.manual_seed(n_blocks)
    f = RealNVP(n_blocks=n_blocks, device="cuda")
    with torch.no_grad():
        f.w3.copy_(0.05 * torch.randn_like(f.w3))
        f.b3.copy_(0.02 * torch.randn_like(f.b3))
    eng = f.bind()
    try:
        for n in (300, 148 * 32 * 128 * 2 + 1000):
            eps = torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n_blocks))
            with torch.no_grad():
                th_r, lq_r = f.sample_from(eps)
            for mode, tol in (("fast", 2e-3), ("precise", 2e-5)):
                th, lq = f.fused_sample_from(eps, eng, precision=mode)
                assert float(((th - th_r).abs() / (1 + th_r.abs())).max()) < 10 * tol, (mode, n)
                assert float((lq - lq_r).abs().median()) < tol and float((lq - lq_r).abs().max()) < 50 * tol, (mode, n)
                lp = f.fused_log_prob(th, eng, precision=mode)
                assert float((lp - lq).abs().median()) < tol, (mode, n)
    finally:
        eng.flow_precision("fast")


def test_sample_log_prob_consistency(flow):
    """the kernel's own pair: log_prob(sample(eps)) reproduces the log q returned with the sample.  sample()'s log q is the
    exact density of the map that produced theta (same s values in the transform and the log-det); log_prob() re-derives
    each block's input to ~1e-7, which can flip the FP16 rounding of a hidden unit, hence the 1e-3-level tolerance."""
    eps = torch.randn(20000, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    th, lq = flow.fused_sample_from(eps)
    lp = flow.fused_log_prob(th)
    err = (lp - lq).abs()
    assert float(err.median()) < 2e-3 and float(err.quantile(0.99)) < 3e-2, (float(err.median()), float(err.quantile(0.99)))
    assert torch.isfinite(th).all() and torch.isfinite(lq).all()


def test_density_integrates_to_one(flow):
    """exp(log_prob) on a grid sums to ~1 and to the same mass as the fp32 torch path (far cells overflow exp(-s) in
    fp32 for both paths and are dropped the same way)"""
    g = torch.linspace(-6, 6, 601, device="cuda")
    xx, yy = torch.meshgrid(g, g, indexing="ij")
    pts = torch.stack([xx.reshape(-1), yy.reshape(-1)], 1)
    with torch.no_grad():
        lp, lp_r = flow.fused_log_prob(pts), flow.log_prob(pts)
    cell = float((g[1] - g[0]) ** 2)
    mass = float(torch.exp(torch.nan_to_num(lp.double(), nan=-1e30, posinf=-1e30)).sum() * cell)
    mass_r = float(torch.exp(torch.nan_to_num(lp_r.double(), nan=-1e30, posinf=-1e30)).sum() * cell)
    assert abs(mass - mass_r) < 5e-3 and abs(mass - 1.0) < 3e-2, (mass, mass_r)


# ---------------------------------------------------------------------------------------------
# GLMCMC_NF sampler (block iSIR against the shared flow)
# ---------------------------------------------------------------------------------------------
def readme_objects():
    import glabc_b200 as g
    model = g.Mixture_set(epsilon=0.05)
    lp = g.DiagGaussian(2, loc=torch.zeros(1, 2), log_scale=torch.log(torch.tensor([0.35, 0.35])))
    return g, model, lp


def test_block_isir_equals_glmcmc_semantics():
    """With the untrained flow (identity map, proposal = N(0, I) exactly) and no training, GLMCMC_NF is iSIR with an
    N(0, I) importance proposal whose candidates are pre-generated: its chains must follow the same law as run_glmcmc
    with ip = N(0, I) — same closed-form posterior, same move rate and ESJD bands (reference: 0.92 %, 0.0295)."""
    from scipy import stats as sst
    g, model, lp = readme_objects()
    out, st = g.GLMCMC_NF(model, 3001, torch.zeros(2), None, lp, None, 0.9, 50, 5, None, 0, num_chains=8192, seed=3,
                          trace="none", return_stats=True)
    assert out is None
    move, e = float(st.move_rate.mean()), float(st.esjd().mean())
    assert 0.0075 < move < 0.0110, move
    assert 0.024 < e < 0.035, e
    out2 = g.GLMCMC_NF(model, 2001, torch.zeros(2), None, lp, None, 0.9, 50, 5, None, 0, num_chains=8192, seed=4, trace="time")
    a = out2[-1].abs().cpu().numpy().astype(np.float64)
    for i in range(2):
        assert sst.kstest(a[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.03
    # chains pause / resume individually (lq refresh after local accepts): every row of every chain was written
    assert torch.isfinite(out2).all() and torch.equal(out2[0], torch.zeros(8192, 2, device=out2.device))


def test_glmcmc_nf_training_improves_the_proposal():
    """Mixture.py:78-79 structure (gf 0.5, K 5, 50 training steps; a shorter block and a larger Adam step so that the 50
    steps fit a short test), many chains sharing one flow: the forward-KL loss falls, the trained flow moves its mass
    onto the four posterior modes, and the chains still target the posterior"""
    from scipy import stats as sst
    g, model, lp = readme_objects()
    # `resample` takes its offset from torch's GLOBAL generator, one torch.rand(1) per training batch (GLMCMC_NFs.py:33, as the
    # reference does): seeded here so that the 50-step trajectory does not depend on what earlier tests drew
    torch.manual_seed(1234)
    res, st, flow, losses = g.GLMCMC_NF(model, 4001, torch.zeros(2), None, lp, None, 0.5, 25, 5, None, 50, num_chains=2048,
                                        seed=1, trace="time", return_stats=True, return_flow=True, lr=3e-3)
    assert len(losses) == 50 and np.mean(losses[-10:]) < np.mean(losses[:5]) - 0.3, losses
    th, _ = flow.fused_sample_from(torch.randn(50000, 2, device="cuda"))
    near_mode = ((th.abs() - 1.425).abs() < 0.7).all(1).float().mean()
    assert float(near_mode) > 0.25, float(near_mode)            # N(0, I) puts ~9 % there
    a = res[-1].abs().cpu().numpy().astype(np.float64)
    for i in range(2):
        assert sst.kstest(a[:, i], sst.norm(1.42518, np.sqrt(0.049881)).cdf).statistic < 0.05
    assert float(st.move_rate.mean()) > 0.012                   # the untrained proposal moves 0.9 % of the time


def test_public_api_glmcmc_nf(tmp_path):
    """examples/Mixture.py:78-79: run_glmcmc_nf(num_ite, theta0, y0, 0.5, lp, gp_base, 5, 200, 50)"""
    g, model, lp = readme_objects()
    torch.manual_seed(0)
    theta0 = torch.tensor([0.0, 0.0])
    y0 = model.generate_samples(theta0)
    base = g.DiagGaussian(2, torch.zeros(1, 2), torch.zeros(1, 2))      # stands in for nf.distributions.base.DiagGaussian(2)
    runner = g.MCMCRunner(model, output_dir=str(tmp_path))
    chain = runner.run_glmcmc_nf(1500, theta0, y0, 0.5, lp, base, 5, 200, 50, output_file="glmcmc_nf_results.csv", verbose=False)
    assert chain.shape == (1500, 2) and chain.dtype == torch.float32 and torch.equal(chain[0], theta0)
    assert (tmp_path / "glmcmc_nf_results.csv").exists()


def test_glmcmc_nf_checkpoint_resume_is_bit_identical(tmp_path):
    """SURVEY.md 8(f) n4 for GLMCMC-NFs: chain state, candidate blocks, the flow's weights AND its Adam moments (glabc_flow_get /
    glabc_flow_train_state), the generators.  With every move global the chains consume their blocks in step, so a run cut in
    two (training steps on both sides of the cut) delivers the same chains, the same losses and the same final flow as the uncut
    run.  With local moves in between the chains reach the end of a block at different iterations and the blocks are refilled
    when EVERY chain is finished or has consumed its block — where a run is cut is then part of the schedule; the checkpoint
    still restores the state exactly: two resumes from one file are bit-identical."""
    g, model, lp = readme_objects()
    C, T, T1 = 512, 601, 257
    kw = dict(num_chains=C, seed=5, trace="time", return_stats=True, return_flow=True, lr=2e-3)
    run = lambda n, gf, **k: g.GLMCMC_NF(model, n, torch.zeros(2), None, lp, None, gf, 20, 5, None, 50, **kw, **k)   # noqa: E731
    torch.manual_seed(3)
    full, st_full, flow_full, loss_full = run(T, 1.0)
    ck = tmp_path / "nf.pt"
    torch.manual_seed(3)
    first, _, _, loss_1 = run(T1, 1.0, checkpoint=str(ck))
    torch.manual_seed(99)                                    # the resumed run takes its generators from the checkpoint
    rest, st_rest, flow_rest, loss_2 = run(T, 1.0, resume=str(ck))
    assert len(loss_1) >= 3 and len(loss_2) > len(loss_1)    # training happened before and after the cut
    assert torch.equal(first, full[:T1]) and torch.equal(rest, full[T1:])
    assert loss_2 == loss_full
    assert torch.equal(flow_rest.flat_params(), flow_full.flat_params())
    assert torch.equal(st_rest.raw[:, :4], st_full.raw[:, :4])
    # local moves in between (gf = 0.6): exact restoration = two resumes agree bit for bit, and the chains keep moving
    ck2 = tmp_path / "nf2.pt"
    torch.manual_seed(3)
    run(T1, 0.6, checkpoint=str(ck2))
    a, st_a, flow_a, loss_a = run(T, 0.6, resume=str(ck2))
    torch.manual_seed(12345)
    b, st_b, flow_b, loss_b = run(T, 0.6, resume=str(ck2))
    assert torch.equal(a, b) and loss_a == loss_b and torch.equal(flow_a.flat_params(), flow_b.flat_params())
    assert torch.equal(st_a.raw, st_b.raw) and float(st_a.move_rate.mean()) > 0.005
