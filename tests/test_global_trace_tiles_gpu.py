"""K1's chain-major trace against its time-major trace of the same native run, bit for bit: the
chain-major writer stages 32-row tiles in shared memory and the steady loop flushes whole tiles, so
these cover the head / full-tile / tail split of the step range, tail warps, partial tiles, chunked
launches that start off a tile boundary, odd and even trace_rows (the 8-byte and the 16-byte flush)
and rows past the last one written."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import abi, gauss_pod, model_pod

pytestmark = pytest.mark.gpu

CHAINS = (1, 31, 33, 1037)
STEPS = (1, 30, 31, 32, 33, 63, 64, 65, 257)
SENTINEL = -1234.5


@pytest.fixture(scope="module")
def eng():
    from glabc_b200.engine import Engine
    return Engine()


def bind(eng, d):
    rng = np.random.default_rng(d)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)  # noqa: E731
    case = dict(y_obs=(1.0 + 0.5 * rng.random(d)).astype(np.float32), noise_loc=0.05 * f(d),
                noise_scale=(0.2 + 0.2 * rng.random(d)).astype(np.float32), prior_loc=0.1 * f(d),
                prior_log_scale=0.2 * f(d), eps_log_scale=np.float32(np.log(0.3)), lp_loc=0.01 * f(d),
                lp_log_scale=np.log(0.2 + 0.3 * rng.random(d)).astype(np.float32), gp_loc=0.2 * f(d),
                gp_log_scale=0.3 * f(d))
    case["prior_scale"], case["eps_scale"] = np.exp(case["prior_log_scale"]), np.exp(case["eps_log_scale"])
    case["lp_scale"], case["gp_scale"] = np.exp(case["lp_log_scale"]), np.exp(case["gp_log_scale"])
    m, lp, gp = model_pod(case), gauss_pod(case, "lp"), gauss_pod(case, "gp")
    eng.ctx.check(eng.lib.glabc_model_set(eng.ctx.handle, C.byref(m), C.sizeof(m)))
    eng.ctx.check(eng.lib.glabc_dist_set(eng.ctx.handle, abi.SLOT_LOCAL, C.byref(lp), C.sizeof(lp)))
    eng.ctx.check(eng.lib.glabc_dist_set(eng.ctx.handle, abi.SLOT_GLOBAL, C.byref(gp), C.sizeof(gp)))


def start(n, d):
    g = torch.Generator().manual_seed(n * 7 + d)
    return (0.3 * torch.randn(n, d, generator=g)).cuda(), (1.0 + 0.3 * torch.randn(n, d, generator=g)).cuda()


def run(eng, theta0, y0, **kw):
    th, yy = theta0.clone(), y0.clone()
    out = eng.run("global", theta=th, y=yy, gf=0.4, seed=17, arith=abi.ARITH_FAST, **kw)
    return out, th, yy


@pytest.mark.parametrize("block", [32, 64, 96])
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_chain_major_is_time_major_transposed(eng, d, block):
    bind(eng, d)
    for n in CHAINS:
        theta0, y0 = start(n, d)
        for steps in STEPS:
            tm, th_t, y_t = run(eng, theta0, y0, n_steps=steps, trace_layout=abi.TRACE_TIME_MAJOR, block_threads=block)
            # trace_rows larger than the steps written: the extra rows must stay as they were
            rows = steps + 1 + 5
            buf = torch.full((n, rows, d), SENTINEL, device="cuda")
            run(eng, theta0, y0, n_steps=steps, trace_layout=abi.TRACE_CHAIN_MAJOR, trace=buf, trace_rows=rows,
                block_threads=block)
            cm, th_c, y_c = run(eng, theta0, y0, n_steps=steps, trace_layout=abi.TRACE_CHAIN_MAJOR, block_threads=block)
            torch.cuda.synchronize()
            where = f"d={d} chains={n} steps={steps} block={block}"
            assert torch.equal(cm.permute(1, 0, 2), tm), where
            assert torch.equal(buf[:, :steps + 1], cm), where
            assert bool((buf[:, steps + 1:] == SENTINEL).all()), where
            assert torch.equal(th_c, th_t) and torch.equal(y_c, y_t), where


@pytest.mark.parametrize("rows", [259, 260])
@pytest.mark.parametrize("write_row0", [True, False])
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_chunked_launches_share_one_buffer(eng, d, write_row0, rows):
    """steps 1..257 in launches at step_base 0, 37 and 100 (off the 32-row tile grid) into one
    [C, rows, d] buffer; an odd row count takes the 8-byte flush, an even one the 16-byte flush"""
    bind(eng, d)
    n, T = 1037, 257
    theta0, y0 = start(n, d)
    tm, th_t, y_t = run(eng, theta0, y0, n_steps=T, trace_layout=abi.TRACE_TIME_MAJOR)
    buf = torch.full((n, rows, d), SENTINEL, device="cuda")
    th, yy = theta0.clone(), y0.clone()
    for base, steps in ((0, 37), (37, 63), (100, T - 100)):
        eng.run("global", theta=th, y=yy, gf=0.4, seed=17, arith=abi.ARITH_FAST, n_steps=steps, step_base=base,
                trace_layout=abi.TRACE_CHAIN_MAJOR, trace=buf, trace_rows=rows, write_row0=write_row0 and base == 0)
    torch.cuda.synchronize()
    first = 0 if write_row0 else 1
    assert torch.equal(buf[:, first:T + 1].permute(1, 0, 2), tm[first:])
    assert bool((buf[:, T + 1:] == SENTINEL).all())
    if not write_row0:
        assert bool((buf[:, 0] == SENTINEL).all())
    assert torch.equal(th, th_t) and torch.equal(yy, y_t)
