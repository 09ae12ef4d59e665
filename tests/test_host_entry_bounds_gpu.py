"""The host-buffer entry points check the bounds of the caller's buffers before anything is allocated or launched: a trace
too small for the run is refused with ERR_INVALID, and the host state, the trace and the memory beyond it keep their
contents."""
import pytest
import torch

from helpers import abi, fresh_mala_state

pytestmark = pytest.mark.gpu

SENTINEL = -7.25
C, T, D, K = 8, 101, 2, 5


@pytest.fixture(scope="module")
def eng():
    import glabc_b200 as g
    from glabc_b200.engine import Engine
    e = Engine()
    e.bind_model(g.Mixture_set(0.05))
    e.bind_proposal(abi.SLOT_LOCAL, g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35]))))
    gp = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    e.bind_proposal(abi.SLOT_GLOBAL, gp)
    e.bind_proposal(abi.SLOT_IMPORTANCE, gp)
    return e


def host_args(eng, sampler):
    """the host state of C chains and the sampler's own arguments; 8 chains and 100 steps keep GlobalMCMC off the event
    transport"""
    y = torch.randn(C, D, generator=torch.Generator().manual_seed(1)) * 0.2236
    kw = dict(theta=torch.zeros(C, D), y=y, stats=torch.zeros(C, abi.nstats(D)), n_steps=T - 1, gf=0.8, seed=3, K=K)
    if sampler == "global":
        kw["chunk_steps"] = 64
    elif sampler == "mala":
        aux, s64 = fresh_mala_state(C)
        kw.update(aux=torch.from_numpy(aux), state64=torch.from_numpy(s64), num_grad=10, tau=0.3)
    elif sampler == "aglmcmc":
        kw["ag"] = eng.aglmcmc_params(step_size=20, alpha=0.8, hat_eps_T=0.2)
    return kw


def assert_refused(eng, sampler, trace, layout, kw):
    before = {k: v.clone() for k, v in kw.items() if isinstance(v, torch.Tensor)}
    with pytest.raises(abi.GlabcError, match="fall outside") as ei:
        eng.run_host(sampler, trace=trace, trace_layout=layout, **kw)
    assert ei.value.status == abi.ERR_INVALID
    for k, v in before.items():
        assert torch.equal(kw[k], v), f"{k} was written"


@pytest.mark.parametrize("sampler", ["global", "mala", "aglmcmc"])
def test_chain_major_trace_with_fewer_chains_than_the_run(eng, sampler):
    """a chain-major host trace holding 4 of the run's 8 chains, a leading view of a bigger buffer: the rows of chains 4..7
    would land in the rest of that buffer"""
    big = torch.full((C, T, D), SENTINEL)
    view = big[:C // 2]
    assert view.is_contiguous()
    assert_refused(eng, sampler, view, abi.TRACE_CHAIN_MAJOR, host_args(eng, sampler))
    assert bool((big == SENTINEL).all())
    eng.run_host(sampler, trace=big, trace_layout=abi.TRACE_CHAIN_MAJOR, **host_args(eng, sampler))   # the same run fits `big`
    assert not bool((big == SENTINEL).any())


@pytest.mark.parametrize("layout", [abi.TRACE_TIME_MAJOR, abi.TRACE_CHAIN_MAJOR], ids=["time", "chain"])
def test_multi_chunk_trace_one_row_short(eng, layout):
    """a run of four 32-step chunks into a host trace one row short is refused before the first chunk, not at the last"""
    kw = host_args(eng, "global")
    kw["chunk_steps"] = 32
    trace = torch.full((T - 1, C, D) if layout == abi.TRACE_TIME_MAJOR else (C, T - 1, D), SENTINEL)
    assert_refused(eng, "global", trace, layout, kw)
    assert bool((trace == SENTINEL).all())
