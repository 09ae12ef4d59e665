"""Host driver of the block-iSIR samplers whose importance proposal is SHARED by all chains: GLMCMC-NFs (one RealNVP,
GLMCMC_NFs.py:90-152) and pooled AGLMCMC (one KernelDensity over the pooled training draws, AGLMCMC.py:124-272).

The chain step is the fused kernel `k_ag_step<EXT>` (csrc/step_aglmcmc.cuh) behind `glabc_run_block_isir` — for a run-time
compiled `models.UserModel` its NVRTC twin `glabc_k_block_isir_user` (csrc/user_model.cu) behind `glabc_run_block_isir_user`,
with the block weights from `glabc_block_weights_user`: a chain pauses
when its block of batch_size * step_size candidates is consumed or when the proposal log-density of a changed state is
needed.  This loop refreshes those log-densities in one batched launch of the proposal's kernel and, when every chain of
the rank has consumed its block, lets the proposal adapt (train / refit — the only place ranks exchange data) and refills.

A proposal object provides
    fill(blk_theta [C,B,d], blk_lq [C,B], round)   fresh candidates and their log-densities (kernels)
    log_prob(theta [n,d]) -> [n]                    proposal log-density of the given states (kernel)
    adapt(block) -> None                            end-of-block training; may run collectives, every rank calls it
"""
import torch

from . import _abi
from .engine import RunStats
from .models import UserModel
from .pooled import RoundSync, _world
from .samplers import _ARITH, _LAYOUT, print_summary, write_csv


class Block:
    """a rank's candidate blocks and per-chain counters (glabc_block_isir_t, include/glabc.h)"""

    def __init__(self, c, K, S, d, yd, dev):
        B = K * S
        self.c, self.K, self.S, self.B, self.d = c, K, S, B, d
        self.theta = torch.empty(c, B, d, device=dev)
        self.x = torch.empty(c, B, yd, device=dev)
        self.w = torch.empty(c, B, device=dev)
        self.lq = torch.empty(c, B, device=dev)
        self.kk = torch.zeros(c, dtype=torch.int32, device=dev)
        self.pending = torch.zeros_like(self.kk)
        self.lq_valid = torch.zeros_like(self.kk)
        self.next_step = torch.ones(c, dtype=torch.int32, device=dev)
        self.lq_cur = torch.zeros(c, device=dev)
        self.pod = _abi.BlockIsirPOD(step_size=S, block=B, blk_theta=self.theta.data_ptr(), blk_x=self.x.data_ptr(),
                                     blk_w=self.w.data_ptr(), blk_lq=self.lq.data_ptr(), kk=self.kk.data_ptr(),
                                     pending=self.pending.data_ptr(), next_step=self.next_step.data_ptr(),
                                     lq_cur=self.lq_cur.data_ptr(), lq_valid=self.lq_valid.data_ptr())


BLOCK_CHECKPOINT_VERSION = 1
_BLOCK_TENSORS = ("theta", "x", "w", "lq", "kk", "pending", "lq_valid", "next_step", "lq_cur")


def run_block_isir(eng, model, proposal, *, num_ite, theta, y, K, S, gf, seed, chain_id_base, arith, trace, single,
                   filelocation, verbose, max_adapt=None, checkpoint=None, resume=None):
    """Advance every chain to iteration num_ite - 1.  Returns (result, RunStats, rounds).
    `model`: the bound built-in model's POD (Engine.bind_model), or a `models.UserModel`, whose kernels run FAST arithmetic
    (`arith` is ignored) and whose checkpoints carry its fingerprint: a resume refuses another model's checkpoint and one written
    by a built-in run, and a built-in run refuses a user model's.
    `checkpoint=path` writes the end-of-run state: chain state, statistics, every chain's candidate block and counters, the
    round / adaptation counters, the proposal's own state (`proposal.state_dict()`: flow weights + Adam moments, or the pooled
    KDE) and the host generators the adaptation draws from; `resume=path` continues from exactly that state (the returned trace
    then holds only the new rows).  The blocks of ALL chains are refilled when every chain has finished or consumed its block,
    so the iteration at which a run is cut is part of that schedule: a cut-and-resumed run equals the uncut one when the chains
    consume their blocks in step (global_frequency = 1; tested), and is a deterministic function of the checkpoint otherwise."""
    c, d = theta.shape
    dev = eng.device
    user = isinstance(model, UserModel)
    blk = Block(c, K, S, d, model.y_dim, dev)
    done0, rnd, n_adapt = 0, 0, 0
    stats = torch.zeros(c, _abi.nstats(d), device=dev)
    if resume is not None:
        ck = resume if isinstance(resume, dict) else torch.load(resume, map_location="cpu", weights_only=False)
        if ck.get("version") != BLOCK_CHECKPOINT_VERSION or ck.get("kind") != type(proposal).__name__:
            raise ValueError("not a block-iSIR checkpoint of this sampler")
        if ck.get("model") != (model.fingerprint() if user else None):
            raise ValueError("the checkpoint was written for another model (a user model's source, dims, params or epsilon differ, "
                             "or one of the two runs used the built-in family)")
        if ck["theta"].shape != theta.shape or (ck["K"], ck["S"]) != (K, S):
            raise ValueError("the checkpoint was written for another number of chains / block shape")
        theta.copy_(ck["theta"])
        y.copy_(ck["y"])
        stats.copy_(ck["stats"])
        for name in _BLOCK_TENSORS:
            getattr(blk, name).copy_(ck["blk"][name])
        done0, rnd, n_adapt, seed, chain_id_base = ck["done"], ck["rnd"], ck["n_adapt"], ck["seed"], ck["chain_id_base"]
        if num_ite - 1 < done0:
            raise ValueError(f"the checkpoint is already at iteration {done0}")
        proposal.load_state_dict(ck["proposal"])
        torch.set_rng_state(ck["torch_rng"])
    common = dict(theta=theta, y=y, gf=gf, seed=seed, chain_id_base=chain_id_base, K=K, blk=blk.pod)

    def refill(rnd):    # GLMCMC_NFs.py:70-85,125-140 / AGLMCMC.py:84-112,219-249
        proposal.fill(blk.theta, blk.lq, rnd)
        if user:
            eng.run_user(model, sampler="block_weights", n_steps=0, round=rnd, trace_layout=_abi.TRACE_NONE, **common)
        else:
            eng.run("block_weights", n_steps=0, step_base=rnd, trace_layout=_abi.TRACE_NONE, **common)

    def refresh_lq(idx=None):   # proposal.log_prob(Theta_old), GLMCMC_NFs.py:96-98 / AGLMCMC.py:137-140, where the state changed
        if idx is None:
            blk.lq_cur.copy_(proposal.log_prob(theta))
            blk.lq_valid.fill_(1)
        else:
            blk.lq_cur[idx] = proposal.log_prob(theta[idx])
            blk.lq_valid[idx] = 1

    if resume is None:
        refill(0)
        refresh_lq()
    layout = _LAYOUT[trace]
    n_steps = num_ite - 1                       # absolute index of the last iteration (chains carry their own next_step)
    rows = num_ite if resume is None else n_steps - done0
    if rows == 0:
        layout = _abi.TRACE_NONE
    out = None
    if layout != _abi.TRACE_NONE:
        out = torch.empty((rows, c, d) if layout == _abi.TRACE_TIME_MAJOR else (c, rows, d), device=dev)
    world = _world()[1]
    sync = RoundSync(dev)
    first = resume is None
    window = dict(step_base=done0, trace_row_base=0 if resume is None else done0 + 1, trace_rows=rows)
    while True:
        if user:
            eng.run_user(model, sampler="block_isir", n_steps=n_steps - done0, trace_layout=layout, trace=out, write_row0=first,
                         stats=stats, **window, **common)
        else:
            eng.run("block_isir", n_steps=n_steps - done0, arith=_ARITH[arith], trace_layout=layout, trace=out,
                    write_row0=first, stats=stats, **window, **common)
        first = False
        need = (blk.pending & 2) != 0
        settled = (blk.next_step > n_steps) | ((blk.pending & 1) != 0)
        n_need, n_done, n_settled = torch.stack([need.sum(), (blk.next_step > n_steps).sum(), settled.sum()]).tolist()
        if n_need:
            refresh_lq(need.nonzero().squeeze(1))
        if world == 1 and n_done == c:
            break
        if n_need == 0 and n_settled == c:      # every chain of this rank consumed its block (GLMCMC_NFs.py:111)
            if world > 1 and sync.round_end(n_done == c):
                break
            if max_adapt is None or n_adapt < max_adapt:
                proposal.adapt(blk)
                n_adapt += 1
            if n_done < c:
                rnd += 1
                refill(rnd)
                refresh_lq()
                blk.kk.zero_()
                blk.pending.zero_()
    if checkpoint is not None:
        cpu = lambda t: t.detach().cpu()  # noqa: E731
        extra = dict(model=model.fingerprint()) if user else {}
        torch.save(dict(version=BLOCK_CHECKPOINT_VERSION, kind=type(proposal).__name__, K=K, S=S, done=n_steps, rnd=rnd, n_adapt=n_adapt,
                        seed=int(seed), chain_id_base=int(chain_id_base), theta=cpu(theta), y=cpu(y), stats=cpu(stats),
                        blk={name: cpu(getattr(blk, name)) for name in _BLOCK_TENSORS}, proposal=proposal.state_dict(),
                        torch_rng=torch.get_rng_state(), **extra), checkpoint)
    rs = RunStats(stats, d)
    if single:
        chain = (out[0] if layout == _abi.TRACE_CHAIN_MAJOR else out[:, 0]).cpu() if out is not None else None
        if filelocation is not None and chain is not None:
            write_csv(filelocation, chain)
        if verbose is not False and chain is not None:
            print_summary(chain)
        result = chain
    else:
        if filelocation is not None and out is not None:
            import numpy as np
            np.save(filelocation if str(filelocation).endswith(".npy") else str(filelocation) + ".npy", out.cpu().numpy())
        result = out
    return result, rs, rnd
