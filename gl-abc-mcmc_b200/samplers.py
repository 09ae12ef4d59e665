"""Shared host driver of the sampler entry points (GlobalMCMC / GLMCMC / ...).

Mirrors what every reference sampler does around its loop — initial state, `Theta_Re` allocation
with row 0 = initial theta (GlobalMCMC.py:31-35), CSV trace (GlobalMCMC.py:27-30,70-76), the
end-of-run summary print (GlobalMCMC.py:77-97) — and hands the loop itself to the fused kernel.
Extension over the reference: `num_chains` independent chains per call, sharded by the caller
across GPUs through `chain_id_base` (see sharding.py).
"""
import csv

import numpy as np
import torch

from . import _abi
from .engine import RunStats, get_engine

_ARITH = {"fast": _abi.ARITH_FAST, "strict": _abi.ARITH_STRICT}
_LAYOUT = {"chain": _abi.TRACE_CHAIN_MAJOR, "time": _abi.TRACE_TIME_MAJOR, "none": _abi.TRACE_NONE}


def default_seed():
    """One draw from torch's global CPU generator: reproducible under torch.manual_seed(s) in the user script, as the
    reference is, and ADVANCING between calls, as the reference's draws from the global generator do — two successive
    sampler calls without seed= are independent runs, not replays of the same Philox streams."""
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def initial_state(eng, model_pod, Initial_theta, Initial_y, num_chains, seed):
    d, yd = model_pod.theta_dim, model_pod.y_dim
    theta = torch.as_tensor(Initial_theta, dtype=torch.float32).reshape(-1, d)
    c = num_chains if num_chains is not None else theta.shape[0]
    if theta.shape[0] not in (1, c):
        raise ValueError(f"Initial_theta has {theta.shape[0]} rows for {c} chains")
    theta = theta.to(eng.device).expand(c, d).contiguous()
    if Initial_y is None:
        # y0 ~ simulator(theta0), one draw per chain (the reference's scripts do this on the host,
        # Mixture.py:66); drawn with a device generator keyed by the seed
        g = torch.Generator(device=eng.device).manual_seed(seed & 0x7FFFFFFFFFFFFFFF)
        eps = torch.randn(c, yd, generator=g, device=eng.device)
        scale = torch.tensor(list(model_pod.noise_scale)[:yd], device=eng.device)
        loc = torch.tensor(list(model_pod.noise_loc)[:yd], device=eng.device)
        mean = theta.abs() if model_pod.family == _abi.MODEL_ABS_NORMAL else theta
        y = mean + (loc + scale * eps)
    else:
        y = torch.as_tensor(Initial_y, dtype=torch.float32).reshape(-1, yd)
        if y.shape[0] not in (1, c):
            raise ValueError(f"Initial_y has {y.shape[0]} rows for {c} chains")
        y = y.to(eng.device).expand(c, yd)
    return theta.clone(), y.contiguous().clone(), c


def write_csv(path, chain):
    """Trace CSV in the reference's format (no header, row 0 = initial theta, one row per
    iteration, str(np.float32) values; GlobalMCMC.py:27-30,70-76) — each row written once
    (the reference's final flush rewrites up to 10,000 rows, SURVEY.md B-9)."""
    arr = chain.detach().cpu().numpy()
    with open(path, "w", newline="", encoding="utf-8") as f:
        w = csv.writer(f)
        for row in arr:
            w.writerow(row)


def print_summary(chain):
    """mean / variance / mean +- 1.96 std per coordinate — the reference's closing print
    (GlobalMCMC.py:77-97; the "95% CI" there is mean +- 1.96*std, reproduced as is)."""
    chain = chain.detach().float().cpu()
    means, variances = torch.mean(chain, dim=0), torch.var(chain, dim=0)
    for i in range(chain.size(1)):
        std = torch.std(chain[:, i])
        m = means[i].item()
        print(f"Theta_Re {i + 1}:")
        print(f"  Mean: {m:.4f}")
        print(f"  Variance: {variances[i].item():.4f}")
        print(f"  95% Confidence Interval: {(m - 1.96 * std, m + 1.96 * std)}")


CHECKPOINT_VERSION = 1


def save_checkpoint(path, *, sampler, step_base, seed, chain_id_base, theta, y, stats, aux=None, state64=None, ag_state=None,
                    model=None):
    """Everything a run needs to continue bit-identically (SURVEY.md 8(f) n4): the chain state, the carried iSIR / MALA
    state, the statistics accumulators and the Philox coordinates (seed, global chain id base, next step index) — the
    generator itself is stateless, so no RNG state exists beyond these three integers.  `model`: a user model's
    fingerprint (models.UserModel.fingerprint)."""
    cpu = lambda t: None if t is None else t.detach().cpu()  # noqa: E731
    extra = {} if model is None else dict(model=model)
    torch.save(dict(version=CHECKPOINT_VERSION, sampler=sampler, step_base=int(step_base), seed=int(seed),
                    chain_id_base=int(chain_id_base), theta=cpu(theta), y=cpu(y), stats=cpu(stats), aux=cpu(aux),
                    state64=cpu(state64), ag_state=cpu(ag_state), **extra), path)


def load_checkpoint(path_or_dict, sampler, device):
    ck = path_or_dict if isinstance(path_or_dict, dict) else torch.load(path_or_dict, map_location="cpu", weights_only=True)
    if ck.get("version") != CHECKPOINT_VERSION:
        raise ValueError(f"checkpoint version {ck.get('version')} (this build reads {CHECKPOINT_VERSION})")
    if ck["sampler"] != sampler:
        raise ValueError(f"checkpoint was written by the {ck['sampler']!r} sampler, not {sampler!r}")
    dev = lambda t: None if t is None else t.to(device).contiguous()  # noqa: E731
    return dict(ck, theta=dev(ck["theta"]), y=dev(ck["y"]), stats=dev(ck["stats"]), aux=dev(ck["aux"]), state64=dev(ck["state64"]),
                ag_state=dev(ck.get("ag_state")))


def continuation(step_base, num_ite, layout):
    """(launch arguments, trace layout) of a run resumed at iteration `step_base` up to iteration num_ite - 1: the launch
    continues the Philox steps and writes only the new rows step_base + 1 .. num_ite - 1; no trace when none is left."""
    if num_ite - 1 < step_base:
        raise ValueError(f"the checkpoint is already at iteration {step_base}")
    kw = dict(step_base=step_base, trace_row_base=step_base + 1, write_row0=False, trace_rows=num_ite - 1 - step_base)
    return kw, (_abi.TRACE_NONE if num_ite - 1 == step_base else layout)


def run_chains(sampler, eng, model_pod, *, num_ite, Initial_theta, Initial_y, global_frequency, filelocation,
               num_chains, seed, chain_id_base, arith, trace, return_stats, verbose, K=0, aux_init=None,
               block_threads=0, checkpoint=None, resume=None, **sampler_kw):
    """`checkpoint=path` writes the end-of-run state; `resume=path` continues a run from such a file up to iteration
    num_ite - 1 (same sampler, model and proposals): the chains continue bit-identically — the returned trace then holds
    only the NEW rows (iterations step_base + 1 .. num_ite - 1)."""
    if num_ite < 1:
        raise ValueError("num_ite must be at least 1")
    if trace not in _LAYOUT:
        raise ValueError(f"trace must be one of {sorted(_LAYOUT)}")
    d = model_pod.theta_dim
    layout = _LAYOUT[trace]
    resumed = {}
    if resume is not None:
        ck = load_checkpoint(resume, sampler, eng.device)
        theta, y, stats, aux = ck["theta"], ck["y"], ck["stats"], ck["aux"]
        seed, chain_id_base, c = ck["seed"], ck["chain_id_base"], ck["theta"].shape[0]
        if theta.shape[1] != d:
            raise ValueError("checkpoint theta_dim does not match the model")
        resumed, layout = continuation(ck["step_base"], num_ite, layout)
        if "state64" in sampler_kw:
            sampler_kw["state64"] = ck["state64"]
        if sampler == "aglmcmc":     # the chains' candidate blocks, KDEs, counters and eps-hat live in the context's workspace
            if ck.get("ag_state") is None:
                raise ValueError("the checkpoint holds no AGLMCMC workspace")
            ag = sampler_kw["ag"]
            eng.aglmcmc_restore(ck["ag_state"], c, int(K) * int(ag.step_size))
            ag.init = 0
    else:
        seed = default_seed() if seed is None else int(seed)
        theta, y, c = initial_state(eng, model_pod, Initial_theta, Initial_y, num_chains, seed)
        stats = torch.zeros(c, _abi.nstats(d), dtype=torch.float32, device=eng.device)
        aux = None
        if aux_init is not None:
            aux = torch.zeros(c, _abi.AUX_SLOTS, dtype=torch.float32, device=eng.device)
            for slot, val in aux_init.items():
                aux[:, slot] = val
    single = num_chains is None and c == 1
    step_base = resumed.get("step_base", 0)
    out = eng.run(sampler, theta=theta, y=y, n_steps=num_ite - 1 - step_base, gf=global_frequency, seed=seed,
                  chain_id_base=chain_id_base, arith=_ARITH[arith], trace_layout=layout, stats=stats, aux=aux, K=K,
                  block_threads=block_threads, **resumed, **sampler_kw)
    if checkpoint is not None:
        save_checkpoint(checkpoint, sampler=sampler, step_base=num_ite - 1, seed=seed, chain_id_base=chain_id_base, theta=theta,
                        y=y, stats=stats, aux=aux, state64=sampler_kw.get("state64"),
                        ag_state=eng.aglmcmc_state() if sampler == "aglmcmc" else None)
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
            np.save(filelocation if str(filelocation).endswith(".npy") else str(filelocation) + ".npy", out.cpu().numpy())
        if verbose and out is not None:
            print_summary(out.reshape(-1, d))
        result = out
    return (result, rs) if return_stats else result
