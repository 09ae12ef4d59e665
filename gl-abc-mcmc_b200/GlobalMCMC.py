"""GlobalMCMC — reference glabcmcmc/GlobalMCMC.py:6-98: each iteration is, with probability
`global_frequency`, an independence Metropolis–Hastings move from `Global_Proposal`, otherwise a
random-walk move from `Local_Proposal`; the ABC likelihood is a Gaussian kernel on the discrepancy
of one simulator draw.  The loop body (GlobalMCMC.py:37-68) runs in the fused kernel
`k_global_mcmc` (csrc/step_global.cu) for all chains at once."""
import torch

from . import _abi
from .engine import RunStats, get_engine
from .models import UserModel
from .samplers import (_LAYOUT, continuation, default_seed, load_checkpoint, print_summary, run_chains, save_checkpoint,
                       write_csv)


def GlobalMCMC(ABCset, num_ite, Initial_theta, Initial_y, Global_Proposal, filelocation, global_frequency,
               Local_Proposal=None, *, num_chains=None, seed=None, chain_id_base=0, arith="fast", trace="chain",
               return_stats=False, verbose=None, device=None, block_threads=0, checkpoint=None, resume=None, chains_per_dataset=None):
    """Same positional signature and return value as the reference (a float32 CPU tensor
    `[num_ite, theta_dim]`, row 0 = `Initial_theta`) when called for one chain.

    Keyword extensions: `num_chains=C` runs C independent chains and returns a device tensor
    `[C, num_ite, d]` (`trace="chain"`), `[num_ite, C, d]` (`trace="time"`) or None
    (`trace="none"`, statistics only); `Initial_theta` / `Initial_y` may then be one row (shared) or
    C rows, and `Initial_y=None` draws y0 from the simulator per chain.  `seed` defaults to
    `torch.initial_seed()`; chain c draws from the Philox stream of global id `chain_id_base + c`.
    `arith="strict"` evaluates in the reference's float32 operation order.  `return_stats=True`
    also returns the in-kernel `RunStats` (accept counts, moments, ESJD numerators).
    `chains_per_dataset=m`: required for a batched `UserModel` (2-D params) and refused otherwise; see
    `run_user_model`."""
    if Local_Proposal is None:
        raise ValueError("Local_Proposal is required (the reference dereferences it on every local move, GlobalMCMC.py:56)")
    eng = get_engine(device)
    if isinstance(ABCset, UserModel):
        eng.bind_proposal(_abi.SLOT_GLOBAL, Global_Proposal)
        return run_user_model(eng, ABCset, "global", num_ite, Initial_theta, Initial_y, Local_Proposal, filelocation,
                              global_frequency, num_chains, seed, chain_id_base, trace, return_stats, verbose, block_threads,
                              checkpoint=checkpoint, resume=resume, chains_per_dataset=chains_per_dataset)
    refuse_chains_per_dataset(chains_per_dataset)
    pod = eng.bind_model(ABCset)
    eng.bind_proposal(_abi.SLOT_LOCAL, Local_Proposal)
    eng.bind_proposal(_abi.SLOT_GLOBAL, Global_Proposal)
    return run_chains("global", eng, pod, num_ite=num_ite, Initial_theta=Initial_theta, Initial_y=Initial_y,
                      global_frequency=global_frequency, filelocation=filelocation, num_chains=num_chains, seed=seed,
                      chain_id_base=chain_id_base, arith=arith, trace=trace, return_stats=return_stats, verbose=verbose,
                      block_threads=block_threads, checkpoint=checkpoint, resume=resume)


def refuse_chains_per_dataset(chains_per_dataset):
    if chains_per_dataset is not None:
        raise ValueError("chains_per_dataset is for a batched UserModel (params of shape [G, n_params]) only")


def check_batched(model, chains_per_dataset, num_chains, chain_id_base):
    """the chain count of a user-model run (None: from Initial_theta) after the batched-model checks: a batched model needs
    chains_per_dataset = m >= 1, defaults num_chains to G m, and its chain ids chain_id_base .. + C - 1 must stay below G m"""
    if not model.batched:
        refuse_chains_per_dataset(chains_per_dataset)
        return num_chains
    if chains_per_dataset is None:
        raise ValueError(f"a batched UserModel ({model.n_datasets} datasets) needs chains_per_dataset=m: chain id g runs "
                         "against dataset g // m")
    m = int(chains_per_dataset)
    if m < 1:
        raise ValueError("chains_per_dataset must be at least 1")
    total = model.n_datasets * m
    c = total if num_chains is None else int(num_chains)
    if chain_id_base < 0 or chain_id_base + c > total:
        raise ValueError(f"chain ids {chain_id_base} .. {chain_id_base + c - 1} reach beyond the {model.n_datasets} datasets x "
                         f"{m} chains of the batched model")
    return c


def _rows(x, width, c, what, per_dataset=None):
    """x as [c, width] on the device: 1 row (shared), c rows, or (batched) one row per dataset, indexed by per_dataset"""
    x = torch.as_tensor(x, dtype=torch.float32).reshape(-1, width)
    if x.shape[0] == c or x.shape[0] == 1:
        return x.expand(c, width).contiguous().clone()
    if per_dataset is not None and x.shape[0] == per_dataset[1]:
        return x[per_dataset[0]].contiguous()
    want = f"1, {per_dataset[1]} (one per dataset) or {c}" if per_dataset is not None else f"1 or {c}"
    raise ValueError(f"{what} must have {want} rows")


def user_initial_state(eng, model, Initial_theta, Initial_y, num_chains, seed, chain_id_base, chains_per_dataset=None):
    """(theta [C, theta_dim], y [C, y_dim], C) of a user-model run: Initial_theta / Initial_y of 1 or C rows (a batched model
    also takes G rows, row g for the m chains of dataset g); Initial_y=None draws y0 of chain c with the model's simulator
    (glabc_user_simulate, Philox id chain_id_base + c at step 0, a batched model's with the chain's dataset)"""
    d, yd = model.theta_dim, model.y_dim
    per_dataset = None
    if model.batched:
        c = num_chains
        ids = torch.arange(chain_id_base, chain_id_base + c, dtype=torch.int64)
        per_dataset = (ids // int(chains_per_dataset), model.n_datasets)
    else:
        c = num_chains if num_chains is not None else torch.as_tensor(Initial_theta).reshape(-1, d).shape[0]
    theta = _rows(Initial_theta, d, c, "Initial_theta", per_dataset).to(eng.device)
    if Initial_y is None:
        y = eng.user_simulate(model, theta, seed, row_base=chain_id_base, chains_per_dataset=chains_per_dataset or 0)
    else:
        y = _rows(Initial_y, yd, c, "Initial_y", per_dataset).to(eng.device)
    return theta, y, c


def run_user_model(eng, model, sampler, num_ite, Initial_theta, Initial_y, Local_Proposal, filelocation, gf, num_chains,
                   seed, chain_id_base, trace, return_stats, verbose, block_threads, K=0, num_grad=0, tau=0.0, checkpoint=None,
                   resume=None, chains_per_dataset=None):
    """GlobalMCMC / GLMCMC / GLMALA for a run-time compiled `UserModel` (glabc_run_{global,isir,mala}_user); the caller has
    bound the sampler's state-independent proposal (GLOBAL / IMPORTANCE slot).  `Initial_y=None` draws y0 of chain c with the
    model's simulator (glabc_user_simulate, Philox id chain_id_base + c at step 0), so y0 does not depend on the sharding.
    `checkpoint=` / `resume=` as in samplers.run_chains; the checkpoint also names the model (UserModel.fingerprint), and a
    resume refuses one written for another model or by another sampler (a built-in run's included).
    A batched model (`model.batched`) needs `chains_per_dataset=m`: chain id g runs against dataset g // m, `num_chains`
    defaults to G m, and the checkpoint records m; a resume with another table or another m is refused."""
    if num_ite < 1:
        raise ValueError("num_ite must be at least 1")
    if trace not in _LAYOUT:
        raise ValueError(f"trace must be one of {sorted(_LAYOUT)}")
    if sampler != "mala":
        eng.bind_proposal(_abi.SLOT_LOCAL, Local_Proposal)
    d, yd = model.theta_dim, model.y_dim
    name = sampler + "_user"
    layout = _LAYOUT[trace]
    resumed = {}
    m = None if chains_per_dataset is None else int(chains_per_dataset)
    if resume is not None:
        ck = load_checkpoint(resume, name, eng.device)
        if ck.get("model") != model.fingerprint():
            raise ValueError("the checkpoint was written for another user model (source, dims, params or epsilon differ)")
        if ck.get("chains_per_dataset") != m:
            raise ValueError(f"the checkpoint was written with chains_per_dataset={ck.get('chains_per_dataset')}, not {m}")
        theta, y, stats, aux = ck["theta"], ck["y"], ck["stats"], ck["aux"]
        seed, chain_id_base, c = ck["seed"], ck["chain_id_base"], theta.shape[0]
        check_batched(model, m, c, chain_id_base)
        resumed, layout = continuation(ck["step_base"], num_ite, layout)
    else:
        seed = default_seed() if seed is None else int(seed)
        num_chains = check_batched(model, m, num_chains, chain_id_base)
        theta, y, c = user_initial_state(eng, model, Initial_theta, Initial_y, num_chains, seed, chain_id_base, m)
        stats = torch.zeros(c, _abi.nstats(d), dtype=torch.float32, device=eng.device)
        aux = None
        if sampler in ("isir", "mala"):
            aux = torch.zeros(c, _abi.AUX_SLOTS, dtype=torch.float32, device=eng.device)
            aux[:, _abi.AUX_LOCAL] = 1.0                        # `local` starts True, GLMCMC.py:49-55
    single = num_chains is None and c == 1 and not model.batched
    step_base = resumed.get("step_base", 0)
    out = eng.run_user(model, theta=theta, y=y, n_steps=num_ite - 1 - step_base, gf=gf, seed=seed, chain_id_base=chain_id_base,
                       trace_layout=layout, stats=stats, block_threads=block_threads, sampler=sampler, K=K, aux=aux,
                       num_grad=num_grad, tau=tau, chains_per_dataset=m or 0, **resumed)
    if checkpoint is not None:
        save_checkpoint(checkpoint, sampler=name, step_base=num_ite - 1, seed=seed, chain_id_base=chain_id_base, theta=theta, y=y,
                        stats=stats, aux=aux, model=model.fingerprint(), chains_per_dataset=m)
    rs = RunStats(stats, d)
    if single:
        result = (out[0] if layout == _abi.TRACE_CHAIN_MAJOR else out[:, 0]).cpu() if out is not None else None
        if filelocation is not None and result is not None:
            write_csv(filelocation, result)
        if verbose is not False and result is not None:
            print_summary(result)
    else:
        result = out
    return (result, rs) if return_stats else result
