"""GLMCMC — reference glabcmcmc/GLMCMC.py:24-137: with probability `global_frequency` an iSIR global
move (`batch_size` fresh candidates from `Importance_Proposal` plus the current state, importance
weights prior*kernel/q, one categorical resample — `weight_sampling`, GLMCMC.py:7-22), otherwise a
random-walk Metropolis–Hastings move from `Local_Proposal`.  The loop body (GLMCMC.py:58-104) runs in
the fused kernel `k_isir` (csrc/step_isir.cuh) for all chains at once."""
from . import _abi
from .engine import get_engine
from .GlobalMCMC import run_user_model
from .models import UserModel
from .samplers import run_chains


def GLMCMC(ABCset, num_ite, Initial_theta, Initial_y, Local_Proposal, filelocation, global_frequency=0,
           Importance_Proposal=None, batch_size=None, *, num_chains=None, seed=None, chain_id_base=0, arith="fast",
           trace="chain", return_stats=False, verbose=None, device=None, block_threads=0, checkpoint=None, resume=None):
    """Same positional signature and return value as the reference for one chain; keyword extensions
    as in `GlobalMCMC` (num_chains, seed, chain_id_base, arith, trace, return_stats)."""
    if Importance_Proposal is None or batch_size is None:
        raise ValueError("Importance_Proposal and batch_size are required (GLMCMC.py:54,66 dereference them)")
    if not 1 <= int(batch_size) <= _abi.MAX_K:
        raise ValueError(f"batch_size must be in 1..{_abi.MAX_K}")
    eng = get_engine(device)
    if isinstance(ABCset, UserModel):       # run-time compiled model (csrc/user_model.cu)
        eng.bind_proposal(_abi.SLOT_IMPORTANCE, Importance_Proposal)
        return run_user_model(eng, ABCset, "isir", num_ite, Initial_theta, Initial_y, Local_Proposal, filelocation, global_frequency,
                              num_chains, seed, chain_id_base, trace, return_stats, verbose, block_threads, K=int(batch_size),
                              checkpoint=checkpoint, resume=resume)
    pod = eng.bind_model(ABCset)
    eng.bind_proposal(_abi.SLOT_LOCAL, Local_Proposal)
    eng.bind_proposal(_abi.SLOT_IMPORTANCE, Importance_Proposal)
    # carried state: cached log-weight (recomputed on first use because `local` starts True, GLMCMC.py:49-55,60-64)
    return run_chains("isir", eng, pod, num_ite=num_ite, Initial_theta=Initial_theta, Initial_y=Initial_y,
                      global_frequency=global_frequency, filelocation=filelocation, num_chains=num_chains, seed=seed,
                      chain_id_base=chain_id_base, arith=arith, trace=trace, return_stats=return_stats, verbose=verbose,
                      K=int(batch_size), aux_init={_abi.AUX_LOCAL: 1.0}, block_threads=block_threads, checkpoint=checkpoint, resume=resume)
