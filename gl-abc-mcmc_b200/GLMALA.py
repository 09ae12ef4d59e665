"""GLMALA — reference glabcmcmc/GLMALA.py:118-230: with probability `global_frequency` the iSIR global
move of GLMCMC (GLMALA.py:151-180), otherwise a MALA local move (GLMALA.py:182-200) drifted by a
finite-difference synthetic-likelihood gradient estimated from 2*d*num_grad simulator draws with common
random numbers (`numberical_gradient_logABC`, GLMALA.py:46-95).  The loop body runs in the fused kernel
`k_mala` (csrc/step_mala.cuh), one warp per chain."""
import torch

from . import _abi
from .engine import get_engine
from .GlobalMCMC import refuse_chains_per_dataset, run_user_model
from .models import UserModel
from .samplers import run_chains


def GLMALA(ABCset, num_ite, Initial_theta, Initial_y, tau, num_grad, filelocation, global_frequency=0,
           Importance_Proposal=None, batch_size=None, *, num_chains=None, seed=None, chain_id_base=0, arith="fast",
           trace="chain", return_stats=False, verbose=None, device=None, block_threads=0, checkpoint=None, resume=None,
           chains_per_dataset=None):
    """Same positional signature and return value as the reference for one chain; keyword extensions as in
    `GlobalMCMC` (num_chains, seed, chain_id_base, arith, trace, return_stats, chains_per_dataset)."""
    if Importance_Proposal is None or batch_size is None:
        raise ValueError("Importance_Proposal and batch_size are required (GLMALA.py:155,158 dereference them)")
    if not 1 <= int(batch_size) <= _abi.MAX_K:
        raise ValueError(f"batch_size must be in 1..{_abi.MAX_K}")
    if not 2 <= int(num_grad) <= _abi.MAX_NUM_GRAD:
        raise ValueError(f"num_grad must be in 2..{_abi.MAX_NUM_GRAD}")
    eng = get_engine(device)
    if isinstance(ABCset, UserModel):       # run-time compiled model (csrc/user_model.cu: glabc_k_mala_user)
        eng.bind_proposal(_abi.SLOT_IMPORTANCE, Importance_Proposal)
        return run_user_model(eng, ABCset, "mala", num_ite, Initial_theta, Initial_y, None, filelocation, global_frequency, num_chains,
                              seed, chain_id_base, trace, return_stats, verbose, block_threads, K=int(batch_size), num_grad=int(num_grad),
                              tau=float(tau), checkpoint=checkpoint, resume=resume, chains_per_dataset=chains_per_dataset)
    refuse_chains_per_dataset(chains_per_dataset)
    pod = eng.bind_model(ABCset)
    eng.bind_proposal(_abi.SLOT_IMPORTANCE, Importance_Proposal)
    state64 = None      # resume: the carried float64 state comes from the checkpoint (Initial_theta / Initial_y are not read)
    if resume is None:
        c = num_chains if num_chains is not None else torch.as_tensor(Initial_theta).reshape(-1, pod.theta_dim).shape[0]
        state64 = torch.zeros(c, _abi.STATE64_SLOTS, dtype=torch.float64, device=eng.device)
    return run_chains("mala", eng, pod, num_ite=num_ite, Initial_theta=Initial_theta, Initial_y=Initial_y,
                      global_frequency=global_frequency, filelocation=filelocation, num_chains=num_chains, seed=seed,
                      chain_id_base=chain_id_base, arith=arith, trace=trace, return_stats=return_stats, verbose=verbose,
                      K=int(batch_size), aux_init={_abi.AUX_LOCAL: 1.0}, block_threads=block_threads,
                      num_grad=int(num_grad), tau=float(tau), state64=state64, checkpoint=checkpoint, resume=resume)
