"""AGLMCMC — reference glabcmcmc/AGLMCMC.py:44-288: iSIR against a block of batch_size * step_size pre-generated
importance candidates; after step_size global moves the auxiliary tolerance eps-hat shrinks by a quantile rule, a
weighted KernelDensity is refit on the block and the next block is sampled from it.  The loop body and the adaptation
run in the kernels of csrc/step_aglmcmc.cuh + csrc/kde.cuh for all chains at once (every chain owns its block and KDE,
as the reference's single chain does).

Deviations from the reference, on purpose (SURVEY.md B-10): the chain is returned (the reference returns None and
crashes past 10,000 iterations) and row 0 holds the initial theta."""
import math

import torch

from . import _abi
from .block_isir import run_block_isir
from .distribution import DiagGaussian
from .engine import get_engine
from .GlobalMCMC import user_initial_state
from .models import UserModel
from .pooled import _world, gather_training_draws, update_hat_eps
from .samplers import default_seed, initial_state, run_chains


class PooledKDEProposal:
    """ONE KernelDensity shared by all chains of all ranks (BASELINE config 5) as the external proposal of
    `block_isir.run_block_isir`.  Until the first adaptation the proposal is `Initial_ISIR_prop` (AGLMCMC.py:84-91,137-138).
    `adapt` is AGLMCMC.py:170-217 on the pooled block: the tolerance eps-hat from the pooled discrepancies (counts
    all-reduced), training weights prior * K_eps-hat / q (:199-203), `kde_train / world` systematic draws per rank
    all-gathered into the training set (:206-214), `KernelDensity.fit` (glabc_kde_fit), then candidates from
    glabc_kde_sample and their log-densities from glabc_kde_log_prob — c * B queries against the pooled points, the
    pairwise kernel the path is named for.  Candidates below the prior floor (:223-224) keep log q = +inf, i.e. weight 0
    (the reference oversamples 4x and takes the first B valid ones; a zero-weight candidate is never selected either).
    `pod` may be a `models.UserModel`: the discrepancies and the prior then come from its compiled plugin methods
    (glabc_user_evaluate), and no slot is bound for the prior."""

    def __init__(self, eng, pod, alpha, hat_eps_T, kde_train, seed, chain_id_base, rule=_abi.BW_SILVERMAN):
        self.eng, self.pod, self.alpha, self.hat_eps_T = eng, pod, float(alpha), float(hat_eps_T)
        self.rank, self.world = _world()
        self.m = max(1, int(kde_train) // self.world)
        self.rule = rule
        self.seed = (int(seed) * 0x9E3779B1 + int(chain_id_base) + 0xA6) & 0x7FFFFFFFFFFFFFFF
        self.gen = torch.Generator(device=eng.device).manual_seed(self.seed)
        self.hat_eps = 1000000.0                      # AGLMCMC.py:119
        self.kde = None                               # (X [n, d], weights [n], bw [d])
        self.history = []                             # (hat_eps, n_train, bandwidth) per adaptation
        self.floor = math.log(1e-10)
        self.user = pod if isinstance(pod, UserModel) else None
        if self.user is not None:
            return
        d = pod.theta_dim
        self.y_obs = torch.tensor(list(pod.y_obs)[:pod.y_dim], device=eng.device)
        # the prior as a device distribution: its log-density of the candidates is the kernel behind glabc_dist_log_prob
        prior = eng.prior_pod if eng.prior_pod is not None else DiagGaussian(d, torch.tensor(list(pod.prior_loc)[:d]),
                                                                              torch.tensor(list(pod.prior_log_scale)[:d]))
        eng.bind_proposal(_abi.SLOT_GLOBAL, prior)

    def _prior(self, theta):
        """log prior of theta [n, d]: the model's compiled prior_log_prob, or the bound prior's kernel"""
        if self.user is not None:
            return self.eng.user_evaluate(self.user, _abi.USER_PRIOR, theta)
        return self.eng.dist_log_prob(_abi.SLOT_GLOBAL, theta)

    def _discrepancy(self, x):
        """discrepancies of the block's simulations x [c, B, y_dim], flattened"""
        if self.user is not None:
            return self.eng.user_evaluate(self.user, _abi.USER_DISCREPANCY, x.reshape(-1, x.shape[-1]))
        return torch.sqrt(torch.sum((x - self.y_obs) ** 2, dim=-1)).reshape(-1)       # Mixture.py:33-36

    def state_dict(self):
        """the pooled KernelDensity (points, normalised weights, bandwidth), eps-hat, the generator of the training draws"""
        kde = None if self.kde is None else tuple(t.cpu() for t in self.kde)
        return dict(kde=kde, hat_eps=self.hat_eps, gen=self.gen.get_state(), history=list(self.history))

    def load_state_dict(self, sd):
        self.kde = None if sd["kde"] is None else tuple(t.to(self.eng.device).contiguous() for t in sd["kde"])
        self.hat_eps = float(sd["hat_eps"])
        self.gen.set_state(sd["gen"])
        self.history = list(sd["history"])

    def fill(self, blk_theta, blk_lq, rnd):
        c, B, d = blk_theta.shape
        s = (self.seed + 0x632BE5AB * (rnd + 1)) & 0x7FFFFFFFFFFFFFFF
        if self.kde is None:
            z, lp = self.eng.dist_sample(_abi.SLOT_IMPORTANCE, c * B, d, seed=s)
        else:
            X, w, bw = self.kde
            z = self.eng.kde_sample(X, w, bw, c * B, seed=s)
            lp = self.eng.kde_log_prob(X, w, bw, z)
            prior = self._prior(z)
            lp = torch.where(prior > self.floor, lp, torch.full_like(lp, float("inf")))
        blk_theta.copy_(z.view(c, B, d))
        blk_lq.copy_(lp.view(c, B))

    def log_prob(self, theta):
        if self.kde is None:
            return self.eng.dist_log_prob(_abi.SLOT_IMPORTANCE, theta)
        X, w, bw = self.kde
        return self.eng.kde_log_prob(X, w, bw, theta.contiguous())

    def adapt(self, blk):
        d = blk.d
        dis = self._discrepancy(blk.x)
        self.hat_eps = update_hat_eps(dis, self.hat_eps, self.alpha, self.hat_eps_T)      # AGLMCMC.py:174-196
        he = torch.tensor(self.hat_eps, dtype=torch.float32, device=dis.device)
        like = -0.5 * math.log(2 * math.pi) - (torch.log(he) + 0.5 * (dis / he) ** 2)     # calculate_log_kernel_dis(dis0, hat_eps)
        prior = self._prior(blk.theta.reshape(-1, d))
        w_train = torch.exp(prior + like - blk.lq.reshape(-1))                            # :199-203
        u = float(torch.rand(1, generator=self.gen, device=dis.device))
        X, w = gather_training_draws(blk.theta.reshape(-1, d), w_train, self.m, u)        # the all-gather of SURVEY 8(e)
        if X.shape[0] < 2:
            return                                                                        # nothing to fit: keep the proposal
        weights, bw = self.eng.kde_fit(X, w, rule=self.rule)                              # :210-214
        self.kde = (X, weights, bw)
        self.history.append((self.hat_eps, int(X.shape[0]), bw.tolist()))


def AGLMCMC(ABCset, num_ite, Initial_theta, Initial_y, Local_Proposal, Initial_ISIR_prop, filelocation, global_frequency,
            step_size, batch_size, alpha, hat_eps_T, device=None, *, num_chains=None, seed=None, chain_id_base=0, arith="fast",
            trace="chain", return_stats=False, verbose=None, block_threads=0, pooled=False, kde_train=100000,
            return_proposal=False, checkpoint=None, resume=None):
    """Same positional signature as the reference; keyword extensions as in `GlobalMCMC`.  `pooled=True`: all chains (of
    all ranks of the process group) share ONE KernelDensity fitted on `kde_train` pooled weighted draws instead of one KDE
    per chain — see `PooledKDEProposal`.  `checkpoint=` / `resume=` (per-chain mode): the end-of-run state incl. every chain's
    candidate block, KernelDensity and eps-hat (pooled mode: the shared KDE); a resumed run continues bit-identically.
    `ABCset` may be a `models.UserModel` of theta_dim <= 4 with `pooled=True`: the block-iSIR step and the block weights run in
    the kernels compiled with the model (FAST arithmetic, `arith` ignored).  The per-chain mode's adaptation kernels are built
    for the fused family only, so it refuses a user model."""

    if not 1 <= int(batch_size) <= _abi.MAX_K:
        raise ValueError(f"batch_size must be in 1..{_abi.MAX_K}")
    if int(step_size) < 1 or int(step_size) * int(batch_size) > _abi.AG_MAX_BLOCK:
        raise ValueError(f"batch_size * step_size must be in 1..{_abi.AG_MAX_BLOCK}")
    eng = get_engine(device)
    user = isinstance(ABCset, UserModel)      # run-time compiled model (csrc/user_model.cu: glabc_k_block_isir_user)
    if user and not pooled:
        raise NotImplementedError("AGLMCMC runs a UserModel with pooled=True (one KernelDensity shared by all chains); the "
                                  "per-chain mode's adaptation kernels are built for the fused model family only")
    if user and ABCset.batched:
        raise ValueError("pooled AGLMCMC pools one KernelDensity over all chains, which is meaningless across the datasets of "
                         "a batched UserModel: run each model.dataset(g) on its own")
    if user and ABCset.theta_dim > 4:
        raise NotImplementedError("pooled AGLMCMC with a UserModel needs theta_dim <= 4 (the KernelDensity and proposal-sampling "
                                  "kernels are built for 1..4 dimensions)")
    pod = ABCset if user else eng.bind_model(ABCset)
    eng.bind_proposal(_abi.SLOT_LOCAL, Local_Proposal)
    eng.bind_proposal(_abi.SLOT_IMPORTANCE, Initial_ISIR_prop)
    if pooled:
        seed = default_seed() if seed is None else int(seed)
        if user:
            theta, y, c = user_initial_state(eng, ABCset, Initial_theta, Initial_y, num_chains, seed, chain_id_base)
        else:
            theta, y, c = initial_state(eng, pod, Initial_theta, Initial_y, num_chains, seed)
        prop = PooledKDEProposal(eng, pod, alpha, hat_eps_T, kde_train, seed, chain_id_base)
        result, rs, _ = run_block_isir(eng, pod, prop, num_ite=num_ite, theta=theta, y=y, K=int(batch_size), S=int(step_size),
                                       gf=global_frequency, seed=seed, chain_id_base=chain_id_base, arith=arith, trace=trace,
                                       single=num_chains is None and c == 1, filelocation=filelocation, verbose=verbose,
                                       checkpoint=checkpoint, resume=resume)
        extra = ((rs,) if return_stats else ()) + ((prop,) if return_proposal else ())
        return (result,) + extra if extra else result
    ag = eng.aglmcmc_params(step_size=step_size, alpha=alpha, hat_eps_T=hat_eps_T)
    return run_chains("aglmcmc", eng, pod, num_ite=num_ite, Initial_theta=Initial_theta, Initial_y=Initial_y,
                      global_frequency=global_frequency, filelocation=filelocation, num_chains=num_chains, seed=seed,
                      chain_id_base=chain_id_base, arith=arith, trace=trace, return_stats=return_stats, verbose=verbose,
                      K=int(batch_size), block_threads=block_threads, ag=ag, checkpoint=checkpoint, resume=resume)
