"""GLMCMC_NF — reference glabcmcmc/GLMCMC_NFs.py:43-186: iSIR whose importance proposal is a 32-block RealNVP trained
online by forward KL on importance-resampled candidates.  Per block of `step_size` global moves: candidates
theta0 ~ flow (GLMCMC_NFs.py:72,127), weights prior * kernel / q (:80-85); each global move resamples among the current
state and the next `batch_size` candidates (:92-110); after the block, at most `Train_step` times, one Adam step on
-mean log q(theta0[resample(w0)]) (:112-124), then a new block from the updated flow.

B200 mapping (many chains, ONE shared flow — the reference's single chain has one flow):
  * flow sample / log_prob for all chains' candidates: tcgen05 tensor-core kernel (csrc/flow.cuh);
  * the chain step against the block: fused kernel `k_ag_step<EXT>` (csrc/step_aglmcmc.cuh) — a chain pauses when its
    block is consumed or when the proposal log-density of a changed state is needed; this host loop then refreshes those
    log-densities in one batched log_prob launch, and at the end of a block trains / rebinds the flow and refills;
  * the <= Train_step training steps (forward KL on systematically resampled candidates, backward, Adam) are kernels of the
    extension too: `resample` -> glabc_resample, forward_kld / backward -> glabc_flow_grad (tcgen05 GEMMs, csrc/flow_train.cuh),
    the flat gradient all-reduced over the ranks, Adam -> glabc_flow_adam_step.  flows.RealNVP keeps an fp32 torch autograd
    restatement of the same network as the tests' checker (`flow_train="torch"`).
Parity note: `normflows` cannot be installed here, so this path is unpinned against it (SURVEY.md 8(c), App. C)."""
import torch

from . import _abi
from .block_isir import run_block_isir
from .engine import get_engine
from .flows import RealNVP
from .GlobalMCMC import user_initial_state
from .models import UserModel
from .pooled import average_flat, average_gradients
from .samplers import default_seed, initial_state


def resample(W, N, eng=None):
    """Systematic resampling, GLMCMC_NFs.py:29-40: u_i = (U + i) / N, index j repeated once per u_i in
    [Psum[j-1], Psum[j]); u_i beyond the last cumulative weight are dropped (the reference returns fewer than N then).
    Device weights go through the kernel `glabc_resample` (csrc/resample.cu); host weights (the reference's own call shape)
    through the equivalent torch.cumsum / searchsorted form.  Both consume ONE torch.rand(1), as the reference does."""
    W = torch.as_tensor(W)
    u0 = torch.rand(1).item()
    if W.is_cuda:
        eng = eng or get_engine(W.device)
        W = W.to(torch.float32).contiguous()
        idx = torch.empty(int(N), dtype=torch.int64, device=W.device)
        count = torch.zeros(1, dtype=torch.int64, device=W.device)
        eng.ctx.check(eng.lib.glabc_resample(eng.ctx.handle, eng._ptr(W), W.numel(), int(N), float(u0), eng._ptr(idx),
                                             eng._ptr(count), eng._stream()))
        return idx[: int(count.item())]
    u = ((u0 + torch.arange(N)) / N).to(W.dtype)
    psum = torch.cumsum(W, dim=0)
    idx = torch.searchsorted(psum, u, right=True)      # first j with Psum[j] > u_i
    return idx[idx < W.shape[0]]


class FlowProposal:
    """the shared RealNVP as the external proposal of `block_isir.run_block_isir`"""

    def __init__(self, flow, eng, seed, chain_id_base, train_batch, lr, weight_decay, precision="precise", train="native"):
        self.flow, self.eng, self.train_batch, self.train = flow, eng, int(train_batch), train
        eng.flow_precision(precision)
        self.seed = (seed * 0x9E3779B1 + chain_id_base + 0x5F) & 0x7FFFFFFFFFFFFFFF
        self.losses = []
        if train == "native":
            flow.train_init(eng, lr=lr, weight_decay=weight_decay)                                # GLMCMC_NFs.py:63, in the context
        else:   # the fp32 torch autograd restatement (the checker of tests/test_flow_train_gpu.py)
            self.opt = torch.optim.Adam(flow.parameters(), lr=lr, weight_decay=weight_decay)
            flow.bind(eng)

    def state_dict(self):
        """flow weights, Adam moments + step count (glabc_flow_get / glabc_flow_train_state), the generator of the base normals"""
        eng, flow = self.eng, self.flow
        sd = dict(train=self.train, params=flow.flat_params().cpu(), losses=list(self.losses))
        if self.train == "native":
            import ctypes as C
            mom = torch.empty(2 * sd["params"].numel(), device=eng.device)
            step = C.c_int64(0)
            eng.ctx.check(eng.lib.glabc_flow_train_state(eng.ctx.handle, eng._ptr(mom), C.byref(step), 0, eng._stream()))
            sd.update(moments=mom.cpu(), step=int(step.value))
        else:
            sd.update(opt=self.opt.state_dict())
        return sd

    def load_state_dict(self, sd):
        import ctypes as C
        eng, flow = self.eng, self.flow
        if sd["train"] != self.train:
            raise ValueError(f"the checkpoint was trained with flow_train={sd['train']!r}")
        flow.load_flat(sd["params"].to(eng.device))
        self.losses = list(sd["losses"])
        if self.train == "native":
            flow.bind(eng)                                   # the restored weights into the context (moments are kept: same architecture)
            mom = sd["moments"].to(eng.device).contiguous()
            step = C.c_int64(sd["step"])
            eng.ctx.check(eng.lib.glabc_flow_train_state(eng.ctx.handle, eng._ptr(mom), C.byref(step), 1, eng._stream()))
            torch.cuda.current_stream(eng.device).synchronize()
        else:
            self.opt.load_state_dict(sd["opt"])
            flow.bind(eng)

    def fill(self, blk_theta, blk_lq, rnd):     # NF_model.sample, GLMCMC_NFs.py:72,127
        c, B, d = blk_theta.shape
        # the base normals are drawn inside the flow kernel (Philox keyed by the proposal's seed and the refill round)
        self.flow.fused_sample(c * B, (self.seed + 0x632BE5AB * (rnd + 1)) & 0x7FFFFFFFFFFFFFFF, self.eng, theta=blk_theta, log_q=blk_lq)

    def log_prob(self, theta):                  # NF_model.log_prob, GLMCMC_NFs.py:98
        return self.flow.fused_log_prob(theta, self.eng)

    def adapt(self, blk):                       # GLMCMC_NFs.py:113-124, pooled over the chains (and, averaged, over the ranks)
        flow, d = self.flow, blk.d
        w = torch.nan_to_num(blk.w.reshape(-1), nan=0.0)
        idx = resample(w / torch.sum(w), min(w.numel(), self.train_batch), self.eng)
        x = blk.theta.reshape(-1, d)[idx].detach().float()
        if self.train == "native":
            # forward_kld, backward and Adam as kernels of libglabc.so (tcgen05 GEMMs, csrc/flow_train.cuh); the flat gradient
            # is the one buffer the ranks all-reduce
            g, loss = flow.grad(x, self.eng)
            average_flat(g, loss)
            flow.adam_step(g, loss, self.eng)    # skipped inside when the loss is NaN / inf (SURVEY.md B-13)
            self.losses.append(float(loss))
            return
        self.opt.zero_grad()
        loss = flow.forward_kld(x)
        if not (torch.isnan(loss) | torch.isinf(loss)):
            loss.backward()
        average_gradients(list(flow.parameters()))
        self.opt.step()
        self.losses.append(float(loss.detach()))
        flow.bind(self.eng)


def _base_params(base):
    if base is None:
        return None, None
    loc, ls = getattr(base, "loc", None), getattr(base, "log_scale", None)
    if loc is None or ls is None:
        raise NotImplementedError("base must be a DiagGaussian(2) with loc / log_scale (Mixture.py:70)")
    return loc.detach().reshape(1, 2).float(), ls.detach().reshape(1, 2).float()


def GLMCMC_NF(ABCset, num_ite, Initial_theta, Initial_y, Local_Proposal, filelocation, global_frequency, step_size, batch_size,
              base, Train_step, *, num_chains=None, seed=None, chain_id_base=0, arith="fast", trace="chain", return_stats=False,
              verbose=None, device=None, n_blocks=32, train_batch=65536, lr=5e-4, weight_decay=1e-5, flow=None,
              return_flow=False, flow_precision="precise", flow_train="native", checkpoint=None, resume=None):
    """Same positional signature and return value as the reference for one chain; keyword extensions as in `GlobalMCMC`,
    plus `flow` (continue with a given RealNVP), `train_batch` (pooled resample size), `return_flow` and `flow_precision`:
    "precise" (default — the flow's log-densities agree with the reference's float32 network to 1e-5, three tensor-core MMAs per
    hidden layer) or "fast" (single FP16 operands, ~3x the flow throughput, 1e-3-class agreement; importance weights stay exact
    either way because sample() returns the density of the map it applied); `flow_train`: "native" (the training step as
    kernels of the extension, the default) or "torch" (the fp32 autograd restatement, kept as the tests' checker);
    `checkpoint=` / `resume=`: the end-of-run state incl. the candidate blocks, the flow's weights and its Adam moments — a
    resumed run continues bit-identically (block_isir.run_block_isir).
    `ABCset` may be a `models.UserModel` of theta_dim 2: its simulator, prior and discrepancy run in the block-iSIR kernels
    compiled with it (FAST arithmetic, `arith` ignored); `Initial_y=None` then draws y0 with the model's simulator, as
    `GlobalMCMC` does for a user model."""
    if num_ite < 1:
        raise ValueError("num_ite must be at least 1")
    K, S = int(batch_size), int(step_size)
    if not 1 <= K <= _abi.MAX_K or S < 1 or K * S > _abi.AG_MAX_BLOCK:
        raise ValueError(f"batch_size in 1..{_abi.MAX_K} and batch_size * step_size <= {_abi.AG_MAX_BLOCK}")
    eng = get_engine(device)
    user = isinstance(ABCset, UserModel)      # run-time compiled model (csrc/user_model.cu: glabc_k_block_isir_user)
    if user and ABCset.batched:
        raise ValueError("GLMCMC_NF trains one flow on all chains, which is meaningless across the datasets of a batched "
                         "UserModel: run each model.dataset(g) on its own")
    pod = ABCset if user else eng.bind_model(ABCset)
    if pod.theta_dim != 2:
        raise NotImplementedError("the reference's flow is MLP([1,128,128,2]) couplings: theta_dim must be 2 (GLMCMC_NFs.py:56)")
    eng.bind_proposal(_abi.SLOT_LOCAL, Local_Proposal)
    seed = default_seed() if seed is None else int(seed)
    if user:
        theta, y, c = user_initial_state(eng, ABCset, Initial_theta, Initial_y, num_chains, seed, chain_id_base)
    else:
        theta, y, c = initial_state(eng, pod, Initial_theta, Initial_y, num_chains, seed)
    single = num_chains is None and c == 1
    dev = eng.device
    if flow is None:
        loc, ls = _base_params(base)
        with torch.random.fork_rng(devices=[]):          # the flow's initial weights: a function of the seed only
            torch.manual_seed(seed & 0x7FFFFFFF)         # (identical on every rank: the flow is shared)
            flow = RealNVP(n_blocks=n_blocks, base_loc=loc, base_log_scale=ls)
    flow.to(dev)
    prop = FlowProposal(flow, eng, seed, chain_id_base, train_batch, lr, weight_decay, precision=flow_precision, train=flow_train)
    result, rs, _ = run_block_isir(eng, pod, prop, num_ite=num_ite, theta=theta, y=y, K=K, S=S, gf=global_frequency, seed=seed,
                                   chain_id_base=chain_id_base, arith=arith, trace=trace, single=single,
                                   filelocation=filelocation, verbose=verbose, max_adapt=int(Train_step), checkpoint=checkpoint,
                                   resume=resume)
    extra = ((rs,) if return_stats else ()) + ((flow, prop.losses) if return_flow else ())
    return (result,) + extra if extra else result
