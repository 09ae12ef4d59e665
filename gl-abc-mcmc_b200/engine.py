"""Host side of the fused samplers: torch tensors <-> the C-ABI of libglabc.so.

PyTorch is plumbing here (device memory, the current stream); all sampler arithmetic runs in the
hand-written kernels behind `glabc_run_*`.  There is no CPU path: `Engine()` raises without a GPU.
"""
import ctypes as C
from dataclasses import dataclass

import torch

from . import _abi
from .models import fused_model, lower_proposal


@dataclass
class RunStats:
    """Per-chain accumulators the kernels keep (include/glabc.h GLABC_STAT_*), as float64 tensors."""
    raw: torch.Tensor  # [C, nstats] float32, device
    dim: int

    @property
    def steps(self):
        return self.raw[:, _abi.STAT_STEPS].double()

    @property
    def global_steps(self):
        return self.raw[:, _abi.STAT_GLOBAL_STEPS].double()

    @property
    def accepted_local(self):
        return self.raw[:, _abi.STAT_ACC_LOCAL].double()

    @property
    def accepted_global(self):
        return self.raw[:, _abi.STAT_ACC_GLOBAL].double()

    @property
    def move_rate(self):
        return (self.accepted_local + self.accepted_global) / self.steps.clamp(min=1)

    @property
    def mean(self):
        d = self.dim
        return self.raw[:, _abi.STAT_SUM:_abi.STAT_SUM + d].double() / self.steps.clamp(min=1)[:, None]

    @property
    def second_moment(self):
        d = self.dim
        return self.raw[:, _abi.STAT_SUM + d:_abi.STAT_SUM + 2 * d].double() / self.steps.clamp(min=1)[:, None]

    def gram(self):
        """[C, d, d] sum of delta delta^T (ESJD.py:17-21 numerator)."""
        d = self.dim
        tri = self.raw[:, _abi.STAT_SUM + 2 * d:_abi.STAT_SUM + 2 * d + d * (d + 1) // 2].double()
        g = torch.zeros(self.raw.shape[0], d, d, dtype=torch.float64, device=self.raw.device)
        t = 0
        for i in range(d):
            for j in range(i, d):
                g[:, i, j] = tri[:, t]
                g[:, j, i] = tri[:, t]
                t += 1
        return g

    def esjd(self):
        """per-chain det(sum delta delta^T / n_delta)^(1/d) — ESJD.py:21-24 without re-reading the trace"""
        g = self.gram() / self.steps.clamp(min=1)[:, None, None]
        return torch.linalg.det(g).clamp(min=0) ** (1.0 / self.dim)


class Engine:
    """One glabc context on the current CUDA device."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("glabc-b200 needs a CUDA device (sm_100a): there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = _abi.Context(self.device.index if self.device.index is not None else torch.cuda.current_device())
        self.lib = self.ctx.lib
        self.dim = None
        self.prior_pod = None   # DistPOD of the bound model's prior when it is not the DiagGaussian of its model POD

    # -- plugin binding -------------------------------------------------------------------------
    def bind_model(self, abc_set):
        model = fused_model(abc_set)
        pod = model.lower()
        prior = model.lower_prior() if hasattr(model, "lower_prior") else None
        self.ctx.check(self.lib.glabc_model_set(self.ctx.handle, C.byref(pod), C.sizeof(pod)))
        if prior is not None:
            self.ctx.check(self.lib.glabc_model_prior_set(self.ctx.handle, C.byref(prior), C.sizeof(prior)))
        self.dim = pod.theta_dim
        self.prior_pod = prior
        return pod

    def bind_proposal(self, slot, dist):
        """`dist`: a distribution object, or its lowered DistPOD"""
        pod = dist if isinstance(dist, _abi.DistPOD) else lower_proposal(dist)
        self.ctx.check(self.lib.glabc_dist_set(self.ctx.handle, slot, C.byref(pod), C.sizeof(pod)))
        return pod

    # -- helpers --------------------------------------------------------------------------------
    def _f32(self, t, shape=None):
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).contiguous()
        return t if shape is None else t.reshape(shape)

    @staticmethod
    def _ptr(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    def run(self, sampler, *, theta, y, n_steps, gf, step_base=0, chain_id_base=0, seed=0,
            rng_mode=_abi.RNG_NATIVE, arith=_abi.ARITH_FAST, trace_layout=_abi.TRACE_CHAIN_MAJOR, trace=None,
            trace_rows=None, trace_chains=None, trace_chain_off=0, trace_row_base=0, write_row0=True,
            stats=None, aux=None, tape32=None, tape64=None, debug=None, tape_dump=None, tape64_dump=None, K=0,
            block_threads=0, num_grad=0, tau=0.0, state64=None, tape_grad0=None, tape_grad0_dump=None, debug64=None,
            ag=None, blk=None):
        """Enqueue `n_steps` transitions of every chain on the current stream (device tensors,
        state updated in place).  Returns the trace tensor (allocated here unless given)."""
        cn, d = theta.shape
        for t in (theta, y, stats, aux, tape32, tape64, debug, tape_dump, tape64_dump, trace, state64, tape_grad0,
                  tape_grad0_dump, debug64):
            if t is not None and (not t.is_cuda or not t.is_contiguous()):
                raise ValueError("device entry point takes contiguous CUDA tensors")
        rows = trace_rows if trace_rows is not None else step_base + n_steps + 1 - trace_row_base
        tchains = trace_chains if trace_chains is not None else cn
        if trace is None and trace_layout == _abi.TRACE_EVENTS:
            raise ValueError("TRACE_EVENTS needs a caller-allocated trace [chains, trace_rows, 1 + d]")
        if trace is None and trace_layout != _abi.TRACE_NONE:
            shape = (rows, tchains, d) if trace_layout == _abi.TRACE_TIME_MAJOR else (tchains, rows, d)
            trace = torch.empty(shape, dtype=torch.float32, device=self.device)
        r = _abi.RunPOD(n_chains=cn, n_steps=n_steps, step_base=step_base, chain_id_base=chain_id_base,
                        seed=int(seed) & 0xFFFFFFFFFFFFFFFF, global_frequency=float(gf), rng_mode=rng_mode,
                        arith_mode=arith, trace_layout=trace_layout, write_row0=int(write_row0),
                        block_threads=block_threads, n_candidates=K, trace_rows=rows, trace_chains=tchains,
                        trace_chain_off=trace_chain_off, trace_row_base=trace_row_base,
                        theta=self._ptr(theta), y=self._ptr(y), aux=self._ptr(aux), trace=self._ptr(trace),
                        stats=self._ptr(stats), tape32=self._ptr(tape32), tape64=self._ptr(tape64),
                        debug=self._ptr(debug), tape_dump=self._ptr(tape_dump), tape64_dump=self._ptr(tape64_dump),
                        num_grad=int(num_grad), tau=float(tau), tau64=float(tau), state64=self._ptr(state64),
                        tape_grad0=self._ptr(tape_grad0), tape_grad0_dump=self._ptr(tape_grad0_dump),
                        debug64=self._ptr(debug64),
                        stream=C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        if sampler == "block_isir":
            self.ctx.check(self.lib.glabc_run_block_isir(self.ctx.handle, C.byref(r), C.byref(blk)))
            return trace
        if sampler == "block_weights":
            self.ctx.check(self.lib.glabc_block_weights(self.ctx.handle, C.byref(r), C.byref(blk), int(step_base) & 0xFFFFFFFF))
            return None
        if sampler == "aglmcmc":
            if ag is None:
                raise ValueError("run('aglmcmc') needs the glabc_aglmcmc_t description (Engine.aglmcmc_params)")
            self.ctx.check(self.lib.glabc_run_aglmcmc(self.ctx.handle, C.byref(r), C.byref(ag)))
            return trace
        fn = getattr(self.lib, "glabc_run_" + sampler)
        self.ctx.check(fn(self.ctx.handle, C.byref(r)))
        return trace

    def run_user(self, model, *, theta, y, n_steps, gf, step_base=0, chain_id_base=0, seed=0, trace_layout=_abi.TRACE_CHAIN_MAJOR,
                 trace=None, trace_rows=None, trace_row_base=0, write_row0=True, stats=None, block_threads=0, sampler="global", K=0,
                 aux=None, num_grad=0, tau=0.0):
        """GlobalMCMC (`sampler="global"`, LOCAL / GLOBAL slots), GLMCMC (`"isir"`, LOCAL / IMPORTANCE slots, K candidates, aux) or
        GLMALA (`"mala"`, IMPORTANCE slot, K, tau, num_grad, aux) transitions for a `models.UserModel` (compiled on first use)"""
        cn, d = theta.shape
        rows = trace_rows if trace_rows is not None else step_base + n_steps + 1 - trace_row_base
        if trace is None and trace_layout != _abi.TRACE_NONE:
            shape = (rows, cn, d) if trace_layout == _abi.TRACE_TIME_MAJOR else (cn, rows, d)
            trace = torch.empty(shape, dtype=torch.float32, device=self.device)
        r = _abi.RunPOD(n_chains=cn, n_steps=n_steps, step_base=step_base, chain_id_base=chain_id_base,
                        seed=int(seed) & 0xFFFFFFFFFFFFFFFF, global_frequency=float(gf), rng_mode=_abi.RNG_NATIVE,
                        arith_mode=_abi.ARITH_FAST, trace_layout=trace_layout, write_row0=int(write_row0),
                        block_threads=block_threads, n_candidates=int(K), trace_rows=rows, trace_chains=cn,
                        trace_row_base=trace_row_base, theta=self._ptr(theta), y=self._ptr(y), aux=self._ptr(aux),
                        trace=self._ptr(trace), stats=self._ptr(stats), stream=self._stream(), num_grad=int(num_grad), tau=float(tau),
                        tau64=float(tau))
        pod = model.user_pod()
        fn = {"isir": self.lib.glabc_run_isir_user, "mala": self.lib.glabc_run_mala_user}.get(sampler, self.lib.glabc_run_global_user)
        self.ctx.check(fn(self.ctx.handle, C.byref(r), C.byref(pod)))
        return trace

    def user_simulate(self, model, theta, seed, row_base=0):
        """y [n, y_dim]: one draw of a `models.UserModel`'s simulator per row of theta [n, theta_dim] (glabc_user_simulate;
        row r draws from the Philox stream of id row_base + r at step 0)"""
        theta = self._f32(theta).reshape(-1, model.theta_dim)
        y = torch.empty(theta.shape[0], model.y_dim, dtype=torch.float32, device=self.device)
        pod = model.user_pod()
        self.ctx.check(self.lib.glabc_user_simulate(self.ctx.handle, C.byref(pod), self._ptr(theta), theta.shape[0],
                                                    int(seed) & 0xFFFFFFFFFFFFFFFF, int(row_base) & 0xFFFFFFFFFFFFFFFF,
                                                    self._ptr(y), self._stream()))
        return y

    def user_evaluate(self, model, op, x):
        """out [n]: the prior (op USER_PRIOR, x = theta rows), discrepancy (USER_DISCREPANCY, x = y rows) or log ABC kernel
        (USER_LOG_KERNEL) of a `models.UserModel` (glabc_user_evaluate)"""
        x = self._f32(x).reshape(-1, model.theta_dim if op == _abi.USER_PRIOR else model.y_dim)
        out = torch.empty(x.shape[0], dtype=torch.float32, device=self.device)
        pod = model.user_pod()
        self.ctx.check(self.lib.glabc_user_evaluate(self.ctx.handle, C.byref(pod), int(op), self._ptr(x), x.shape[0], self._ptr(out),
                                                    self._stream()))
        return out

    def aglmcmc_params(self, *, step_size, alpha, hat_eps_T, rule=_abi.BW_SILVERMAN, init=True, init_p=None, init_s=None,
                       ad_idx=None, ad_noise=None, ad_sim=None, ad_rec=None, ad_blk=None, init_w=None):
        """glabc_aglmcmc_t; the tensors (replay tapes / parity dumps) must stay alive until the run is enqueued"""
        for t in (init_p, init_s, ad_idx, ad_noise, ad_sim, ad_rec, ad_blk, init_w):
            if t is not None and (not t.is_cuda or not t.is_contiguous()):
                raise ValueError("aglmcmc tapes / dumps must be contiguous CUDA tensors")
        rounds = 0 if ad_idx is None else ad_idx.shape[0]
        dump = min([t.shape[0] for t in (ad_rec, ad_blk) if t is not None], default=0)
        return _abi.AglmcmcPOD(step_size=int(step_size), init=int(bool(init)), alpha=float(alpha), hat_eps_T=float(hat_eps_T),
                               kde_rule=int(rule), tape_rounds=rounds, init_p=self._ptr(init_p), init_s=self._ptr(init_s),
                               ad_idx=self._ptr(ad_idx), ad_noise=self._ptr(ad_noise), ad_sim=self._ptr(ad_sim),
                               ad_rec=self._ptr(ad_rec), ad_blk=self._ptr(ad_blk), init_w=self._ptr(init_w), dump_rounds=dump)

    def dist_log_prob(self, slot, z):
        """log_prob of the distribution bound to `slot`, evaluated on the device"""
        z = self._f32(z)
        out = torch.empty(z.shape[0], dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_dist_log_prob(self.ctx.handle, int(slot), self._ptr(z), z.shape[0], self._ptr(out), self._stream()))
        return out

    def dist_sample(self, slot, n, dim, seed=0):
        """forward(n) of the distribution bound to `slot`: (z [n, dim], log_p [n])"""
        z = torch.empty(n, dim, dtype=torch.float32, device=self.device)
        lp = torch.empty(n, dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_dist_sample(self.ctx.handle, int(slot), int(n), int(seed) & 0xFFFFFFFFFFFFFFFF, self._ptr(z),
                                                  self._ptr(lp), self._stream()))
        return z, lp

    # -- KernelDensity (kernel_density.py) ------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def kde_fit(self, X, w=None, n=None, rule=_abi.BW_SILVERMAN):
        """X [sets, cap, d] (or [n, d]), w [sets, cap] or None, n [sets] int32 or None -> (weights, bandwidth)"""
        single = X.dim() == 2
        X3 = X.unsqueeze(0) if single else X
        sets, cap, d = X3.shape
        X3 = self._f32(X3)
        w2 = None if w is None else self._f32(w).reshape(sets, cap)
        weights = torch.empty(sets, cap, dtype=torch.float32, device=self.device)
        bw = torch.empty(sets, d, dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_kde_fit(self.ctx.handle, self._ptr(X3), self._ptr(w2), self._ptr(n), sets, cap, d, int(rule),
                                              self._ptr(weights), self._ptr(bw), self._stream()))
        return (weights[0], bw[0]) if single else (weights, bw)

    def kde_log_prob(self, X, weights, bw, x, n=None, arith=_abi.ARITH_FAST):
        single = X.dim() == 2
        X3, w2, b2, x3 = (X.unsqueeze(0), weights.unsqueeze(0), bw.reshape(1, -1), x.unsqueeze(0)) if single else (X, weights, bw, x)
        sets, cap, d = X3.shape
        X3, w2, b2, x3 = self._f32(X3), self._f32(w2), self._f32(b2), self._f32(x3)
        m = x3.shape[1]
        out = torch.empty(sets, m, dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_kde_log_prob(self.ctx.handle, self._ptr(X3), self._ptr(w2), self._ptr(b2), self._ptr(n), sets,
                                                   cap, d, self._ptr(x3), m, self._ptr(out), int(arith), self._stream()))
        return out[0] if single else out

    def kde_sample(self, X, weights, bw, m, n=None, seed=0, idx_tape=None, noise_tape=None):
        single = X.dim() == 2
        X3, w2, b2 = (X.unsqueeze(0), weights.unsqueeze(0), bw.reshape(1, -1)) if single else (X, weights, bw)
        sets, cap, d = X3.shape
        X3, w2, b2 = self._f32(X3), self._f32(w2), self._f32(b2)
        if idx_tape is not None:
            idx_tape = idx_tape.to(self.device, torch.int32).reshape(sets, m).contiguous()
            noise_tape = self._f32(noise_tape).reshape(sets, m, d)
        out = torch.empty(sets, m, d, dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_kde_sample(self.ctx.handle, self._ptr(X3), self._ptr(w2), self._ptr(b2), self._ptr(n), sets, cap,
                                                 d, int(m), int(seed) & 0xFFFFFFFFFFFFFFFF, self._ptr(idx_tape),
                                                 self._ptr(noise_tape), self._ptr(out), self._stream()))
        return out[0] if single else out

    def run_host(self, sampler, *, theta, y, n_steps, gf, trace, step_base=0, chain_id_base=0, seed=0,
                 arith=_abi.ARITH_FAST, trace_layout=_abi.TRACE_TIME_MAJOR, write_row0=True, stats=None,
                 aux=None, K=0, chunk_steps=0, block_threads=0, num_grad=0, tau=0.0, state64=None, ag=None):
        """The reference-facing call on HOST buffers (numpy-compatible CPU tensors, ideally pinned):
        H2D of the state, kernels, D2H of trace/state/stats — returns when the host buffers hold the
        result."""
        cn, d = theta.shape
        for t in (theta, y, stats, aux, trace):
            if t is not None and (t.is_cuda or not t.is_contiguous() or t.dtype != torch.float32):
                raise ValueError("host entry point takes contiguous float32 CPU tensors")
        if state64 is not None and (state64.is_cuda or not state64.is_contiguous() or state64.dtype != torch.float64):
            raise ValueError("state64 must be a contiguous float64 CPU tensor")
        if trace_layout == _abi.TRACE_NONE:
            rows, tchains = 0, cn
        elif trace_layout == _abi.TRACE_TIME_MAJOR:
            rows, tchains = trace.shape[0], trace.shape[1]
        else:
            tchains, rows = trace.shape[0], trace.shape[1]
        r = _abi.RunPOD(n_chains=cn, n_steps=n_steps, step_base=step_base, chain_id_base=chain_id_base,
                        seed=int(seed) & 0xFFFFFFFFFFFFFFFF, global_frequency=float(gf), rng_mode=_abi.RNG_NATIVE,
                        arith_mode=arith, trace_layout=trace_layout, write_row0=int(write_row0),
                        block_threads=block_threads, n_candidates=K, trace_rows=rows, trace_chains=tchains,
                        trace_chain_off=0, trace_row_base=0, theta=self._ptr(theta), y=self._ptr(y),
                        aux=self._ptr(aux), trace=self._ptr(trace), stats=self._ptr(stats), num_grad=int(num_grad),
                        tau=float(tau), tau64=float(tau), state64=self._ptr(state64))
        if sampler == "aglmcmc":
            if ag is None:
                raise ValueError("run_host('aglmcmc') needs the glabc_aglmcmc_t description (Engine.aglmcmc_params)")
            self.ctx.check(self.lib.glabc_run_aglmcmc_host(self.ctx.handle, C.byref(r), C.byref(ag), int(chunk_steps)))
            return trace
        fn = getattr(self.lib, f"glabc_run_{sampler}_host")
        self.ctx.check(fn(self.ctx.handle, C.byref(r), int(chunk_steps)))
        return trace

    def aglmcmc_state(self):
        """the context's AGLMCMC workspace (candidate blocks, per-chain KDEs, counters, eps-hat) as a uint8 device tensor"""
        n = C.c_int64(0)
        self.ctx.check(self.lib.glabc_aglmcmc_state(self.ctx.handle, None, C.byref(n), 0, 0, 0, self._stream()))
        blob = torch.empty(n.value, dtype=torch.uint8, device=self.device)
        self.ctx.check(self.lib.glabc_aglmcmc_state(self.ctx.handle, self._ptr(blob), C.byref(n), 0, 0, 0, self._stream()))
        return blob

    def aglmcmc_restore(self, blob, n_chains, block):
        blob = blob.to(self.device).contiguous()
        n = C.c_int64(blob.numel())
        self.ctx.check(self.lib.glabc_aglmcmc_state(self.ctx.handle, self._ptr(blob), C.byref(n), int(n_chains), int(block), 1, self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def flow_precision(self, mode):
        """operand precision of the flow's hidden layer for the following glabc_flow_sample / glabc_flow_log_prob calls of this
        context: "precise" (FP16 hi + lo split, 1e-5-class log-densities; the default) or "fast" (single FP16 operands)"""
        code = {"fast": _abi.FLOW_FAST, "precise": _abi.FLOW_PRECISE}[mode] if isinstance(mode, str) else int(mode)
        self.ctx.check(self.lib.glabc_flow_precision(self.ctx.handle, code))

    def summarize(self, stats_raw, dim):
        """[chains, steps, global steps, acc local, acc global, sum esjd, sum theta (d), sum theta^2 (d)] of a shard, float64,
        one kernel (glabc_summarize)"""
        out = torch.zeros(6 + 2 * dim, dtype=torch.float64, device=self.device)
        self.ctx.check(self.lib.glabc_summarize(self.ctx.handle, self._ptr(stats_raw), stats_raw.shape[0], int(dim), self._ptr(out),
                                                self._stream()))
        return out

    def esjd(self, trace, layout):
        """per-chain esjd of a device trace ([rows, C, d] time-major / [C, rows, d] chain-major)."""
        if layout == _abi.TRACE_TIME_MAJOR:
            rows, chains, d = trace.shape
        else:
            chains, rows, d = trace.shape
        out = torch.empty(chains, dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.glabc_esjd(self.ctx.handle, self._ptr(trace), layout, rows, chains, d, self._ptr(out),
                                           C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out

    def philox(self, ctr, key):
        ctr = torch.as_tensor(ctr, dtype=torch.int64).to(self.device).to(torch.int32).contiguous()   # wraps mod 2^32
        key = torch.as_tensor(key, dtype=torch.int64).to(self.device).to(torch.int32).contiguous()
        out = torch.empty_like(ctr)
        self.ctx.check(self.lib.glabc_philox_kat(self.ctx.handle, self._ptr(ctr), self._ptr(key), ctr.shape[0],
                                                 self._ptr(out), None))
        torch.cuda.synchronize(self.device)
        return out.to(torch.int64) & 0xFFFFFFFF


_engines = {}


def get_engine(device=None):
    """process-wide engine per device (contexts are cheap but hold scratch buffers)"""
    if not torch.cuda.is_available():
        raise RuntimeError("glabc-b200 needs a CUDA device (sm_100a): there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx not in _engines:
        _engines[idx] = Engine(torch.device("cuda", idx))
    return _engines[idx]
