#!/usr/bin/env python
"""Headline benchmark: ABC-MCMC chain-steps/s of the fused GlobalMCMC step kernel on the README
Mixture_set workload (BASELINE.json configs[1]: 65,536 independent chains x 1e4 iterations per GPU,
gf=0.5, local sigma 0.35, global N(0,I), epsilon 0.05), full float32 trace written.

  python bench.py [--gpus N] [--steps K] [--warmup W]           # this repo's CUDA path
  python bench.py --impl reference [...]                          # the CPU port of the reference path

One "step" = one pass of the hot path over the whole batch (C chains x (T-1) transitions).  Prints
ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_STEP = 8       # one float32 trace row of d=2
# SURVEY.md §8(d): algorithmic thread-instructions per chain-step (Philox4x32-10 + Box-Muller floor)
#   global: GlobalMCMC.py:37-68 = 186;  glmcmc: GLMCMC.py:58-104, K=5, gf=0.9 = 0.9*760 + 0.1*186 = 703
SAMPLERS = {
    "global": dict(entry="global", gf=0.5, K=0, alg_inst=186,
                   workload="README Mixture_set GlobalMCMC (BASELINE configs[1])"),
    "glmcmc": dict(entry="isir", gf=0.9, K=5, alg_inst=703,
                   workload="README Mixture_set GLMCMC iSIR K=5, gf=0.9 (BASELINE configs[2], run_glmcmc)"),
    # GLMALA.py:150-200, gf=0.8, K=5, tau=0.3, num_grad=100: 0.2 * ~22,000 (400 CRN simulator draws) + 0.8 * 760
    # AGLMCMC.py:124-272 with the example's settings (Mixture.py:74): gf=1, K=5, step 200, alpha 0.8, eps-hat_T 0.2.
    # Dominant work: KDE.log_prob of each new block, B x n pairs per chain per adaptation = K * n ~ 5,000 pairs per
    # chain-step at 7 thread-instructions per pair (kde.cuh) + ~100 for the step itself
    "aglmcmc": dict(entry="aglmcmc", gf=1.0, K=5, alg_inst=35100, step_size=200, alpha=0.8, hat_eps_T=0.2,
                    workload="README Mixture_set AGLMCMC K=5, gf=1, step 200, alpha 0.8, eps_hat_T 0.2 (BASELINE configs[4], run_aglmcmc)"),
    "glmala": dict(entry="mala", gf=0.8, K=5, alg_inst=5000, num_grad=100, tau=0.3,
                   workload="README Mixture_set GLMALA K=5, gf=0.8, tau=0.3, num_grad=100 (BASELINE configs[2], run_glmala)"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="native", choices=["native", "reference"])
    p.add_argument("--sampler", default="global", choices=sorted(SAMPLERS) + ["kde", "glmcmc_nf", "aglmcmc_pooled"],
                   help="which fused step kernel to time")
    p.add_argument("--kde-train", type=int, default=100000, help="aglmcmc_pooled: pooled KDE training draws (all ranks together)")
    p.add_argument("--kde-points", type=int, default=100000)
    p.add_argument("--chains", type=int, default=65536, help="chains per GPU (weak scaling)")
    p.add_argument("--iters", type=int, default=10000, help="num_ite per chain (trace rows)")
    p.add_argument("--layout", default="chain", choices=["chain", "time", "none"])
    p.add_argument("--block", type=int, default=0)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip the short device-resident timings of the other kernels")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--no-ref-python", action="store_true", help="skip timing the unmodified reference package (baseline/_ref)")
    p.add_argument("--ref-python-its", type=int, default=10001, help="iterations per reference chain (one chain per host core)")
    p.add_argument("--no-other-configs", action="store_true", help="skip BASELINE configs 3-5 / strong scaling (other_configs)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / float64, "
                        f"at most {DUMP_BYTES >> 20} MB in all; an array over its share keeps a fixed, seeded sample of its "
                        "chains); rank 0 only")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        p.error("--dump-outputs: the reference arm sizes its sample by the host's speed, so its outputs differ from run to run")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> (tensor, chain axis or None).  Writes out_dir/<name>.npy.  Each array gets an equal share of
    DUMP_BYTES; a larger one keeps the chains of a fixed permutation's head (sorted), so the same arguments dump the same
    chains in every run and the smaller samples are subsets of the larger ones."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, (t, axis) in arrays.items():
        t = t.detach()
        if t.dtype not in (torch.float32, torch.float64):
            t = t.float()
        if axis is not None and t.numel() * t.element_size() > share:
            n = t.shape[axis]
            keep = share // (t.numel() // n * t.element_size())
            if keep < 1:
                raise ValueError(f"--dump-outputs: one chain of '{name}' {tuple(t.shape)} is larger than {share} bytes")
            idx = np.sort(np.random.default_rng(0).permutation(n)[:keep])
            t = t.index_select(axis, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def workload_objects():
    import torch
    import glabc_b200 as g
    model = g.Mixture_set(0.05)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))   # README.md:120
    gp = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    return model, lp, gp


class CpuPort:
    """The oracle (C restatement of GlobalMCMC.py:37-68, native Philox mode) on the host cores, run on
    bounded samples of the workload (the full 65,536 x 1e4 job would take ~10 s per pass per 100 M
    steps/s of host throughput)."""

    def __init__(self, threads=0, sampler="global"):
        self.spec = SAMPLERS[sampler]
        from glabc_b200.models import lower_model, lower_proposal
        from oracle import oracle
        self.oracle = oracle
        model, lp, gp = workload_objects()
        self.pods = (lower_model(model), lower_proposal(lp), lower_proposal(gp))
        self.threads = threads
        oracle.lib().oracle_set_num_threads(threads)
        self.cores = oracle.lib().oracle_num_threads()

    def run(self, c, t):
        import numpy as np
        from glabc_b200 import _abi as abi
        theta = np.zeros((c, 2), np.float32)
        y = (np.random.default_rng(0).standard_normal((c, 2)) * 0.2236).astype(np.float32)
        trace = np.zeros((c, t + 1, 2), np.float32)
        aux, extra = None, {}
        if self.spec["K"]:
            aux = np.zeros((c, abi.AUX_SLOTS), np.float32)
            aux[:, abi.AUX_LOCAL] = 1.0
        if self.spec["entry"] == "mala":
            extra = dict(num_grad=self.spec["num_grad"], tau=self.spec["tau"], state64=np.zeros((c, abi.STATE64_SLOTS)))
        if self.spec["entry"] == "aglmcmc":
            aux = None
            extra = dict(ag=self.oracle.aglmcmc_params(S=self.spec["step_size"], alpha=self.spec["alpha"],
                                                       hat_eps_T=self.spec["hat_eps_T"]))
        stats = np.zeros((c, abi.nstats(2)), np.float32)
        t0 = time.perf_counter()
        self.oracle.run(self.spec["entry"], *self.pods, theta=theta, y=y, n_steps=t, gf=self.spec["gf"], seed=0,
                        trace=trace, trace_layout=abi.TRACE_CHAIN_MAJOR, threads=self.threads, K=self.spec["K"], aux=aux,
                        stats=stats, **extra)
        dt = time.perf_counter() - t0
        # ESJD.py:17-24 from the Gram accumulators: det(sum dd^T / n)^(1/2) per chain, averaged
        n = np.maximum(stats[:, abi.STAT_STEPS].astype(np.float64), 1.0)
        g00, g01, g11 = (stats[:, abi.STAT_SUM + 4 + k].astype(np.float64) / n for k in range(3))
        self.mean_esjd = float(np.sqrt(np.maximum(g00 * g11 - g01 * g01, 0.0)).mean())
        return dt

    def size_sample(self, chains, iters, seconds):
        """chains x transitions of the workload that take about `seconds` on this host"""
        t = min(iters - 1, 9999)
        c = max(self.cores * 4, 64)
        dt = self.run(c, t)                     # calibration (thread start-up dominates tiny runs)
        while dt < min(1.0, seconds / 4) and c < chains:
            c = min(chains, c * 4)
            dt = self.run(c, t)
        c = int(max(self.cores, min(chains, c * seconds / dt)))
        return c, t


def cpu_port_rate(chains, iters, seconds, threads=0, sampler="global"):
    port = CpuPort(threads, sampler)
    c, t = port.size_sample(chains, iters, seconds)
    dt = port.run(c, t)
    return (c * t / dt, port.cores, f"{c} chains x {t} transitions of the same workload, full trace in host memory, {dt:.1f} s",
            port.mean_esjd)


def bench_reference(a, rank):
    """--impl reference: the reference's CPU path (its C port, all host threads), one bounded sample per step,
    sized so the whole run ends within ~2 minutes."""
    if rank != 0:
        return
    port = CpuPort(sampler=a.sampler)
    per_step = max(0.2, min(a.cpu_seconds, 100.0 / max(1, a.steps + a.warmup)))
    c, t = port.size_sample(a.chains, a.iters, per_step)
    times = []
    for i in range(a.warmup + a.steps):
        dt = port.run(c, t)
        if i >= a.warmup:
            times.append(dt)
    value = c * t * len(times) / sum(times)
    sample = f"{c} chains x {t} transitions of the same workload per step, full trace in host memory, {sum(times) / len(times):.2f} s per step"
    line = {"impl": "reference", "metric": "abc_mcmc_chain_steps_per_sec", "value": value, "unit": "chain-steps/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a, cpu=dict(chains_per_step=c, transitions=t, threads=port.cores)),
            "cpu_baseline": {"value": value, "unit": "chain-steps/s", "cores": port.cores, "kind": "port", "sample": sample,
                             "esjd": {"mean_per_chain": port.mean_esjd, "aggregate_esjd_per_sec": port.mean_esjd * value}},
            "e2e": {"value": value, "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if a.sampler in ("global", "glmcmc") and not a.no_ref_python:
        # the reference's own Python (unmodified, baseline/_ref), beside its C port: ~1e4 chain-steps/s on 8 cores
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import ref_python
        line["cpu_baseline"]["reference_python"] = ref_python.measure(a.ref_python_its, sampler=a.sampler)
    emit(line)


def bench_kde(a, rank, world, local_rank):
    """--sampler kde: KernelDensity.fit + log_prob of 1e5 queries against 1e5 weighted training draws, d = 2
    (BASELINE configs[4]: the pairwise Gaussian KDE of AGLMCMC at pooled size).  One step = fit + log_prob."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = get_engine()
    info = eng.ctx.device_info()
    n = m = a.kde_points
    g = torch.Generator(device="cuda").manual_seed(77 + rank)
    signs = torch.randint(0, 2, (n, 2), device="cuda", generator=g) * 2 - 1
    X = (signs * (1.42518 + 0.2233 * torch.randn(n, 2, device="cuda", generator=g))).contiguous()   # SURVEY.md App. D posterior
    w = torch.rand(n, device="cuda", generator=g) ** 2
    x = (X[torch.randperm(n, device="cuda", generator=g)[:m]] + 0.1 * torch.randn(m, 2, device="cuda", generator=g)).contiguous()

    def one_step():
        weights, bw = eng.kde_fit(X, w)
        return weights, bw, eng.kde_log_prob(X, weights, bw, x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(a.warmup):
        one_step()
    barrier()
    n_idle = len(sampler.rows)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        fit_w, fit_bw, out = one_step()
    e1.record()
    barrier()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"weights": (fit_w, 0), "bandwidth": (fit_bw, None), "log_prob": (out, 0)})
    sampler.rows = sampler.rows[max(0, n_idle - 1):]
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    pairs = float(n) * m * world
    value = pairs * a.steps / (total_ms * 1e-3)
    weights, bw = eng.kde_fit(X, w)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kms = []
    for _ in range(min(a.steps, 20)):
        k0.record()
        eng.kde_log_prob(X, weights, bw, x)
        k1.record()
        torch.cuda.synchronize()
        kms.append(k0.elapsed_time(k1))
    kms = sum(kms) / len(kms)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    sm_max_mhz = float(peaks.get("sm_max_mhz", clocks.get("sm_max_mhz") or 1965.0))
    inst_peak = info["sm_count"] * 128 * sm_max_mhz * 1e6 / 1e9
    rate = float(n) * m / (kms * 1e-3)
    inst_ach = rate * 7 / 1e9
    mufu_peak = info["sm_count"] * 16 * sm_max_mhz * 1e6 / 1e9
    roofline = {"bound": "alu-issue", "achieved": inst_ach, "peak": inst_peak, "unit": "Gthread-inst/s", "frac": inst_ach / inst_peak,
                "traffic": None, "kernel_ms": kms, "kernel_pairs_per_sec": rate,
                "note": "7 algorithmic thread-instructions per (query, point) pair at d = 2: 2 sub, 2 fma, 1 fma, 1 ex2, 1 add",
                "mufu": {"achieved": rate / 1e9, "peak": mufu_peak, "unit": "Gex2/s", "frac": rate / 1e9 / mufu_peak}}
    line = {"metric": "kde_pairs_per_sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": "KernelDensity.fit + log_prob, weighted Silverman KDE (BASELINE configs[4] / SURVEY 6)",
                                            "train_points": n, "queries": m, "dim": 2, "arith": "fast",
                                            "l2": "inputs 2.4 MB, L2-resident by design; compute-bound pair loop"},
            "clocks": clocks, "gpu_launches": 2 * a.steps, "roofline": roofline}
    if not a.no_e2e:
        hX, hw, hx = X.cpu().pin_memory(), w.cpu().pin_memory(), x.cpu().pin_memory()
        hout = torch.empty(m).pin_memory()

        def e2e():
            dX, dw, dx = hX.cuda(non_blocking=True), hw.cuda(non_blocking=True), hx.cuda(non_blocking=True)
            ww, bb = eng.kde_fit(dX, dw)
            hout.copy_(eng.kde_log_prob(dX, ww, bb, dx), non_blocking=True)
            torch.cuda.synchronize()
        e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(1, min(a.steps, 5))):
            e2e()
        barrier()
        dt = (time.perf_counter() - t0) / max(1, min(a.steps, 5))
        line["e2e"] = {"value": pairs / dt, "unit": "pairs/s", "h2d_bytes_per_step": (hX.numel() + hw.numel() + hx.numel()) * 4,
                       "d2h_bytes_per_step": m * 4}
    if rank == 0 and not a.no_cpu:
        from oracle import oracle
        Xn, wn = X.cpu().numpy(), w.cpu().numpy()
        wo, bo = oracle.kde_fit(Xn, wn)
        q = 64
        t0 = time.perf_counter()
        oracle.kde_log_prob(Xn, wo, bo, x[:q].cpu().numpy())
        dt = time.perf_counter() - t0
        q = int(max(64, min(m, q * a.cpu_seconds / max(dt, 1e-3))))
        t0 = time.perf_counter()
        ref = oracle.kde_log_prob(Xn, wo, bo, x[:q].cpu().numpy())
        dt = time.perf_counter() - t0
        err = float(np.abs(out[:q].cpu().numpy() - ref).max())
        line["cpu_baseline"] = {"value": q * n / dt, "unit": "pairs/s", "cores": 1, "kind": "port",
                                "sample": f"{q} queries x {n} training points, {dt:.1f} s; max |gpu - cpu| = {err:.2e}"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


# samplers whose importance proposal is SHARED by all chains of all ranks (the two places the path exchanges data):
#   glmcmc_nf      BASELINE configs[3]: one RealNVP, flow sample / log_prob on tcgen05, gradients all-reduced per Adam step
#   aglmcmc_pooled BASELINE configs[4]: one KernelDensity over `--kde-train` pooled draws, all-gathered before every fit
SHARED = {
    "glmcmc_nf": dict(gf=0.5, K=5, step_size=200, train_steps=50, chains=131072, iters=1001,
                      workload="README Mixture_set GLMCMC-NFs: shared RealNVP(32 blocks), gf 0.5, K 5, step 200, 50 train steps "
                               "(BASELINE configs[3], run_glmcmc_nf)"),
    "aglmcmc_pooled": dict(gf=1.0, K=5, step_size=200, alpha=0.8, hat_eps_T=0.2, chains=16384, iters=1001,
                           workload="README Mixture_set AGLMCMC with ONE pooled KernelDensity (BASELINE configs[4]), gf 1, K 5, "
                                    "step 200, alpha 0.8, eps_hat_T 0.2"),
}


def bench_shared(a, rank, world, local_rank):
    """One step = one whole sampler call through the public entry point (C chains x (T - 1) iterations per GPU, statistics
    only), device-resident inputs; e2e = the same call with host tensors in and the statistics copied back."""
    import torch
    import torch.distributed as dist
    import glabc_b200 as g
    from glabc_b200 import _abi as abi
    from glabc_b200.engine import get_engine
    from glabc_b200.flows import RealNVP
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    spec = SHARED[a.sampler]
    C = a.chains if a.chains != 65536 else spec["chains"]
    T = a.iters if a.iters != 10000 else spec["iters"]
    eng = get_engine()
    info = eng.ctx.device_info()
    model, lp, gp = workload_objects()
    K, S, gf = spec["K"], spec["step_size"], spec["gf"]
    base = rank * C
    z_dev = torch.zeros(2, device="cuda")
    z_host = torch.zeros(2)

    def call(theta0, seed):
        if a.sampler == "glmcmc_nf":
            return g.GLMCMC_NF(model, T, theta0, None, lp, None, gf, S, K, None, spec["train_steps"], num_chains=C, seed=seed,
                               chain_id_base=base, trace="none", return_stats=True, verbose=False)
        return g.AGLMCMC(model, T, theta0, None, lp, gp, None, gf, S, K, spec["alpha"], spec["hat_eps_T"], num_chains=C, seed=seed,
                         chain_id_base=base, trace="none", return_stats=True, verbose=False, pooled=True, kde_train=a.kde_train)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for w in range(a.warmup):
        call(z_dev, w)
    barrier()
    n_idle = len(sampler.rows)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls0 = eng.ctx.n_calls
    e0.record()
    for s in range(a.steps):
        _, st = call(z_dev, a.warmup + s)
    e1.record()
    barrier()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"stats": (st.raw, 0)})
    n_launch_calls = eng.ctx.n_calls - calls0    # every one launches at least one kernel of libglabc.so (3 binds per call aside)
    sampler.rows = sampler.rows[max(0, n_idle - 1):]
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    steps_per_pass = float(C) * (T - 1) * world
    value = steps_per_pass * a.steps / (total_ms * 1e-3)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    sm_max_mhz = float(peaks.get("sm_max_mhz", clocks.get("sm_max_mhz") or 1965.0))

    # the dominant kernel, timed alone at the size one block refill launches it (CUDA events on the launching stream)
    def timed(fn, reps=5):
        fn()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        k0.record()
        for _ in range(reps):
            fn()
        k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / reps
    n_cand = C * K * S
    if a.sampler == "glmcmc_nf":
        flow = RealNVP(device="cuda")
        with torch.no_grad():
            flow.w3.copy_(0.05 * torch.randn_like(flow.w3))
        flow.bind(eng)
        eps = torch.randn(n_cand, 2, device="cuda")
        th, lq = torch.empty(n_cand, 2, device="cuda"), torch.empty(n_cand, device="cuda")
        kms = timed(lambda: flow.fused_sample_from(eps, eng, theta=th, log_q=lq))
        tf = n_cand * 1.049e6 / (kms * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops", 1654.4))
        roofline = {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "traffic": None,
                    "kernel_ms": kms, "samples_per_sec": n_cand / (kms * 1e-3),
                    "note": f"k_flow sample of one block refill ({n_cand} candidates x 32 coupling blocks, 1.049 MFLOP dense per "
                    "sample, FP16 operands / FP32 accumulate on tcgen05 kind::f16); peak = measured dense bf16 / fp16 rate "
                    "(MEASURED_PEAKS.json); the kernel's binding unit is the shared-memory broadcast of the layer vectors "
                    "(DESIGN.md K4), not the tensor pipe"}
        del eps, th, lq
    else:
        n = a.kde_train
        X = torch.randn(n, 2, device="cuda")
        wn, bw = eng.kde_fit(X, torch.rand(n, device="cuda"))
        q = torch.randn(n_cand, 2, device="cuda")
        kms = timed(lambda: eng.kde_log_prob(X, wn, bw, q), reps=2)
        rate = float(n_cand) * n / (kms * 1e-3)
        mufu_peak = info["sm_count"] * 16 * sm_max_mhz * 1e6
        roofline = {"bound": "mufu", "achieved": rate / 1e9, "peak": mufu_peak / 1e9, "unit": "Gex2/s", "frac": rate / mufu_peak,
                    "traffic": None, "kernel_ms": kms, "note": f"k_kde_logprob of one block refill: {n_cand} candidates x {n} pooled "
                    "training draws, one MUFU.EX2 per pair (16 / clk / SM)"}
        del X, q
    torch.cuda.empty_cache()
    cfg = {"workload": spec["workload"], "chains_per_gpu": C, "iterations": T, "theta_dim": 2, "epsilon": 0.05, "global_frequency": gf,
           "isir_candidates": K, "step_size": S, "trace": "statistics only", "rng": "philox4x32-10 native", "arith": "fast",
           "l2": "candidate blocks (C x 1000 x 24 B) stream through HBM once per refill, >> 126 MB L2",
           "parallelism": f"chains sharded over {world} GPU(s); shared proposal: " +
                          ("gradients all-reduced per Adam step" if a.sampler == "glmcmc_nf" else
                           f"{a.kde_train} training draws all-gathered per fit")}
    line = {"metric": "abc_mcmc_chain_steps_per_sec", "value": value, "unit": "chain-steps/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16/f32" if a.sampler == "glmcmc_nf" else "f32", "data": "synthetic", "config": cfg, "clocks": clocks,
            "gpu_launches": n_launch_calls - 4 * a.steps, "roofline": roofline,
            "esjd": {"mean_per_chain": float(st.esjd().mean()), "move_rate": float(st.move_rate.mean())}}
    line["esjd"]["aggregate_esjd_per_sec"] = line["esjd"]["mean_per_chain"] * value
    if not a.no_e2e:
        call(z_host, 1000)
        barrier()
        t0 = time.perf_counter()
        e_steps = max(1, min(a.steps, 2))
        for i in range(e_steps):
            _, st = call(z_host, 1001 + i)
            h = st.raw.cpu()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        line["e2e"] = {"value": steps_per_pass * e_steps / float(dt.item()), "unit": "chain-steps/s", "h2d_bytes_per_step": 8,
                       "d2h_bytes_per_step": h.numel() * 4, "steps": e_steps,
                       "note": "public entry point with host tensors in (theta0 broadcast to the chains on the device), per-chain statistics out"}
    if rank == 0 and not a.no_cpu:
        if a.sampler == "aglmcmc_pooled":
            r, cores, sample, cpu_esjd = cpu_port_rate(C, T, a.cpu_seconds, sampler="aglmcmc")
            line["cpu_baseline"] = {"value": r, "unit": "chain-steps/s", "cores": cores, "kind": "port",
                                    "sample": sample + " (the reference's own per-chain KDE: it has no pooled mode)"}
        else:
            cf = RealNVP()
            n_eval = 4096
            torch.set_num_threads(os.cpu_count() or 1)
            with torch.no_grad():
                t0 = time.perf_counter()
                reps = 0
                while time.perf_counter() - t0 < a.cpu_seconds:
                    xs, _ = cf.sample(n_eval)
                    cf.log_prob(xs[: n_eval // K])
                    reps += 1
                dt = time.perf_counter() - t0
            moves = reps * (n_eval // K)                 # a global move = K fresh samples + 1 log_prob (GLMCMC_NFs.py:98,127)
            line["cpu_baseline"] = {"value": moves / dt / gf, "unit": "chain-steps/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"fp32 torch RealNVP (flows.py restatement of the normflows model) on the host: {reps} x "
                                              f"({n_eval} samples + {n_eval // K} log_probs) in {dt:.1f} s; flow evaluations only "
                                              "(the step arithmetic is negligible beside them), batched — the reference evaluates log_prob on a batch of one"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


def other_kernels(eng, model, lp, gp):
    """Short device-resident timings of the other hot-path kernels (the headline line stays GlobalMCMC, BASELINE configs[1]);
    full lines with e2e / cpu_baseline: `bench.py --sampler glmcmc|glmala|aglmcmc|kde`.  CUDA events, 3 warm-up + 5 timed."""
    import torch
    import glabc_b200 as g
    from glabc_b200.flows import RealNVP

    def timed(fn, units):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        return {"ms": ms, "per_sec": units / (ms * 1e-3)}

    z = torch.zeros(2)
    out = {}
    out["glmcmc_isir_K5"] = dict(timed(lambda: g.GLMCMC(model, 10000, z, None, lp, None, 0.9, gp, 5, num_chains=65536, seed=1, trace="none"),
                                       65536 * 9999), unit="chain-steps/s", workload="65,536 chains x 1e4, gf 0.9, statistics only")
    out["glmala"] = dict(timed(lambda: g.GLMALA(model, 1001, z, None, 0.3, 100, None, 0.8, gp, 5, num_chains=32768, seed=1, trace="none"),
                               32768 * 1000), unit="chain-steps/s", workload="32,768 chains x 1e3, gf 0.8, tau 0.3, num_grad 100")
    out["aglmcmc"] = dict(timed(lambda: g.AGLMCMC(model, 2001, z, None, lp, gp, None, 1.0, 200, 5, 0.8, 0.2, num_chains=16384, seed=1,
                                                  trace="none"), 16384 * 2000), unit="chain-steps/s",
                          workload="16,384 chains x 2e3, gf 1, K 5, step 200")
    from glabc_b200.models import mixture_user_model
    um, y0 = mixture_user_model(0.05), torch.randn(65536, 2, device="cuda") * 0.2236
    out["global_user_model_nvrtc"] = dict(timed(lambda: g.GlobalMCMC(um, 10000, z, y0, gp, None, 0.5, lp, num_chains=65536, seed=1,
                                                                     trace="none"), 65536 * 9999), unit="chain-steps/s",
                                          workload="65,536 chains x 1e4, the README model given as CUDA source and compiled by NVRTC "
                                                   "into the step kernel, statistics only")
    X = torch.randn(100000, 2, device="cuda")
    w, bw = eng.kde_fit(X, None)
    out["kde_log_prob"] = dict(timed(lambda: eng.kde_log_prob(X, w, bw, X), 1e10), unit="pairs/s", workload="1e5 queries x 1e5 points, d = 2")
    flow = RealNVP(device="cuda")
    with torch.no_grad():
        flow.w3.copy_(0.05 * torch.randn_like(flow.w3))
    flow.bind(eng)
    eps = torch.randn(1 << 21, 2, device="cuda")
    r = timed(lambda: flow.fused_sample_from(eps, eng, precision="fast"), float(1 << 21))
    out["realnvp_sample_tcgen05"] = dict(r, unit="samples/s", tflops_f16=r["per_sec"] * 1.049e6 / 1e12,
                                         workload="2,097,152 samples through 32 coupling blocks (128x128 hidden layer on tensor cores), "
                                                  "GLABC_FLOW_FAST: single FP16 operands")
    r = timed(lambda: flow.fused_sample_from(eps, eng, precision="precise"), float(1 << 21))
    out["realnvp_sample_tcgen05_precise"] = dict(r, unit="samples/s", tflops_f16_issued=3 * r["per_sec"] * 1.049e6 / 1e12,
                                                 workload="same, GLABC_FLOW_PRECISE (the samplers' default): FP16 hi + lo split, three MMAs per "
                                                          "K step, 1e-5-class log-densities")
    return out


def other_configs(a, eng, model, lp, gp, rank, world, info, sm_max_mhz, peaks):
    """BASELINE configs 3-5 and the strong-scaling form of config 2, at THIS world size (every rank takes part; chains are
    sharded by rank with Philox keyed by the global chain id).  Short runs: CUDA events on the launching stream, barrier on both
    sides, max over ranks; `value` = chain-steps of all ranks / that time; `kernel_ms` = one launch of the dominant kernel timed
    alone on rank 0's GPU; `roofline.frac` against the same peaks as the headline line."""
    import torch
    import torch.distributed as dist
    import glabc_b200 as g
    from glabc_b200 import _abi as abi
    from glabc_b200 import sweeps
    from glabc_b200.flows import RealNVP
    inst_peak = info["sm_count"] * 128 * sm_max_mhz * 1e6

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, reps, warm=1):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def step_kernel(entry, C, T, gf, K, layout, alg_inst, reps, **extra):
        """device-resident pass of a fused step kernel: C chains per rank x (T - 1) transitions"""
        d = 2
        theta0 = torch.zeros(C, d, device="cuda")
        y0 = torch.randn(C, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(99 + rank)) * 0.22360679507255554
        theta, y = theta0.clone(), y0.clone()
        stats = torch.zeros(C, abi.nstats(d), device="cuda")
        aux0 = None
        if K:
            aux0 = torch.zeros(C, abi.AUX_SLOTS, device="cuda")
            aux0[:, abi.AUX_LOCAL] = 1.0
        aux = None if aux0 is None else aux0.clone()
        if entry == "mala":
            extra = dict(extra, state64=torch.zeros(C, abi.STATE64_SLOTS, device="cuda", dtype=torch.float64))
        trace = None if layout == abi.TRACE_NONE else torch.empty(C, T, d, device="cuda")

        def fn():
            theta.copy_(theta0)
            y.copy_(y0)
            stats.zero_()
            if aux is not None:
                aux.copy_(aux0)
            if "state64" in extra:
                extra["state64"].zero_()
            eng.run(entry, theta=theta, y=y, n_steps=T - 1, gf=gf, seed=3, chain_id_base=rank * C, trace_layout=layout,
                    trace=trace, trace_rows=T, stats=stats, K=K, aux=aux, **extra)
        ms = timed(fn, reps)
        rate = float(C) * (T - 1) * world / (ms * 1e-3)
        frac = rate / world * alg_inst / inst_peak
        return {"value": rate, "unit": "chain-steps/s", "ms_per_pass": ms, "kernel_ms": ms, "chains_total": C * world, "chains_per_gpu": C,
                "iterations": T, "roofline": {"bound": "alu-issue", "frac": frac, "alg_inst_per_chain_step": alg_inst,
                                              "note": "state reset + one fused step kernel per pass; frac = per-GPU rate x algorithmic "
                                                      "thread-instructions / (SMs x 128 x max clock)"}}

    out = {}
    # (iv) BASELINE metric's own size: 65,536 chains IN TOTAL (strong scaling), full chain-major trace on the device
    out["global_strong_65536"] = dict(step_kernel("global", 65536 // world, a.iters, 0.5, 0, abi.TRACE_CHAIN_MAJOR, 186, reps=20),
                                      scaling="strong", workload="BASELINE configs[1]: GlobalMCMC, 65,536 chains in total, full [C,T,2] trace")
    # (i) BASELINE configs[2]: 262,144 chains in total
    out["glmcmc_262144"] = dict(step_kernel("isir", 262144 // world, 10000, 0.9, 5, abi.TRACE_NONE, 703, reps=3), scaling="strong",
                                workload="BASELINE configs[2]: run_glmcmc iSIR K=5 gf=0.9, 262,144 chains in total x 1e4, statistics only")
    out["glmala_262144"] = dict(step_kernel("mala", 262144 // world, 1001, 0.8, 5, abi.TRACE_NONE, 5000, reps=2, num_grad=100, tau=0.3),
                                scaling="strong",
                                workload="BASELINE configs[2]: run_glmala K=5 gf=0.8 tau=0.3 num_grad=100, 262,144 chains in total x 1e3, statistics only")
    torch.cuda.empty_cache()

    # (ii) BASELINE configs[3]: GLMCMC-NFs, 1,048,576 chains in total, one shared flow (gradients all-reduced per Adam step)
    C_nf, T_nf = 1048576 // world, 401
    z = torch.zeros(2, device="cuda")

    def nf_call():
        return g.GLMCMC_NF(model, T_nf, z, None, lp, None, 0.5, 200, 5, None, 50, num_chains=C_nf, seed=5, chain_id_base=rank * C_nf,
                           trace="none", return_stats=True, verbose=False)
    ms = timed(nf_call, reps=1, warm=1)
    flow = RealNVP(device="cuda")
    with torch.no_grad():
        flow.w3.copy_(0.05 * torch.randn_like(flow.w3))
    flow.bind(eng)
    n_s = 1 << 21
    eps = torch.randn(n_s, 2, device="cuda")
    th, lq = torch.empty(n_s, 2, device="cuda"), torch.empty(n_s, device="cuda")
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def flow_ms(precision):
        flow.fused_sample_from(eps, eng, theta=th, log_q=lq, precision=precision)
        torch.cuda.synchronize()
        k0.record()
        for _ in range(3):
            flow.fused_sample_from(eps, eng, theta=th, log_q=lq)
        k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / 3
    kms_fast = flow_ms("fast")
    kms = flow_ms("precise")      # the mode the sampler call above ran in
    tf = 3 * n_s * 1.049e6 / (kms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops", 1654.4))
    out["glmcmc_nf_1M"] = {"value": float(C_nf) * (T_nf - 1) * world / (ms * 1e-3), "unit": "chain-steps/s", "ms_per_pass": ms,
                           "kernel_ms": kms, "chains_total": C_nf * world, "chains_per_gpu": C_nf, "iterations": T_nf, "scaling": "strong",
                           "flow_precision": "precise (FP16 hi + lo split, three MMAs; log-densities within 1e-5 of float64)",
                           "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                                        "samples_per_sec": n_s / (kms * 1e-3),
                                        "fast_mode": {"kernel_ms": kms_fast, "samples_per_sec": n_s / (kms_fast * 1e-3),
                                                      "tflops": n_s * 1.049e6 / (kms_fast * 1e-3) / 1e12,
                                                      "frac": n_s * 1.049e6 / (kms_fast * 1e-3) / 1e12 / peak},
                                        "note": f"k_flow sample, {n_s} samples x 32 coupling blocks; achieved = tensor-core FLOPs ISSUED "
                                                "(3 x 1.049 MFLOP per sample in the split-precision mode the sampler runs; fast_mode: one MMA)"},
                           "workload": "BASELINE configs[3]: run_glmcmc_nf gf=0.5 K=5 step 200, 50 train steps, 1,048,576 chains in total, "
                                       "statistics only (one sampler call per pass: block refills + flow training inside)"}
    del eps, th, lq, flow
    torch.cuda.empty_cache()

    # (iii) BASELINE configs[4]: AGLMCMC with ONE pooled KernelDensity over 1e5 draws (all-gathered before every fit) ...
    C_ag, T_ag = 16384, 1001

    def ag_call():
        return g.AGLMCMC(model, T_ag, z, None, lp, gp, None, 1.0, 200, 5, 0.8, 0.2, num_chains=C_ag, seed=6, chain_id_base=rank * C_ag,
                         trace="none", return_stats=True, verbose=False, pooled=True, kde_train=a.kde_train)
    ms = timed(ag_call, reps=1, warm=1)
    n = a.kde_train
    X = torch.randn(n, 2, device="cuda")
    wn, bw = eng.kde_fit(X, torch.rand(n, device="cuda"))
    q = torch.randn(C_ag * 250, 2, device="cuda")
    eng.kde_log_prob(X, wn, bw, q)
    torch.cuda.synchronize()
    k0.record()
    eng.kde_log_prob(X, wn, bw, q)
    k1.record()
    torch.cuda.synchronize()
    kms = k0.elapsed_time(k1)
    pair_rate = float(q.shape[0]) * n / (kms * 1e-3)
    mufu_peak = info["sm_count"] * 16 * sm_max_mhz * 1e6
    out["aglmcmc_pooled_kde1e5"] = {"value": float(C_ag) * (T_ag - 1) * world / (ms * 1e-3), "unit": "chain-steps/s", "ms_per_pass": ms,
                                    "kernel_ms": kms, "chains_total": C_ag * world, "chains_per_gpu": C_ag, "iterations": T_ag,
                                    "scaling": "weak", "kde_train_total": n,
                                    "roofline": {"bound": "mufu", "achieved": pair_rate / 1e9, "peak": mufu_peak / 1e9, "unit": "Gex2/s",
                                                 "frac": pair_rate / mufu_peak,
                                                 "note": f"k_kde_logprob, {q.shape[0]} queries x {n} pooled points, one ex2 per pair"},
                                    "workload": "BASELINE configs[4]: run_aglmcmc gf=1 K=5 step 200 alpha 0.8 eps_hat_T 0.2 with one pooled "
                                                "KernelDensity (1e5 training draws all-gathered per fit), 16,384 chains per GPU"}
    del X, q
    torch.cuda.empty_cache()
    # ... plus the ESJD hyper-parameter sweep of examples/Mixture_hyper.py:23-41 (11 global_frequency values, run_glmcmc K=5),
    # grid points dealt to the ranks, score table all-reduced
    barrier()
    t0 = time.perf_counter()
    best, table = sweeps.esjd_sweep(lambda gf, **kw: g.GLMCMC(model, 1000, z, None, lp, None, gf, gp, 5, verbose=False, **kw),
                                    num_chains=8192, seed=7, rank=rank, world=world)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    out["esjd_sweep_mixture_hyper"] = {"best_global_frequency": best, "seconds": float(dt.item()), "grid_points": int(table.shape[0]),
                                       "chains_per_point": 8192, "iterations": 1000,
                                       "esjd_per_sec": [float(v) for v in table[:, 3]], "mean_esjd": [float(v) for v in table[:, 1]],
                                       "workload": "Mixture_hyper.py:23-41: esjd / seconds-per-iteration of run_glmcmc(1000 its, K=5) over "
                                                   "global_frequency in {0, 0.1, .., 1}; the reference's 10 seeds become 8,192 chains per point"}
    return out


def replay_parity_bit(eng, abi, entry, gf, T, trace_first64, theta0, y0, seed, chain_base):
    """SURVEY.md 8(d) config 2: the first 64 chains of the TIMED configuration against the oracle.  The kernel re-runs them in
    the reference's float32 operation order (STRICT) dumping every Philox draw it uses; the oracle replays the dump; and the rows
    the timed FAST launch wrote for those chains are compared with that replay."""
    import numpy as np
    import torch
    from glabc_b200.models import lower_model, lower_proposal
    from oracle import oracle
    model, lp, gp = workload_objects()
    n = 64
    th, yy = theta0[:n].clone(), y0[:n].clone()
    dump = torch.zeros(T - 1, 6, n, device="cuda")
    got = eng.run(entry, theta=th, y=yy, n_steps=T - 1, gf=gf, seed=seed, chain_id_base=chain_base, arith=abi.ARITH_STRICT,
                  trace_layout=abi.TRACE_TIME_MAJOR, tape_dump=dump)
    torch.cuda.synchronize()
    th_o, y_o = theta0[:n].cpu().numpy().copy(), y0[:n].cpu().numpy().copy()
    want = oracle.run(entry, lower_model(model), lower_proposal(lp), lower_proposal(gp), theta=th_o, y=y_o, n_steps=T - 1, gf=gf,
                      rng_mode=abi.RNG_REPLAY, tape32=dump.cpu().numpy())
    strict_equal = bool(np.array_equal(got.cpu().numpy(), want))
    fast = trace_first64.cpu().numpy()                       # [64, T, 2] rows of the timed launch
    same = float((fast.transpose(1, 0, 2) == want).all(-1).mean())
    return {"chains": n, "transitions": T - 1, "strict_kernel_equals_oracle_bitwise": strict_equal, "timed_fast_rows_equal_oracle": same,
            "note": "oracle = C restatement of GlobalMCMC.py:37-68 pinned by tests/golden; draws = the kernel's own Philox stream"}


def workload_config(a, cpu=None):
    spec = SAMPLERS[a.sampler]
    cfg = {"workload": spec["workload"], "chains_per_gpu": a.chains,
           "iterations": a.iters, "theta_dim": 2, "epsilon": 0.05, "global_frequency": spec["gf"],
           "local_sigma": 0.35, "global_proposal": "N(0,I)", "isir_candidates": spec["K"], "trace": {"chain": "full float32 [C,T,2]",
           "time": "full float32 [T,C,2]", "none": "statistics only"}[a.layout], "rng": "philox4x32-10 native"}
    if cpu is None:
        cfg.update({"arith": "fast", "l2": "no re-read inputs; 5.2 GB trace written per step >> 126 MB L2",
                    "parallelism": f"chains sharded over {a.gpus} GPU(s), no data-path collective"})
    else:   # the CPU arm: the oracle port in the reference's float32 operation order, a bounded sample of the workload per step
        cfg.update({"arith": "reference float32 order (C port of GlobalMCMC.py:37-68 / GLMCMC.py:58-104)",
                    "sample_per_step": f"{cpu['chains_per_step']} chains x {cpu['transitions']} transitions (of {a.chains} x {a.iters - 1})",
                    "parallelism": f"{cpu['threads']} host threads, chains split over them"})
    return cfg


def main():
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL's version banner, ...) are sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    try:
        _main()
    finally:
        sys.stdout.flush()
        os.dup2(json_fd, 1)
        os.close(json_fd)
        if _RESULT:
            print(_RESULT[-1], flush=True)


_RESULT = []


def emit(line):
    _RESULT.append(json.dumps(line))


def _main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.sampler == "kde":
        if a.impl == "reference":
            if rank == 0:
                emit({"impl": "reference", "unavailable": "--sampler kde has no reference arm; see cpu_baseline of the native line"})
            return
        bench_kde(a, rank, world, local_rank)
        return
    if a.sampler in SHARED:
        if a.impl == "reference":
            if rank == 0:
                emit({"impl": "reference", "unavailable": f"--sampler {a.sampler}: see cpu_baseline of the native line"})
            return
        bench_shared(a, rank, world, local_rank)
        return
    if a.impl == "reference":
        bench_reference(a, rank)
        return

    import torch
    import torch.distributed as dist
    import glabc_b200 as g  # noqa: F401
    from glabc_b200 import _abi as abi
    from glabc_b200 import sharding
    from glabc_b200.engine import RunStats, get_engine

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = get_engine()
    model, lp, gp = workload_objects()
    eng.bind_model(model)
    eng.bind_proposal(abi.SLOT_LOCAL, lp)
    eng.bind_proposal(abi.SLOT_GLOBAL, gp)
    eng.bind_proposal(abi.SLOT_IMPORTANCE, gp)   # README.md:125: the iSIR importance proposal is the same N(0,I)
    spec = SAMPLERS[a.sampler]
    entry, gf, K = spec["entry"], spec["gf"], spec["K"]
    info = eng.ctx.device_info()

    C, T, d = a.chains, a.iters, 2
    layout = {"chain": abi.TRACE_CHAIN_MAJOR, "time": abi.TRACE_TIME_MAJOR, "none": abi.TRACE_NONE}[a.layout]
    chain_base = rank * C
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    theta0 = torch.zeros(C, d, device="cuda")
    y0 = torch.randn(C, d, device="cuda", generator=gen) * 0.22360679507255554
    trace = None
    if layout != abi.TRACE_NONE:
        trace = torch.empty((C, T, d) if layout == abi.TRACE_CHAIN_MAJOR else (T, C, d), device="cuda")
    theta, y = theta0.clone(), y0.clone()
    stats = torch.zeros(C, abi.nstats(d), device="cuda")
    aux0 = aux = None
    if K and entry != "aglmcmc":
        aux0 = torch.zeros(C, abi.AUX_SLOTS, device="cuda")
        aux0[:, abi.AUX_LOCAL] = 1.0
        aux = aux0.clone()
    summary = None
    extra, s64 = {}, None
    if entry == "mala":
        s64 = torch.zeros(C, abi.STATE64_SLOTS, device="cuda", dtype=torch.float64)
        extra = dict(num_grad=spec["num_grad"], tau=spec["tau"], state64=s64)

    if entry == "aglmcmc":
        extra = dict(ag=eng.aglmcmc_params(step_size=spec["step_size"], alpha=spec["alpha"], hat_eps_T=spec["hat_eps_T"]))

    def reset_state():
        theta.copy_(theta0)
        y.copy_(y0)
        if aux is not None:
            aux.copy_(aux0)
        if s64 is not None:
            s64.zero_()

    pending = []   # (summary tensor, NCCL work handle) of the passes whose all-reduce is still in flight

    def one_step(step_idx):
        nonlocal summary
        reset_state()
        stats.zero_()
        eng.run(entry, theta=theta, y=y, n_steps=T - 1, gf=gf, seed=step_idx, chain_id_base=chain_base,
                trace_layout=layout, trace=trace, trace_rows=T, stats=stats, block_threads=a.block, K=K, aux=aux, **extra)
        rs = RunStats(stats, d)
        summary = sharding.summarize(rs).to(torch.float64)
        if world > 1:
            # the one collective of the path (6 + 2d float64 scalars): asynchronous, on NCCL's own stream, so the next pass's
            # kernel does not wait for it; all of them are waited for before the timed region closes
            pending.append((summary, dist.all_reduce(summary, op=dist.ReduceOp.SUM, async_op=True)))

    def drain():
        for _, work in pending:
            work.wait()
        pending.clear()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for w in range(a.warmup):
        one_step(w)
    drain()
    # kernel-only duration of the dominant kernel, CUDA events on the launching stream
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    barrier()
    n_idle = len(sampler.rows)   # samples taken before the timed region are dropped
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(a.steps):
        one_step(a.warmup + s)
    drain()
    e1.record()
    barrier()
    sampler.rows = sampler.rows[max(0, n_idle - 1):]
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    steps_per_pass = C * (T - 1) * world
    last_seed = a.warmup + a.steps - 1
    first64 = trace[:64].clone() if (layout == abi.TRACE_CHAIN_MAJOR and entry == "global" and C >= 64) else None
    value = steps_per_pass * a.steps / (total_ms * 1e-3)
    if a.dump_outputs and rank == 0:
        # before the kernel-only timings below overwrite the state, stats and trace
        outs = {"theta": (theta, 0), "y": (y, 0), "stats": (stats, 0), "summary": (summary, None)}
        if trace is not None:
            outs["trace"] = (trace, 0 if layout == abi.TRACE_CHAIN_MAJOR else 1)
        if aux is not None:
            outs["aux"] = (aux, 0)
        if s64 is not None:
            outs["state64"] = (s64, 0)
        dump_outputs(a.dump_outputs, outs)

    # the step kernel alone (no state reset / summary kernels around it)
    for s in range(min(a.steps, 20)):
        reset_state()
        k0.record()
        eng.run(entry, theta=theta, y=y, n_steps=T - 1, gf=gf, seed=s, chain_id_base=chain_base,
                trace_layout=layout, trace=trace, trace_rows=T, stats=stats, block_threads=a.block, K=K, aux=aux, **extra)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms.append(k0.elapsed_time(k1))
    kms = sum(kernel_ms) / len(kernel_ms)
    kernel_rate = C * (T - 1) / (kms * 1e-3)

    # kernels of ours per pass: one fused step kernel, or for AGLMCMC the init pair + per round (step + 8 adaptation kernels)
    # (+ 1: the fused summary kernel glabc_summarize that closes every pass)
    launches_per_pass = 1 + (1 if entry != "aglmcmc" else 3 + ((T - 1) // spec["step_size"] + 2) * 9)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    sm_max_mhz = float(peaks.get("sm_max_mhz", clocks.get("sm_max_mhz") or 1965.0))
    inst_peak = info["sm_count"] * 128 * sm_max_mhz * 1e6 / 1e9            # G thread-inst/s at max clock
    inst_ach = kernel_rate * spec["alg_inst"] / 1e9
    hbm_ach = kernel_rate * ALG_BYTES_PER_STEP / 1e9 if layout != abi.TRACE_NONE else 0.0
    traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of the step kernel, one ncu --set full capture per workload
    try:
        with open(os.path.join(ROOT, "profiles", "r1_traffic.json")) as f:
            tr = json.load(f).get(f"{a.sampler}:{C}x{T}:{a.layout}")
            traffic = tr["bytes"] if tr else None
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "alu-issue", "achieved": inst_ach, "peak": inst_peak, "unit": "Gthread-inst/s",
                "frac": inst_ach / inst_peak, "traffic": traffic,
                "note": f"{spec['alg_inst']} algorithmic thread-instructions per chain-step (SURVEY.md 8(d)); peak = "
                        f"{info['sm_count']} SMs x 128 lanes x {sm_max_mhz:.0f} MHz; kernel {kms:.3f} ms per launch",
                "hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
                "kernel_ms": kms, "kernel_chain_steps_per_sec": kernel_rate}

    line = {"metric": "abc_mcmc_chain_steps_per_sec", "value": value, "unit": "chain-steps/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": total_ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(a),
            "clocks": clocks, "gpu_launches": a.steps * launches_per_pass, "roofline": roofline}
    if summary is not None:
        desc = sharding.describe(summary.cpu(), d)
        line["esjd"] = {"mean_per_chain": desc["mean_esjd"], "aggregate_esjd_per_sec": desc["mean_esjd"] * value,
                        "move_rate": desc["move_rate"]}

    # end-to-end through the reference-facing call with HOST buffers (pinned): H2D state, kernels in time
    # chunks, D2H of the full trace overlapped, D2H state + stats — every step.
    if not a.no_e2e and entry == "aglmcmc":
        # no host-buffer C entry for AGLMCMC yet: e2e through the public Python call with host tensors in and the
        # chains copied back (run_chains: H2D of theta / y, device run, D2H of the full trace)
        import glabc_b200 as g
        e_steps = max(1, min(a.steps, 3))
        del trace
        torch.cuda.empty_cache()
        h_theta0, h_y0 = theta0.cpu(), y0.cpu()

        h_out = torch.empty((T, C, d)).pin_memory()     # the caller's (pinned) result buffer, reused every step

        def e2e_step(i):
            out = g.AGLMCMC(model, T, h_theta0, h_y0, lp, gp, None, gf, spec["step_size"], K, spec["alpha"], spec["hat_eps_T"],
                            num_chains=C, seed=i, chain_id_base=chain_base, trace="time", verbose=False)
            h_out.copy_(out, non_blocking=True)
            torch.cuda.synchronize()
            return h_out
        e2e_step(0)
        barrier()
        t0 = time.perf_counter()
        for i in range(e_steps):
            res = e2e_step(1 + i)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        line["e2e"] = {"value": steps_per_pass * e_steps / float(dt.item()), "unit": "chain-steps/s",
                       "h2d_bytes_per_step": (h_theta0.numel() + h_y0.numel()) * 4, "d2h_bytes_per_step": res.numel() * 4,
                       "steps": e_steps, "note": "glabc_b200.AGLMCMC(...) with host tensors in, full [T,C,2] trace copied into a pinned host buffer"}
    elif not a.no_e2e:
        e_steps = max(1, min(a.steps, 3))
        h_theta0, h_y0 = theta0.cpu().pin_memory(), y0.cpu().pin_memory()
        h_theta, h_y = torch.empty_like(h_theta0).pin_memory(), torch.empty_like(h_y0).pin_memory()
        h_stats = torch.zeros(C, abi.nstats(d)).pin_memory()
        h_aux0 = aux0.cpu().pin_memory() if K else None
        h_aux = torch.empty_like(h_aux0).pin_memory() if K else None
        h_extra = dict(extra)
        if s64 is not None:
            h_extra["state64"] = torch.zeros(C, abi.STATE64_SLOTS, dtype=torch.float64).pin_memory()
        # host view: chain-major [C, T, 2] for GlobalMCMC (out[c] is a reference-shaped chain; glabc_run_global_host brings part
        # of the chains back as move events and expands them on the host cores), time-major for the other samplers
        chain_host = entry in ("global", "isir") and layout != abi.TRACE_NONE
        h_layout = abi.TRACE_NONE if layout == abi.TRACE_NONE else (abi.TRACE_CHAIN_MAJOR if chain_host else abi.TRACE_TIME_MAJOR)
        del trace
        torch.cuda.empty_cache()
        h_trace = None if h_layout == abi.TRACE_NONE else torch.empty((C, T, d) if chain_host else (T, C, d)).pin_memory()

        def e2e_step(i):
            h_theta.copy_(h_theta0)
            h_y.copy_(h_y0)
            h_stats.zero_()
            if K:
                h_aux.copy_(h_aux0)
            if s64 is not None:
                h_extra["state64"].zero_()
            eng.run_host(entry, theta=h_theta, y=h_y, n_steps=T - 1, gf=gf, seed=i, chain_id_base=chain_base,
                         trace=h_trace, trace_layout=h_layout, stats=h_stats, block_threads=a.block, K=K, aux=h_aux,
                         **h_extra)
        e2e_step(0)
        barrier()
        t0 = time.perf_counter()
        for i in range(e_steps):
            e2e_step(1 + i)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = (h_theta.numel() + h_y.numel() + h_stats.numel()) * 4
        d2h = h2d + (h_trace.numel() * 4 if h_trace is not None else 0)
        # the same call when the caller wants the in-kernel statistics (ESJD Gram, moments, acceptance) instead of the chain
        def e2e_stats_step(i):
            h_theta.copy_(h_theta0)
            h_y.copy_(h_y0)
            h_stats.zero_()
            if K:
                h_aux.copy_(h_aux0)
            if s64 is not None:
                h_extra["state64"].zero_()
            eng.run_host(entry, theta=h_theta, y=h_y, n_steps=T - 1, gf=gf, seed=i, chain_id_base=chain_base, trace=None,
                         trace_layout=abi.TRACE_NONE, stats=h_stats, block_threads=a.block, K=K, aux=h_aux, **h_extra)
        e2e_stats_step(0)
        barrier()
        t1 = time.perf_counter()
        for i in range(e_steps):
            e2e_stats_step(1 + i)
        barrier()
        dt_s = torch.tensor([time.perf_counter() - t1], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt_s, op=dist.ReduceOp.MAX)
        line["e2e_stats_only"] = {"value": steps_per_pass * e_steps / float(dt_s.item()), "unit": "chain-steps/s",
                                  "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h2d,
                                  "note": "same host-buffer call with trace_layout NONE: state + statistics copied back, no chain"}
        wire = None
        if chain_host and os.environ.get("GLABC_HOST_EVENTS", "1") != "0":
            cap = min(T + 1, max(64, (T - 1) // 32))            # event capacity per chain (csrc/abi.cu run_global_host_hybrid)
            wire = h2d + C * cap * (1 + d) * 4
        line["e2e"] = {"value": steps_per_pass * e_steps / float(dt.item()), "unit": "chain-steps/s",
                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e_steps,
                       "pcie_d2h_bytes_per_step": wire if wire is not None else d2h,
                       "note": (f"glabc_run_{entry}_host: pinned host buffers, the full dense float32 trace [C,T,2] delivered to the host: "
                                "the chains travel as run-length (move) events (a chain moves on ~1 % of its steps) and the host cores "
                                "expand them into the dense buffer with full-line non-temporal stores, group by group while the next "
                                "group's kernel runs; bit-identical to the dense PCIe copy (GLABC_HOST_EVENTS=0), bounded by the "
                                "host's DRAM write rate instead of PCIe") if chain_host else
                               (f"glabc_run_{entry}_host: pinned host buffers, full trace copied back in time chunks "
                                "overlapped with the kernels; host view [T,C,2] (chain c = trace[:, c])")}

    if a.sampler == "global" and not a.no_extra and not a.no_other_configs:
        torch.cuda.empty_cache()
        oc = other_configs(a, eng, model, lp, gp, rank, world, info, sm_max_mhz, peaks)   # every rank takes part
        if rank == 0:
            line["other_configs"] = oc
        eng.bind_model(model)
        eng.bind_proposal(abi.SLOT_LOCAL, lp)
        eng.bind_proposal(abi.SLOT_GLOBAL, gp)
        eng.bind_proposal(abi.SLOT_IMPORTANCE, gp)
    if rank == 0 and world == 1 and a.sampler == "global" and not a.no_extra:
        line["other_kernels"] = other_kernels(eng, model, lp, gp)
    if rank == 0 and not a.no_cpu:
        r, cores, sample, cpu_esjd = cpu_port_rate(C, T, a.cpu_seconds, sampler=a.sampler)
        line["cpu_baseline"] = {"value": r, "unit": "chain-steps/s", "cores": cores, "kind": "port", "sample": sample,
                                "esjd": {"mean_per_chain": cpu_esjd, "aggregate_esjd_per_sec": cpu_esjd * r}}
        if first64 is not None:
            eng.bind_model(model)
            eng.bind_proposal(abi.SLOT_LOCAL, lp)
            eng.bind_proposal(abi.SLOT_GLOBAL, gp)
            line["parity"] = replay_parity_bit(eng, abi, entry, gf, T, first64, theta0, y0, last_seed, chain_base)
        if world == 1 and a.sampler in ("global", "glmcmc") and not a.no_ref_python:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import ref_python
            line["cpu_baseline"]["reference_python"] = ref_python.measure(a.ref_python_its, sampler=a.sampler)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


if __name__ == "__main__":
    main()
