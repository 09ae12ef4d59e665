"""Chain-steps/s of batched user models (many observed datasets in one run, csrc/user_model.cu -DGLABC_BATCHED) against the
one-dataset kernels, GlobalMCMC, 1e4 iterations, gf 0.5, statistics only.  The model is the README Mixture model as CUDA
source (models.MIXTURE_USER_SOURCE, params y_obs0, y_obs1, noise sd), each dataset with its own y_obs.
  (a) G = 1024 datasets x m = 64 chains: one batched call against 1024 one-dataset calls of 64 chains (the workflow a
      batched model replaces);
  (b) G = 1 x 65,536 chains against the one-dataset kernel at 65,536 chains: the cost of reading the row from the table;
  (c) m = 1, G = 65,536 (every chain its own dataset): the worst case for row locality.
The (b) / (c) / (a)-batched variants alternate in one process, one warm-up each (incl. the NVRTC compile), CUDA events
around each call; the 1024 one-dataset calls are timed once after their warm-up.  Prints one JSON object with the device
name and power limit it ran on.

    python profiles/user_batched_bench.py [--reps 3] [--out results.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import glabc_b200 as g  # noqa: E402
from glabc_b200.models import MIXTURE_USER_SOURCE, mixture_user_model  # noqa: E402
from prior_bench import device_info  # noqa: E402

C, T = 65536, 10000


def model(G):
    y_obs = 1.5 + 0.1 * torch.randn(G, 2, generator=torch.Generator().manual_seed(G))
    params = torch.cat([y_obs, torch.full((G, 1), 0.05 ** 0.5)], dim=1)
    return g.UserModel(MIXTURE_USER_SOURCE, theta_dim=2, y_dim=2, n_noise=2, epsilon=0.05, params=params)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    gp = g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0]))
    z = torch.zeros(2)
    y0 = torch.randn(C, 2, generator=torch.Generator().manual_seed(1)) * 0.2236
    one = mixture_user_model(0.05)

    def run(um, m=None, n=C, base=0, y=y0):
        return g.GlobalMCMC(um, T, z, y, gp, None, 0.5, lp, num_chains=n, seed=1, trace="none", chains_per_dataset=m,
                            chain_id_base=base)

    variants = {
        "unbatched_65536": lambda: run(one),
        "b_G1_m65536": lambda um=model(1): run(um, C),
        "c_G65536_m1": lambda um=model(C): run(um, 1),
        "a_G1024_m64_batched": lambda um=model(1024): run(um, 64),
    }
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for fn in variants.values():
        fn()                               # warm-up: NVRTC compile, module load, table copy
    ms = {k: [] for k in variants}
    for _ in range(args.reps):             # alternated
        for k, fn in variants.items():
            ms[k].append(timed(fn))
    res = {"workload": f"GlobalMCMC, {T} iterations, gf 0.5, statistics only; README model as CUDA source, one y_obs per dataset",
           **device_info(), "reps": args.reps, "variants": {}}
    for k, v in ms.items():
        med = statistics.median(v)
        res["variants"][k] = {"ms": [round(x, 2) for x in v], "median_ms": round(med, 2),
                              "chain_steps_per_s": C * (T - 1) / (med * 1e-3)}
    # (a) the same 1024 x 64 chains as 1024 one-dataset calls (chain ids g m .., so they draw the batched run's numbers)
    um = model(1024)
    ones = [um.dataset(i) for i in range(1024)]
    y64 = y0[:64]
    run(ones[0], n=64, y=y64)              # warm-up
    total = timed(lambda: [run(ones[i], n=64, base=64 * i, y=y0[64 * i:64 * (i + 1)]) for i in range(1024)])
    res["variants"]["a_G1024_m64_1024_calls"] = {"ms": [round(total, 2)], "median_ms": round(total, 2),
                                                 "chain_steps_per_s": C * (T - 1) / (total * 1e-3)}
    base = res["variants"]["unbatched_65536"]["median_ms"]
    res["b_over_unbatched"] = round(res["variants"]["b_G1_m65536"]["median_ms"] / base, 4)
    res["c_over_unbatched"] = round(res["variants"]["c_G65536_m1"]["median_ms"] / base, 4)
    res["a_speedup"] = round(total / res["variants"]["a_G1024_m64_batched"]["median_ms"], 2)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
