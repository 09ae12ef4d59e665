"""Chain-steps/s of the run-time compiled user-model kernels with each proposal kind in the Global (GlobalMCMC) and
Importance (GLMCMC) slot, next to the built-in kernels on the same proposals (the general k_global_generic /
k_isir_generic for Uniform / Gamma / GaussianMixture, the tuned kernels for DiagGaussian), at bench.py's sizes:
65,536 chains x 1e4 steps, gf 0.5 (GlobalMCMC) / 0.9 with K 5 (GLMCMC), statistics only.  The model is the README
Mixture model, as `Mixture_set` and as CUDA source (models.mixture_user_model).  CUDA events around `reps` runs after one
warm-up run (module load / NVRTC compile); prints one JSON object with the device name and power limit it ran on.

    python profiles/user_proposal_bench.py [--reps 3] [--out results.json]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import glabc_b200 as g  # noqa: E402
from glabc_b200.models import mixture_user_model  # noqa: E402
from prior_bench import device_info, timed  # noqa: E402

C, T = 65536, 10000


def proposals():
    two = lambda v: torch.full((2,), float(v))  # noqa: E731
    return dict(
        gauss=g.DiagGaussian(2, torch.tensor([0.0, 0.0]), torch.tensor([0.0, 0.0])),
        uniform=g.Uniform(2, two(-3.0), two(3.0)),
        gamma=g.Gamma(two(2.0), two(1.5)),
        mix=g.GaussianMixture(2, 2, loc=[[1.4, 1.4], [-1.4, -1.4]], scale=[[0.5, 0.5]] * 2, weights=[0.5, 0.5]),
    )


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    z = torch.zeros(2)
    y0 = torch.randn(C, 2, generator=torch.Generator().manual_seed(1)) * 0.2236
    models = {"user": mixture_user_model(0.05), "builtin": g.Mixture_set(0.05)}
    res = {"workload": f"{C} chains x {T} steps, statistics only; GlobalMCMC gf 0.5, GLMCMC gf 0.9 K 5; local DiagGaussian",
           **device_info(), "reps": args.reps, "global": {}, "glmcmc": {}}
    for kind, q in proposals().items():
        for name, m in models.items():
            run_g = lambda m=m, q=q: g.GlobalMCMC(m, T, z, y0, q, None, 0.5, lp, num_chains=C, seed=1, trace="none")  # noqa: E731
            run_i = lambda m=m, q=q: g.GLMCMC(m, T, z, y0, lp, None, 0.9, q, 5, num_chains=C, seed=1, trace="none")  # noqa: E731
            res["global"].setdefault(kind, {})[name] = timed(run_g, C * (T - 1), args.reps)
            res["glmcmc"].setdefault(kind, {})[name] = timed(run_i, C * (T - 1), args.reps)
            print(kind, name, res["global"][kind][name], res["glmcmc"][kind][name], file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
