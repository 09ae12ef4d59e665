"""Chain-steps/s of the block-iSIR samplers with the README model as a run-time compiled `UserModel`
(models.mixture_user_model: glabc_k_block_isir_user + glabc_k_block_weights_user) next to the built-in `Mixture_set`
(k_ag_step<EXT> + k_blk_weights), same proposals, same seeds, statistics only:
  * GLMCMC-NFs: 131,072 chains x 1,000 iterations, gf 0.5, K 5, step_size 200, `--train` training steps (shared RealNVP);
  * pooled AGLMCMC: 16,384 chains x 1,000 iterations, gf 0.5, K 5, step_size 50, alpha 0.8, hat_eps_T 0.2, kde_train 1e5.
One warm-up call per (sampler, model) — module load and the NVRTC compile — then `reps` timed calls of each, the two models
alternating, CUDA events around each call.  Prints one JSON object with the device name and power limit it ran on.

    python profiles/user_block_isir_bench.py [--reps 3] [--train 3] [--out results.json]
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
from prior_bench import device_info  # noqa: E402

T = 1001


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--train", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    ip = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    z = torch.zeros(2)
    models = {"user": mixture_user_model(0.05), "builtin": g.Mixture_set(0.05)}
    runs = {
        "glmcmc_nf": (131072, lambda m, C, y0: g.GLMCMC_NF(m, T, z, y0, lp, None, 0.5, 200, 5, None, args.train, num_chains=C, seed=5,
                                                           trace="none", verbose=False)),
        "aglmcmc_pooled": (16384, lambda m, C, y0: g.AGLMCMC(m, T, z, y0, lp, ip, None, 0.5, 50, 5, 0.8, 0.2, num_chains=C, seed=5,
                                                             trace="none", verbose=False, pooled=True, kde_train=100000)),
    }
    res = {"workload": f"README model, {T - 1} iterations, statistics only; GLMCMC-NFs 131072 chains gf 0.5 K 5 step 200 "
                       f"train {args.train}; pooled AGLMCMC 16384 chains gf 0.5 K 5 step 50 kde_train 1e5",
           **device_info(), "reps": args.reps}
    for name, (C, fn) in runs.items():
        y0 = torch.randn(C, 2, generator=torch.Generator().manual_seed(1)) * 0.2236
        for m in models.values():
            fn(m, C, y0)                       # warm-up: NVRTC compile, module load, workspaces
        ms = {k: [] for k in models}
        for _ in range(args.reps):
            for k, m in models.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                fn(m, C, y0)
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1))
        res[name] = {k: {"ms": [round(v, 2) for v in ms[k]], "chain_steps_per_s": C * (T - 1) / (min(ms[k]) * 1e-3)}
                     for k in models}
        res[name]["user_over_builtin"] = res[name]["user"]["chain_steps_per_s"] / res[name]["builtin"]["chain_steps_per_s"]
        print(name, res[name], file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
