"""Rows/s of the user-model evaluation kernel glabc_k_eval_user: a posterior-predictive check of a whole GlobalMCMC trace of
the README Mixture model as a `UserModel` (models.mixture_user_model) -- SIMULATE (generate_samples) and PRIOR
(prior_log_prob) over 65,536 chains x 10,000 rows = 6.55e8 theta rows, 5.2 GB of input, far larger than the 126 MB L2.
The trace comes from one run with Initial_y=None.  CUDA events around `reps` calls after one warm-up call (module load /
NVRTC compile); bytes are the input and output rows each call must move (SIMULATE 16 B/row, PRIOR 12 B/row), against the
7.7 TB/s of the B200's data sheet.  Prints one JSON object with the device name and power limit it ran on.

    python profiles/user_eval_bench.py [--reps 100] [--out results.json]
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

C, T = 65536, 10000
HBM_BYTES_PER_S = 7.7e12


def timed(fn, rows, bytes_per_row, reps):
    out = fn()   # warm-up: module load
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / reps
    bps = rows * bytes_per_row / s
    return out, {"ms": round(s * 1e3, 3), "rows_per_s": rows / s, "bytes_per_s": bps, "of_7.7TB_s": round(bps / HBM_BYTES_PER_S, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    um = mixture_user_model(0.05)
    d, yd = um.theta_dim, um.y_dim
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    gp = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    trace = g.GlobalMCMC(um, T, torch.zeros(2), None, gp, None, 0.5, lp, num_chains=C, seed=1, trace="chain")
    theta = trace.reshape(-1, d)
    rows = theta.shape[0]
    res = {"workload": f"README model as a UserModel; posterior predictive over a {C} x {T} GlobalMCMC trace ({rows} rows)",
           **device_info(), "reps": args.reps}
    y, res["simulate"] = timed(lambda: um.generate_samples(theta, seed=2), rows, 4 * (d + yd), args.reps)
    lpr, res["prior"] = timed(lambda: um.prior_log_prob(theta), rows, 4 * (d + 1), args.reps)
    # the draws are the model's: mean of y - |theta| is 0, its variance the noise variance 0.05
    resid = (y - theta.abs()).double()
    res["check"] = {"resid_mean": float(resid.mean()), "resid_var": float(resid.var()), "prior_finite": bool(torch.isfinite(lpr).all())}
    res["device_after"] = torch.cuda.get_device_name(0)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
