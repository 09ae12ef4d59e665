"""Chain-steps/s of every sampler with the model's DiagGaussian prior (the tuned kernels) and with a Uniform and a Gamma
prior (glabc_model_prior_set: the general GlobalMCMC / GLMCMC kernels, k_mala_fast<GPRIOR>, k_ag_step<GPRIOR>), at the
sizes bench.py times the samplers.  Prints one JSON object, with the device name and power limit it ran on.

    python profiles/prior_bench.py [--reps 3] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import glabc_b200 as g  # noqa: E402


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def timed(fn, units, reps):
    fn()   # warm-up: module load, workspace allocation
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {"ms": round(ms, 3), "chain_steps_per_s": units / (ms * 1e-3)}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    torch.cuda.set_device(0)
    priors = {"gaussian": None,
              "uniform": g.Uniform(2, torch.tensor([-3.0, -3.0]), torch.tensor([3.0, 3.0])),
              "gamma": g.Gamma(torch.tensor([2.0, 2.0]), torch.tensor([1.0, 1.0]))}
    lp = g.DiagGaussian(2, torch.zeros(1, 2), torch.log(torch.tensor([0.35, 0.35])))
    gp = g.DiagGaussian(2, torch.zeros(2), torch.zeros(2))
    z = torch.tensor([1.0, 1.0])   # inside every prior's support
    work = {
        "global": (lambda m: g.GlobalMCMC(m, 10000, z, None, gp, None, 0.5, lp, num_chains=65536, seed=1, trace="none"),
                   65536 * 9999, "65,536 chains x 1e4, gf 0.5, statistics only"),
        "glmcmc": (lambda m: g.GLMCMC(m, 10000, z, None, lp, None, 0.9, gp, 5, num_chains=65536, seed=1, trace="none"),
                   65536 * 9999, "65,536 chains x 1e4, gf 0.9, K 5, statistics only"),
        "glmala": (lambda m: g.GLMALA(m, 1001, z, None, 0.3, 100, None, 0.8, gp, 5, num_chains=32768, seed=1, trace="none"),
                   32768 * 1000, "32,768 chains x 1e3, gf 0.8, tau 0.3, num_grad 100"),
        "aglmcmc": (lambda m: g.AGLMCMC(m, 2001, z, None, lp, gp, None, 1.0, 200, 5, 0.8, 0.2, num_chains=16384, seed=1,
                                        trace="none"), 16384 * 2000, "16,384 chains x 2e3, gf 1, K 5, step 200"),
    }
    out = {"info": device_info(), "unit": "chain-steps/s", "results": {}}
    for name, (fn, units, desc) in work.items():
        row = {"workload": desc}
        for pname, prior in priors.items():
            model = g.AbsNormalModel(0.05, y_obs=(1.5, 1.5), noise_var=0.05, prior=prior)
            row[pname] = timed(lambda: fn(model), units, a.reps)
        out["results"][name] = row
    out["info"]["device_after"] = torch.cuda.get_device_name(0)
    text = json.dumps(out)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
