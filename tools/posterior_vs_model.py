"""Does the MNLE estimator's gap to the model's own likelihood move the posterior?

A few sessions are simulated at prior draws (configs[3] shape: T = 50 trials, one pulse train per trial).  Each is
sampled twice with ``run_inference_mcmc`` from the same starting points and the same uniforms: once under the trained
estimator (``tests/golden/mnle_trained.npz``) and once under the grid likelihood (``GridLikelihood``, the simulator's
exact first-passage law).  Per coordinate it prints the difference of the posterior means in units of the grid
posterior's sd, the ratio of the posterior sds (estimator / grid), the two-sample KS statistic on the chains' last
draws, and theta_true's rank (fraction of draws below it) under each posterior.  The card's name and power limit are
read in the same run.

    python tools/posterior_vs_model.py [--sessions N] [--warmup N] [--samples N] [--chains N] [--out FILE]

The defaults are the reference settings (100 warm-up sweeps, 1000 draws, 128 chains).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from scipy.stats import ks_2samp  # noqa: E402

from sbi_for_diffusion_models_b200 import mnle  # noqa: E402
from sbi_for_diffusion_models_b200.likelihood import GridLikelihood  # noqa: E402
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE  # noqa: E402
from sbi_for_diffusion_models_b200.priors import build_prior_theta  # noqa: E402
from sbi_for_diffusion_models_b200.pulses import generate_pulse_matrix_device  # noqa: E402
from sbi_for_diffusion_models_b200.run_config import RunConfig  # noqa: E402
from sbi_for_diffusion_models_b200.simulator import simulate_trials  # noqa: E402

NAMES = ("a0", "lam", "v", "B", "tau")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sessions", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--chains", type=int, default=128)
    ap.add_argument("--trials", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    d = np.load(os.path.join(ROOT, "tests", "golden", "mnle_trained.npz"))
    est = DeviceMNLE(PackedMNLE(d["packed"], int(d["n_choices"])))
    grid = GridLikelihood()
    prior = build_prior_theta(dev)
    cfg = RunConfig(WARMUP_STEPS=args.warmup, POSTERIOR_SAMPLES=args.samples)
    res = {"card": card(), "settings": vars(args), "sessions": []}
    print(json.dumps({"card": res["card"]}), flush=True)
    torch.manual_seed(2026)
    rng = np.random.default_rng(11)
    for i in range(args.sessions):
        theta_true = prior.sample((1,)).to(dev, torch.float32)
        pulses = generate_pulse_matrix_device(rng, args.trials, 80, p_success=0.75).to(dev, torch.float32)
        x = simulate_trials(theta_true.expand(args.trials, 5).contiguous(), pulses, seed=1000 + i)
        draws, secs = {}, {}
        for name, lik in (("mnle", est), ("grid", grid)):
            torch.manual_seed(77 + i)                          # the same starting points
            t0 = time.perf_counter()
            draws[name] = mnle.run_inference_mcmc(cfg, prior, lik, x, pulses, num_chains=args.chains,
                                                  generator=torch.Generator(device=dev).manual_seed(5 + i)).double()
            secs[name] = round(time.perf_counter() - t0, 1)
        # run_inference_mcmc returns the first POSTERIOR_SAMPLES of the (draw, chain)-ordered draws: chain c's last
        # kept draw is row c + chains * ((samples - 1 - c) // chains)
        rows = [c + args.chains * ((args.samples - 1 - c) // args.chains) for c in range(min(args.chains, args.samples))]
        last = {k: v[rows] for k, v in draws.items()}
        tt = theta_true[0].double().cpu()
        row = {"theta_true": [round(float(v), 4) for v in tt], "seconds": secs, "coords": {}}
        for j, nm in enumerate(NAMES):
            m, g = draws["mnle"][:, j], draws["grid"][:, j]
            row["coords"][nm] = {
                "mean_diff_in_grid_sd": round(float((m.mean() - g.mean()) / g.std()), 3),
                "sd_ratio_mnle_over_grid": round(float(m.std() / g.std()), 3),
                "ks_last_draws": round(float(ks_2samp(last["mnle"][:, j].numpy(), last["grid"][:, j].numpy()).statistic), 3),
                "rank_mnle": round(float((m < tt[j]).double().mean()), 3),
                "rank_grid": round(float((g < tt[j]).double().mean()), 3),
            }
        res["sessions"].append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
