"""Rows per second of the grid likelihood kernels, in steady state with CUDA events, against the float64 CPU spec.

Sessions shaped like configs[3] (T = 50 trials, C = 128 and 1024 chains at prior draws, trials simulated at one
prior draw) through ``GridLikelihood.loglik_sum``, and the full law (``first_passage_law``, W steps per row) of
prior draws.  The card's name and power limit are read in the same run.

    python tools/time_grid_likelihood.py [--out FILE]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle import ddm_grid_spec as spec  # noqa: E402
from oracle import ddm_oracle as orc  # noqa: E402
from sbi_for_diffusion_models_b200 import likelihood  # noqa: E402
from sbi_for_diffusion_models_b200.simulator import simulate_trials  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def main():
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"card": card()}
    rng = np.random.default_rng(5)
    T = 50
    pulses = torch.from_numpy(np.where(rng.random((T, 80)) < 0.5, 1.0, -1.0).astype(np.float32)).to(dev)
    theta_true = orc.prior_sample(1, seed=8).to(dev)
    x = simulate_trials(theta_true.expand(T, 5), pulses, seed=31)
    gl = likelihood.GridLikelihood()
    for C in (128, 1024):
        th = orc.prior_sample(C, seed=C).to(dev)
        s = timed(lambda: gl.loglik_sum(th, x, pulses), 3 if C == 128 else 1)
        res[f"loglik_sum_T{T}_C{C}"] = {"seconds": round(s, 4), "rows_per_s": round(T * C / s, 1)}
        print(json.dumps({f"T{T}_C{C}": res[f"loglik_sum_T{T}_C{C}"]}), flush=True)
    N = 1024
    th = orc.prior_sample(N, seed=3).to(dev)
    pl = torch.from_numpy(np.where(rng.random((N, 80)) < 0.5, 1.0, -1.0).astype(np.float32)).to(dev)
    s = timed(lambda: likelihood.first_passage_law(th, pl), 1)
    res["law_prior_N1024"] = {"seconds": round(s, 4), "rows_per_s": round(N / s, 1)}
    print(json.dumps({"law": res["law_prior_N1024"]}), flush=True)
    # the float64 CPU spec on a few of the same session rows
    thc, xc, pc = th[:4].cpu().numpy(), x.cpu().numpy(), pulses.cpu().numpy()
    t0 = time.perf_counter()
    for i in range(4):
        spec.loglik(thc[i], xc[i], pc[i])
    cpu = (time.perf_counter() - t0) / 4
    res["cpu_spec_loglik_row_seconds"] = round(cpu, 3)
    res["cpu_spec_rows_per_s"] = round(1.0 / cpu, 3)
    print(json.dumps(res, indent=1), flush=True)
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
