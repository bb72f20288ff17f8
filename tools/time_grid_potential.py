"""The grid potential per call, row kernel against the batched kernel, and one posterior under the grid likelihood.

* configs[3]-shaped calls (T = 50 trials simulated at one prior draw, C = 128 and 1024 chains at prior draws): the
  row path (``ddm_grid_loglik_sum_f32``, one CTA per (trial, chain)) and the batched path
  (``GridLikelihood.loglik_sum_batched``) alternated, timed with CUDA events, their outputs required bit-equal;
* the wall time of ``run_inference_mcmc`` with the grid likelihood at the reference settings (T = 50, 128 chains,
  100 warm-up sweeps, 1000 draws), or with ``--warmup N`` a shorter run whose time per sweep is scaled to them
  (reported as ``reference_measured: false``).

The card's name and power limit are read in the same run.

    python tools/time_grid_potential.py [--reps N] [--warmup N] [--out FILE]
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

from oracle import ddm_oracle as orc  # noqa: E402
from sbi_for_diffusion_models_b200 import _native, likelihood  # noqa: E402
from sbi_for_diffusion_models_b200.simulator import simulate_trials  # noqa: E402

def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def row_path(gl, th, x, pl):
    """The parent's potential: one row-kernel CTA per (trial, chain), then the fixed-order chain sum."""
    L, s = _native.lib(), gl.schedule
    T, C = x.shape[0], th.shape[0]
    out = torch.empty(C, dtype=torch.float32, device=th.device)
    ws = torch.empty(L.ddm_grid_loglik_sum_workspace_floats(T, C), dtype=torch.float32, device=th.device)
    rc = L.ddm_grid_loglik_sum_f32(th.data_ptr(), 5, x.data_ptr(), pl.data_ptr(), pl.shape[1], T, C, pl.shape[1],
                                   s.n_max, s.steps_per_pulse, s.dt, s.t_max, s.t_nd_hi, s.noise_scale,
                                   gl.cells_per_sigma, out.data_ptr(), ws.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "ddm_grid_loglik_sum_f32")
    return out


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=None,
                    help="run the sampler with this many warm-up sweeps and one draw per chain, and scale its wall "
                         "time per sweep to the reference settings (default: run the reference settings)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"card": card()}
    print(json.dumps(res), flush=True)
    rng = np.random.default_rng(5)
    T = 50
    pulses = torch.from_numpy(np.where(rng.random((T, 80)) < 0.5, 1.0, -1.0).astype(np.float32)).to(dev)
    theta_true = orc.prior_sample(1, seed=8).to(dev)
    x = simulate_trials(theta_true.expand(T, 5), pulses, seed=31)
    gl = likelihood.GridLikelihood()
    for C in (128, 1024):
        th = orc.prior_sample(C, seed=C).to(dev)
        new = lambda: gl.loglik_sum_batched(th[None], x[None], pulses[None])[0]
        new()
        torch.cuda.synchronize()
        t_row, t_new, equal = [], [], True
        for _ in range(args.reps if C == 128 else 1):
            s, a = timed(lambda: row_path(gl, th, x, pulses))
            t_row.append(s)
            s, b = timed(new)
            t_new.append(s)
            equal = equal and torch.equal(a.view(torch.int32), b.view(torch.int32))
        r = {"row_s": [round(v, 4) for v in t_row], "batched_s": [round(v, 4) for v in t_new],
             "ratio": round(min(t_row) / min(t_new), 2), "bit_equal": equal}
        res[f"T{T}_C{C}"] = r
        print(json.dumps({f"T{T}_C{C}": r}), flush=True)

    from sbi_for_diffusion_models_b200 import mnle
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    # the reference settings: 100 warm-up sweeps and 1000 draws from 128 chains (8 sweeps)
    sweeps = 100 + -(-1000 // 128)
    warmup = 100 if args.warmup is None else args.warmup
    cfg = RunConfig(WARMUP_STEPS=warmup, POSTERIOR_SAMPLES=1000 if args.warmup is None else 128)
    torch.manual_seed(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    draws = mnle.run_inference_mcmc(cfg, build_prior_theta(dev), gl, x, pulses, num_chains=128,
                                    generator=torch.Generator(device=dev).manual_seed(1))
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ran = warmup + -(-cfg.POSTERIOR_SAMPLES // 128)
    # wall_s includes the search for starting points, so the scaled figure overstates a long run
    mc = {"sweeps_run": ran, "wall_s": round(wall, 2), "reference_sweeps": sweeps,
          "scaled_to_reference_s": round(wall / ran * sweeps, 1), "reference_measured": args.warmup is None,
          "posterior_mean": [round(float(v), 4) for v in draws.mean(0)],
          "theta_true": [round(float(v), 4) for v in theta_true[0]]}
    res["run_inference_mcmc_T50_C128"] = mc
    print(json.dumps(res, indent=1), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
