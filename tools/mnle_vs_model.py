"""How far is the trained MNLE estimator (tests/golden/mnle_trained.npz) from the model it emulates?  A diagnostic,
not a test.  Sessions of T trials are simulated at prior draws theta_true (fixed pulse trains per trial); for every
trial the estimator's log-likelihood (``DeviceMNLE.log_prob``, precise kernel) is set against the simulator's own
grid log-likelihood (``likelihood.loglik_rows``).  Printed:

* per choice, the per-trial difference ``DeviceMNLE.log_prob - grid log-lik`` as median, mean and worst (choice 2's
  grid value is a probability mass, not a density, so its difference is listed but not comparable);
* the estimator's choice probabilities (frequencies of ``DeviceMNLE.sample``, --draws per condition) against the
  law's P(c) = sum_k P(c, k) and P(2);
* the mean log-likelihood gap per choice-0/1 trial at theta_true, grid minus estimator: with x drawn from the model
  this estimates KL(model || estimator) restricted to decided trials, in nats per trial;
* the card's name and power limit, read in the same run.

    python tools/mnle_vs_model.py [--sessions D] [--trials T] [--draws S] [--out FILE]
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle import ddm_oracle as orc  # noqa: E402
from sbi_for_diffusion_models_b200 import likelihood  # noqa: E402
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE  # noqa: E402
from sbi_for_diffusion_models_b200.pulses import generate_pulse_matrix_device  # noqa: E402
from sbi_for_diffusion_models_b200.run_config import RunConfig  # noqa: E402
from sbi_for_diffusion_models_b200.simulator import simulate_trials  # noqa: E402


def _arg(name, default):
    return int(sys.argv[sys.argv.index(name) + 1]) if name in sys.argv else default


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    D, T, S = _arg("--sessions", 32), _arg("--trials", 50), _arg("--draws", 4096)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    d = np.load(os.path.join(ROOT, "tests", "golden", "mnle_trained.npz"))
    est = DeviceMNLE(PackedMNLE(d["packed"], int(d["n_choices"])))
    K = int(d["n_choices"])
    cfg = RunConfig()
    thetas = orc.prior_sample(D, seed=2026)
    pulses = generate_pulse_matrix_device(np.random.default_rng(77), D * T, 80, p_success=cfg.P_SUCCESS, device=dev)
    theta_rows = thetas.repeat_interleave(T, 0).to(dev)
    x = simulate_trials(theta_rows, pulses, mu_sensory=cfg.MU_SENSORY, seed=4242)
    cond = torch.cat([theta_rows, pulses], 1)
    lp_est = est.log_prob(x, cond, kernel="precise")[0].double().cpu().numpy()
    lp_grid = likelihood.loglik_rows(theta_rows, x, pulses, mu_sensory=cfg.MU_SENSORY).double().cpu().numpy()
    ch = x[:, 1].cpu().numpy().astype(int)
    diff = lp_est - lp_grid
    res = {"card": card(), "sessions": D, "trials": T, "rows": D * T, "per_choice": {}}
    for c in range(3):
        sel = (ch == c) & np.isfinite(diff)
        if not sel.any():
            continue
        dd = diff[sel]
        res["per_choice"][c] = {"n": int(sel.sum()), "median": round(float(np.median(dd)), 4),
                                "mean": round(float(dd.mean()), 4),
                                "worst": round(float(dd[np.argmax(np.abs(dd))]), 4),
                                "non_finite_grid": int(((ch == c) & ~np.isfinite(lp_grid)).sum())}
    dec = (ch < 2) & np.isfinite(diff)
    res["kl_nats_per_decided_trial"] = round(float(-diff[dec].mean()), 4)
    # choice probabilities: the law against the estimator's sampled choices, one condition per theta (first trial)
    first = torch.arange(D, device=dev) * T
    law, surv, _ = likelihood.first_passage_law(theta_rows[first], pulses[first], mu_sensory=cfg.MU_SENSORY)
    p_law = torch.cat([law.double().sum(2), surv.double()[:, None]], 1).cpu().numpy()
    xe = est.sample((S,), condition=cond[first], seed=99).cpu().numpy()
    p_est = np.stack([(xe[:, :, 1] == c).mean(0) for c in range(3)], 1)
    gap = np.abs(p_est[:, :K] - p_law[:, :K])
    res["choice_prob"] = {"draws_per_condition": S, "max_abs_gap": round(float(gap.max()), 4),
                          "mean_abs_gap": round(float(gap.mean()), 4),
                          "rows": [{"theta": [round(float(v), 3) for v in thetas[i]],
                                    "law": p_law[i].round(4).tolist(), "mnle": p_est[i].round(4).tolist()}
                                   for i in range(min(D, 8))]}
    print(json.dumps(res, indent=1), flush=True)
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
