"""How well does the trained estimator (tests/golden/mnle_trained.npz) emulate the simulator?  A diagnostic, not a
test: for the test session's theta and four prior draws, N trials (default 2e5) with the same fixed pulse trains are
drawn from the estimator (``DeviceMNLE.sample``) and from the simulator; printed per theta: the choice fractions, the
chi^2 of the 2 x K table of choice counts, and per choice the two-sample KS statistic and p-value of rt.

    python tools/mnle_emulator_check.py [--n N] [--out FILE]
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from scipy import stats  # noqa: E402

from oracle import ddm_oracle as orc  # noqa: E402
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE  # noqa: E402
from sbi_for_diffusion_models_b200.pulses import generate_pulse_matrix_device  # noqa: E402
from sbi_for_diffusion_models_b200.run_config import RunConfig  # noqa: E402
from sbi_for_diffusion_models_b200.simulator import simulate_trials  # noqa: E402


def main():
    N = int(sys.argv[sys.argv.index("--n") + 1]) if "--n" in sys.argv else 200_000
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    d = np.load(os.path.join(ROOT, "tests", "golden", "mnle_trained.npz"))
    est = DeviceMNLE(PackedMNLE(d["packed"], int(d["n_choices"])))
    K = int(d["n_choices"])
    cfg = RunConfig()
    pulses = generate_pulse_matrix_device(np.random.default_rng(123), N, 80, p_success=cfg.P_SUCCESS, device=dev)
    thetas = torch.cat([torch.tensor([[0.45, 0.6, 1.3, 14.0, 0.25]]), orc.prior_sample(4, seed=11)])
    out = []
    for i, th in enumerate(thetas):
        theta = th[None, :].expand(N, 5).to(dev)
        xs = simulate_trials(theta, pulses, mu_sensory=cfg.MU_SENSORY, seed=100 + i).cpu().numpy()
        xe = est.sample((), condition=torch.cat([theta, pulses], 1), seed=200 + i).cpu().numpy()
        cs = np.bincount(xs[:, 1].astype(int), minlength=K)
        ce = np.bincount(xe[:, 1].astype(int), minlength=K)
        table = np.stack([cs, ce])
        table = table[:, table.sum(0) > 0]
        chi2, pv, dof, _ = stats.chi2_contingency(table)
        row = {"theta": [round(float(v), 4) for v in th], "n": N, "choice_frac_sim": (cs / N).round(4).tolist(),
               "choice_frac_mnle": (ce / N).round(4).tolist(), "chi2": round(float(chi2), 2), "chi2_dof": int(dof),
               "chi2_p": float(f"{pv:.3g}"), "ks": {}}
        for c in range(K):
            a, b = xs[xs[:, 1] == c, 0], xe[xe[:, 1] == c, 0]
            if a.size < 20 or b.size < 20:
                continue
            r = stats.ks_2samp(a, b)
            row["ks"][c] = {"D": round(float(r.statistic), 4), "p": float(f"{r.pvalue:.3g}"),
                            "median_rt_sim": round(float(np.median(a)), 4), "median_rt_mnle": round(float(np.median(b)), 4),
                            "rt_max_sim": round(float(a.max()), 4), "rt_max_mnle": round(float(b.max()), 4)}
        print(json.dumps(row), flush=True)
        out.append(row)
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
