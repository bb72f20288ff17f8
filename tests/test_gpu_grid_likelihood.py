"""The grid likelihood kernels (csrc/ddm_grid.cu) against the float64 spec (oracle/ddm_grid_spec.py) row by row,
their batch invariance and chain sum, the law against 2e6 trials of the native simulator per theta (with the
power to reject a 2 % gain or 1 % bound change), and the host's refusals."""
import math

import numpy as np
import pytest
import torch
from scipy.stats import chi2

from oracle import ddm_grid_spec as g
from oracle import ddm_oracle as orc

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24


def _lik():
    from sbi_for_diffusion_models_b200 import likelihood
    return likelihood


def _pulses(seed, n=1, P=80):
    rng = np.random.default_rng(seed)
    return np.where(rng.random((n, P)) < 0.5, 1.0, -1.0).astype(np.float32)


def _rtol(k):
    # fp32 rounding: each step rounds every mass a few times and erfcf is good to a few ulp; those errors add like
    # a random walk over the steps.  On top, one step's fp32 weights sum to 1 only within rounding, so the mass that
    # stays inside drifts by a fraction of an ulp per step (measured: 6e-4 on a survival mass after 14617 steps,
    # 0.7 ulp per step); 2 ulp per step bounds it.
    k = np.asarray(k, dtype=np.float64)
    return 64.0 * U32 * np.sqrt(k + 1.0) + 2.0 * U32 * k


ROWS = np.array([
    *orc.prior_sample(4, seed=11).numpy().tolist(),
    [0.0, 0.3, 0.5, 2.0, 0.3],          # start on the lower bound
    [1.0, 0.3, 0.5, 2.0, 0.3],          # start on the upper bound
    [0.5, 0.2, 0.5, 0.0, 0.3],          # B at its 1e-6 clamp, kick larger than B
    [0.5, 0.0, 3.0, 1.0, 0.3],          # kick larger than B
    [0.5, 0.3, 0.4, 1.5, 7.9999],       # W = 0
    [0.5, 0.3, 0.4, 1.5, 8.0 - 0.0007], # W = 1
    [0.4, 7.0, 0.5, 3.0, 0.0],          # strong leak, W = 16000
    [0.5, 0.1, 0.3, 60.0, 4.0],         # B above the cap: coarser cells
    [0.5, -0.5, 0.2, 1.0, 0.0],         # negative leak
], dtype=np.float32)


def test_law_matches_float64_spec_row_by_row():
    lik = _lik()
    pl = _pulses(7, len(ROWS))
    pl[4] *= np.float32(0.37)            # a row of non-+-1 pulse values
    law, surv, hs = lik.first_passage_law(torch.from_numpy(ROWS), torch.from_numpy(pl))
    law, surv, hs = law.cpu().numpy().astype(np.float64), surv.cpu().numpy(), hs.cpu().numpy()
    worst = 0.0
    for r, th in enumerate(ROWS):
        P, p2 = g.first_passage_law(th, pl[r])
        assert abs(hs[r] - g.grid_h_over_s(th)) <= 1e-6 * g.grid_h_over_s(th)
        m = P > 1e-6
        k = np.nonzero(m)[1] + 1
        rel = np.abs(law[r][m] - P[m]) / P[m]
        worst = max(worst, float((rel / _rtol(k)).max(initial=0.0)))
        assert (rel <= _rtol(k)).all(), (r, th, float(rel.max()))
        assert (law[r][~m] <= 2e-6).all()
        if p2 > 1e-6:
            assert abs(surv[r] - p2) <= _rtol(g.row_scalars(th)["W"]) * p2
        else:
            assert surv[r] <= 2e-6
    assert hs[-2] > 0.25 and hs[0] <= 0.25
    print(f"worst |law - spec| / tolerance: {worst:.3f}")


def test_loglik_matches_float64_spec_row_by_row():
    lik = _lik()
    theta = orc.prior_sample(16, seed=3)
    pl = _pulses(9, 16)
    x = orc.sim_rng_c(theta.numpy(), pl, seed=5)[0]
    x[-1] = [8.0, 2.0]
    x[-2] = [float(theta[-2, 4]) - 0.01, 0.0]          # before t_nd: -inf
    got = lik.loglik_rows(theta, torch.from_numpy(x), torch.from_numpy(pl)).cpu().numpy().astype(np.float64)
    for r in range(16):
        want = g.loglik(theta[r].numpy(), x[r], pl[r])
        if not math.isfinite(want):
            assert got[r] == want
            continue
        k = g.observed_step(theta[r].numpy(), x[r, 0])
        assert abs(got[r] - want) <= _rtol(k) + 2e-6, (r, got[r], want)


def test_rows_are_batch_invariant_and_chain_sum_is_the_fixed_order_row_sum():
    lik = _lik()
    C, T = 12, 5
    theta = orc.prior_sample(C, seed=21)
    theta[:, 3] = theta[:, 3].clamp(max=8.0)          # keep the rows short
    pl = _pulses(4, T)
    x = torch.from_numpy(orc.sim_rng_c(theta[:T].numpy(), pl, seed=9)[0])
    rows_th = theta.repeat(T, 1)                       # row r = t * C + c
    rows_x = x.repeat_interleave(C, 0)
    rows_pl = torch.from_numpy(pl).repeat_interleave(C, 0)
    full = lik.loglik_rows(rows_th, rows_x, rows_pl).cpu()
    perm = torch.randperm(T * C, generator=torch.Generator().manual_seed(0))
    shuffled = lik.loglik_rows(rows_th[perm], rows_x[perm], rows_pl[perm]).cpu()
    assert torch.equal(shuffled, full[perm])
    half = T * C // 2
    parts = torch.cat([lik.loglik_rows(rows_th[:half], rows_x[:half], rows_pl[:half]).cpu(),
                       lik.loglik_rows(rows_th[half:], rows_x[half:], rows_pl[half:]).cpu()])
    assert torch.equal(parts, full)
    law_a = lik.first_passage_law(theta[:4], torch.from_numpy(_pulses(1, 4)))[0]
    law_b = lik.first_passage_law(theta[2:3], torch.from_numpy(_pulses(1, 4)[2:3]))[0]
    assert torch.equal(law_a[2], law_b[0])
    got = lik.GridLikelihood().loglik_sum(theta, x, torch.from_numpy(pl))
    want = full.double().view(T, C)
    acc = torch.zeros(C, dtype=torch.float64)
    for t in range(T):
        acc = acc + want[t]
    assert torch.equal(got.cpu(), acc.float())


# eight theta: strong leak, large gain, small and large B, late t_nd; one fixed pulse train each
MC_THETA = np.array([
    [0.5, 0.37, 1.0, 2.0, 0.3],
    [0.4, 5.0, 0.6, 2.0, 0.3],         # strong leak
    [0.5, 0.3, 1.5, 6.0, 0.2],         # large gain
    [0.6, 0.2, 0.3, 0.6, 0.1],         # small B
    [0.5, 0.3, 1.5, 12.0, 0.3],        # large B
    [0.5, 0.3, 0.5, 1.5, 6.5],         # late t_nd: a short window, censored trials
    [0.3, 1.0, 0.8, 4.0, 0.5],
    [0.7, 0.0, 0.4, 1.2, 0.0],
], dtype=np.float32)
MC_N, MC_BIN = 2_000_000, 50


def _chi2_p(law, surv, steps, ch):
    law, surv = law.cpu().numpy().astype(np.float64), float(surv)
    n_max = law.shape[1]
    nb = (n_max + MC_BIN - 1) // MC_BIN
    obs, exp = [], []
    for c in (0, 1):
        sel = steps[ch == c]
        obs.append(np.bincount((sel - 1) // MC_BIN, minlength=nb))
        exp.append(np.add.reduceat(law[c], np.arange(0, n_max, MC_BIN)) * MC_N)
    obs.append(np.array([np.sum(ch == 2)]))
    exp.append(np.array([surv * MC_N]))
    o, e = np.concatenate(obs).astype(np.float64), np.concatenate(exp)
    keep = e >= 5
    o = np.append(o[keep], o[~keep].sum())
    e = np.append(e[keep], max(e[~keep].sum(), 1e-9))
    e *= o.sum() / e.sum()       # the kernel's fp32 mass sums to 1 within rounding
    stat = float(((o - e) ** 2 / e).sum())
    return float(chi2.sf(stat, len(o) - 1))


def test_law_matches_native_simulator_and_rejects_perturbed_laws():
    lik = _lik()
    from sbi_for_diffusion_models_b200 import simulator as sim
    alpha = 1e-3 / len(MC_THETA)
    report = []
    for i, th in enumerate(MC_THETA):
        pl = _pulses(100 + i)
        theta = torch.from_numpy(np.tile(th, (MC_N, 1))).cuda()
        x, steps = sim.simulate_trials(theta, torch.from_numpy(pl).cuda(), seed=1234 + i, return_steps=True)
        steps = steps.cpu().numpy().astype(np.int64)
        ch = x[:, 1].cpu().numpy().astype(np.int64)
        variants = np.stack([th, th * np.float32([1, 1, 1.02, 1, 1]), th * np.float32([1, 1, 1, 1.01, 1])])
        law, surv, _ = lik.first_passage_law(torch.from_numpy(variants), torch.from_numpy(np.tile(pl, (3, 1))))
        p = [_chi2_p(law[v], surv[v], steps, ch) for v in range(3)]
        report.append(p)
    print("chi2 p-values (law, gain x 1.02, B x 1.01):", [[f"{v:.2e}" for v in r] for r in report])
    for th, p in zip(MC_THETA, report):
        assert p[0] > alpha, (th, p)
        assert p[1] < alpha and p[2] < alpha, (th, p)


@pytest.mark.parametrize("bad", ["theta_shape", "theta_nan", "x_shape", "x_choice", "pulses_short", "leak"])
def test_refusals_on_the_host(bad):
    lik = _lik()
    theta = torch.tensor([[0.5, 0.3, 0.5, 2.0, 0.3]])
    x = torch.tensor([[0.8, 1.0]])
    pl = torch.ones(1, 80)
    if bad == "theta_shape":
        theta = torch.ones(1, 4)
    elif bad == "theta_nan":
        theta[0, 3] = float("nan")
    elif bad == "x_shape":
        x = torch.ones(2, 2)
    elif bad == "x_choice":
        x[0, 1] = 3.0
    elif bad == "pulses_short":
        pl = torch.ones(1, 79)
    elif bad == "leak":
        theta[0, 1] = 5000.0
    with pytest.raises(ValueError):
        lik.loglik_rows(theta, x, pl)
    if bad not in ("x_shape", "x_choice"):
        with pytest.raises(ValueError):
            lik.first_passage_law(theta, pl)
