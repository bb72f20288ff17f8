"""The float64 grid specification of the DDM's first-passage law (oracle/ddm_grid_spec.py), on the CPU: mass
conservation, closed forms of pure diffusion, grid convergence, agreement with the C simulator, edge cases."""
import math

import numpy as np
import pytest
from scipy.stats import chi2

from oracle import ddm_grid_spec as g
from oracle import ddm_oracle as orc

S = float(np.float32(math.sqrt(orc.DT_CHOICE)))      # the step's noise scale at mu_sensory = 1
BETA = 0.5826                                         # -zeta(1/2) / sqrt(2 pi): discrete-monitoring bound shift


def _pulses(seed, P=80):
    rng = np.random.default_rng(seed)
    return np.where(rng.random(P) < 0.5, 1.0, -1.0).astype(np.float32)


@pytest.mark.parametrize("theta", [[0.5, 0.0, 0.0, 1.0, 0.3], [0.3, 0.4, 1.0, 3.0, 0.3], [0.7, 2.0, 0.5, 2.0, 7.5],
                                   [0.5, 0.3, 4.0, 1.0, 0.3], [0.2, -1.0, 0.3, 1.2, 0.0]])
def test_total_mass_is_one(theta):
    P, p2 = g.first_passage_law(theta, _pulses(1))
    assert abs(P.sum() + p2 - 1.0) < 1e-12
    assert (P >= 0).all() and p2 >= 0


@pytest.mark.parametrize("a0,B", [(0.5, 1.0), (0.3, 1.5)])
def test_pure_diffusion_closed_forms(a0, B):
    # lam = 0, v = 0: P(upper) = a / B and E[exit] = a (B - a) / sigma^2 (sigma^2 = s^2 / dt = 1) for the
    # continuous process.  The Euler chain is watched only at the steps, which moves both bounds out by
    # BETA * s = O(sqrt dt) (Broadie, Glasserman & Kou 1997); the grid adds O(h).  Bound: that shift on each side
    # plus one cell.
    theta = [a0, 0.0, 0.0, B, 0.0]
    P, p2 = g.first_passage_law(theta, np.ones(80, np.float32))
    r = g.row_scalars(theta)
    a = a0 * B
    k = np.arange(1, P.shape[1] + 1)
    e_exit = float((P.sum(0) * k).sum()) * r["dt"]
    shift = BETA * S
    assert p2 < 1e-6
    assert abs(P[1].sum() - a0) <= shift / B + r["h"] / B
    assert abs(e_exit - a * (B - a)) <= 2 * shift * B + r["h"] * B
    # and the shifted closed form is much closer than the bound
    a_s, B_s = a + shift, B + 2 * shift
    assert abs(e_exit - a_s * (B_s - a_s)) <= 0.1 * shift * B


def test_grid_convergence():
    # Halving h (cells_per_sigma 4 -> 8) moves log P(c, k) by at most 0.021 (median 0.0039 and 0.0002) over the
    # entries with P > 1e-4 at these two rows; the largest changes are on the first steps after a kick, where the
    # density is narrowest.  Bound 0.03.
    for theta in ([0.5, 0.3, 0.8, 1.5, 0.3], [0.4, 1.0, 0.4, 2.5, 0.2]):
        pl = _pulses(0)
        P4, p4 = g.first_passage_law(theta, pl, cells_per_sigma=4)
        P8, p8 = g.first_passage_law(theta, pl, cells_per_sigma=8)
        m = P8 > 1e-4
        d = np.abs(np.log(P4[m]) - np.log(P8[m]))
        assert d.max() < 0.03, d.max()
        assert abs(P4[1].sum() - P8[1].sum()) < 1e-4


@pytest.mark.parametrize("theta", [[0.5, 0.3, 0.8, 1.5, 0.3], [0.4, 1.0, 0.4, 2.5, 0.2], [0.6, 0.0, 0.2, 0.8, 0.5]])
def test_spec_matches_c_simulator(theta):
    # chi^2 on (choice, 50-step bin) counts of 2e5 trials of the C oracle against the law
    n, binw = 200_000, 50
    pl = _pulses(3)
    P, p2 = g.first_passage_law(theta, pl)
    x, steps = orc.sim_rng_c(np.tile(np.float32(theta), (n, 1)), pl, seed=17)
    ch = x[:, 1].astype(int)
    n_max = P.shape[1]
    nb = (n_max + binw - 1) // binw
    obs, exp = [], []
    for c in (0, 1):
        cnt = np.bincount((steps[ch == c] - 1) // binw, minlength=nb)
        pb = np.add.reduceat(P[c], np.arange(0, n_max, binw))
        obs.append(cnt)
        exp.append(pb * n)
    obs.append(np.array([np.sum(ch == 2)]))
    exp.append(np.array([p2 * n]))
    obs, exp = np.concatenate(obs).astype(float), np.concatenate(exp)
    keep = exp >= 5
    rest_o, rest_e = obs[~keep].sum(), exp[~keep].sum()
    o = np.append(obs[keep], rest_o)
    e = np.append(exp[keep], rest_e)
    stat = float(((o - e) ** 2 / np.maximum(e, 1e-300)).sum())
    p = float(chi2.sf(stat, len(o) - 1))
    assert p > 1e-3, (stat, len(o), p)


def test_start_on_a_bound():
    for a0, c in ((0.0, 0), (1.0, 1)):
        P, p2 = g.first_passage_law([a0, 0.0, 0.0, 1.0, 0.3], np.ones(80, np.float32))
        assert abs(P[c, 0] - 0.5) < 1e-12
        assert abs(P.sum() + p2 - 1.0) < 1e-12


def test_windows_of_zero_and_one_step():
    dt = float(np.float32(orc.DT_CHOICE))
    P, p2 = g.first_passage_law([0.5, 0.1, 1.0, 1.0, 8.0], np.ones(80, np.float32))
    assert g.row_scalars([0.5, 0.1, 1.0, 1.0, 8.0])["W"] == 0 and p2 == 1.0 and not P.any()
    theta = [0.5, 0.1, 0.0, 0.05, 8.0 - 1.5 * dt]
    assert g.row_scalars(theta)["W"] == 1
    P, p2 = g.first_passage_law(theta, np.ones(80, np.float32))
    assert not P[:, 1:].any() and abs(P[:, 0].sum() + p2 - 1.0) < 1e-12 and p2 > 0.05
    # observed step outside the window: -inf
    assert g.loglik(theta, [8.0 - 1.5 * dt + 2 * dt, 0.0], np.ones(80, np.float32)) == -math.inf


def test_bound_at_its_clamp_and_kick_beyond_the_bound():
    P, p2 = g.first_passage_law([0.5, 0.2, 0.5, 0.0, 0.3], np.ones(80, np.float32))
    assert g.row_scalars([0.5, 0.2, 0.5, 0.0, 0.3])["M"] == 1
    assert abs(P.sum() + p2 - 1.0) < 1e-12 and P[1, 0] > 0.999   # the first kick (0.5 >> B) sends it up
    P, p2 = g.first_passage_law([0.5, 0.0, 0.0, 1e-6, 0.3], np.ones(80, np.float32))
    assert abs(P[0, 0] - 0.5) < 1e-4 and abs(P[1, 0] - 0.5) < 1e-4
    P, p2 = g.first_passage_law([0.5, 0.1, 3.0, 1.0, 0.3], -np.ones(80, np.float32))
    assert P[0, 0] > 1 - 1e-12


def test_non_unit_pulses_kick_by_gain_times_value():
    pl = _pulses(5) * np.float32(0.5)
    P1, q1 = g.first_passage_law([0.5, 0.3, 0.5, 2.0, 0.3], pl)
    P2, q2 = g.first_passage_law([0.5, 0.3, 0.25, 2.0, 0.3], _pulses(5))
    np.testing.assert_allclose(P1, P2, rtol=1e-12, atol=1e-300)
    # and the pulse value enters: a different train gives a different law
    P3, _ = g.first_passage_law([0.5, 0.3, 0.5, 2.0, 0.3], _pulses(5))
    assert np.abs(P3 - P1).max() > 1e-3


def test_loglik_units():
    theta, pl = [0.5, 0.3, 0.8, 1.5, 0.3], _pulses(0)
    P, p2 = g.first_passage_law(theta, pl)
    r = g.row_scalars(theta)
    k = int(np.argmax(P[0])) + 1
    rt = float(np.float32(np.float32(r["t_nd"]) + np.float32(k) * np.float32(r["dt"])))
    assert abs(g.loglik(theta, [rt, 0.0], pl) - (math.log(P[0, k - 1]) - math.log(r["dt"]))) < 1e-9
    assert abs(g.loglik(theta, [8.0, 2.0], pl) - math.log(p2)) < 1e-9
