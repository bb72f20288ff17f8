"""Float64 specification of the pulse DDM's first-passage law by density propagation --
TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The simulator (``ddm_oracle.sim_lockstep_torch``) is a Markov chain

    a <- a - lam a dt + s xi          (xi ~ N(0,1), s = mu_sensory sqrt(dt))
    a <- a + gain pulse[k / spp]      on steps k with k % spp == 0
    a >= B absorbs as choice 1, a <= 0 as choice 0, at step k + 1,

started at a0 = clamp(theta0, 0, 1) B and run for at most W steps.  Its law is computed
here by propagating the accumulator's density on a grid; ``csrc/ddm_grid.cu`` is held to
this module row by row.

Discretisation (what the kernel implements in fp32):

* Cells.  (0, B) is cut into M = clamp(ceil(B q / s), 1, max_cells) cells of width
  h = B / M, q = ``cells_per_sigma`` (default 4: h <= s / 4).  The bounds sit on cell
  edges.  Rows with B q / s > max_cells get coarser cells; ``grid_h_over_s`` says which
  h / s a row used.
* Representation.  The mass of cell j sits at its centre c_j = (j + 1/2) h.  The first
  step starts from the exact point a0 instead (a0 = 0 and a0 = B are allowed: half the
  mass is absorbed on step 1).
* One Euler step.  The mass at c sends to cell i the integral over cell i of the
  Gaussian with mean c (1 - lam dt) + kick and standard deviation sigma_eff, truncated at
  +-R sigma_eff (R = ``SIGMAS``) and renormalised; the tail masses beyond 0 and B are the
  step's absorptions.  Every (source, cell) weight is a difference of the truncated CDF at
  the two cell edges, taken between the two smaller tails so that no weight is the
  difference of two numbers close to 1.
* Variance.  Moving each cell's mass to its centre adds h^2 / 12 of variance per step on
  average (Sheppard's correction), which would compound over thousands of steps into a
  drift of the RT law's time scale by h^2 / (12 s^2) (0.5 % at q = 4).  The step's
  Gaussian therefore has sigma_eff^2 = s^2 - h^2 / 12 (at least s^2 / 4), so that step
  plus re-projection keeps the Euler step's variance.  What error remains is measured,
  not assumed: see ``tests/test_ddm_grid_spec.py`` and DESIGN section 4b.

Outputs per row: P(c, k) for c in {0, 1} and k = 1..W, and P(2) = the mass that survives
W steps.  Log-likelihood of an observed (rt seconds, choice):
    choice 0 / 1: log P(c, k) - log dt with k = round((rt - t_nd) / dt), -inf unless
                  1 <= k <= W -- a density in rt seconds, piecewise constant over a step,
                  in the unit DeviceMNLE.log_prob uses;
    choice 2:     log P(2) -- a probability MASS, not comparable with the estimator's
                  density for choice 2.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import numpy as np
import scipy.sparse as sp
from scipy.special import ndtr

from .ddm_oracle import DT_CHOICE, PULSE_INTERVAL, T_MAX, fp32_scalars, schedule

CELLS_PER_SIGMA = 4.0
MAX_CELLS = 8192
SIGMAS = 6.0                      # Gaussian truncation, in sigma_eff
TAIL_R = float(ndtr(-SIGMAS))     # mass beyond one truncation point


def _f32(v) -> np.float32:
    return np.float32(v)


def row_scalars(theta, *, dt: float = DT_CHOICE, t_max: float = T_MAX, mu_sensory: float = 1.0,
                cells_per_sigma: float = CELLS_PER_SIGMA, max_cells: int = MAX_CELLS, n_max: Optional[int] = None):
    """The per-row quantities of the scheme, from the fp32 theta the simulator sees."""
    th = np.asarray(theta, dtype=np.float32).reshape(5)
    sc = fp32_scalars(dt, t_max, mu_sensory)
    if n_max is None:
        n_max = int(np.floor(float(t_max) / float(dt)))
    a0f = np.float32(min(max(float(th[0]), 0.0), 1.0))
    lam = float(th[1])
    gain = float(abs(th[2]))
    B = float(max(np.float32(abs(th[3])), np.float32(1e-6)))
    t_nd = np.float32(min(max(float(th[4]), 0.0), sc["t_nd_hi"]))
    win = np.floor(np.float32(np.float32(sc["t_max"]) - t_nd) / np.float32(sc["dt"]))   # fp32, as the simulator
    W = int(min(max(win, 0), n_max))
    s = float(sc["noise_scale"])
    M = int(min(max(math.ceil(B * float(cells_per_sigma) / s), 1), int(max_cells)))
    h = B / M
    sig = math.sqrt(max(s * s - h * h / 12.0, 0.25 * s * s))
    return dict(a0=float(a0f) * B, lam=lam, gain=gain, B=B, t_nd=float(t_nd), W=W, M=M, h=h, s=s, sigma=sig,
                decay=1.0 - lam * float(sc["dt"]), dt=float(sc["dt"]))


def grid_h_over_s(theta, **kw) -> float:
    r = row_scalars(theta, **kw)
    return r["h"] / r["s"]


def _tail(x: np.ndarray) -> np.ndarray:
    """Truncated, renormalised N(0,1) mass below -|x| (the smaller tail at x)."""
    t = (ndtr(-np.abs(x)) - TAIL_R) / (1.0 - 2.0 * TAIL_R)
    return np.maximum(t, 0.0)


def _cell_mass(xa: np.ndarray, xb: np.ndarray) -> np.ndarray:
    """Truncated-normal mass of (xa, xb), xa < xb, from the two smaller tails."""
    ta, tb = _tail(xa), _tail(xb)
    return np.where(xb <= 0.0, tb - ta, np.where(xa >= 0.0, ta - tb, 1.0 - ta - tb))


def _lower_mass(x: np.ndarray) -> np.ndarray:
    t = _tail(x)
    return np.where(x <= 0.0, t, 1.0 - t)


def step_operator(mu: np.ndarray, r: dict):
    """(W (M, n_src) sparse, bottom (n_src,), top (n_src,)) for point sources at positions mu (absolute units)."""
    M, h, sig = r["M"], r["h"], r["sigma"]
    reach = int(math.ceil(SIGMAS * sig / h)) + 2
    centre = np.floor(mu / h).astype(np.int64)
    rows, cols, vals = [], [], []
    for d in range(max(-reach, -int(centre.max())), min(reach, M - 1 - int(centre.min())) + 1):
        i = centre + d
        ok = (i >= 0) & (i < M)
        if not ok.any():
            continue
        src = np.nonzero(ok)[0]
        ii = i[ok]
        xa = (ii * h - mu[ok]) / sig
        xb = ((ii + 1) * h - mu[ok]) / sig
        rows.append(ii)
        cols.append(src)
        vals.append(_cell_mass(xa, xb))
    if rows:
        Wm = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(M, mu.size))
    else:
        Wm = sp.csr_matrix((M, mu.size))
    bottom = _lower_mass((0.0 - mu) / sig)
    top = _lower_mass((mu - r["B"]) / sig)
    return Wm, bottom, top


def first_passage_law(theta, pulses, *, dt: float = DT_CHOICE, t_max: float = T_MAX,
                      pulse_interval: float = PULSE_INTERVAL, mu_sensory: float = 1.0,
                      cells_per_sigma: float = CELLS_PER_SIGMA, max_cells: int = MAX_CELLS,
                      n_steps: Optional[int] = None) -> Tuple[np.ndarray, float]:
    """(P (2, n_max) float64 with P[c, k - 1] = P(choice c at step k), P(2)) for one row.

    ``n_steps`` stops the propagation early (entries past it stay 0 and P(2) is then the
    mass still inside after n_steps)."""
    n_max, spp, n_p = schedule(dt, t_max, pulse_interval)
    r = row_scalars(theta, dt=dt, t_max=t_max, mu_sensory=mu_sensory, cells_per_sigma=cells_per_sigma,
                    max_cells=max_cells, n_max=n_max)
    pl = np.asarray(pulses, dtype=np.float32).reshape(-1)
    if pl.size < n_p:
        raise ValueError(f"pulses must hold at least {n_p} values, got {pl.size}")
    W = r["W"] if n_steps is None else min(r["W"], int(n_steps))
    P = np.zeros((2, n_max), dtype=np.float64)
    if W == 0:
        return P, 1.0
    M, h = r["M"], r["h"]
    centres = (np.arange(M) + 0.5) * h
    W0 = None
    m = None
    for k in range(W):
        kick = r["gain"] * float(pl[k // spp]) if k % spp == 0 else 0.0
        if k == 0:
            Wk, bot, top = step_operator(np.array([r["a0"] * r["decay"] + kick]), r)
            P[0, 0], P[1, 0] = bot[0], top[0]
            m = Wk.toarray()[:, 0]
            continue
        if kick != 0.0:
            Wk, bot, top = step_operator(centres * r["decay"] + kick, r)
        else:
            if W0 is None:
                W0 = step_operator(centres * r["decay"], r)
            Wk, bot, top = W0
        P[0, k], P[1, k] = float(bot @ m), float(top @ m)
        m = Wk @ m
    return P, float(m.sum())


def observed_step(theta, rt: float, *, dt: float = DT_CHOICE, t_max: float = T_MAX) -> int:
    r = row_scalars(theta, dt=dt, t_max=t_max)
    return int(np.rint((float(np.float32(rt)) - r["t_nd"]) / r["dt"]))


def loglik(theta, x, pulses, *, dt: float = DT_CHOICE, t_max: float = T_MAX,
           pulse_interval: float = PULSE_INTERVAL, mu_sensory: float = 1.0,
           cells_per_sigma: float = CELLS_PER_SIGMA, max_cells: int = MAX_CELLS) -> float:
    """log-likelihood of x = (rt seconds, choice) under the grid law (see the module docstring)."""
    rt, c = float(np.float32(x[0])), int(x[1])
    kw = dict(dt=dt, t_max=t_max, pulse_interval=pulse_interval, mu_sensory=mu_sensory,
              cells_per_sigma=cells_per_sigma, max_cells=max_cells)
    r = row_scalars(theta, dt=dt, t_max=t_max, mu_sensory=mu_sensory, cells_per_sigma=cells_per_sigma,
                    max_cells=max_cells)
    if c == 2:
        _, p2 = first_passage_law(theta, pulses, **kw)
        return math.log(p2) if p2 > 0 else -math.inf
    k = observed_step(theta, rt, dt=dt, t_max=t_max)
    if k < 1 or k > r["W"]:
        return -math.inf
    P, _ = first_passage_law(theta, pulses, n_steps=k, **kw)
    p = P[c, k - 1]
    return math.log(p) - math.log(r["dt"]) if p > 0 else -math.inf
