"""CPU specification of the MNLE density estimator's ``sample`` -- TEST INFRASTRUCTURE.

sbi's ``MixedDensityEstimator.sample`` draws the choice from the categorical net and then log rt from the conditional
spline flow given that choice, running the ten rational-quadratic splines in inverse.  This module restates that on
top of ``mnle_spec`` (same parameter names, same spline construction), from caller-given draws, in the dtype of the
parameters: with the float64 parameters it is the row-by-row oracle of ``mnle_sample_tc_f32`` under injected draws.

The inverse spline (``rqs_inverse``) is pinned against the nflows-derived VITS spline shipped in ``transformers``
(``reverse=True``, ``tests/test_mnle_sample_spec.py``).  The wiring around it -- choice first, then the flow given the
choice -- is unpinned, like the rest of ``mnle_spec`` (sbi is not installable where this package is built).
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

from .mnle_spec import HIDDEN, MIN_BIN, MIN_DERIV, NUM_BINS, NUM_TRANSFORMS, TAIL_BOUND, rqs_forward


def rqs_inverse(y: torch.Tensor, q: torch.Tensor):
    """Inverse of ``rqs_forward``: y (R,), q (R, 3K-1) -> (u (R,), logabsdet (R,)) with rqs_forward(u, q)[0] == y and
    logabsdet = -(the forward log-det at u).  Identity outside the tail bound; inside, the bin is located on the HEIGHT
    knots and the rational quadratic is solved for the position in the bin (nflows ``rational_quadratic_spline(...,
    inverse=True)``: root = 2c / (-b - sqrt(b^2 - 4ac)))."""
    K = NUM_BINS
    uw = q[:, :K] / math.sqrt(HIDDEN)
    uh = q[:, K:2 * K] / math.sqrt(HIDDEN)
    ud = q[:, 2 * K:]
    const = math.log(math.exp(1.0 - MIN_DERIV) - 1.0)
    ud = F.pad(ud, (1, 1), value=const)

    inside = (y >= -TAIL_BOUND) & (y <= TAIL_BOUND)
    yi = torch.where(inside, y, torch.zeros_like(y))

    def knots(unnorm):
        w = MIN_BIN + (1.0 - MIN_BIN * K) * torch.softmax(unnorm, dim=-1)
        cw = torch.cumsum(w, dim=-1)
        cw = F.pad(cw, (1, 0), value=0.0)
        cw = 2.0 * TAIL_BOUND * cw - TAIL_BOUND
        cw[:, 0] = -TAIL_BOUND
        cw[:, -1] = TAIL_BOUND
        return cw, cw[:, 1:] - cw[:, :-1]

    cw, w = knots(uw)
    ch, h = knots(uh)
    d = MIN_DERIV + F.softplus(ud)

    edges = ch.clone()
    edges[:, -1] += 1e-6
    b = (yi[:, None] >= edges).sum(dim=-1) - 1
    b = b.clamp(0, K - 1)[:, None]
    in_cw, in_w = cw.gather(1, b)[:, 0], w.gather(1, b)[:, 0]
    in_ch, in_h = ch.gather(1, b)[:, 0], h.gather(1, b)[:, 0]
    delta = in_h / in_w
    d0, d1 = d.gather(1, b)[:, 0], d.gather(1, b + 1)[:, 0]

    i1 = d0 + d1 - 2.0 * delta
    i2 = yi - in_ch
    i3 = i2 * i1
    a = in_h * (delta - d0) + i3
    bq = in_h * d0 - i3
    c = -delta * i2
    disc = (bq * bq - 4.0 * a * c).clamp_min(0.0)
    th = (2.0 * c) / (-bq - torch.sqrt(disc))
    out = th * in_w + in_cw
    t1 = th * (1.0 - th)
    den = delta + i1 * t1
    dnum = delta * delta * (d1 * th * th + 2.0 * delta * t1 + d0 * (1.0 - th) * (1.0 - th))
    lad = -(torch.log(dnum) - 2.0 * torch.log(den))
    return torch.where(inside, out, y), torch.where(inside, lad, torch.zeros_like(lad))


def choice_logits(p: Dict[str, torch.Tensor], cond: torch.Tensor) -> torch.Tensor:
    """cond (R,85) -> the categorical net's logits (R,K), in the dtype of the parameters."""
    dt = p["cat.W0"].dtype
    zt = (cond.to(dt) - p["cond_mean"]) / p["cond_std"]
    h = torch.sigmoid(zt @ p["cat.W0"].T + p["cat.b0"])
    h = torch.sigmoid(h @ p["cat.W1"].T + p["cat.b1"])
    h = torch.sigmoid(h @ p["cat.W2"].T + p["cat.b2"])
    return h @ p["cat.Wo"].T + p["cat.bo"]


def choice_from_uniform(logits: torch.Tensor, u_choice: torch.Tensor) -> torch.Tensor:
    """The smallest j with u < sum_{i<=j} softmax(logits)_i, in float64; K - 1 when rounding leaves u at or above the
    total.  -> int64 (R,)."""
    cdf = torch.cumsum(torch.softmax(logits.to(torch.float64), dim=-1), dim=-1)
    c = (u_choice.to(torch.float64)[:, None] >= cdf).sum(dim=-1)
    return c.clamp(max=logits.shape[1] - 1)


def spline_params(p: Dict[str, torch.Tensor], cond: torch.Tensor, choice: torch.Tensor):
    """The raw outputs (R, 71) of the ten conditioners on the context [z-scored condition, choice]."""
    dt = p["cat.W0"].dtype
    zt = (cond.to(dt) - p["cond_mean"]) / p["cond_std"]
    ctx = torch.cat([zt, choice.to(dt)[:, None]], dim=1)
    out = []
    for k in range(NUM_TRANSFORMS):
        a = torch.relu(ctx @ p[f"flow.{k}.W1"].T + p[f"flow.{k}.b1"])
        a = torch.relu(a @ p[f"flow.{k}.W2"].T + p[f"flow.{k}.b2"])
        out.append(a @ p[f"flow.{k}.W3"].T + p[f"flow.{k}.b3"])
    return out


def sample(p: Dict[str, torch.Tensor], cond: torch.Tensor, u_choice: torch.Tensor, normal: torch.Tensor) -> torch.Tensor:
    """estimator.sample from caller-given draws: cond (R,85), u_choice (R,) in (0,1), normal (R,) ~ N(0,1) ->
    x (R,2) = [rt seconds, choice].  The choice is drawn from the categorical net (float64 CDF), then u = normal goes
    through the ten splines inverted in reverse order, and rt = exp(mu_y + sigma_y * u).  rt is not clamped.  Computed
    in the dtype of the parameters."""
    dt = p["cat.W0"].dtype
    c = choice_from_uniform(choice_logits(p, cond), u_choice)
    u = normal.to(dt)
    for q in reversed(spline_params(p, cond, c)):
        u, _ = rqs_inverse(u, q)
    y = p["flow.mu_y"] + p["flow.sigma_y"] * u
    return torch.stack([torch.exp(y), c.to(dt)], dim=1)


def flow_forward(p: Dict[str, torch.Tensor], x: torch.Tensor, cond: torch.Tensor) -> torch.Tensor:
    """The flow's base variable of rows x (R,2) = [rt, choice]: the ten splines forward from (log rt - mu_y) / sigma_y.
    For a sample of the estimator it is N(0,1)-distributed given the choice."""
    dt = p["cat.W0"].dtype
    x = x.to(dt)
    u = (torch.log(x[:, 0]) - p["flow.mu_y"]) / p["flow.sigma_y"]
    for q in spline_params(p, cond, x[:, 1]):
        u, _ = rqs_forward(u, q)
    return u
