"""Row-by-row checks of the MNLE gradient kernels -- TEST INFRASTRUCTURE (CPU, float64 unless the params are float32).

The tensor-core kernels run their networks on bf16 hi / lo operands, which leave pre-activations ~1e-5 from fp32
(DESIGN §3.5 / §3.6).  A ReLU unit, a spline knot or a probability clamp that close to its kink lands on the other
side, and single gradient entries move by a whole row's contribution.  Comparing such rows with float64 says nothing
about the kernel; comparing only the rows that are clear of every kink does, entry by entry and tightly.

* ``kink_margins``: per row, how far it sits from every place where d log p is discontinuous.
* ``theta_grad_by_plane``: the float64 d log p / d theta of every (trial, chain) row, split into the 22 (net, column
  half) planes the reverse-mode kernel forms (``kGradPlanes`` in ``csrc/mnle_train.cu``).
* ``check_rows`` / ``check_sum`` / ``check_named``: the comparisons the GPU tests make, and that
  ``tests/test_mnle_grad_spec.py`` shows to reject mutated gradients.

The wiring restates ``oracle.mnle_spec.log_prob`` (the CPU tests hold the two to 1e-12) with the first-layer
pre-activations of each net kept, so that autograd can stop there.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import torch

from oracle import mnle_spec as ms

N_NETS = 1 + ms.NUM_TRANSFORMS      # net 0: categorical head, net 1 + k: conditioner of flow transform k
N_PLANES = 2 * N_NETS               # (net, first-layer units 0-63 / 64-127)
HALF = ms.HIDDEN // 2


def _first_weight(p, net):
    return p["cat.W0"] if net == 0 else p[f"flow.{net - 1}.W1"]


def _forward(p: Dict[str, torch.Tensor], x: torch.Tensor, cond: torch.Tensor):
    """log p (R,) as ``ms.log_prob`` computes it, plus what the margins and the planes need: the first-layer
    pre-activation of every net, the second-layer ones of the conditioners, each transform's input u_k and raw
    parameters q_k, and the probability of the observed choice before the clamp."""
    dt = p["cat.W0"].dtype
    x, cond = x.to(dt), cond.to(dt)
    zt = (cond - p["cond_mean"]) / p["cond_std"]
    choice = x[:, 1]
    pre1 = [zt @ p["cat.W0"].T + p["cat.b0"]]
    h = torch.sigmoid(pre1[0])
    h = torch.sigmoid(h @ p["cat.W1"].T + p["cat.b1"])
    h = torch.sigmoid(h @ p["cat.W2"].T + p["cat.b2"])
    probs = torch.softmax(h @ p["cat.Wo"].T + p["cat.bo"], dim=-1)
    pc = probs.gather(1, choice.to(torch.int64)[:, None])[:, 0]
    lp_choice = torch.log(pc.clamp(ms.PROB_EPS, 1.0 - ms.PROB_EPS))
    ctx = torch.cat([zt, choice[:, None]], dim=1)
    y = torch.log(x[:, 0])
    u = (y - p["flow.mu_y"]) / p["flow.sigma_y"]
    lad = -torch.log(p["flow.sigma_y"]) * torch.ones_like(u)
    pre2, us, qs = [], [], []
    for k in range(ms.NUM_TRANSFORMS):
        pre1.append(ctx @ p[f"flow.{k}.W1"].T + p[f"flow.{k}.b1"])
        pre2.append(torch.relu(pre1[-1]) @ p[f"flow.{k}.W2"].T + p[f"flow.{k}.b2"])
        qs.append(torch.relu(pre2[-1]) @ p[f"flow.{k}.W3"].T + p[f"flow.{k}.b3"])
        us.append(u)
        u, l = ms.rqs_forward(u, qs[-1])
        lad = lad + l
    base = -0.5 * u * u - 0.5 * math.log(2.0 * math.pi)
    return dict(lp=lp_choice + base + lad - y, pre1=pre1, pre2=pre2, u=us, q=qs, pc=pc)


def log_prob(p, x, cond):
    return _forward(p, x, cond)["lp"]


def kink_margins(p: Dict[str, torch.Tensor], x: torch.Tensor, cond: torch.Tensor) -> Dict[str, torch.Tensor]:
    """Per row (R,) float64, each kind of gradient discontinuity on its own:
    ``relu``  smallest |pre-activation| over both ReLU layers of the ten conditioners;
    ``knot``  smallest distance of a transform's input u_k to an interior knot of its bin grid (``cw`` in
              ``ms.rqs_forward``), over the transforms whose input lies inside the tail bound;
    ``tail``  smallest distance of a u_k to +-TAIL_BOUND, where the spline meets its linear tails;
    ``prob``  min(p, 1 - p) / PROB_EPS of the observed choice's probability: the log-probability is clamped below 1."""
    with torch.no_grad():
        f = _forward(ms.cast_params(p, torch.float64), x.double(), cond.double())
        relu = torch.stack([t.abs().min(dim=1).values for t in f["pre1"][1:] + f["pre2"]]).min(dim=0).values
        knot = torch.full_like(f["lp"], float("inf"))
        tail = torch.full_like(f["lp"], float("inf"))
        K = ms.NUM_BINS
        for u, q in zip(f["u"], f["q"]):
            w = ms.MIN_BIN + (1.0 - ms.MIN_BIN * K) * torch.softmax(q[:, :K] / math.sqrt(ms.HIDDEN), dim=-1)
            cw = 2.0 * ms.TAIL_BOUND * torch.cumsum(w, dim=-1)[:, :-1] - ms.TAIL_BOUND    # the K - 1 interior knots
            inside = u.abs() <= ms.TAIL_BOUND
            d = (u[:, None] - cw).abs().min(dim=1).values
            knot = torch.minimum(knot, torch.where(inside, d, torch.full_like(d, float("inf"))))
            tail = torch.minimum(tail, (u.abs() - ms.TAIL_BOUND).abs())
        prob = torch.minimum(f["pc"], 1.0 - f["pc"]) / ms.PROB_EPS
    return dict(relu=relu, knot=knot, tail=tail, prob=prob)


KINDS = ("relu", "knot", "tail", "prob")


def kink_kind(m: Dict[str, torch.Tensor], delta: float) -> List[str]:
    """The first kind of kink each row is within ``delta`` of ("" when it is clear of all):
    pre-activations and u-distances against ``delta``, the probability against a factor of 2 of its clamp."""
    lim = dict(relu=delta, knot=delta, tail=delta, prob=2.0)
    out = [""] * m["relu"].shape[0]
    for k in reversed(KINDS):
        for r in torch.nonzero(m[k] <= lim[k]).flatten().tolist():
            out[r] = k
    return out


def kept_rows(m: Dict[str, torch.Tensor], delta: float) -> torch.Tensor:
    """(R,) bool: rows clear of every kink by ``delta`` (and of the probability clamps by a factor of 2)."""
    return (m["relu"] > delta) & (m["knot"] > delta) & (m["tail"] > delta) & (m["prob"] > 2.0)


def theta_grad_by_plane(p: Dict[str, torch.Tensor], theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor):
    """(lp (T,C), planes (T,C,22,5)) in the dtype of ``p``: row r = t*C + c of ``ms.potential_rows``, and
    planes[t,c, 2*net + half] = d log p_r / d theta through net ``net``'s first-layer units half*64 .. half*64+63 --
    d log p / d (those pre-activations) contracted with the theta columns of the net's first weight, z-scoring
    included, as the backward kernel's last epilogue does.  Summed over the planes: autograd's d log p_r / d theta_c."""
    C, T = theta.shape[0], x_o.shape[0]
    dt = p["cat.W0"].dtype
    xr, cond = ms.potential_rows(theta.to(dt).detach().requires_grad_(True), x_o.to(dt), pulses.to(dt))
    f = _forward(p, xr, cond)
    g = torch.autograd.grad(f["lp"].sum(), f["pre1"])
    planes = []
    for net in range(N_NETS):
        w = _first_weight(p, net)[:, :5] / p["cond_std"][:5]
        for half in range(2):
            s = slice(half * HALF, (half + 1) * HALF)
            planes.append(g[net][:, s] @ w[s])
    planes = torch.stack(planes, dim=1).detach()
    return f["lp"].detach().reshape(T, C), planes.reshape(T, C, N_PLANES, 5)


# ---- bounds (tests/test_gpu_mnle_grad_rows.py; tests/test_mnle_grad_spec.py shows they reject mutated gradients) ----

# Rows within DELTA of a ReLU kink, a knot or the tail bound are left out.  Measured on a B200 (NVIDIA B200, 1000 W), 8
# trials x 512 thetas per net: at 1e-4 only 0.41 of the init nets' rows stay (0.58 trained), at 5e-5 0.55-0.66, and the
# kept rows' errors do not change between 2e-5 and 2e-4 -- the tensor cores flip a unit only within ~2e-5 of its kink.
DELTA = 5e-5
# check_rows bounds: kernel error <= 3 x the fp32 CPU spec's own + an absolute term, per column in units of its RMS.
# Measured (excess over 3 x floor, largest column): init / init-K2 / init-K8 -- gradient tc <= -4e-5, simt <= 7e-6,
# value <= 7e-7; trained -- gradient tc 2.5e-2 (max) / 1.3e-5 (mean) (worst row 0.039 of the column RMS against a
# floor of 0.0047; the older bound allowed 5 x |ref|), simt < 0; value tc 3.1e-5.
ROW_BOUNDS = {(kind, kernel, what): dict(k=3.0, atol_max=3e-5 if what == "grad" else 2e-6, atol_mean=0.0)
              for kind in ("init", "trained", "init-K2", "init-K8") for kernel in ("tc", "simt") for what in ("value", "grad")}
ROW_BOUNDS[("trained", "tc", "grad")] = dict(k=3.0, atol_max=5e-2, atol_mean=4e-5)
ROW_BOUNDS[("trained", "tc", "value")] = dict(k=3.0, atol_max=1e-4, atol_mean=0.0)
# a T-trial call against its T single-trial calls: measured <= 8.0e-7 of the parts' L1 (tc and simt, both nets)
SUM_TOL = 2e-6
# training step on kink-free rows: every tensor measured within 6.3e-5 of its largest float64 entry (R = 300, 4096,
# 8325; K = 2, 3, 8; the older bound was 1e-2), loss within 6.5e-7 relative
TRAIN_TOL = 1.5e-4
TRAIN_LOSS_TOL = 2e-6
# R g_R against the sum over the pieces of a split minibatch: measured <= 4.0e-5 of the tensor's largest L1
TRAIN_SUM_TOL = 1e-4
TRAIN_SUM_FLOOR = 1.0


# ---- checks -------------------------------------------------------------------------------------------------------

def row_errors(got: torch.Tensor, ref: torch.Tensor, floor: torch.Tensor, kept: torch.Tensor):
    """Per-entry errors on the kept rows of (R, m) tensors, in units of each column's RMS over those rows:
    (kernel error e, fp32-spec error f), both (n_kept, m) float64."""
    ref = ref.double()[kept]
    scale = ref.pow(2).mean(dim=0).sqrt().clamp_min(1e-300)
    return (got.double()[kept] - ref).abs() / scale, (floor.double()[kept] - ref).abs() / scale


def check_rows(got, ref, floor, kept, *, k: float, atol_max: float, atol_mean: float):
    """Entry-by-entry check of per-row results ``got`` (R, m) against the float64 ``ref`` on the ``kept`` rows.
    ``floor`` is the fp32 CPU spec's result on the same rows (what the reference's own arithmetic gets): the max and
    the mean error of every column, in units of the column's RMS, must be within ``k`` x the floor's plus an absolute
    term (the tensor-core operands carry ~17 bits, fp32 24).  Returns (ok, stats); stats["over_max"] and
    stats["over_mean"] are the largest excess over k x floor among the columns, i.e. the absolute terms the rows need."""
    e, f = row_errors(got, ref, floor, kept)
    over_max = float((e.max(dim=0).values - k * f.max(dim=0).values).max())
    over_mean = float((e.mean(dim=0) - k * f.mean(dim=0)).max())
    st = dict(max=float(e.max()), mean=float(e.mean(dim=0).max()), floor_max=float(f.max()),
              floor_mean=float(f.mean(dim=0).max()), over_max=over_max, over_mean=over_mean)
    return over_max <= atol_max and over_mean <= atol_mean, st


def sum_error(total: torch.Tensor, parts: Sequence[torch.Tensor], floor: float = 1e-3) -> float:
    """max over entries of |total - sum(parts)| / L1, sum and L1 = sum |parts| entrywise in float64; L1 is floored at
    ``floor`` x its largest entry so that entries whose parts are all ~0 do not divide by ~0 (floor = 1: the error in
    units of the tensor's largest L1, for sums whose parts themselves cancel, like a weight gradient's)."""
    P = torch.stack([q.double() for q in parts])
    l1 = P.abs().sum(dim=0)
    den = l1 + floor * float(l1.max()) + 1e-300
    return float(((total.double() - P.sum(dim=0)).abs() / den).max())


def check_sum(total, parts, *, tol: float, floor: float = 1e-3):
    """A sum computed by the kernel against the float64 sum of parts computed by the same kernel: the rows are the
    same numbers wherever they sit, so only fp32 summation may separate them.  Returns (ok, error)."""
    e = sum_error(total, parts, floor)
    return e <= tol, e


def check_named(got: Dict[str, torch.Tensor], want: Dict[str, torch.Tensor], *, tol: float):
    """Every named tensor within ``tol`` of its own largest float64 entry.  Returns (ok, {name: error / max})."""
    errs = {}
    for name, w in want.items():
        ref = float(w.double().abs().max())
        errs[name] = float((got[name].double() - w.double()).abs().max()) / max(ref, 1e-300)
    return all(v <= tol for v in errs.values()), errs


def nll_grads(p: Dict[str, torch.Tensor], x: torch.Tensor, cond: torch.Tensor, rows: torch.Tensor = None):
    """(loss, {name: d loss / d name}) of loss = -mean log p over the rows, in the dtype of ``p``: the training step's
    reference.  ``rows`` (bool or index) restricts the sum to those rows while still dividing by all R."""
    frozen = ("cond_mean", "cond_std", "flow.mu_y", "flow.sigma_y")
    q = {k: v.clone().requires_grad_(k not in frozen) for k, v in p.items()}
    lp = log_prob(q, x, cond)
    R = lp.shape[0]
    loss = -(lp if rows is None else lp[rows]).sum() / R
    names = [k for k in q if k not in frozen]
    g = torch.autograd.grad(loss, [q[k] for k in names])
    return float(loss.detach()), dict(zip(names, g))
