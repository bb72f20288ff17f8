"""One-chain-at-a-time specification of ``samplers.VectorizedSliceSampler`` -- TEST INFRASTRUCTURE.

Neal (2003), "Slice sampling", Fig. 3 (stepping out with a limit of m expansions) and Fig. 5 (shrinkage), applied to
one coordinate after another, written as plain nested loops for a single chain.  It shares no code with the sampler's
vectorised state machine (``samplers.py`` on torch, ``csrc/mnle_sampler.cu`` on the device); given the same uniforms
it reproduces every chain of theirs bit for bit.  The project's conventions, all of which the loops below follow:

* Coordinates are updated in order 0..D-1; one sweep is D updates.
* An update of coordinate d with width w from the point x, log-probability lp:
  slice level ``log_y = lp + log(u1)``; bracket ``lo = x[d] - w*u2``, ``hi = lo + w``; limits
  ``J = clamp(floor(m*u3), 0, m-1)``, ``K = m-1-J``.  Step out left while J > 0 and the potential at lo is above the
  slice (lo -= w, J -= 1), then right the same way with K.  A point is inside when its potential is > log_y.
* Shrinkage proposes ``lo + (hi-lo)*u0``; an accepted proposal becomes x[d].  A rejected one left of x[d] moves lo,
  otherwise hi.  After ``max_shrink`` failed proposals the update gives up and the chain keeps its point.
* During the first ``warmup`` sweeps every finished update moves the width of its coordinate to the running mean of
  the final bracket, ``w + ((hi-lo) - w)/(n+1)`` after n earlier tunings, clamped below at 1e-6.  Widths never change
  otherwise.
* After warm-up every ``thin``-th sweep is recorded, up to S draws; after ``warmup + S*thin`` sweeps the chain stops.
* A NaN potential counts as -inf.
* The uniform clock: iteration ``it0`` supplies u1..u3 of the first update.  Every potential evaluation of the chain
  is the next iteration k and a shrinkage proposal uses u0 of that iteration.  An update that finishes at iteration k
  starts the next one with u1..u3 of iteration k.  In the sampler, iteration ``it`` is draws 4*it + j (j = 0..3) of the
  ``uniforms`` callable, and ``run()`` starts at the sampler's ``_it``.

Every operation is rounded in ``dtype`` (numpy float32 or float64), in the order written.  ``log(u1)`` comes from
``log_fn`` because the logarithm of a device library is not correctly rounded: to replay a device run, pass the
device's own logarithm.
"""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import numpy as np


def slice_chain(log_prob: Callable[[np.ndarray], float], x: Sequence[float], width: Sequence[float],
                uniforms: Callable[[int], Sequence[float]], *, it0: int = 0, lp: Optional[float] = None,
                max_step_out: int = 8, max_shrink: int = 64, warmup: int = 0, S: int = 1, thin: int = 1,
                dtype=np.float32, log_fn: Callable[[float], float] = np.log) -> dict:
    """Run one chain for ``warmup + S*thin`` sweeps.

    ``log_prob``: (D,) array of ``dtype`` -> log-probability (-inf outside the support); ``x``, ``width``: (D,) start
    and slice widths; ``uniforms(k)`` -> (u0, u1, u2, u3) of iteration k; ``lp``: log-probability at ``x`` (evaluated
    when None, not counted).  Returns ``draws`` (S, D), final ``x``, ``lp``, ``width``, ``tuned`` (tunings per
    coordinate), ``sweeps`` and ``evals`` (iterations the chain used after ``it0``)."""
    t = np.dtype(dtype).type
    x = np.array(x, dtype=dtype)
    width = np.array(width, dtype=dtype)
    D = x.shape[0]
    tuned = np.zeros(D, dtype=dtype)
    m, thin = int(max_step_out), max(int(thin), 1)
    total = int(warmup) + int(S) * thin

    def f(v):
        y = t(log_prob(v))
        return t(-np.inf) if math.isnan(y) else y

    def at(d, v):
        p = x.copy()
        p[d] = v
        return p

    lp = f(x) if lp is None else t(lp)
    draws = []
    it = int(it0)
    u = [t(v) for v in uniforms(it)]
    sweeps = 0
    while sweeps < total:
        for d in range(D):
            w, x0 = width[d], x[d]
            # Fig. 3: slice level, randomly placed bracket, limits split at random between the two ends
            log_y = t(lp + t(log_fn(u[1])))
            lo = t(x0 - t(w * u[2]))
            hi = t(lo + w)
            J = min(max(math.floor(t(t(m) * u[3])), 0), m - 1)
            K = (m - 1) - J
            while J > 0:
                it += 1
                u = [t(v) for v in uniforms(it)]
                if not f(at(d, lo)) > log_y:
                    break
                lo = t(lo - w)
                J -= 1
            while K > 0:
                it += 1
                u = [t(v) for v in uniforms(it)]
                if not f(at(d, hi)) > log_y:
                    break
                hi = t(hi + w)
                K -= 1
            # Fig. 5: shrinkage, giving up after max_shrink proposals
            n = 0
            while True:
                it += 1
                u = [t(v) for v in uniforms(it)]
                q = t(lo + t(t(hi - lo) * u[0]))
                fq = f(at(d, q))
                n += 1
                if fq > log_y:
                    x[d], lp = q, fq
                    break
                if n >= max_shrink:
                    break
                if q < x0:
                    lo = q
                else:
                    hi = q
            if sweeps < warmup:
                nw = t(w + t(t(t(hi - lo) - w) / t(tuned[d] + t(1))))
                width[d] = max(nw, t(1e-6))
                tuned[d] = t(tuned[d] + t(1))
        sweeps += 1
        past = sweeps - warmup
        if past > 0 and past % thin == 0 and len(draws) < S:
            draws.append(x.copy())
    return dict(draws=np.array(draws, dtype=dtype).reshape(len(draws), D), x=x, lp=lp, width=width, tuned=tuned,
                sweeps=sweeps, evals=it - int(it0))


class SeededUniforms:
    """Uniforms for n chains in which draw k of every chain is a pure function of (seed, k):
    ``default_rng([seed, k])``, 24 random bits per value -> (bits + 0.5) * 2^-24, in (0, 1) and exact in float32 like
    the sampler's Philox uniforms.  ``override(k, u)`` may overwrite entries of draw k in place to force a branch.
    ``draw(k)`` -> (n,) float32; ``chain(c)`` -> the ``uniforms`` argument of ``slice_chain`` for chain c."""

    def __init__(self, seed: int, n: int, override: Optional[Callable[[int, np.ndarray], None]] = None):
        self.seed, self.n, self.override = int(seed), int(n), override
        self._cache = {}

    def draw(self, k: int) -> np.ndarray:
        k = int(k)
        if k not in self._cache:
            bits = np.random.default_rng([self.seed, k]).integers(0, 1 << 24, self.n, dtype=np.int64)
            u = ((bits.astype(np.float64) + 0.5) * 2.0 ** -24).astype(np.float32)
            if self.override is not None:
                self.override(k, u)
            self._cache[k] = u
        return self._cache[k]

    def chain(self, c: int) -> Callable[[int], Sequence[float]]:
        return lambda it: [self.draw(4 * it + j)[c] for j in range(4)]


INF = float("inf")


# Targets for replaying a run: written once for numpy (n, D) float32 arrays (xp = numpy) and torch (n, D) tensors
# (xp = torch), elementwise in a fixed order or with exactly representable values, so that numpy and torch on any
# device give the same bits
def gauss(x, xp):
    acc = None
    for j in range(x.shape[1]):
        t = (x[:, j] - 0.25) * (x[:, j] - 0.25)
        acc = t if acc is None else acc + t
    return acc * -0.5


def gauss_nan(x, xp):           # NaN on 0.5 < x_0 < 1, which the sampler treats as -inf
    return xp.where((x[:, 0] > 0.5) & (x[:, 0] < 1.0), float("nan"), gauss(x, xp))


def box(x, xp):                 # flat on (-40, 40)^D: stepping out always runs to its limit
    return xp.where((xp.abs(x) < 40.0).all(1), x[:, 0] * 0.0, -INF)


def spike(x, xp):               # finite only on |x_0 - 0.1| < 0.01
    return xp.where(xp.abs(x[:, 0] - 0.1) < 0.01, x[:, 0] * 0.0, -INF)


def trunc_exp(x, xp):           # exp(-x_0) on [0, 3) x uniform on [-1, 1): chains may start on the edge x_0 = 0
    ok = (x[:, 0] >= 0.0) & (x[:, 0] < 3.0) & (x[:, -1] >= -1.0) & (x[:, -1] < 1.0)
    return xp.where(ok, -x[:, 0], -INF)


def staircase(x, xp):           # -floor(2|x_j|) summed (exact integers) on (-3, 3)^D
    ok = (xp.abs(x) < 3.0).all(1)
    return xp.where(ok, -xp.floor(xp.abs(x) * 2.0).sum(1), -INF)


def bits(a):
    a = np.asarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)
