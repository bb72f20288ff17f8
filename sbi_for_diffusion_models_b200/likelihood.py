"""The pulse DDM's own likelihood on the GPU, by propagating the accumulator's density.

The simulator is a one-dimensional Markov chain with Gaussian steps, two absorbing bounds and a known kick
schedule, so its law can be computed rather than sampled: the density is propagated on a grid of cells over
(0, B) one Euler step at a time, and the mass absorbed at each bound on each step is the probability of that
(choice, step).  This is a reference likelihood for the model users simulate, against which the MNLE estimator's
error can be stated in nats per trial (``tools/mnle_vs_model.py``).

* ``first_passage_law``: P(c, k) for c in {0, 1}, k = 1..W, and P(2), the mass that survives the W steps.
* ``loglik_rows``: log-likelihood of (rt seconds, choice) rows.  For choice 0 / 1 it is log P(c, k) - log dt with
  k = round((rt - t_nd) / dt): a density in rt seconds, piecewise constant over each step, in the unit
  ``DeviceMNLE.log_prob`` uses.  For choice 2 it is log P(2), a probability MASS, which is not comparable with the
  estimator's density for choice 2.
* ``GridLikelihood.loglik_sum`` / ``loglik_sum_batched``: the call shapes of ``DeviceMNLE.loglik_sum`` /
  ``loglik_sum_batched``, so the MCMC drivers can sample the posterior under the model's own likelihood.  Each
  theta's weights of the steps without a kick are tabulated once per call and shared by its trials; every value has
  the bits of ``loglik_rows``.

The discretisation, its truncation and its error are defined by ``oracle/ddm_grid_spec.py`` (float64) and
DESIGN section 4b; the kernels are ``csrc/ddm_grid.cu``.  Schedule arguments default to the simulator's.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import _native
from .simulator import Schedule, _as_f32_rows, compute_device

CELLS_PER_SIGMA = 4.0


def _schedule(mu_sensory: float, dt, t_max, pulse_interval) -> Schedule:
    return Schedule.from_constants(mu_sensory, dt=dt, t_max=t_max, pulse_interval=pulse_interval)


def _check_theta(theta: torch.Tensor, sched: Schedule, what: str) -> torch.Tensor:
    if not isinstance(theta, torch.Tensor):
        theta = torch.as_tensor(np.asarray(theta))
    if theta.ndim == 1:
        theta = theta.view(1, -1)
    if theta.ndim != 2 or theta.shape[1] != 5:
        raise ValueError(f"{what}: theta must be (N,5), got {tuple(theta.shape)}")
    th = theta.detach().to("cpu", torch.float32)
    if not bool(torch.isfinite(th).all()):
        raise ValueError(f"{what}: theta must be finite")
    if bool((th[:, 1].double() * sched.dt >= 0.5).any()):
        raise ValueError(f"{what}: the leak must satisfy lam * dt < 0.5")
    return theta


def _check_pulses(pulses, n: int, sched: Schedule, what: str) -> torch.Tensor:
    s = pulses if isinstance(pulses, torch.Tensor) else torch.as_tensor(np.asarray(pulses))
    if s.ndim == 1:
        s = s.view(1, -1)
    if s.ndim != 2 or s.shape[0] != n or s.shape[1] < sched.n_pulses:
        raise ValueError(f"{what}: pulses must be ({n}, >={sched.n_pulses}), got {tuple(s.shape)}")
    if not bool(torch.isfinite(s.detach().to("cpu", torch.float32)).all()):
        raise ValueError(f"{what}: pulses must be finite")
    return s


def _check_x(x, n: int, what: str) -> torch.Tensor:
    x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))
    if x.ndim != 2 or x.shape != (n, 2):
        raise ValueError(f"{what}: x must be ({n}, 2) = [rt seconds, choice], got {tuple(x.shape)}")
    xc = x.detach().to("cpu", torch.float32)
    if not bool(torch.isfinite(xc).all()):
        raise ValueError(f"{what}: x must be finite")
    c = xc[:, 1]
    if not bool(((c == 0) | (c == 1) | (c == 2)).all()):
        raise ValueError(f"{what}: choices must be 0, 1 or 2")
    return x


def _cells_per_sigma(q: float) -> float:
    q = float(q)
    if not (0.0 < q <= 64.0):
        raise ValueError(f"cells_per_sigma must be in (0, 64], got {q}")
    return q


def first_passage_law(theta: torch.Tensor, pulses, *, mu_sensory: float = 1.0, dt: Optional[float] = None,
                      t_max: Optional[float] = None, pulse_interval: Optional[float] = None,
                      cells_per_sigma: float = CELLS_PER_SIGMA, device=None
                      ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """theta (N,5), pulses (N,>=n_pulses) -> (law (N, 2, n_max), survive (N,), h_over_s (N,)) fp32 on the device.

    law[r, c, k - 1] = P(choice c at step k) for k = 1..W (0 after W), survive[r] = P(2).  h_over_s is the cell
    width over the step's noise scale the row used: 1 / cells_per_sigma or less, more for rows whose B needs more
    than ``ddm_grid_max_cells()`` cells."""
    sched = _schedule(mu_sensory, dt, t_max, pulse_interval)
    q = _cells_per_sigma(cells_per_sigma)
    theta = _check_theta(theta, sched, "first_passage_law")
    n = theta.shape[0]
    pl = _check_pulses(pulses, n, sched, "first_passage_law")
    L = _native.lib()
    dev = compute_device(device if device is not None else (theta.device if theta.is_cuda else None))
    with torch.cuda.device(dev):
        th = _as_f32_rows(theta, dev).contiguous()
        s = _as_f32_rows(pl, dev).contiguous()
        law = torch.empty((n, 2, sched.n_max), dtype=torch.float32, device=dev)
        survive = torch.empty((n,), dtype=torch.float32, device=dev)
        cells = torch.empty((n,), dtype=torch.int32, device=dev)
        if n:
            rc = L.ddm_grid_law_f32(th.data_ptr(), 5, s.data_ptr(), s.shape[1], n, s.shape[1], sched.n_max,
                                    sched.steps_per_pulse, sched.dt, sched.t_max, sched.t_nd_hi, sched.noise_scale, q,
                                    law.data_ptr(), survive.data_ptr(), cells.data_ptr(),
                                    torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "ddm_grid_law_f32")
        B = th[:, 3].abs().clamp_min(1e-6).double()
        h_over_s = (B / cells.double() / sched.noise_scale).float()
    return law, survive, h_over_s


def loglik_rows(theta: torch.Tensor, x: torch.Tensor, pulses, *, mu_sensory: float = 1.0, dt: Optional[float] = None,
                t_max: Optional[float] = None, pulse_interval: Optional[float] = None,
                cells_per_sigma: float = CELLS_PER_SIGMA, device=None) -> torch.Tensor:
    """theta (N,5), x (N,2) = [rt seconds, choice], pulses (N,>=n_pulses) -> (N,) fp32 grid log-likelihoods on the
    device (see the module docstring for the units of choice 0 / 1 and of choice 2)."""
    sched = _schedule(mu_sensory, dt, t_max, pulse_interval)
    q = _cells_per_sigma(cells_per_sigma)
    theta = _check_theta(theta, sched, "loglik_rows")
    n = theta.shape[0]
    x = _check_x(x, n, "loglik_rows")
    pl = _check_pulses(pulses, n, sched, "loglik_rows")
    L = _native.lib()
    dev = compute_device(device if device is not None else (theta.device if theta.is_cuda else None))
    with torch.cuda.device(dev):
        th = _as_f32_rows(theta, dev).contiguous()
        xr = _as_f32_rows(x, dev).contiguous()
        s = _as_f32_rows(pl, dev).contiguous()
        out = torch.empty((n,), dtype=torch.float32, device=dev)
        if n:
            rc = L.ddm_grid_loglik_f32(th.data_ptr(), 5, xr.data_ptr(), s.data_ptr(), s.shape[1], n, s.shape[1],
                                       sched.n_max, sched.steps_per_pulse, sched.dt, sched.t_max, sched.t_nd_hi,
                                       sched.noise_scale, q, out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "ddm_grid_loglik_f32")
    return out


class GridLikelihood:
    """Summed grid log-likelihood over the trials of a session, with the call shape of ``DeviceMNLE.loglik_sum``:
    ``loglik_sum(theta (C,5), x_o (T,2), pulses (T,>=80)) -> (C,)`` with out[c] = sum_t log p(x_o[t] | theta[c],
    pulses[t]), summed over t in order in fp64.  A choice-2 trial contributes log P(2), a probability mass."""

    def __init__(self, *, mu_sensory: float = 1.0, dt: Optional[float] = None, t_max: Optional[float] = None,
                 pulse_interval: Optional[float] = None, cells_per_sigma: float = CELLS_PER_SIGMA, device=None):
        self.schedule = _schedule(mu_sensory, dt, t_max, pulse_interval)
        self.cells_per_sigma = _cells_per_sigma(cells_per_sigma)
        self._device = device

    def loglik_sum(self, theta: torch.Tensor, x_o: torch.Tensor, pulses) -> torch.Tensor:
        """The D = 1 case of ``loglik_sum_batched``, with the values of theta, x_o and pulses checked on the host."""
        sched = self.schedule
        theta = _check_theta(theta, sched, "GridLikelihood.loglik_sum")
        x_o = x_o if isinstance(x_o, torch.Tensor) else torch.as_tensor(np.asarray(x_o))
        x_o = x_o.reshape(-1, 2)
        T = x_o.shape[0]
        x_o = _check_x(x_o, T, "GridLikelihood.loglik_sum")
        pl = _check_pulses(pulses, T, sched, "GridLikelihood.loglik_sum")
        return self.loglik_sum_batched(theta[None], x_o[None], pl[None])[0]

    def loglik_sum_batched(self, theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor) -> torch.Tensor:
        """theta (D,C,5), x_o (D,T,2) = [rt seconds, choice], pulses (D,T,>=n_pulses) -> (D,C) fp32 with out[d,c] =
        sum_t log p(x_o[d,t] | theta[d,c], pulses[d,t]), summed over t in order in fp64: the contract of
        ``DeviceMNLE.loglik_sum_batched``.  Only shapes are checked and nothing is read back to the host, so a CUDA
        graph can record the call; check the values of x_o and pulses once with the host checks of ``loglik_sum``.
        A theta that is not finite or has lam * dt >= 0.5 gives NaN."""
        sched = self.schedule
        if theta.ndim != 3 or theta.shape[2] != 5:
            raise ValueError(f"GridLikelihood.loglik_sum_batched: theta must be (D,C,5), got {tuple(theta.shape)}")
        D, C = theta.shape[0], theta.shape[1]
        if x_o.ndim != 3 or x_o.shape[0] != D or x_o.shape[2] != 2:
            raise ValueError(f"GridLikelihood.loglik_sum_batched: x_o must be (D,T,2) with D={D}, got {tuple(x_o.shape)}")
        T = x_o.shape[1]
        if pulses.ndim != 3 or pulses.shape[0] != D or pulses.shape[1] != T or pulses.shape[2] < sched.n_pulses:
            raise ValueError(f"GridLikelihood.loglik_sum_batched: pulses must be (D,T,>={sched.n_pulses}) with D={D}, "
                             f"T={T}, got {tuple(pulses.shape)}")
        if D * C >= 2**31 or D * T >= 2**31:
            raise ValueError(f"GridLikelihood.loglik_sum_batched: D * C and D * T must be < 2^31, got {D * C}, {D * T}")
        L = _native.lib()
        dev = compute_device(self._device if self._device is not None else (theta.device if theta.is_cuda else None))
        with torch.cuda.device(dev):
            th = theta.to(device=dev, dtype=torch.float32).contiguous()
            xr = x_o.to(device=dev, dtype=torch.float32).contiguous()
            s = pulses.to(device=dev, dtype=torch.float32).contiguous()
            out = torch.empty((D, C), dtype=torch.float32, device=dev)
            n_ws = L.ddm_grid_loglik_sum_batched_workspace_floats(D, T, C, self.cells_per_sigma)
            ws = torch.empty((max(n_ws, 1),), dtype=torch.float32, device=dev)
            rc = L.ddm_grid_loglik_sum_batched_f32(th.data_ptr() if D * C else None, 5, xr.data_ptr() if D * T else None,
                                                   s.data_ptr() if D * T else None, s.shape[2], D, T, C, s.shape[2],
                                                   sched.n_max, sched.steps_per_pulse, sched.dt, sched.t_max,
                                                   sched.t_nd_hi, sched.noise_scale, self.cells_per_sigma,
                                                   out.data_ptr() if D * C else None, ws.data_ptr(),
                                                   torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "ddm_grid_loglik_sum_batched_f32")
        return out.to(theta.device)
