"""Inference and calibration drivers around the fused MNLE potential (reference mnle.py:52-237).

``run_inference_mcmc`` and ``run_sbc`` keep the reference's arguments and return values.  What
changes is where the work happens: the potential is the tcgen05 kernel, and the sampler is the
device-resident many-chain slice sampler of ``samplers.py`` instead of sbi's ``MCMCPosterior`` /
pyro NUTS (third-party, CPU, one process per chain).  ``run_sbc`` pre-draws every dataset in the
reference's order, simulates all sessions of a rank in one launch, samples all
(dataset, chain) pairs in lock-step through the batched potential, and shards datasets over the
GPUs of the box (all-gather of the ranks at the end).

Training the estimator (reference mnle.py:16-50, ``sbi.inference.MNLE``) is not part of the hot
path; estimators arrive here as ``DeviceMNLE`` / ``PackedMNLE`` or anything exposing an
MNLE-shaped ``state_dict()``.
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import numpy as np
import torch

from .potentials import as_device_estimator, prior_log_prob
from .samplers import GraphedLogProb, PhiloxUniforms, VectorizedSliceSampler
from .sbc import compute_ranks, draw_sbc_datasets, simulate_sbc_sessions
from .sharding import _world, all_gather_rows, gather_sbc, shard_bounds
from .simulator import compute_device

MIN_VECTOR_CHAINS = 128   # one row tile of the potential kernel


def _init_from_prior(prior_theta, log_prob_fn, n: int, device, max_tries: int = 20) -> torch.Tensor:
    """``init_strategy="proposal"`` (reference mnle.py:85): prior draws, redrawn where the
    posterior potential is not finite."""
    x = prior_theta.sample((n,)).to(device=device, dtype=torch.float32)
    for _ in range(max_tries):
        bad = ~torch.isfinite(log_prob_fn(x))
        if not bool(bad.any()):
            return x
        x[bad] = prior_theta.sample((int(bad.sum()),)).to(device=device, dtype=torch.float32)
    raise RuntimeError("could not find starting points with finite posterior potential")


@torch.no_grad()
def run_inference_mcmc(cfg, prior_theta, density_estimator, x_o, pulses_o, *, num_chains: Optional[int] = None,
                       device=None, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """Posterior samples over theta (dim 5) given one observed session (reference mnle.py:52-95).

    Returns (cfg.POSTERIOR_SAMPLES, 5) on the CPU.  ``num_chains`` defaults to
    max(cfg.NUM_CHAINS, 128): the sampler advances all chains with one potential call per step, so
    fewer chains than one row tile would leave the kernel idle.  Each chain contributes
    ceil(POSTERIOR_SAMPLES / num_chains) draws after cfg.WARMUP_STEPS tuning sweeps."""
    dev = compute_device(device)
    chains = int(num_chains) if num_chains is not None else max(int(cfg.NUM_CHAINS), MIN_VECTOR_CHAINS)
    # the same potential as ThetaOnlyPosteriorPotential(ConditionedMNLELogLikelihood(...)) (reference
    # mnle.py:61-73), in the sync-free form a CUDA graph can record: every row is evaluated and rows
    # outside the prior's support keep their -inf
    x = x_o.to(device=dev, dtype=torch.float32)
    if x.dim() == 3:
        assert x.shape[1] == 1, "This implementation supports a single observed x batch (num_xs=1)."
        x = x[:, 0, :]
    pulses = pulses_o.to(device=dev, dtype=torch.float32)
    assert pulses.shape[0] == x.shape[0], f"local_theta must have shape (num_trials, P). Got {tuple(pulses.shape)}"
    fn = _BatchedPotential(as_device_estimator(density_estimator), prior_theta, x[None], pulses[None], float(cfg.TEMPERATURE))
    init = _init_from_prior(prior_theta, fn, chains, dev)
    sampler = VectorizedSliceSampler(GraphedLogProb(fn, init), init, generator=generator)
    want = int(cfg.POSTERIOR_SAMPLES)
    per_chain = -(-want // chains)
    draws = sampler.run(per_chain, warmup=int(cfg.WARMUP_STEPS), thin=1)          # (per_chain, chains, 5)
    return draws.reshape(-1, draws.shape[-1])[:want].detach().cpu()


class _BatchedPotential:
    """log prior + loglik / temperature for D datasets x C chains as one flat (D*C, 5) batch: datasets of equal
    length (x (D,T,2), pulses (D,T,>=80)), or with ``plan`` (a ``SessionPlan``) ragged sessions one after the other
    (x (N,2), pulses (N,>=80))."""

    def __init__(self, estimator, prior_theta, x, pulses, temperature: float, plan=None):
        self.est, self.prior, self.x, self.pulses, self.plan = estimator, prior_theta, x, pulses, plan
        self.D, self.temperature = (x.shape[0] if plan is None else plan.D), float(temperature)

    def __call__(self, theta_flat: torch.Tensor) -> torch.Tensor:
        lp = prior_log_prob(self.prior, theta_flat)
        th = theta_flat.view(self.D, -1, theta_flat.shape[-1])
        if self.plan is None:
            ll = self.est.loglik_sum_batched(th, self.x, self.pulses)
        else:
            ll = self.est.loglik_sum_sessions(th, self.x, self.pulses, self.plan, kernel=self.plan.kernel)
        return torch.where(torch.isfinite(lp), lp + ll.reshape(-1) / self.temperature, lp)


def _sample_groups(cfg, potential, init: torch.Tensor, G: int, first: int, num_samples: int, seed: int, what: str
                   ) -> torch.Tensor:
    """The sampling core of ``sbc_shard`` and ``sessions_shard``: G groups (datasets / sessions, global numbers
    first .. first + G - 1) of C chains each, all in lock-step through one potential call per iteration, each group
    with its own slice widths and every chain with its own counter-based uniforms (Philox rows of the GLOBAL chain
    numbers).  -> (G, num_samples, 5) CPU."""
    S, C = int(num_samples), init.shape[0] // G
    ok = torch.isfinite(potential(init)).view(G, C).all(dim=1)
    if not bool(ok.all()):
        raise RuntimeError(f"a prior draw of {what} {first + int((~ok).nonzero()[0])} has a non-finite posterior potential")
    sampler = VectorizedSliceSampler(GraphedLogProb(potential, init), init, chain_groups=G,
                                     uniforms=PhiloxUniforms(int(seed) * 1_000_003 + 17, first * C, G * C, init.device))
    per_chain = -(-S // C)
    draws = sampler.run(per_chain, warmup=int(cfg.WARMUP_STEPS), thin=1)                  # (per_chain, G*C, 5)
    return draws.view(per_chain, G, C, 5).permute(1, 0, 2, 3).reshape(G, per_chain * C, 5)[:, :S].cpu()


@torch.no_grad()
def sbc_shard(cfg, prior_theta, estimator, thetas_true: torch.Tensor, ds_seeds, init_all: torch.Tensor, lo: int, hi: int,
              num_samples: int, seed: int, device=None):
    """Datasets [lo, hi) of an SBC run: simulate their sessions (one launch), sample all their chains
    in lock-step through the batched potential, rank.  -> (ranks (hi-lo,5) int64 CPU, samples
    (hi-lo,S,5) float32 CPU).  Everything random is indexed by the GLOBAL dataset / chain number
    (Philox trial offsets in the simulator, starting points ``init_all`` drawn for all datasets,
    counter-based uniforms, per-dataset slice widths), so the result for a dataset does not depend on
    which other datasets share its launch -- any split into shards reproduces the unsplit run."""
    dev = compute_device(device)
    D, S, T = hi - lo, int(num_samples), int(cfg.NUM_TRIALS_OBS)
    C = init_all.shape[0] // thetas_true.shape[0]
    ranks = torch.empty((D, 5), dtype=torch.int64)
    if D == 0:
        return ranks, torch.empty((0, S, 5), dtype=torch.float32)
    x, pulses = simulate_sbc_sessions(thetas_true[lo:hi], ds_seeds[lo:hi], T, mu_sensory=float(cfg.MU_SENSORY),
                                      p_success=float(cfg.P_SUCCESS), noise_seed=seed, first_dataset=lo, device=dev)
    if bool(cfg.LOG_RT_MANUALLY):
        x = x.clone()
        x[..., 0] = torch.log(x[..., 0].clamp_min(1e-6))
    potential = _BatchedPotential(estimator, prior_theta, x, pulses, float(cfg.TEMPERATURE))
    init = init_all[lo * C:hi * C].to(device=dev, dtype=torch.float32)
    samples = _sample_groups(cfg, potential, init, D, lo, S, seed, "dataset")
    for i in range(D):
        ranks[i] = compute_ranks(thetas_true[lo + i], samples[i])
    return ranks, samples


@torch.no_grad()
def run_sbc(cfg, *, prior_theta, density_estimator, device: str = "cpu", num_datasets: int = 25,
            posterior_samples_per_dataset: Optional[int] = None, seed: int = 0,
            param_names: Sequence[str] = ("a0", "lam", "v", "B", "tau"), outdir: str = "sbc_outputs", plot_bins: int = 30,
            chains_per_dataset: int = MIN_VECTOR_CHAINS, group=None, save: bool = True) -> dict:
    """Simulation-based calibration (reference mnle.py:128-237): for every dataset draw
    theta_true ~ prior, simulate a session, sample the posterior, rank theta_true among the draws.

    Returns {"thetas_true": (N,5) float32 ndarray, "ranks": (N,5) int64 ndarray,
    "all_samples": list of N CPU tensors (S,5)} on every rank, identical for any number of ranks.
    ``device`` is accepted for signature compatibility; the work runs on this rank's GPU."""
    dev = compute_device(None)
    rank, world = _world(group)
    N = int(num_datasets)
    S = int(posterior_samples_per_dataset) if posterior_samples_per_dataset is not None else int(cfg.POSTERIOR_SAMPLES)
    thetas_true, ds_seeds = draw_sbc_datasets(prior_theta, N, seed)                       # reference order
    init_all = prior_theta.sample((N * int(chains_per_dataset),)).to(torch.float32)       # same on every rank
    lo, hi = shard_bounds(N, rank, world)
    ranks_local, samples_local = sbc_shard(cfg, prior_theta, as_device_estimator(density_estimator), thetas_true, ds_seeds,
                                           init_all, lo, hi, S, seed, dev)
    thetas_all, ranks_all = gather_sbc(thetas_true[lo:hi].to(dev), ranks_local.to(dev), N, group)
    samples_all = all_gather_rows(samples_local.to(dev), N, group).cpu()
    out = {"thetas_true": thetas_all.cpu().numpy(), "ranks": ranks_all.cpu().numpy(),
           "all_samples": [samples_all[i] for i in range(N)]}
    if save and rank == 0:
        os.makedirs(outdir, exist_ok=True)
        np.save(os.path.join(outdir, "sbc_thetas_true.npy"), out["thetas_true"])
        np.save(os.path.join(outdir, "sbc_ranks.npy"), out["ranks"])   # (the reference also draws a histogram: not on this path)
    return out


def _session_tensors(sessions, first: int, dev):
    """(x (T_i,2), pulses (T_i,80)) fp32 on ``dev`` of every session, checked on the host."""
    xs, pls = [], []
    for i, (x, pl) in enumerate(sessions):
        x = x.to(device=dev, dtype=torch.float32)
        if x.dim() == 3 and x.shape[1] == 1:
            x = x[:, 0, :]
        if x.dim() != 2 or x.shape[1] != 2:
            raise ValueError(f"session {first + i}: x_o must be (T,2), got {tuple(x.shape)}")
        if pl.dim() != 2 or pl.shape[0] != x.shape[0] or pl.shape[1] < 80:
            raise ValueError(f"session {first + i}: pulses must be (T,>=80) with T={x.shape[0]}, got {tuple(pl.shape)}")
        xs.append(x)
        pls.append(pl[:, :80].to(device=dev, dtype=torch.float32))
    return xs, pls


@torch.no_grad()
def sessions_shard(cfg, prior_theta, estimator, sessions, init_all: torch.Tensor, lo: int, hi: int, seed: int,
                   kernel: str = "tc", device=None) -> torch.Tensor:
    """Sessions [lo, hi) of ``run_inference_sessions``: all their chains sampled in lock-step through one ragged
    potential call per iteration (the counterpart of ``sbc_shard``, same sampling core).  ``init_all``: the starting
    points of ALL sessions, C per session.  -> (hi-lo, cfg.POSTERIOR_SAMPLES, 5) float32 CPU.  Everything random is
    indexed by the global session / chain number, so any split into shards reproduces the unsplit run bit for bit."""
    dev = compute_device(device)
    G, S = hi - lo, int(cfg.POSTERIOR_SAMPLES)
    if G == 0:
        return torch.empty((0, S, 5), dtype=torch.float32)
    C = init_all.shape[0] // len(sessions)
    xs, pls = _session_tensors(sessions[lo:hi], lo, dev)
    est = as_device_estimator(estimator)
    plan = est.session_plan([x.shape[0] for x in xs], C, kernel=kernel, device=dev)
    potential = _BatchedPotential(est, prior_theta, torch.cat(xs), torch.cat(pls), float(cfg.TEMPERATURE), plan=plan)
    init = init_all[lo * C:hi * C].to(device=dev, dtype=torch.float32)
    return _sample_groups(cfg, potential, init, G, lo, S, seed, "session")


@torch.no_grad()
def run_inference_sessions(cfg, prior_theta, density_estimator, sessions, *, num_chains: Optional[int] = None, seed: int = 0,
                           kernel: str = "tc", device=None, group=None) -> list:
    """Posterior samples over theta (dim 5) for each of several observed sessions of any lengths, from one estimator
    in one run: ``sessions`` is a sequence of (x_o (T_i,2), pulses_o (T_i,>=80)); x_o is used as given, as
    ``run_inference_mcmc`` uses it.  Returns one (cfg.POSTERIOR_SAMPLES, 5) float32 CPU tensor per session.

    ``num_chains`` per session defaults to max(cfg.NUM_CHAINS, 128); cfg.WARMUP_STEPS tuning sweeps and
    cfg.TEMPERATURE as in ``run_inference_mcmc``.  ``kernel``: "tc" or "tc64" (``DeviceMNLE.loglik_sum_sessions``).
    The starting points are prior draws under ``torch.manual_seed(seed)`` in a forked RNG state (the caller's stream
    is left alone), the sampler's uniforms are keyed by ``seed`` and the global chain number.  Under torchrun the
    sessions are split over the ranks (``shard_bounds``) and the draws all-gathered: every rank returns the full
    list, identical for any world size."""
    sessions = list(sessions)
    n = len(sessions)
    if n == 0:
        return []
    dev = compute_device(device)
    C = int(num_chains) if num_chains is not None else max(int(cfg.NUM_CHAINS), MIN_VECTOR_CHAINS)
    cuda_devices = list(range(torch.cuda.device_count())) if torch.cuda.is_initialized() else []
    with torch.random.fork_rng(devices=cuda_devices):
        torch.manual_seed(int(seed))
        init_all = prior_theta.sample((n * C,)).to(torch.float32)
    rank, world = _world(group)
    lo, hi = shard_bounds(n, rank, world)
    local = sessions_shard(cfg, prior_theta, density_estimator, sessions, init_all, lo, hi, seed, kernel, dev)
    samples = all_gather_rows(local.to(dev), n, group).cpu()
    return [samples[i] for i in range(n)]


# ---- checkpoints (reference mnle.py:241-297) ---------------------------------------------------------------

def _model_dir() -> str:
    path = os.path.join(os.path.expanduser("~"), "models")
    os.makedirs(path, exist_ok=True)
    return path


def save_model(density_estimator, cfg, filename: str = "mnle_rt_choice_model.pt") -> str:
    """``torch.save({"state_dict": ..., "config": ...})`` under ``~/models`` like the reference (mnle.py:247-259);
    the state of a device estimator is its packed parameter buffer.  Returns the path."""
    est = as_device_estimator(density_estimator)
    path = os.path.join(_model_dir(), filename)
    torch.save({"state_dict": est.state_dict(), "config": cfg}, path)
    return path


def load_model(cfg=None, filename: str = "mnle_rt_choice.pt"):
    """The estimator saved by ``save_model`` (``None`` when the file does not exist, as the reference's
    mnle.py:262-266; its default file names differ between save and load, which is kept).  ``cfg`` is accepted for
    signature compatibility: the architecture is fixed by the packed layout, nothing has to be rebuilt."""
    from .mnle_net import DeviceMNLE, PackedMNLE
    path = os.path.join(_model_dir(), filename)
    if not os.path.exists(path):
        return None
    blob = torch.load(path, map_location="cpu", weights_only=False)
    sd = blob["state_dict"]
    if "packed_params" in sd:
        return DeviceMNLE(PackedMNLE(sd["packed_params"].numpy(), int(sd["n_choices"])))
    return DeviceMNLE(PackedMNLE.from_state_dict(sd))      # a checkpoint written by sbi itself (see from_state_dict)


@torch.no_grad()
def posterior_predictive(density_estimator, theta: torch.Tensor, pulses: torch.Tensor, *, seed: Optional[int] = None
                         ) -> torch.Tensor:
    """One emulated session per parameter draw: theta (C,5) (e.g. from ``run_inference_mcmc``) and the session's pulse
    trains (T,>=80) -> x (C,T,2) = [rt seconds, choice], x[c,t] drawn from the estimator at [theta_c, pulses_t].  One
    ``sample`` call on the (C*T, 85) condition rows, row c*T + t; rt is not clamped (see ``DeviceMNLE.sample``)."""
    est = as_device_estimator(density_estimator)
    if theta.ndim != 2 or theta.shape[1] != 5:
        raise ValueError(f"theta must be (C,5), got {tuple(theta.shape)}")
    if pulses.ndim != 2 or pulses.shape[1] < 80:
        raise ValueError(f"pulses must be (T,>=80), got {tuple(pulses.shape)}")
    C, T = theta.shape[0], pulses.shape[0]
    pl = pulses[:, :80].to(device=theta.device, dtype=torch.float32)
    cond = torch.cat([theta.to(torch.float32)[:, None, :].expand(C, T, 5), pl[None, :, :].expand(C, T, 80)], dim=2)
    return est.sample((), condition=cond.reshape(C * T, 85), seed=seed).reshape(C, T, 2)
