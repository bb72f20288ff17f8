"""Posteriors of many observed sessions of different lengths in one run: the ragged potential
(``DeviceMNLE.loglik_sum_sessions``, tc and tc64) against per-session calls, and the driver
``run_inference_sessions`` / ``sessions_shard`` against itself and against ``sbc_shard``.

Equalities are bit for bit: every (trial, chain) row is computed independently of the other rows of
its tile, and a session's sum over its trials runs in a fixed order, whichever other sessions share
the launch."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ddm_oracle as orc
from oracle import mnle_spec as ms
from sbi_for_diffusion_models_b200.mnle import run_inference_sessions, sbc_shard, sessions_shard
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE
from sbi_for_diffusion_models_b200.priors import build_prior_theta
from sbi_for_diffusion_models_b200.run_config import RunConfig
from sbi_for_diffusion_models_b200.sbc import draw_sbc_datasets, simulate_sbc_sessions

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRAINED = os.path.join(ROOT, "tests", "golden", "mnle_trained.npz")
LENGTHS = ([50, 7, 1, 0, 130, 64], [3], [0, 0, 0])


@pytest.fixture(scope="module", params=["init", "trained"])
def est(request):
    if request.param == "init":
        return DeviceMNLE(PackedMNLE.from_params(ms.init_params(0)))
    d = np.load(TRAINED)
    return DeviceMNLE(PackedMNLE(d["packed"], int(d["n_choices"])))


def _sessions(lengths, seed=1):
    """Simulated sessions with the given numbers of trials: lists of x (T_i,2) and pulses (T_i,80) on the GPU."""
    D = max(len(lengths), 1)
    thetas, seeds = draw_sbc_datasets(build_prior_theta(), D, seed=seed)
    x, pulses = simulate_sbc_sessions(thetas, seeds, max(max(lengths, default=1), 1), mu_sensory=1.0, p_success=0.75,
                                      noise_seed=2)
    return [x[d, :T] for d, T in enumerate(lengths)], [pulses[d, :T] for d, T in enumerate(lengths)]


def _thetas(D, C, seed=0):
    torch.manual_seed(seed)
    return build_prior_theta().sample((D * C,)).view(D, C, 5).cuda()


@pytest.mark.parametrize("kernel", ["tc", "tc64"])
@pytest.mark.parametrize("C", [1, 37, 128, 130, 300])
@pytest.mark.parametrize("lengths", LENGTHS, ids=["mixed", "one", "empty"])
def test_sessions_equal_per_session_calls(est, lengths, C, kernel):
    xs, pls = _sessions(lengths)
    th = _thetas(len(lengths), C)
    got = est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), lengths, kernel=kernel)
    assert tuple(got.shape) == (len(lengths), C) and got.is_cuda and got.dtype == torch.float32
    for d, T in enumerate(lengths):
        want = est.loglik_sum(th[d], xs[d], pls[d], kernel=kernel)
        assert torch.equal(got[d], want), (d, T, float((got[d] - want).abs().max()))
        if T == 0:
            assert bool((got[d] == 0).all())
    assert torch.equal(got, est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), torch.tensor(lengths), kernel=kernel))


@pytest.mark.parametrize("C", [37, 128])
def test_equal_lengths_equal_the_batched_call(est, C):
    D, T = 4, 50
    xs, pls = _sessions([T] * D)
    th = _thetas(D, C)
    got = est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), [T] * D)
    assert torch.equal(got, est.loglik_sum_batched(th, torch.stack(xs), torch.stack(pls)))


@pytest.mark.parametrize("kernel", ["tc", "tc64"])
def test_permuting_the_sessions_permutes_the_outputs(est, kernel):
    lengths, C = LENGTHS[0], 130
    xs, pls = _sessions(lengths)
    th = _thetas(len(lengths), C)
    got = est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), lengths, kernel=kernel)
    perm = [4, 2, 0, 5, 3, 1]
    again = est.loglik_sum_sessions(th[perm], torch.cat([xs[i] for i in perm]), torch.cat([pls[i] for i in perm]),
                                    [lengths[i] for i in perm], kernel=kernel)
    assert torch.equal(again, got[perm])


@pytest.mark.parametrize("kernel", ["tc", "tc64"])
def test_split_over_several_launches_keeps_the_bits(est, kernel, monkeypatch):
    lengths, C = LENGTHS[0], 130
    xs, pls = _sessions(lengths)
    th = _thetas(len(lengths), C)
    whole = est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), lengths, kernel=kernel)
    monkeypatch.setattr(DeviceMNLE, "SESSIONS_MAX_TRIALS", 140)
    monkeypatch.setattr(DeviceMNLE, "SESSIONS_TC64_MAX_ROWS", 140 * C)
    monkeypatch.setattr(DeviceMNLE, "SESSIONS_TC64_MAX_SESSIONS", 2)
    plan = est.session_plan(lengths, C, kernel=kernel)
    assert len(plan.chunks) >= 3 and plan.chunks[0][0] == 0 and plan.chunks[-1][1] == len(lengths)
    assert torch.equal(est.loglik_sum_sessions(th, torch.cat(xs), torch.cat(pls), plan, kernel=kernel), whole)


def test_refusals(est, monkeypatch):
    lengths, C = [50, 7, 1, 0, 130, 64], 37
    xs, pls = _sessions(lengths)
    x, pl, th = torch.cat(xs), torch.cat(pls), _thetas(len(lengths), C)
    for bad in ([50, 7, 1, 0, 130, 63], [50, 7, 2, -1, 130, 64], [50, 7, 1, 0, 130], [50.0, 7, 1, 0, 130, 64]):
        with pytest.raises(ValueError):
            est.loglik_sum_sessions(th, x, pl, bad)
    with pytest.raises(ValueError, match="theta must be"):
        est.loglik_sum_sessions(th[..., :4], x, pl, lengths)
    with pytest.raises(ValueError, match="theta must be"):
        est.loglik_sum_sessions(th[0], x, pl, lengths)
    with pytest.raises(ValueError, match="x_o must be"):
        est.loglik_sum_sessions(th, torch.cat([x, x[:, :1]], dim=1), pl, lengths)
    with pytest.raises(ValueError, match="pulses must be"):
        est.loglik_sum_sessions(th, x, pl[:, :79], lengths)
    with pytest.raises(ValueError, match="pulses must be"):
        est.loglik_sum_sessions(th, x, pl[1:], lengths)
    with pytest.raises(ValueError, match="unknown kernel"):
        est.loglik_sum_sessions(th, x, pl, lengths, kernel="simt")
    monkeypatch.setattr(DeviceMNLE, "SESSIONS_MAX_TRIALS", 100)
    with pytest.raises(ValueError, match="session 4 has 130 trials"):
        est.loglik_sum_sessions(th, x, pl, lengths)


def _observed(lengths, theta=(0.45, 0.6, 1.3, 14.0, 0.25), seed=123):
    out = []
    for i, T in enumerate(lengths):
        pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(seed + i)), 0, T, 80, 0.75))
        x, _ = orc.sim_rng_c(np.repeat(np.array([theta], np.float32), T, 0), pulses.numpy(), 7 + i)
        out.append((torch.from_numpy(x), pulses))
    return out


def test_run_inference_sessions_outputs_and_posteriors_concentrate(est):
    from sbi_for_diffusion_models_b200.potentials import ConditionedMNLELogLikelihood, ThetaOnlyPosteriorPotential
    cfg = RunConfig(POSTERIOR_SAMPLES=600, WARMUP_STEPS=15, NUM_CHAINS=2)
    prior = build_prior_theta()
    sessions = _observed([50, 35, 60])
    state = torch.random.get_rng_state()
    out = run_inference_sessions(cfg, prior, est, sessions, seed=4)
    assert torch.equal(torch.random.get_rng_state(), state)          # the caller's stream is left alone
    assert len(out) == 3
    torch.manual_seed(1)
    prior_draws = prior.sample((600,))
    for (x, pulses), s in zip(sessions, out):
        assert tuple(s.shape) == (600, 5) and s.device.type == "cpu" and s.dtype == torch.float32
        assert bool(torch.isfinite(prior.log_prob(s)).all())
        pot = ThetaOnlyPosteriorPotential(conditioned_loglike=ConditionedMNLELogLikelihood(est, pulses, "cpu"),
                                          prior_theta=prior, x_o=x, device="cpu", temperature=1.0)
        assert float(pot(s, track_gradients=False).median()) > float(pot(prior_draws, track_gradients=False).median()) + 1.0
    assert run_inference_sessions(cfg, prior, est, []) == []


def test_sessions_shard_does_not_depend_on_the_sharding(est):
    cfg = RunConfig(WARMUP_STEPS=4, POSTERIOR_SAMPLES=200)
    prior = build_prior_theta()
    lengths, C = [12, 5, 0, 20, 9], 128
    xs, pls = _sessions(lengths, seed=3)
    sessions = list(zip(xs, pls))
    torch.manual_seed(0)
    init_all = prior.sample((len(lengths) * C,)).to(torch.float32)
    whole = sessions_shard(cfg, prior, est, sessions, init_all, 0, len(lengths), 3)
    assert tuple(whole.shape) == (len(lengths), 200, 5) and whole.dtype == torch.float32 and whole.device.type == "cpu"
    for lo, hi in ((0, 2), (2, 5), (4, 5), (3, 3), (3, 4)):
        assert torch.equal(sessions_shard(cfg, prior, est, sessions, init_all, lo, hi, 3), whole[lo:hi]), (lo, hi)
    assert torch.equal(sessions_shard(cfg, prior, est, sessions, init_all, 0, len(lengths), 3), whole)
    other = sessions_shard(cfg, prior, est, sessions, init_all, 0, len(lengths), 4)
    assert not torch.equal(other, whole)


def test_equal_length_sessions_reproduce_sbc_shard(est):
    T, N, C, S, seed = 12, 4, 128, 200, 3
    cfg = RunConfig(WARMUP_STEPS=4, NUM_TRIALS_OBS=T, POSTERIOR_SAMPLES=S)
    prior = build_prior_theta()
    thetas, seeds = draw_sbc_datasets(prior, N, seed=seed)
    init_all = prior.sample((N * C,)).to(torch.float32)
    _, want = sbc_shard(cfg, prior, est, thetas, seeds, init_all, 0, N, S, seed)
    x, pulses = simulate_sbc_sessions(thetas, seeds, T, mu_sensory=float(cfg.MU_SENSORY), p_success=float(cfg.P_SUCCESS),
                                      noise_seed=seed, first_dataset=0)
    got = sessions_shard(cfg, prior, est, [(x[i], pulses[i]) for i in range(N)], init_all, 0, N, seed)
    assert torch.equal(got, want)


def test_two_gpu_sessions_match_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs; the shards' union is checked on one GPU by "
                    "test_sessions_shard_does_not_depend_on_the_sharding")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29531", os.path.join(ROOT, "tools", "check_sessions_sharded.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "sessions sharded over 2 GPUs == single GPU: True" in r.stdout
