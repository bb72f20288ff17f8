"""The batched grid potential (``GridLikelihood.loglik_sum_batched`` over ``ddm_grid_loglik_sum_batched_f32``): every
(trial, theta) value has the bits of ``loglik_rows``, the result does not depend on how chains and datasets are split
or chunked, the sampler's potential and its CUDA graph give the bits of direct calls, posterior draws of
``run_inference_mcmc`` follow the posterior computed by quadrature with the same likelihood, and the drivers refuse
what the grid cannot score."""
import math
from dataclasses import replace

import numpy as np
import pytest
import torch
from scipy.stats import kstwo

from oracle import ddm_oracle as orc

pytestmark = pytest.mark.gpu


def _lik():
    from sbi_for_diffusion_models_b200 import likelihood
    return likelihood


def _pulses(seed, shape, P=80):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(np.where(rng.random((*shape, P)) < 0.5, 1.0, -1.0).astype(np.float32))


SIM_THETA = [0.5, 0.3, 0.15, 2.0, 0.12]   # small gain, B = 2: rt from 0.12 s to several s, k up to thousands


def _chains(C, seed, late=False):
    """Prior draws with small gains (long propagation, many kick-free steps) and 0.8 <= B <= 2.5 (rows short enough
    to run every shape through loglik_rows); t_nd below 0.1, or in [7, 7.5] (windows of 1000-2000 steps)."""
    th = orc.prior_sample(C, seed=seed)
    th[:, 2] = th[:, 2].clamp(max=0.3)
    th[:, 3] = th[:, 3].clamp(0.8, 2.5)
    th[:, 4] = 7.0 + 0.5 * th[:, 4] if late else 0.1 * th[:, 4]
    return th


def _case(D, C, T, seed):
    """theta (D,C,5), x (D,T,2), pulses (D,T,80); each dataset has its own chains.
    dataset 0: trials simulated at SIM_THETA (t_nd 0.12) against chains with t_nd < 0.1: every value finite unless a
      density underflows, observed steps from 40 to thousands;
    dataset 1: censored trials (choice 2) alternating with choices 0 / 1 at rt in (7.6, 7.99), against chains with t_nd
      in [7, 7.5]: finite P(2) and densities;
    dataset 2: dataset 0's kind of trials plus one before every t_nd and one past every window: -inf.
    Every dataset has one pulse row scaled by 0.37 and one pulse equal to 0."""
    from sbi_for_diffusion_models_b200.simulator import simulate_trials
    pl = _pulses(seed, (D, T))
    th = torch.tensor([SIM_THETA]).expand(D * T, 5).contiguous()
    x = simulate_trials(th, pl.view(D * T, 80).cuda(), seed=seed).cpu().view(D, T, 2).clone()
    theta = torch.stack([_chains(C, seed + 17 * d, late=(d == 1)) for d in range(D)])
    rng = np.random.default_rng(seed)
    if D > 1:
        x[1, :, 0] = torch.from_numpy(rng.uniform(7.6, 7.99, T).astype(np.float32))
        x[1, :, 1] = torch.tensor([2.0 if t % 2 == 0 else float((t // 2) % 2) for t in range(T)])
    if D > 2:
        x[2, 0] = torch.tensor([0.0, 1.0])                    # before every t_nd
        if T > 1:
            x[2, 1] = torch.tensor([8.5, 0.0])                # past every window
    for d in range(D):
        pl[d, -1] *= 0.37
        pl[d, 0, 3] = 0.0
    return theta, x, pl


def _mostly_finite(want):
    assert torch.isfinite(want).float().mean() > 0.5, "the comparison would be between -inf values"


def _rows_reference(lik, theta, x, pl):
    """out[d, c] = float(sum over t in order, in fp64, of loglik_rows(theta[d, c], x[d, t], pl[d, t]))."""
    D, C, T = theta.shape[0], theta.shape[1], x.shape[1]
    rows_th = theta[:, None, :, :].expand(D, T, C, 5).reshape(-1, 5)
    rows_x = x[:, :, None, :].expand(D, T, C, 2).reshape(-1, 2)
    rows_pl = pl[:, :, None, :].expand(D, T, C, pl.shape[2]).reshape(-1, pl.shape[2])
    v = lik.loglik_rows(rows_th, rows_x, rows_pl).cpu().double().view(D, T, C)
    acc = torch.zeros(D, C, dtype=torch.float64)
    for t in range(T):
        acc = acc + v[:, t]
    return acc.float(), v.float()


def _same_bits(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.parametrize("D", [1, 3])
@pytest.mark.parametrize("C", [1, 5, 129])
@pytest.mark.parametrize("T", [1, 7, 50])
def test_bits_of_the_row_kernel(D, C, T):
    lik = _lik()
    theta, x, pl = _case(D, C, T, seed=100 + 10 * T + 7 * D + C)
    got = lik.GridLikelihood().loglik_sum_batched(theta.cuda(), x.cuda(), pl.cuda()).cpu()
    want, rows = _rows_reference(lik, theta, x, pl)
    _mostly_finite(want)
    assert _same_bits(got, want)
    if T == 1:
        assert _same_bits(got, rows[:, 0])


# the edge rows of tests/test_gpu_grid_likelihood.py
EDGE = torch.tensor([
    [0.0, 0.3, 0.5, 2.0, 0.3],          # start on the lower bound
    [1.0, 0.3, 0.5, 2.0, 0.3],          # start on the upper bound
    [0.5, 0.2, 0.5, 0.0, 0.3],          # B at its 1e-6 clamp, kick larger than B
    [0.5, 0.0, 3.0, 1.0, 0.3],          # kick larger than B
    [0.5, 0.3, 0.4, 1.5, 7.9999],       # W = 0
    [0.5, 0.3, 0.4, 1.5, 8.0 - 0.0007], # W = 1
    [0.4, 7.0, 0.5, 3.0, 0.0],          # strong leak, W = 16000
    [0.5, 0.1, 0.3, 60.0, 4.0],         # B above the cap: coarser cells
    [0.5, -0.5, 0.2, 1.0, 0.0],         # negative leak
], dtype=torch.float32)


def test_bits_of_the_row_kernel_on_edge_rows():
    """Every edge row against every trial, one trial per dataset (each value is one row of loglik_rows), and the
    same trials as one group of seven."""
    lik = _lik()
    _, x, pl = _case(1, 1, 7, seed=77)
    x[0, 3] = torch.tensor([7.9998, 1.0])                   # the one step of the W = 1 row
    x[0, 4] = torch.tensor([8.0, 2.0])                      # censored
    x[0, 5] = torch.tensor([4.3, 0.0])                      # inside the coarse row's window
    theta = torch.cat([EDGE, _chains(4, seed=5)])
    th7 = theta[None].expand(7, -1, -1).contiguous()
    gl = lik.GridLikelihood()
    got = gl.loglik_sum_batched(th7.cuda(), x[0, :, None].cuda(), pl[0, :, None].cuda()).cpu()
    want, _ = _rows_reference(lik, th7, x[0, :, None], pl[0, :, None])
    assert _same_bits(got, want)
    assert torch.isfinite(want).float().mean() > 0.4 and torch.isneginf(want).any()
    got = gl.loglik_sum_batched(theta[None].cuda(), x.cuda(), pl.cuda()).cpu()
    want, _ = _rows_reference(lik, theta[None], x, pl)
    assert _same_bits(got, want)


def test_invalid_theta_gives_nan_on_the_device():
    lik = _lik()
    theta, x, pl = _case(1, 6, 7, seed=3)
    theta[0, 1, 3] = float("nan")
    theta[0, 2, 0] = float("inf")
    theta[0, 3, 1] = 1000.0                               # lam dt = 0.5
    got = lik.GridLikelihood().loglik_sum_batched(theta.cuda(), x.cuda(), pl.cuda()).cpu()
    assert torch.isnan(got[0, 1:4]).all()
    keep = [0, 4, 5]
    want, _ = _rows_reference(lik, theta[:, keep], x, pl)
    _mostly_finite(want)
    assert _same_bits(got[:, keep], want)


def test_invariance_under_permutation_splitting_and_chunking():
    lik = _lik()
    gl = lik.GridLikelihood()
    # tables are built for floor(1.75 GiB / table bytes per theta) theta at a time: 265 at cells_per_sigma 4
    per_theta = (math.ceil(48 * gl.cells_per_sigma) + 24) * 2048 * 16
    chunk = (7 << 28) // per_theta
    D, C, T = 3, 100, 12
    assert D * C > chunk
    theta, x, pl = _case(D, C, T, seed=45)
    want, _ = _rows_reference(lik, theta, x, pl)
    _mostly_finite(want)
    theta, x, pl = theta.cuda(), x.cuda(), pl.cuda()
    full = gl.loglik_sum_batched(theta, x, pl)
    assert _same_bits(full.cpu(), want)
    perm = torch.randperm(C, generator=torch.Generator().manual_seed(1)).cuda()
    assert _same_bits(gl.loglik_sum_batched(theta[:, perm], x, pl), full[:, perm])
    by_d = torch.cat([gl.loglik_sum_batched(theta[d:d + 1], x[d:d + 1], pl[d:d + 1]) for d in range(D)])
    assert _same_bits(by_d, full)
    by_c = torch.cat([gl.loglik_sum_batched(theta[:, :37], x, pl), gl.loglik_sum_batched(theta[:, 37:], x, pl)], dim=1)
    assert _same_bits(by_c, full)
    for d in range(D):
        assert _same_bits(gl.loglik_sum(theta[d], x[d], pl[d]), full[d])


def test_potential_and_its_graph():
    lik = _lik()
    from sbi_for_diffusion_models_b200.mnle import _BatchedPotential
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.samplers import GraphedLogProb
    gl = lik.GridLikelihood()
    prior = build_prior_theta("cuda")
    theta, x, pl = _case(1, 130, 7, seed=12)
    x, pl = x.cuda(), pl.cuda()
    pot = _BatchedPotential(gl, prior, x, pl, 2.0)
    th = theta[0].cuda()
    th[1, 0] = 1.5                                        # outside the prior: -inf
    th[2, 3] = float("nan")                               # not finite
    th[3, 1] = 1000.0                                     # lam dt = 0.5: NaN from the likelihood
    got = pot(th)
    lp = prior.log_prob(th)
    ll = gl.loglik_sum_batched(th[None], x, pl)[0]
    _mostly_finite(got.cpu())
    assert _same_bits(got, torch.where(torch.isfinite(lp), lp + ll / 2.0, lp))
    assert torch.isneginf(got[1]) and torch.isnan(ll[3]) and torch.isnan(got[3])
    graphed = GraphedLogProb(pot, th)
    assert graphed.graph is not None
    th2 = _chains(130, seed=14).cuda()
    for t in (th2, th):
        want = pot(t)
        _mostly_finite(want.cpu())
        assert _same_bits(graphed(t), want)


# ---- end to end: posterior draws against the posterior by quadrature ----------------------------------------------

# a0, lam, B, t_nd pinned by LogNormal(log m, s) components; t_nd sits half a step inside its window so that +-3 sds
# change neither W nor any trial's observed step
PIN = {0: (0.5, 1e-3), 1: (0.5, 1e-3), 3: (1.0, 1e-3), 4: (0.10025, 5e-4)}
V_LOC, V_SCALE, V_TRUE = math.log(0.3), 0.5, 0.3
SCHED = dict(t_max=0.5)                                                 # 1000 steps, 5 pulses
E2E_T, E2E_CHAINS = 100, 1024


def _e2e_prior(v_loc=V_LOC, v_scale=V_SCALE):
    from torch.distributions import LogNormal
    from sbi_for_diffusion_models_b200.priors import MultipleIndependentPrior
    comps = []
    for i in range(5):
        m, s = PIN.get(i, (None, None))
        comps.append(LogNormal(torch.tensor([math.log(m) if m else v_loc]), torch.tensor([s if s else v_scale])))
    return MultipleIndependentPrior(comps)


def _e2e_session():
    """T trials drawn from the grid law itself at theta_true (rt = t_nd + k dt), so the model is exact."""
    lik = _lik()
    gl = lik.GridLikelihood(**SCHED)
    sched = gl.schedule
    theta_true = torch.tensor([[PIN[0][0], PIN[1][0], V_TRUE, PIN[3][0], PIN[4][0]]]).expand(E2E_T, 5).contiguous()
    pl = _pulses(2024, (E2E_T,), P=sched.n_pulses)
    law, surv, _ = lik.first_passage_law(theta_true, pl, **SCHED)
    law, surv = law.cpu().double().numpy(), surv.cpu().double().numpy()
    rng = np.random.default_rng(7)
    x = np.zeros((E2E_T, 2), dtype=np.float32)
    for t in range(E2E_T):
        p = np.concatenate([law[t, 0], law[t, 1], [surv[t]]])
        i = rng.choice(p.size, p=p / p.sum())
        n = sched.n_max
        if i == 2 * n:
            x[t] = [sched.t_max, 2.0]
        else:
            x[t] = [np.float32(PIN[4][0]) + (i % n + 1) * np.float32(sched.dt), i // n]
    return gl, torch.from_numpy(x), pl


def _quadrature_cdf(gl, x, pl, v, shift=None):
    """Posterior CDF of v on the grid v (1-D, theta's other coordinates at their pinned values, optionally one of
    them moved by k prior sds) by the trapezoid rule on the log-density."""
    th = torch.zeros(v.numel(), 5)
    for i, (m, s) in PIN.items():
        th[:, i] = m
    if shift is not None:
        i, k = shift
        th[:, i] = PIN[i][0] * math.exp(k * PIN[i][1])
    th[:, 2] = v
    ll = gl.loglik_sum(th.cuda(), x.cuda(), pl.cuda()).cpu().double()
    lv = torch.log(v.double())
    logp = ll - lv - (lv - V_LOC) ** 2 / (2 * V_SCALE ** 2)
    dens = torch.exp(logp - logp.max()).numpy()
    vv = v.double().numpy()
    cum = np.concatenate([[0.0], np.cumsum(0.5 * (dens[1:] + dens[:-1]) * np.diff(vv))])
    return vv, cum / cum[-1]


def _ks(draws, vv, cdf):
    s = np.sort(draws)
    F = np.interp(s, vv, cdf)
    n = s.size
    d = max(float((np.arange(1, n + 1) / n - F).max()), float((F - np.arange(n) / n).max()))
    return d, float(kstwo.sf(d, n))


def test_run_inference_mcmc_draws_follow_the_quadrature_posterior():
    from sbi_for_diffusion_models_b200 import mnle
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    lik = _lik()
    gl, x, pl = _e2e_session()
    # a coarse log-spaced pass finds the posterior's support, a fine pass over it is the reference
    vc = torch.logspace(-2, math.log10(5.0), 801)
    vvc, cdfc = _quadrature_cdf(gl, x, pl, vc)
    lo, hi = float(np.interp(1e-9, cdfc, vvc)), float(np.interp(1 - 1e-9, cdfc, vvc))
    v = torch.linspace(lo * 0.9, hi * 1.1, 2001)
    vv, cdf = _quadrature_cdf(gl, x, pl, v)
    assert cdf[20] < 1e-6 and cdf[-20] > 1 - 1e-6, "the v grid does not cover the posterior"
    crit = float(kstwo.isf(1e-3, E2E_CHAINS))
    # the pinning is below the statistic's resolution: 3 prior sds of any pinned coordinate move the CDF less
    moved = max(float(np.abs(_quadrature_cdf(gl, x, pl, v, (i, k))[1] - cdf).max()) for i in PIN for k in (-3, 3))
    assert moved < crit, (moved, crit)
    cfg = RunConfig(WARMUP_STEPS=20, POSTERIOR_SAMPLES=E2E_CHAINS)
    torch.manual_seed(3)
    draws = mnle.run_inference_mcmc(cfg, _e2e_prior(), gl, x, pl, num_chains=E2E_CHAINS,
                                    generator=torch.Generator(device="cuda").manual_seed(5))
    d, p = _ks(draws[:, 2].double().numpy(), vv, cdf)
    # power: the same statistic rejects the posterior of a model whose noise is 5 % larger (mu_sensory x 1.05), a
    # misspecification of the size the estimator's own errors reach
    vv_b, cdf_b = _quadrature_cdf(lik.GridLikelihood(mu_sensory=1.05, **SCHED), x, pl, v)
    d_b, p_b = _ks(draws[:, 2].double().numpy(), vv_b, cdf_b)
    print(f"KS against the quadrature posterior: D={d:.4f} p={p:.3g}; pinning moves the CDF by {moved:.4f} "
          f"(critical {crit:.4f}); against mu_sensory x 1.05: D={d_b:.4f} p={p_b:.3g}; posterior of v in "
          f"[{lo:.3f}, {hi:.3f}]")
    assert p > 1e-3
    assert p_b < 1e-6


def test_run_sbc_completes_under_the_grid():
    """run_sbc with the grid likelihood under a prior whose every draw gives the simulated sessions a non-zero
    likelihood: a0, lam, B and t_nd pinned (t_nd within a fraction of a step of the true one) and small gains
    (v ~ LogNormal(log 0.1, 0.2)), so that no trial is absorbed within the few steps that the +-6 sigma truncation
    would make impossible for a smaller gain.  -> ranks and finite draws for every dataset."""
    from sbi_for_diffusion_models_b200 import mnle
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    lik = _lik()
    cfg = RunConfig(NUM_TRIALS_OBS=20, WARMUP_STEPS=3)
    out = mnle.run_sbc(cfg, prior_theta=_e2e_prior(math.log(0.1), 0.2), density_estimator=lik.GridLikelihood(),
                       num_datasets=2,
                       posterior_samples_per_dataset=128, chains_per_dataset=128, seed=4, save=False)
    assert out["ranks"].shape == (2, 5)
    for d in range(2):
        s = out["all_samples"][d]
        assert s.shape == (128, 5) and bool(torch.isfinite(s).all())
        assert abs(float(s[:, 3].mean()) - PIN[3][0]) < 0.01


# ---- refusals --------------------------------------------------------------------------------------------------

def test_drivers_refuse_what_the_grid_cannot_score():
    from sbi_for_diffusion_models_b200 import mnle
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    lik = _lik()
    prior = build_prior_theta()
    cfg = RunConfig()
    with pytest.raises(ValueError, match="schedule"):
        mnle.run_sbc(cfg, prior_theta=prior, density_estimator=lik.GridLikelihood(mu_sensory=1.05), num_datasets=1,
                     save=False)
    with pytest.raises(ValueError, match="schedule"):
        mnle.run_sbc(cfg, prior_theta=prior, density_estimator=lik.GridLikelihood(t_max=4.0), num_datasets=1,
                     save=False)
    with pytest.raises(ValueError, match="LOG_RT_MANUALLY"):
        mnle.run_sbc(replace(cfg, LOG_RT_MANUALLY=True), prior_theta=prior, density_estimator=lik.GridLikelihood(),
                     num_datasets=1, save=False)
    _, x, pl = _case(1, 1, 3, seed=1)
    with pytest.raises(TypeError, match="grid"):
        mnle.run_inference_sessions(cfg, prior, lik.GridLikelihood(), [(x[0], pl[0])])
