"""The one-chain slice-sampler reference (oracle/slice_spec.py) against closed forms, and the elementwise torch
implementation of samplers.VectorizedSliceSampler on the CPU against the reference, bit for bit in float32."""
import math

import numpy as np
import pytest
import torch
from scipy import stats

from oracle.slice_spec import (INF, SeededUniforms, bits, box, gauss, gauss_nan, slice_chain, spike, staircase,
                               trunc_exp)
from sbi_for_diffusion_models_b200.samplers import VectorizedSliceSampler

def cpu_log(N, c):
    """torch.log as the CPU sampler applies it to chain c of N: vectorised lanes and the scalar tail of ATen's CPU
    loop may round differently, so the value is taken at the chain's own position."""
    return lambda u: np.float32(torch.log(torch.full((N,), float(u)))[c].item())


def check_against_reference(target, init, *, seed=0, override=None, runs=1, warmup=2, S=3, thin=1, max_step_out=8,
                            max_shrink=64, init_width=0.1, chain_groups=1, width=None):
    N, D = init.shape
    src = SeededUniforms(seed, N, override)
    s = VectorizedSliceSampler(lambda x: target(x, torch), torch.from_numpy(init), init_width=init_width,
                               max_step_out=max_step_out, max_shrink=max_shrink, chain_groups=chain_groups,
                               uniforms=lambda k: torch.from_numpy(src.draw(k)))
    if width is not None:
        s.width[:] = width
    log_prob = lambda v: target(v[None, :], np)[0]
    for _ in range(runs):
        x0, w0, lp0, it0, ev0 = s.x.numpy().copy(), s.width.numpy().copy(), s.lp.numpy().copy(), s._it, s.n_evals
        out = s.run(S, warmup=warmup, thin=thin).numpy()
        most = 0
        for c in range(N):
            r = slice_chain(log_prob, x0[c], w0[c], src.chain(c), it0=it0, lp=lp0[c], max_step_out=max_step_out,
                            max_shrink=max_shrink, warmup=warmup, S=S, thin=thin, log_fn=cpu_log(N, c))
            assert np.array_equal(bits(out[:, c]), bits(r["draws"])), c
            assert np.array_equal(bits(s.x[c].numpy()), bits(r["x"])), c
            assert bits(s.lp[c].numpy()) == bits(r["lp"]), c
            assert np.array_equal(bits(s.width[c].numpy()), bits(r["width"])), c
            assert np.array_equal(s.tuned[c].numpy(), r["tuned"]) and int(s.sweeps[c]) == r["sweeps"], c
            most = max(most, r["evals"])
        # one evaluation per iteration; the host looks for unfinished chains every 16 iterations
        assert most <= s.n_evals - ev0 <= most + 15
    return s


def _start(N, D, seed, lo=-1.0, hi=0.5):
    return np.random.default_rng(seed).uniform(lo, hi, (N, D)).astype(np.float32)


def _set(j, value):
    """override: uniform j of every iteration (0 shrink, 1 slice level, 2 bracket offset, 3 step-out split) := value"""
    def f(k, u):
        if k % 4 == j:
            u[:] = value
    return f


CASES = {
    "gauss_d3_m8": dict(target=gauss, D=3, warmup=3, S=4),
    "gauss_d2_m1": dict(target=gauss, D=2, max_step_out=1, warmup=2, S=3, thin=2),
    "gauss_d2_m2": dict(target=gauss, D=2, max_step_out=2),
    "gauss_J0": dict(target=gauss, D=2, override=_set(3, 2.0 ** -25)),
    "gauss_Jmax": dict(target=gauss, D=2, override=_set(3, 1.0 - 2.0 ** -25)),
    "box_limit_both_sides": dict(target=box, D=2, override=_set(1, 2.0 ** -25)),
    "spike_give_up": dict(target=spike, D=1, start=0.1, width=1.0, max_shrink=2, warmup=2, S=3),
    "edge_start": dict(target=trunc_exp, D=2, start=0.0, warmup=1),
    "nan_region": dict(target=gauss_nan, D=2, warmup=2),
    "staircase_d5": dict(target=staircase, D=5, warmup=1, S=2),
    "thin3": dict(target=gauss, D=2, warmup=1, S=3, thin=3),
    "groups4": dict(target=gauss, D=2, chain_groups=4),
    "warmup0_tiny_width": dict(target=gauss, D=2, start=0.0, init_width=1e-4, warmup=0, S=2),
    "two_runs": dict(target=gauss, D=2, runs=2, warmup=2, S=2),
    "d65_torch": dict(target=staircase, D=65, warmup=0, S=1),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_torch_path_on_the_cpu_replays_the_reference_bit_for_bit(name):
    case = dict(CASES[name])
    target, D = case.pop("target"), case.pop("D")
    N = 24 if D > 5 else 40
    start = case.pop("start", None)
    init = _start(N, D, seed=len(name)) if start is None else np.full((N, D), start, np.float32)
    if start is not None and target is trunc_exp:
        init[:, 1] = _start(N, 1, seed=3)[:, 0]
    s = check_against_reference(target, init, seed=11, **case)
    if case.get("warmup", 2) == 0:
        assert torch.equal(s.tuned, torch.zeros_like(s.tuned))


def test_widths_below_the_tuning_floor_are_left_alone_without_tuning():
    """warmup = 0 tunes nothing, so no width may move -- not even up to the 1e-6 floor a tuned width is held to."""
    init = torch.zeros((4, 2))
    s = VectorizedSliceSampler(lambda x: gauss(x, torch), init, init_width=1e-4,
                               uniforms=lambda k: torch.from_numpy(SeededUniforms(5, 4).draw(k)))
    w0 = s.width.clone()
    assert float(w0.max()) < 1e-6
    s.run(1, warmup=0)
    assert torch.equal(s.width, w0)


def test_more_than_64_coordinates_run_the_torch_path():
    init = torch.zeros((2, 65))
    assert not VectorizedSliceSampler(lambda x: gauss(x, torch), init)._fused
    with pytest.raises(ValueError, match="fused"):
        VectorizedSliceSampler(lambda x: gauss(x, torch), init, fused=True)


# ---------------------------------------------------------------------------------------------------------------------
# the reference's own laws (float64, one chain at a time)

def _chains(log_prob, starts, width, seed, **kw):
    rng = np.random.default_rng(seed)
    return [slice_chain(log_prob, s, width, lambda k: rng.random(4), dtype=np.float64, **kw) for s in starts]


def test_reference_leaves_a_truncated_exponential_invariant():
    """Started at exact draws of exp(-x) on (0, 3), two sweeps with a fixed width must keep the law exactly."""
    n = 20000
    Z = 1.0 - math.exp(-3.0)
    u = np.random.default_rng(1).random(n)
    starts = -np.log1p(-u * Z)[:, None]
    log_prob = lambda v: -v[0] if 0.0 < v[0] < 3.0 else -INF
    runs = _chains(log_prob, starts, [0.7], seed=2, warmup=0, S=1, thin=2)
    x = np.array([r["draws"][0, 0] for r in runs])
    p = stats.kstest(x, lambda t: (1.0 - np.exp(-np.clip(t, 0, 3))) / Z).pvalue
    assert p > 1e-3, p
    assert not np.array_equal(x, starts[:, 0])                     # the chains moved
    # power: the same statistic on the start scaled by 1.05 rejects
    assert stats.kstest(starts[:, 0] * 1.05, lambda t: (1.0 - np.exp(-np.clip(t, 0, 3))) / Z).pvalue < 1e-3


def test_reference_is_uniform_in_rank_for_a_known_posterior():
    """The conjugate model of test_sampler_prior: theta ~ N(0,1), x | theta ~ N(theta, 1), one chain per dataset
    started at 0 with width tuning; the rank of theta_true among each chain's thinned draws must be uniform."""
    g = np.random.default_rng(5)
    n_data, n_draws = 400, 31
    theta = g.standard_normal(n_data)
    xs = theta + g.standard_normal(n_data)
    ranks = []
    for i in range(n_data):
        lp = lambda v, xo=xs[i]: -0.5 * v[0] ** 2 - 0.5 * (xo - v[0]) ** 2
        r = _chains(lp, [[0.0]], [1.0], seed=100 + i, warmup=20, S=n_draws, thin=3)[0]
        assert r["tuned"][0] == 20
        ranks.append(int((r["draws"][:, 0] < theta[i]).sum()))
    hist = np.bincount(np.array(ranks) // 4, minlength=8)[:8]
    p = stats.chisquare(hist).pvalue
    assert p > 1e-3, (p, hist)
