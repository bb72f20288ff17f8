"""The device slice sampler (csrc/mnle_sampler.cu with and without CUDA-graph replay, and the torch implementation
on CUDA and on the CPU) against the one-chain reference oracle/slice_spec.py, bit for bit, branch by branch; and its
draws against exact laws, from chains started at stationarity."""
import math

import numpy as np
import pytest
import torch
from scipy import stats
from scipy.special import ndtr

from oracle.slice_spec import (INF, SeededUniforms, bits, box, gauss, gauss_nan, slice_chain, spike, staircase,
                               trunc_exp)
from sbi_for_diffusion_models_b200.samplers import PhiloxUniforms, VectorizedSliceSampler

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")

# (fused, use_graph, device)
PATHS = ((True, True, "cuda"), (True, False, "cuda"), (False, False, "cuda"))


def cuda_log(u):
    return np.float32(torch.log(torch.tensor([float(u)], device=DEV)).item())


def cpu_log(N, c):     # ATen's vectorised lanes and scalar tail may round differently: take chain c's own lane
    return lambda u: np.float32(torch.log(torch.full((N,), float(u)))[c].item())


def chain_subset(N, n=64, seed=0):
    """~n chains: 0, N-1, the last (partial) 256-block's first and last chains, and a seeded sample of the rest."""
    if N <= n:
        return np.arange(N)
    tail = np.arange(256 * ((N - 1) // 256), N)
    pick = {0, N - 1, *tail[:8].tolist(), *tail[-8:].tolist()}
    rest = np.random.default_rng(seed).choice(N, n, replace=False)
    for c in rest.tolist():
        if len(pick) >= n:
            break
        pick.add(c)
    return np.array(sorted(pick))


class Recorded:
    """A device uniform source whose draws the reference replays: keeps the values of the chain subset."""

    def __init__(self, fn, chains):
        self.fn, self.idx, self.rec = fn, torch.as_tensor(chains, device=DEV), {}

    def __call__(self, k):
        u = self.fn(k)
        self.rec[k] = u[self.idx].cpu().numpy()
        return u

    def chain(self, i):
        def get(k):
            if k not in self.rec:
                self(k)
            return self.rec[k][i]
        return lambda it: [get(4 * it + j) for j in range(4)]


def replay(target, init, *, seed=11, override=None, philox=False, paths=PATHS, runs=1, warmup=2, S=3, thin=1,
           max_step_out=8, max_shrink=64, init_width=0.1, chain_groups=1, width=None):
    """Run every path on all N chains with the same uniforms; require each chain of the subset to give the bits of
    the reference: draws, final x / lp, widths, tuning counts, sweeps; and the global evaluation count."""
    N, D = init.shape
    chains = chain_subset(N)
    src = SeededUniforms(seed, N, override)
    log_prob = lambda v: target(v[None, :], np)[0]
    refs = {}
    samplers = []
    for fused, graph, dev in paths:
        if philox:
            ufn = Recorded(PhiloxUniforms(seed, 0, N, DEV), chains)
            uni = [ufn.chain(i) for i in range(len(chains))]
        else:
            ufn = lambda k, dev=dev: torch.from_numpy(src.draw(k)).to(dev)
            uni = [src.chain(c) for c in chains]
        s = VectorizedSliceSampler(lambda x: target(x, torch), init.to(dev), init_width=init_width,
                                   max_step_out=max_step_out, max_shrink=max_shrink, chain_groups=chain_groups,
                                   uniforms=ufn, fused=fused, use_graph=graph)
        assert fused is None or s._fused == fused
        if width is not None:
            s.width[:] = width
        for r in range(runs):
            x0, w0, lp0 = (t[chains].cpu().numpy() for t in (s.x, s.width, s.lp))
            it0, ev0 = s._it, s.n_evals
            out = s.run(S, warmup=warmup, thin=thin)[:, chains].cpu().numpy()
            key = (dev, r)
            if key not in refs:
                refs[key] = [slice_chain(log_prob, x0[i], w0[i], uni[i], it0=it0, lp=lp0[i], max_step_out=max_step_out,
                                         max_shrink=max_shrink, warmup=warmup, S=S, thin=thin,
                                         log_fn=cuda_log if dev == "cuda" else cpu_log(N, c))
                             for i, c in enumerate(chains)]
            x, lp, w, tuned, sweeps = (t[chains].cpu().numpy() for t in (s.x, s.lp, s.width, s.tuned, s.sweeps))
            tag = (fused, graph, dev, r)
            most = 0
            for i, (c, ref) in enumerate(zip(chains, refs[key])):
                assert np.array_equal(bits(out[:, i]), bits(ref["draws"])), (tag, c)
                assert np.array_equal(bits(x[i]), bits(ref["x"])), (tag, c)
                assert bits(lp[i]) == bits(ref["lp"]), (tag, c)
                assert np.array_equal(bits(w[i]), bits(ref["width"])), (tag, c)
                assert np.array_equal(tuned[i], ref["tuned"]) and sweeps[i] == ref["sweeps"], (tag, c)
                most = max(most, ref["evals"])
            # one evaluation per iteration, finished chains looked for every 16 iterations; with a subset of the
            # chains only the lower bound is known
            assert most <= s.n_evals - ev0, tag
            if len(chains) == N:
                assert s.n_evals - ev0 <= most + 15, tag
        samplers.append(s)
    return samplers


def _start(N, D, seed, lo=-1.0, hi=0.5):
    return torch.from_numpy(np.random.default_rng(seed).uniform(lo, hi, (N, D)).astype(np.float32))


def _set(j, value):
    """override: uniform j of every iteration (0 shrink, 1 slice level, 2 bracket offset, 3 step-out split) := value"""
    def f(k, u):
        if k % 4 == j:
            u[:] = value
    return f


CASES = {
    "m1": dict(target=gauss, D=3, max_step_out=1, warmup=2, S=3, thin=2),
    "m2": dict(target=gauss, D=3, max_step_out=2),
    "m8": dict(target=gauss, D=3, warmup=3, S=4, cpu=True),
    "J0": dict(target=gauss, D=2, override=_set(3, 2.0 ** -25)),
    "Jmax": dict(target=gauss, D=2, override=_set(3, 1.0 - 2.0 ** -25)),
    "box_limit_both_sides": dict(target=box, D=2, override=_set(1, 2.0 ** -25), cpu=True),
    "spike_shrink1": dict(target=spike, D=1, start=0.1, width=1.0, max_shrink=1, warmup=2, S=3),
    "spike_shrink2": dict(target=spike, D=1, start=0.1, width=1.0, max_shrink=2, warmup=2, S=3, cpu=True),
    "spike_shrink3": dict(target=spike, D=1, start=0.1, width=1.0, max_shrink=3, warmup=3, S=2, thin=2),
    "edge_start": dict(target=trunc_exp, D=2, start=0.0, warmup=1),
    "nan_region": dict(target=gauss_nan, D=2, warmup=2, cpu=True),
    "d1": dict(target=gauss, D=1, warmup=3, S=3),
    "d5_staircase": dict(target=staircase, D=5, warmup=1, S=2),
    "d64_staircase": dict(target=staircase, D=64, warmup=1, S=1),
    "warmup0_tiny_width": dict(target=gauss, D=2, start=0.0, init_width=1e-4, warmup=0, S=2, cpu=True),
    "thin3_uneven_finish": dict(target=gauss, D=2, warmup=1, S=3, thin=3),
    "groups4": dict(target=gauss, D=2, N=256, chain_groups=4),
    "two_runs": dict(target=gauss, D=2, runs=2, warmup=2, S=2, cpu=True),
    "n1": dict(target=gauss, D=2, N=1, warmup=2, S=3),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_sampler_replays_the_one_chain_reference_bit_for_bit(name):
    case = dict(CASES[name])
    target, D, N = case.pop("target"), case.pop("D"), case.pop("N", 257)
    start = case.pop("start", None)
    paths = PATHS + (((False, False, "cpu"),) if case.pop("cpu", False) else ())
    init = _start(N, D, seed=len(name)) if start is None else torch.full((N, D), float(start))
    if start is not None and target is trunc_exp:
        init[:, 1] = _start(N, 1, seed=3)[:, 0]
    samplers = replay(target, init, paths=paths, **case)
    s = samplers[0]
    if case.get("warmup", 2) == 0:
        assert torch.equal(s.tuned, torch.zeros_like(s.tuned))
    else:
        assert bool((s.tuned == case.get("warmup", 2)).all())         # every update of a warm-up sweep tunes, no other
    if case.get("chain_groups", 1) > 1:                           # one starting width per group
        w0 = VectorizedSliceSampler(lambda x: target(x, torch), init.to(DEV), chain_groups=4).width
        g = w0.view(4, -1, D)
        assert torch.equal(g, g[:, :1].expand_as(g)) and not torch.equal(g[0], g[1])


def test_device_sampler_replays_the_reference_on_a_million_chains():
    """2^20 chains with Philox uniforms, as production draws them; the reference replays a subset."""
    init = _start(1 << 20, 2, seed=9)
    replay(gauss, init, philox=True, paths=PATHS[:1] + PATHS[2:], warmup=1, S=2)


def test_more_than_64_coordinates_fall_back_to_torch_and_refuse_the_kernels():
    init = _start(257, 65, seed=4).to(DEV)
    s = VectorizedSliceSampler(lambda x: staircase(x, torch), init)
    assert not s._fused
    assert VectorizedSliceSampler(lambda x: staircase(x, torch), init[:, :64])._fused
    with pytest.raises(ValueError, match="fused"):
        VectorizedSliceSampler(lambda x: staircase(x, torch), init, fused=True)
    replay(staircase, init.cpu(), paths=((None, False, "cuda"),), warmup=0, S=1)


# ---------------------------------------------------------------------------------------------------------------------
# exact laws.  With fixed widths (warmup = 0) a slice-sampler transition leaves the target invariant for any width and
# step-out limit, so N independent chains started at exact draws must still follow the target after a few sweeps:
# one draw per chain, Philox uniforms, fused kernels.

N_LAW = 1 << 16
P_MIN = 1e-3
Z_EXP = 1.0 - math.exp(-3.0)
STAIR_EDGES = np.arange(-3.0, 3.01, 0.5)
STAIR_MASS = np.exp(-np.floor(2.0 * np.abs(0.5 * (STAIR_EDGES[:-1] + STAIR_EDGES[1:]))))
W_MIX, MU_MIX, SD_MIX = (0.3, 0.7), (-4.0, 4.0), 0.5


def _exp_lp(x):
    return torch.where((x[:, 0] > 0) & (x[:, 0] < 3), -x[:, 0], torch.full_like(x[:, 0], -INF))


def _exp_cdf(t):
    return (1.0 - np.exp(-np.clip(t, 0.0, 3.0))) / Z_EXP


def _exp_draw(rng, n):
    return -np.log1p(-rng.random(n) * Z_EXP)


def _stair_lp(x):
    return staircase(x, torch)


def _stair_cdf(t, mass=STAIR_MASS):
    return np.interp(t, STAIR_EDGES, np.concatenate([[0.0], np.cumsum(mass) / mass.sum()]))


def _stair_draw(rng, n, mass=STAIR_MASS):
    k = rng.choice(len(mass), n, p=mass / mass.sum())
    return STAIR_EDGES[k] + 0.5 * rng.random(n)


def _mix_lp(x):
    a = math.log(W_MIX[0]) - 0.5 * ((x[:, 0] - MU_MIX[0]) / SD_MIX) ** 2
    b = math.log(W_MIX[1]) - 0.5 * ((x[:, 0] - MU_MIX[1]) / SD_MIX) ** 2
    return torch.logaddexp(a, b)


def _mix_cdf(t):
    return W_MIX[0] * ndtr((t - MU_MIX[0]) / SD_MIX) + W_MIX[1] * ndtr((t - MU_MIX[1]) / SD_MIX)


def _mix_draw(rng, n):
    comp = rng.random(n) < W_MIX[0]
    return np.where(comp, MU_MIX[0], MU_MIX[1]) + SD_MIX * rng.standard_normal(n)


LAWS = {"exp": (_exp_lp, _exp_cdf, _exp_draw, 1.0), "stair": (_stair_lp, _stair_cdf, _stair_draw, 0.5),
        "mix": (_mix_lp, _mix_cdf, _mix_draw, SD_MIX)}


def _sample(lp, start, width, *, max_step_out=8, sweeps=3, seed=0, warmup=0):
    init = torch.as_tensor(start, dtype=torch.float32, device=DEV).reshape(len(start), -1).contiguous()
    s = VectorizedSliceSampler(lp, init, max_step_out=max_step_out, uniforms=PhiloxUniforms(seed, 0, len(start), DEV),
                               fused=True)
    if width is not None:
        s.width[:] = width
    return s.run(1, warmup=warmup, thin=sweeps)[0].double().cpu().numpy()


@pytest.mark.parametrize("law,scale,m", [("exp", 1.0, 8), ("stair", 1.0, 8), ("mix", 1.0, 8), ("exp", 1e-2, 8),
                                         ("exp", 100.0, 8), ("stair", 1e-2, 1), ("mix", 100.0, 1), ("stair", 100.0, 1)])
def test_transition_leaves_the_target_invariant(law, scale, m):
    lp, cdf, draw, unit = LAWS[law]
    start = draw(np.random.default_rng(1), N_LAW)
    x = _sample(lp, start, scale * unit, max_step_out=m, seed=2)[:, 0]
    moved = float(np.mean(x != start.astype(np.float32)))
    res = stats.kstest(x, cdf)
    print(f"{law} width {scale}x m={m}: KS D = {res.statistic:.5f}, p = {res.pvalue:.3g}, moved {moved:.3f}")
    assert res.pvalue > P_MIN, (res.statistic, res.pvalue)
    assert moved > 0.3


def test_law_statistics_reject_a_wrong_law_at_the_same_size():
    """The KS statistic of the invariance tests, at the same N, rejects the exact start scaled by 1.05 (zero sweeps)
    and the staircase with one step's mass moved to its neighbour."""
    rng = np.random.default_rng(1)
    p_scaled = stats.kstest(1.05 * _exp_draw(rng, N_LAW), _exp_cdf).pvalue
    moved = STAIR_MASS.copy()
    moved[7], moved[8] = 0.0, moved[8] + moved[7]              # [0.5, 1) -> [1, 1.5)
    p_step = stats.kstest(_stair_draw(rng, N_LAW, moved), _stair_cdf).pvalue
    print(f"power: scaled start p = {p_scaled:.3g}, moved step p = {p_step:.3g}")
    assert p_scaled < P_MIN and p_step < P_MIN


MEAN3 = np.array([0.5, -1.0, 2.0])
COV3 = np.array([[1.0, 0.6, 0.0], [0.6, 2.0, 0.3], [0.0, 0.3, 0.5]])


def test_truncated_correlated_gaussian_stays_exact():
    """The 3-D target of test_gpu_inference (correlated Gaussian truncated to x_2 > 0): KS on each marginal and
    the correlations of the truncated law."""
    mean, prec = torch.tensor(MEAN3, dtype=torch.float32, device=DEV), torch.linalg.inv(
        torch.tensor(COV3, dtype=torch.float32, device=DEV))

    def lp(x):
        d = x - mean
        v = -0.5 * torch.einsum("ni,ij,nj->n", d, prec, d)
        return torch.where(x[:, 2] > 0, v, torch.full_like(v, -INF))

    rng = np.random.default_rng(6)
    z = rng.multivariate_normal(MEAN3, COV3, 2 * N_LAW)
    z = z[z[:, 2] > 0][:N_LAW]
    x = _sample(lp, z, torch.tensor([0.5, 0.7, 0.3], device=DEV), seed=7)
    # x_2 | x_2 > 0 is a truncated normal; x_0 is independent of x_2 (cov 0): N(0.5, 1); x_1 | x_2 is normal
    s2 = math.sqrt(COV3[2, 2])
    a = -MEAN3[2] / s2
    Za = 1.0 - ndtr(a)
    cdf2 = lambda t: (ndtr((np.maximum(t, 0.0) - MEAN3[2]) / s2) - ndtr(a)) / Za
    cdf0 = lambda t: ndtr(t - MEAN3[0])
    g = np.linspace(0.0, MEAN3[2] + 12 * s2, 2001)
    wq = np.exp(-0.5 * ((g - MEAN3[2]) / s2) ** 2)
    wq /= wq.sum()
    b, sc = COV3[1, 2] / COV3[2, 2], math.sqrt(COV3[1, 1] - COV3[1, 2] ** 2 / COV3[2, 2])
    cdf1 = lambda t: (ndtr((np.asarray(t)[:, None] - (MEAN3[1] + b * (g[None, :] - MEAN3[2]))) / sc) * wq).sum(1)
    grid = np.linspace(x[:, 1].min() - 1e-6, x[:, 1].max() + 1e-6, 2001)
    tab = cdf1(grid)
    for j, cdf in enumerate((cdf0, lambda t: np.interp(t, grid, tab), cdf2)):
        res = stats.kstest(x[:, j], cdf)
        print(f"x_{j}: KS D = {res.statistic:.5f}, p = {res.pvalue:.3g}")
        assert res.pvalue > P_MIN, (j, res.statistic, res.pvalue)
    lam = math.exp(-0.5 * a * a) / math.sqrt(2 * math.pi) / Za
    var2 = COV3[2, 2] * (1 + a * lam - lam * lam)
    beta = COV3[:, 2] / COV3[2, 2]
    cov = COV3 - np.outer(COV3[:, 2], COV3[:, 2]) / COV3[2, 2] + np.outer(beta, beta) * var2
    cov[2, :2] = cov[:2, 2] = beta[:2] * var2
    cov[2, 2] = var2
    want = cov / np.sqrt(np.outer(np.diag(cov), np.diag(cov)))
    got = np.corrcoef(x.T)
    print("correlation error", np.abs(got - want).max())
    assert np.abs(got - want).max() < 0.02, (got, want)


def test_production_shaped_run_converges_to_the_exact_law():
    """Every chain starts at the same point; default warm-up (100 sweeps) and width tuning, then one draw per chain:
    KS against N(0.5, 0.25^2)."""
    mu, sd = 0.5, 0.25
    lp = lambda x: -0.5 * ((x[:, 0] - mu) / sd) ** 2
    x = _sample(lp, np.full(N_LAW, 1.0), None, warmup=100, sweeps=1, seed=8)[:, 0]
    res = stats.kstest(x, lambda t: ndtr((t - mu) / sd))
    print(f"converged: KS D = {res.statistic:.5f}, p = {res.pvalue:.3g}")
    assert res.pvalue > P_MIN, (res.statistic, res.pvalue)
