"""``DeviceMNLE.sample`` (``mnle_sample_tc_f32``) against the float64 CPU specification, on the default-init net and on
the trained net of ``tests/golden/mnle_trained.npz``.

With injected draws the spec sees the same (u_choice, n) as the kernel, so the two are compared row by row: the choice
must agree except where u_choice sits within 1e-4 of a boundary of the spec's CDF, and log rt must be in the class of
the ``tc`` log_prob kernel (tensor-core networks, fp64 spline chain).  With native Philox draws the law is checked:
choice counts by chi^2 against the spec's softmax, and per choice the spec's forward flow must map the sampled rt back
to N(0,1) (KS)."""
import os

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import ddm_oracle as orc
from oracle import mnle_sample_spec as mss
from oracle import mnle_spec as ms
from sbi_for_diffusion_models_b200.mnle import posterior_predictive
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE, unpack_params

pytestmark = pytest.mark.gpu

TRAINED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mnle_trained.npz")


def trained_net():
    d = np.load(TRAINED)
    packed, K = d["packed"], int(d["n_choices"])
    p = {k: v.clone() for k, v in unpack_params(torch.from_numpy(packed.copy()), K).items()}
    p["cond_mean"], p["cond_std"] = torch.zeros(85), torch.ones(85)
    return p, PackedMNLE(packed, K)


def _make_net(kind):
    """(fp32 spec params, float64 spec params, estimator, kind); "init-K<k>" is a default-init net with k choices."""
    if kind == "trained":
        p, packed = trained_net()
        return p, ms.cast_params(p, torch.float64), DeviceMNLE(packed), kind
    p = ms.init_params(0) if kind == "init" else ms.init_params(0, n_choices=int(kind[len("init-K"):]))
    return p, ms.cast_params(p, torch.float64), DeviceMNLE(PackedMNLE.from_params(p)), kind


# K = 3 (the reference's choices: left, right, censored) on both nets, and default-init nets with 1, 2, 5 and 8 choices
@pytest.fixture(scope="module", params=["init", "trained", "init-K1", "init-K2", "init-K5", "init-K8"])
def net(request):
    return _make_net(request.param)


@pytest.fixture(scope="module", params=["init", "trained"])
def net3(request):
    return _make_net(request.param)


def _conditions(B, seed=2):
    theta = orc.prior_sample(B, seed=seed)
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(seed + 1)), 0, B, 80, 0.75))
    return torch.cat([theta, pulses], dim=1)


def _draws(R, seed):
    rng = np.random.default_rng(seed)
    uc = ((rng.integers(0, 2**32, R) + 0.5) * 2.0**-32).astype(np.float32)
    n = rng.standard_normal(R).astype(np.float32)
    return torch.from_numpy(np.stack([uc, n], 1))


def _cuda(p):
    return {k: v.cuda() for k, v in p.items()}


def check_against_spec(got, rows, uc, n, p32, p64, kind, what=""):
    """Kernel samples got (R,2) of condition rows (R,85) under injected draws (uc, n) against the float64 spec, row by
    row: the choice equal except where uc lies within 1e-4 of a boundary of the spec's CDF, and log rt in the class of
    the tensor-core log_prob kernel (init nets: every row within 2e-3; trained net: mean error within 4x of the fp32
    CPU spec's on the same rows and draws; median below 1e-4 on both)."""
    got = got.reshape(-1, 2).double().cpu()
    cd = rows.double().cuda()                         # the float64 spec runs on the GPU with torch: same arithmetic
    uc, n = uc.double().cuda(), n.double().cuda()
    p64c = _cuda(p64)
    want = mss.sample(p64c, cd, uc, n).cpu()
    cdf = torch.cumsum(torch.softmax(mss.choice_logits(p64c, cd), dim=-1), dim=-1).cpu()
    near = ((uc.cpu()[:, None] - cdf[:, :-1]).abs() < 1e-4).any(dim=1)
    differ = got[:, 1] != want[:, 1]
    assert not bool((differ & ~near).any()), int((differ & ~near).sum())
    same = ~differ
    dy = (torch.log(got[same, 0]) - torch.log(want[same, 0])).abs()
    print(f"\n{kind} {what}: choice differs on {int(differ.sum())} of {got.shape[0]} rows ({int(near.sum())} near a boundary); "
          f"|d log rt| max {float(dy.max()):.3g} mean {float(dy.mean()):.3g} median {float(dy.median()):.3g}")
    assert float(dy.median()) <= 1e-4, float(dy.median())
    if kind != "trained":
        assert float(dy.max()) <= 2e-3, float(dy.max())
    else:   # no further from float64 than the fp32 CPU spec on the same rows and draws
        w32 = mss.sample(_cuda(p32), cd.float(), uc, n).cpu().double()
        both = same & (w32[:, 1] == want[:, 1])
        floor = (torch.log(w32[both, 0]) - torch.log(want[both, 0])).abs()
        dyb = (torch.log(got[both, 0]) - torch.log(want[both, 0])).abs()
        print(f"fp32 spec: mean {float(floor.mean()):.3g} max {float(floor.max()):.3g}")
        assert float(dyb.mean()) <= 4.0 * float(floor.mean()), (float(dyb.mean()), float(floor.mean()))
    assert bool((got[:, 0] > 0).all() and torch.isfinite(got).all())


@pytest.mark.parametrize("B,S", [(1000, 3), (12800, 4)])
def test_injected_draws_match_the_float64_spec(net, B, S):
    p32, p64, est, kind = net
    cond = _conditions(B)
    draws = _draws(B * S, seed=B + S)
    got = est.sample((S,), condition=cond, draws=draws)
    assert tuple(got.shape) == (S, B, 2) and got.device.type == "cpu"
    rows = cond.repeat(S, 1)                          # row s*B + b holds condition b
    check_against_spec(got, rows, draws[:, 0], draws[:, 1], p32, p64, kind, f"B={B} S={S}")


def test_native_draws_are_reproducible_and_split_invariant(net, monkeypatch):
    _, _, est, _ = net
    cond = _conditions(300, seed=4).cuda()
    a = est.sample((7,), condition=cond, seed=1234)
    assert a.is_cuda and tuple(a.shape) == (7, 300, 2)
    assert torch.equal(a, est.sample((7,), condition=cond, seed=1234))
    assert not torch.equal(a, est.sample((7,), condition=cond, seed=1235))
    # S split over calls with matching sample offsets: 600 rows per call -> samples [0, 2), [2, 4), [4, 6), [6, 7)
    monkeypatch.setattr(est, "SAMPLE_MAX_ROWS", 600)
    assert torch.equal(a, est.sample((7,), condition=cond, seed=1234))
    monkeypatch.undo()
    # sample s of condition b does not depend on how many conditions the call has (ragged last tiles)
    for r in (1, 127, 129):
        assert torch.equal(est.sample((7,), condition=cond[:r], seed=1234), a[:, :r])
    # seed=None draws the key from torch's global generator
    torch.manual_seed(5)
    b = est.sample((2,), condition=cond, seed=None)
    torch.manual_seed(5)
    assert torch.equal(b, est.sample((2,), condition=cond, seed=None))
    # CPU condition in, CPU out, (*sample_shape, B, 2)
    c = est.sample((2, 3), condition=cond[:5].cpu(), seed=9)
    assert c.device.type == "cpu" and tuple(c.shape) == (2, 3, 5, 2)
    assert torch.equal(c.reshape(6, 5, 2), est.sample((6,), condition=cond[:5], seed=9).cpu())
    assert tuple(est.sample(condition=cond[:5].cpu(), seed=9).shape) == (5, 2)
    assert set(torch.unique(a[..., 1]).tolist()) <= set(float(k) for k in range(est.packed.n_choices))


def test_native_draws_have_the_estimators_law(net):
    """2^20 samples of four conditions (2^18 on the nets with other numbers of choices): per condition the choice
    counts by chi^2 against the float64 spec's softmax, and per (condition, choice) the spec's forward flow maps log rt
    to N(0,1) (KS); alpha = 1e-3 with Bonferroni."""
    _, p64, est, kind = net
    B, S = 4, (2**18 if kind in ("init", "trained") else 2**16)
    cond = _conditions(B, seed=8).cuda()
    x = est.sample((S,), condition=cond, seed=77).reshape(-1, 2)
    p64c = {k: v.cuda() for k, v in p64.items()}
    rows = cond.double().repeat(S, 1)
    z = mss.flow_forward(p64c, x.double(), rows).cpu().numpy()
    probs = torch.softmax(mss.choice_logits(p64c, cond.double()), dim=-1).cpu().numpy()
    xc = x[:, 1].long().cpu().numpy().reshape(S, B)
    z = z.reshape(S, B)
    n_tests = B * (1 + probs.shape[1])
    for b in range(B):
        counts = np.bincount(xc[:, b], minlength=probs.shape[1])
        keep = probs[b] * S >= 5                    # chi^2 over the categories with enough expected counts
        exp_ = probs[b][keep] * S
        obs = counts[keep]
        assert counts[~keep].sum() <= max(5.0, 3 * probs[b][~keep].sum() * S + 5), (b, counts, probs[b] * S)
        if keep.sum() > 1:                          # (one choice category: nothing to test beyond the line above)
            pv = stats.chisquare(obs, exp_ * obs.sum() / exp_.sum()).pvalue
            assert pv > 1e-3 / n_tests, (kind, b, counts, probs[b] * S, pv)
        for c in range(probs.shape[1]):
            zc = z[xc[:, b] == c, b]
            if zc.size < 100:
                continue
            pv = stats.kstest(zc, "norm").pvalue
            assert pv > 1e-3 / n_tests, (kind, b, c, zc.size, pv)


def test_posterior_predictive_is_one_sample_call(net):
    _, _, est, _ = net
    C, T = 6, 50
    theta = orc.prior_sample(C, seed=3).cuda()
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(3)), 0, T, 80, 0.75)).cuda()
    x = posterior_predictive(est, theta, pulses, seed=21)
    assert tuple(x.shape) == (C, T, 2) and x.is_cuda
    rows = torch.cat([theta.repeat_interleave(T, 0), pulses.repeat(C, 1)], dim=1)   # row c*T + t
    assert torch.equal(x, est.sample((), condition=rows, seed=21).reshape(C, T, 2))


# ---- sampler edges under injected draws, on the K = 3 nets ----------------------------------------------------------

def _rt_of_u(p32, u):
    """float32(exp(float64(mu_y) + float64(sigma_y) * u)) with the packed fp32 mu_y, sigma_y: the rt of a base value u
    that no spline moves."""
    mu, sg = float(p32["flow.mu_y"]), float(p32["flow.sigma_y"])
    return np.exp(mu + sg * np.asarray(u, np.float64)).astype(np.float32)


def test_identity_tails_and_edge_bins_are_exact(net3):
    """n outside [-10, 10]: every inverse spline is the identity, so rt = exp(mu_y + sigma_y n) to 1 fp32 ulp.  n = +-10
    exactly lies inside: in the last bin d1 = 1 makes the discriminant h^2 and the root 1, in the first bin the constant
    term is 0 and so is the root, so every spline maps +-10 to itself and rt is again exp(mu_y +- 10 sigma_y).  n =
    +-9.9999 and 0 go through the splines and are compared with the float64 spec like any other row; the choices of
    all rows too."""
    p32, p64, est, kind = net3
    B = 512
    cond = _conditions(B, seed=12)
    exact = [10.0001, -10.0001, 10.5, -10.5, 25.0, -25.0, -60.0, 10.0, -10.0]
    ns = np.array(exact + [9.9999, -9.9999, 0.0], np.float32)
    S, E = len(ns), len(exact) * B
    rng = np.random.default_rng(5)
    uc = ((rng.integers(0, 2**32, S * B) + 0.5) * 2.0**-32).astype(np.float32)
    n = np.repeat(ns, B)                                         # row s*B + b: n = ns[s]
    draws = torch.from_numpy(np.stack([uc, n], 1))
    got = est.sample((S,), condition=cond, draws=draws).reshape(-1, 2)
    rows = cond.repeat(S, 1)
    want = _rt_of_u(p32, n[:E])
    ulps = np.abs(got[:E, 0].numpy().astype(np.float64) - want) / np.spacing(want).astype(np.float64)
    print(f"\n{kind}: tails and edge bins: at most {ulps.max():.3g} fp32 ulp from exp(mu_y + sigma_y n)")   # measured: 0
    assert ulps.max() <= 1.0, (np.unique(n[:E][ulps > 1.0]), ulps.max())
    check_against_spec(got[:E], rows[:E], draws[:E, 0], draws[:E, 1], p32, p64, kind, "tails (choices)")
    check_against_spec(got[E:], rows[E:], draws[E:, 0], draws[E:, 1], p32, p64, kind, "n = +-9.9999, 0")


def test_every_sample_maps_back_to_its_normal(net3):
    """50 000 rows of N(0,1) draws: the spec's forward flow, in float64, on the kernel's (rt, choice) gives back the
    injected n on every row.  No row is excused: where the kernel's choice differs from the spec's next to a CDF
    boundary, the flow is the one of the kernel's choice and must still invert."""
    p32, p64, est, kind = net3
    B, S = 12500, 4
    cond = _conditions(B, seed=13)
    draws = _draws(B * S, seed=14)
    got = est.sample((S,), condition=cond, draws=draws).reshape(-1, 2).double().cuda()
    rows = cond.repeat(S, 1).double().cuda()
    p64c = _cuda(p64)
    n = draws[:, 1].double()
    err = (mss.flow_forward(p64c, got, rows).cpu() - n).abs()
    print(f"\n{kind}: round trip |z - n| max {float(err.max()):.3g} mean {float(err.mean()):.3g}")
    # measured on a B200: init net max 5.3e-5, mean 5.0e-6; trained net max 1.9e-3, mean 6.6e-5 against the fp32 spec's
    # round trip max 3.8e-2, mean 8.4e-4
    if kind != "trained":
        assert float(err.max()) <= 2e-4, float(err.max())
    else:   # the float32 spec's own samples, mapped back the same way, set the floor
        x32 = mss.sample(_cuda(p32), rows.float(), draws[:, 0].cuda(), draws[:, 1].cuda()).double()
        floor = (mss.flow_forward(p64c, x32, rows).cpu() - n).abs()
        print(f"fp32 spec round trip: max {float(floor.max()):.3g} mean {float(floor.mean()):.3g}")
        assert float(err.mean()) <= 4.0 * float(floor.mean()), (float(err.mean()), float(floor.mean()))
        assert float(err.max()) <= 4.0 * float(floor.max()), (float(err.max()), float(floor.max()))


def test_choice_at_the_ends_of_the_unit_interval(net3):
    """u_c = 2^-33 (the smallest native draw), 1e-30 and 1 - 2^-24 (the largest float32 below 1) pick the spec's
    class; u_c = 1 exactly, which injected draws can reach, takes the documented fallback K - 1."""
    p32, p64, est, kind = net3
    K, B = est.packed.n_choices, 256
    cond = _conditions(B, seed=15)
    ucs = np.array([2.0**-33, 1e-30, 1.0 - 2.0**-24, 1.0], np.float32)
    n = np.random.default_rng(16).standard_normal(len(ucs) * B).astype(np.float32)
    draws = torch.from_numpy(np.stack([np.repeat(ucs, B), n], 1))
    got = est.sample((len(ucs),), condition=cond, draws=draws).reshape(-1, 2)
    logits = mss.choice_logits(_cuda(p64), cond.double().cuda()).repeat(len(ucs), 1)
    want = mss.choice_from_uniform(logits, draws[:, 0].cuda()).cpu()
    assert torch.equal(got[:, 1].long(), want), [int((got[s * B:(s + 1) * B, 1].long() != want[s * B:(s + 1) * B]).sum())
                                                 for s in range(len(ucs))]
    assert bool((got[-B:, 1] == K - 1).all())


@pytest.mark.parametrize("shift", [(-24.0, -12.0, 0.0), (0.0, -12.0, -24.0)], ids=["rising", "falling"])
def test_choice_next_to_the_boundaries_of_a_peaked_categorical(net3, shift):
    """cat.bo shifted so that the class probabilities span ~1e-11 .. 1.  u_c at F_j (1 +- 1e-2) and 1 - (1 - F_j)
    (1 +- 1e-2) for every boundary F_j of the spec's float64 CDF, rounded to float32, picks exactly the spec's class:
    these points are far outside the tensor-core logit error in relative terms, so no row is excused.  Native draws
    never produce a class of probability below 1e-9."""
    p32, _, _, kind = net3
    p = dict(p32)
    p["cat.bo"] = p32["cat.bo"] + torch.tensor(shift, dtype=torch.float32)
    p64 = ms.cast_params(p, torch.float64)
    est = DeviceMNLE(PackedMNLE.from_params(p))
    B = 512
    cond = _conditions(B, seed=19)
    p64c = _cuda(p64)
    probs = torch.softmax(mss.choice_logits(p64c, cond.double().cuda()), dim=-1).cpu()
    F = torch.cumsum(probs, dim=-1)[:, :-1]                        # (B, K-1) boundaries
    pts = torch.stack([F * (1 - 1e-2), F * (1 + 1e-2), 1 - (1 - F) * (1 - 1e-2), 1 - (1 - F) * (1 + 1e-2)], -1)
    b_idx = torch.arange(B)[:, None, None].expand_as(pts).reshape(-1)
    u = pts.reshape(-1).float().double()                          # rounded to float32
    # keep the points in (0, 1] whose rounding left them at least 2e-3 (relative) from every boundary of their row
    Fb = F[b_idx]
    margin = ((u[:, None] - Fb).abs() / torch.minimum(Fb, 1 - Fb)).min(dim=1).values
    keep = (u > 0) & (u <= 1) & (margin >= 2e-3)
    u, b_idx = u[keep], b_idx[keep]
    # measured on a B200: 2921 .. 3177 points per (net, shift), the least margin 2.3e-3, every choice equal
    print(f"\n{kind} {shift}: class probabilities {float(probs.min()):.2g} .. {float(probs.max()):.2g}; {int(keep.sum())} "
          f"points, least margin {float(margin[keep].min()):.3g}")
    assert float(probs.min()) < 1e-9 and int(keep.sum()) >= 4 * B
    rows = cond[b_idx]
    n = torch.from_numpy(np.random.default_rng(20).standard_normal(u.shape[0]).astype(np.float32))
    got = est.sample((), condition=rows, draws=torch.stack([u.float(), n], 1))
    want = mss.choice_from_uniform(mss.choice_logits(p64c, rows.double().cuda()), u.cuda()).cpu()
    bad = got[:, 1].long() != want
    assert not bool(bad.any()), (int(bad.sum()), u[bad][:8].tolist(), want[bad][:8].tolist())
    # native draws: u_c >= 2^-33 and <= 1 - 2^-33 never reach a class of probability below 1e-9
    S = 2048
    x = est.sample((S,), condition=cond.cuda(), seed=31).reshape(S, B, 2)
    c = x[..., 1].long().cpu()
    pc = probs.gather(1, c.t()).t()
    assert float(pc.min()) >= 1e-9, float(pc.min())


def test_strided_and_broadcast_conditions_give_the_same_bits(net3):
    """The same samples whatever the condition's memory layout: a column view of a wider CUDA matrix (ld_cond > 85 in
    the kernel), non-contiguous CPU matrices, one condition at a time (B = 1, with that condition's injected draws),
    and a broadcast row (row stride 0)."""
    _, _, est, _ = net3
    B, S = 300, 5
    cond = _conditions(B, seed=17)
    draws = _draws(B * S, seed=18)
    want = est.sample((S,), condition=cond.cuda(), draws=draws)
    native = est.sample((S,), condition=cond.cuda(), seed=99)
    views = (torch.cat([cond, torch.randn(B, 11)], 1).cuda()[:, :85],      # CUDA view, row stride 96
             torch.cat([cond, torch.zeros(B, 3)], 1)[:, :85],              # CPU view, row stride 88
             cond.t().contiguous().t())                                     # CPU, column-major
    for c in views:
        assert not c.is_contiguous()
        assert torch.equal(est.sample((S,), condition=c, draws=draws).cuda(), want)
        assert torch.equal(est.sample((S,), condition=c, seed=99).cuda(), native)
    d3 = draws.reshape(S, B, 2)
    for b in (0, 1, 137, B - 1):
        assert torch.equal(est.sample((S,), condition=cond[b:b + 1].cuda(), draws=d3[:, b]), want[:, b:b + 1])
    one = cond.cuda()[7:8]
    assert torch.equal(est.sample((S,), condition=one.expand(B, 85), draws=draws),
                       est.sample((S,), condition=one.repeat(B, 1), draws=draws))
