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


@pytest.fixture(scope="module", params=["init", "trained"])
def net(request):
    if request.param == "init":
        p = ms.init_params(0)
        return p, ms.cast_params(p, torch.float64), DeviceMNLE(PackedMNLE.from_params(p)), "init"
    p, packed = trained_net()
    return p, ms.cast_params(p, torch.float64), DeviceMNLE(packed), "trained"


def _conditions(B, seed=2):
    theta = orc.prior_sample(B, seed=seed)
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(seed + 1)), 0, B, 80, 0.75))
    return torch.cat([theta, pulses], dim=1)


def _draws(R, seed):
    rng = np.random.default_rng(seed)
    uc = ((rng.integers(0, 2**32, R) + 0.5) * 2.0**-32).astype(np.float32)
    n = rng.standard_normal(R).astype(np.float32)
    return torch.from_numpy(np.stack([uc, n], 1))


@pytest.mark.parametrize("B,S", [(1000, 3), (12800, 4)])
def test_injected_draws_match_the_float64_spec(net, B, S):
    p32, p64, est, kind = net
    cond = _conditions(B)
    draws = _draws(B * S, seed=B + S)
    got = est.sample((S,), condition=cond, draws=draws)
    assert tuple(got.shape) == (S, B, 2) and got.device.type == "cpu"
    got = got.reshape(-1, 2).double()
    rows = cond.repeat(S, 1).double()                 # row s*B + b holds condition b
    uc, n = draws[:, 0].double(), draws[:, 1].double()
    cd = rows.cuda()                                  # the float64 spec runs on the GPU with torch: same arithmetic
    p64c = {k: v.cuda() for k, v in p64.items()}
    want = mss.sample(p64c, cd, uc.cuda(), n.cuda()).cpu()
    # choice: equal except within 1e-4 of a CDF boundary of the spec
    cdf = torch.cumsum(torch.softmax(mss.choice_logits(p64c, cd), dim=-1), dim=-1).cpu()
    near = ((uc[:, None] - cdf[:, :-1]).abs() < 1e-4).any(dim=1)
    differ = got[:, 1] != want[:, 1]
    assert not bool((differ & ~near).any()), int((differ & ~near).sum())
    same = ~differ
    dy = (torch.log(got[same, 0]) - torch.log(want[same, 0])).abs()
    print(f"\n{kind} B={B} S={S}: choice differs on {int(differ.sum())} rows ({int(near.sum())} near a boundary); "
          f"|d log rt| max {float(dy.max()):.3g} mean {float(dy.mean()):.3g} median {float(dy.median()):.3g}")
    assert float(dy.median()) <= 1e-4, float(dy.median())
    if kind == "init":
        assert float(dy.max()) <= 2e-3, float(dy.max())
    else:   # no further from float64 than the fp32 CPU spec on the same rows and draws
        p32c = {k: v.cuda() for k, v in p32.items()}
        w32 = mss.sample(p32c, cd.float(), uc.cuda(), n.cuda()).cpu().double()
        both = same & (w32[:, 1] == want[:, 1])
        floor = (torch.log(w32[both, 0]) - torch.log(want[both, 0])).abs()
        dyb = (torch.log(got[both, 0]) - torch.log(want[both, 0])).abs()
        print(f"fp32 spec: mean {float(floor.mean()):.3g} max {float(floor.max()):.3g}")
        assert float(dyb.mean()) <= 4.0 * float(floor.mean()), (float(dyb.mean()), float(floor.mean()))
    assert bool((got[:, 0] > 0).all() and torch.isfinite(got).all())


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
    assert set(torch.unique(a[..., 1]).tolist()) <= {0.0, 1.0, 2.0}


def test_native_draws_have_the_estimators_law(net):
    """2^20 samples of four conditions: per condition the choice counts by chi^2 against the float64 spec's softmax,
    and per (condition, choice) the spec's forward flow maps log rt to N(0,1) (KS); alpha = 1e-3 with Bonferroni."""
    _, p64, est, kind = net
    B, S = 4, 2**18
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
