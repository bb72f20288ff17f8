"""CPU: the row-by-row gradient specification (oracle/mnle_grad_spec.py) and its checks.

The planes add up to autograd's gradient, the margins see the kinks, and the checks that tests/test_gpu_mnle_grad_rows.py
applies to the kernels -- with the same bounds -- accept the fp32 CPU spec's gradient and reject it once it is
mutated the way a wrong kernel would be: a (net, column half) plane dropped, theta columns swapped, a trial missing
from or doubled in a chain's sum, a chain's gradient in another chain's place, a gradient tensor off by 1 %, the last
row of a minibatch or a 64-row chunk of one layer's rows dropped.  Whether the bounds the older tests apply accept the
same mutations is printed next to each verdict."""
import math

import numpy as np
import pytest
import torch

from oracle import ddm_oracle as orc
from oracle import mnle_grad_spec as gs
from oracle import mnle_spec as ms


def _trained():
    from sbi_for_diffusion_models_b200.mnle_net import unpack_params
    import os
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mnle_trained.npz"))
    p = {k: v.clone() for k, v in unpack_params(torch.from_numpy(d["packed"].copy()), int(d["n_choices"])).items()}
    p["cond_mean"], p["cond_std"] = torch.zeros(85), torch.ones(85)
    return p


def _net(kind):
    return _trained() if kind == "trained" else ms.init_params(0, n_choices=int(kind[len("init-K"):]) if "-K" in kind else 3)


def _trials(T, K, seed=0):
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(seed + 5)), 0, T, 80, 0.75))
    rs = np.random.RandomState(seed)
    x = torch.from_numpy(np.stack([np.exp(rs.uniform(-3, 2.1, T)), rs.randint(0, K, T)], 1).astype(np.float32))
    return x, pulses


def test_forward_restates_the_spec():
    for kind in ("init", "init-K8", "trained"):
        p = ms.cast_params(_net(kind), torch.float64)
        x, pulses = _trials(300, int(p["cat.Wo"].shape[0]), 1)
        cond = torch.cat([orc.prior_sample(300, seed=3), pulses], 1)
        x[:3, 0] = torch.tensor([1e-6, 1e4, 8.0])
        assert torch.equal(gs.log_prob(p, x, cond), ms.log_prob(p, x, cond)), kind


@pytest.mark.parametrize("kind", ["init", "init-K2", "trained"])
def test_planes_add_up_to_the_autograd_gradient(kind):
    p = ms.cast_params(_net(kind), torch.float64)
    x, pulses = _trials(3, int(p["cat.Wo"].shape[0]))
    theta = orc.prior_sample(40, seed=9)
    lp, planes = gs.theta_grad_by_plane(p, theta, x, pulses)
    assert tuple(planes.shape) == (3, 40, gs.N_PLANES, 5)
    assert torch.allclose(lp.sum(0), ms.loglik_sum(p, theta, x, pulses), rtol=1e-12, atol=0)
    th = theta.double().requires_grad_(True)
    (want,) = torch.autograd.grad(ms.loglik_sum(p, th, x, pulses).sum(), th)
    assert float((planes.sum((0, 2)) - want).abs().max()) <= 1e-12 * float(want.abs().max())
    # row by row: trial 1 alone
    th = theta.double().requires_grad_(True)
    (want1,) = torch.autograd.grad(ms.loglik_sum(p, th, x[1:2], pulses[1:2]).sum(), th)
    assert float((planes[1].sum(1) - want1).abs().max()) <= 1e-12 * float(want1.abs().max())
    # each plane is what its net contributes: the categorical net alone (planes 0, 1) through the choice term
    th = theta.double().requires_grad_(True)
    xr, cond = ms.potential_rows(th, x, pulses)
    zt = (cond - p["cond_mean"]) / p["cond_std"]
    h = torch.sigmoid(zt @ p["cat.W0"].T + p["cat.b0"])
    h = torch.sigmoid(torch.sigmoid(h @ p["cat.W1"].T + p["cat.b1"]) @ p["cat.W2"].T + p["cat.b2"])
    lpc = torch.log_softmax(h @ p["cat.Wo"].T + p["cat.bo"], -1).gather(1, xr[:, 1:].long())[:, 0]
    (want_cat,) = torch.autograd.grad(lpc.sum(), th)
    assert float((planes[:, :, :2].sum((0, 2)) - want_cat).abs().max()) <= 1e-10 * float(want_cat.abs().max())


def test_margins_see_the_kinks():
    p = ms.init_params(0)
    x, pulses = _trials(6, 3, 2)
    cond = torch.cat([orc.prior_sample(6, seed=4), pulses], 1)
    m = gs.kink_margins(p, x, cond)
    assert all(float(v.min()) > 0 for v in m.values())
    f = gs._forward(ms.cast_params(p, torch.float64), x.double(), cond.double())
    # row 0 on the fifth interior knot of transform 0, row 1 (in float64 rt) on the upper tail bound
    K = ms.NUM_BINS
    w = ms.MIN_BIN + (1 - ms.MIN_BIN * K) * torch.softmax(f["q"][0][0, :K] / math.sqrt(ms.HIDDEN), -1)
    knot = float(2 * ms.TAIL_BOUND * w[:5].sum() - ms.TAIL_BOUND)
    mu, sg = float(p["flow.mu_y"]), float(p["flow.sigma_y"])
    x[0, 0] = float(np.exp(mu + sg * knot))
    x[1, 0] = float(np.exp(mu + sg * ms.TAIL_BOUND))
    m = gs.kink_margins(p, x, cond)
    assert float(m["knot"][0]) < 1e-6 and float(m["tail"][1]) < 1e-6
    assert not bool(gs.kept_rows(m, gs.DELTA)[:2].any())
    # a categorical head that puts all mass on choice 0: choice 1 sits on the probability clamp
    p["cat.bo"] = torch.tensor([40.0, -40.0, -40.0])
    x[2, 1] = 1.0
    m = gs.kink_margins(p, x, cond)
    assert float(m["prob"][2]) <= 2.0 and not bool(gs.kept_rows(m, gs.DELTA)[2])
    kinds = gs.kink_kind(m, gs.DELTA)
    assert all((kinds[r] == "") == bool(gs.kept_rows(m, gs.DELTA)[r]) for r in range(6))


def _old_chain_bound(g, ref):
    """What test_potential_gradient_matches_autograd_of_the_spec accepts of a reverse-mode gradient (chain sums)."""
    e = (g.double() - ref).abs() / (ref.abs() + 1e-2 * ref.abs().max())
    return float(e.median()) < 5e-3 and float(e.mean()) < 5e-2 and float(e.max()) < 5.0


@pytest.fixture(scope="module", params=["init", "trained"])
def rows(request):
    """fp32 CPU spec (the stand-in for a kernel) and float64 planes of 6 trials x 256 thetas, with tail trials."""
    p32 = _net(request.param)
    x, pulses = _trials(6, 3, 3)
    x[4, 0], x[5, 0] = 1e-6, 1e4
    theta = orc.prior_sample(256, seed=12)
    lp64, pl64 = gs.theta_grad_by_plane(ms.cast_params(p32, torch.float64), theta, x, pulses)
    lp32, pl32 = gs.theta_grad_by_plane(p32, theta, x, pulses)
    xr, cond = ms.potential_rows(theta, x, pulses)
    kept = gs.kept_rows(gs.kink_margins(p32, xr, cond), gs.DELTA)
    return request.param, pl32.double().reshape(-1, gs.N_PLANES, 5), pl64.reshape(-1, gs.N_PLANES, 5), kept, (6, 256)


def _row_mutations(pl):
    """(name, per-row gradient) of a wrong kernel, from the fp32 spec's planes (R, 22, 5)."""
    out = []
    g = pl.clone()
    g[:, 0:2, 4] = 0                                 # net 0 (categorical) adds nothing to theta column 4
    out.append(("net 0 without theta column 4", g.sum(1)))
    g = pl.clone()
    g[:, 2 * 10 + 1] = 0                             # flow.9's units 64-127
    out.append(("flow.9 units 64-127 dropped", g.sum(1)))
    g = pl.clone()
    g[:, 2:4, 3], g[:, 2:4, 4] = pl[:, 2:4, 4], pl[:, 2:4, 3]   # flow.0 reads theta columns 3 and 4 swapped
    out.append(("flow.0 theta columns 3 and 4 swapped", g.sum(1)))
    return out


@pytest.mark.parametrize("kernel", ["tc", "simt"])
def test_row_check_rejects_wrong_planes(rows, kernel):
    kind, pl32, pl64, kept, (T, C) = rows
    g64, g32 = pl64.sum(1), pl32.sum(1)
    bounds = gs.ROW_BOUNDS[(kind, kernel, "grad")]
    ok, st = gs.check_rows(g32, g64, g32, kept, **bounds)
    assert ok, st
    for name, g in _row_mutations(pl32):
        ok, st = gs.check_rows(g, g64, g32, kept, **bounds)
        old = _old_chain_bound(g.reshape(T, C, 5).sum(0), g64.reshape(T, C, 5).sum(0))
        print(f"\n{kind} {kernel} {name}: over k x floor by {st['over_max']:.3g} (max) {st['over_mean']:.3g} (mean) -> "
              f"{'accepted' if ok else 'rejected'}; the older chain-sum bound {'accepts' if old else 'rejects'} it")
        assert not ok, (name, st)


def test_sum_check_rejects_wrong_trial_and_chain_sums():
    """A chain's value and gradient against its trials' (fp32 spec as the kernel: T = 50 x C = 130)."""
    p32 = ms.init_params(0)
    T, C = 50, 130
    x, pulses = _trials(T, 3, 4)
    theta = orc.prior_sample(C, seed=6)
    lp, pl = gs.theta_grad_by_plane(p32, theta, x, pulses)
    lp64, pl64 = gs.theta_grad_by_plane(ms.cast_params(p32, torch.float64), theta, x, pulses)
    gv = torch.cat([lp[..., None], pl.sum(2)], -1)       # (T, C, 6): value and gradient of every row
    ref = torch.cat([lp64.sum(0)[:, None], pl64.sum((0, 2))], -1)
    total = _fp32_trial_sum(gv)
    ok, e = gs.check_sum(total, list(gv), tol=gs.SUM_TOL)
    assert ok, e
    bad = []
    t = total.clone(); t[5] -= gv[17, 5]
    bad.append(("trial 17 missing from chain 5", t))
    t = total.clone(); t[5] += gv[17, 5]
    bad.append(("trial 17 doubled in chain 5", t))
    t = total.clone(); t[127] = t[128]
    bad.append(("chain 127 given chain 128's sum", t))
    for name, t in bad:
        ok, e = gs.check_sum(t, list(gv), tol=gs.SUM_TOL)
        print(f"\n{name}: {e:.3g} of the parts' L1 -> {'accepted' if ok else 'rejected'}; the older chain-sum bound "
              f"{'accepts' if _old_chain_bound(t[:, 1:], ref[:, 1:]) else 'rejects'} the gradient")
        assert not ok, (name, e)


def _fp32_trial_sum(parts):
    acc = torch.zeros_like(parts[0])
    for q in parts:
        acc = acc + q
    return acc


@pytest.fixture(scope="module")
def train():
    """R = 300 kink-free rows of a default-init net; the fp32 spec's gradient stands in for the kernel's."""
    p = ms.init_params(1)
    x, pulses = _trials(900, 3, 7)
    cond = torch.cat([orc.prior_sample(900, seed=8), pulses], 1)
    kept = gs.kept_rows(gs.kink_margins(p, x, cond), gs.DELTA)
    x, cond = x[kept][:300].contiguous(), cond[kept][:300].contiguous()
    assert x.shape[0] == 300
    return p, x, cond


def _old_train_bound(got, want):
    """test_loss_and_gradient_match_float64_autograd, forward="tc": every tensor within 1e-2 of its largest entry."""
    return all(float((got[k].double() - w).abs().max()) <= 1e-2 * float(w.abs().max()) + 1e-9 for k, w in want.items())


def test_training_checks_reject_a_wrong_gradient(train):
    p, x, cond = train
    R = x.shape[0]
    _, want = gs.nll_grads(ms.cast_params(p, torch.float64), x, cond)
    _, got = gs.nll_grads(p, x, cond)
    ok, errs = gs.check_named(got, want, tol=gs.TRAIN_TOL)
    assert ok, max(errs.values())

    def pieces(rows_of):
        return [{k: v.double() * (b - a) for k, v in gs.nll_grads(p, x[a:b], cond[a:b])[1].items()} for a, b in rows_of]

    splits = [(a, b) for a, b in zip([0, 1, 63, 64, 127, 129], [1, 63, 64, 127, 129, R])]
    parts = pieces(splits)

    def split_error(g):
        return max(gs.sum_error(g[k].double() * R, [q[k] for q in parts], gs.TRAIN_SUM_FLOOR) for k in g)

    assert split_error(got) <= gs.TRAIN_SUM_TOL, split_error(got)
    scaled = dict(got, **{"flow.9.b2": got["flow.9.b2"] * 1.01})
    no_last = gs.nll_grads(p, x, cond, rows=torch.arange(R) < R - 1)[1]
    chunk = gs.nll_grads(p, x, cond, rows=(torch.arange(R) < 64) | (torch.arange(R) >= 128))[1]
    no_chunk = dict(got, **{"flow.3.W2": chunk["flow.3.W2"]})
    for name, g in (("flow.9.b2 x 1.01", scaled), ("last row dropped", no_last),
                    ("rows 64-127 dropped from flow.3.W2", no_chunk)):
        ok, errs = gs.check_named(g, want, tol=gs.TRAIN_TOL)
        e_split = split_error(g)
        print(f"\n{name}: float64 check {'accepts' if ok else 'rejects'} (worst {max(errs.values()):.3g}), row-split check "
              f"{'accepts' if e_split <= gs.TRAIN_SUM_TOL else 'rejects'} ({e_split:.3g}); the older 1e-2-of-max bound "
              f"{'accepts' if _old_train_bound(g, want) else 'rejects'} it")
        assert not (ok and e_split <= gs.TRAIN_SUM_TOL), name
    # each wrong gradient is caught by the check meant for it
    assert not gs.check_named(scaled, want, tol=gs.TRAIN_TOL)[0]
    assert split_error(no_last) > gs.TRAIN_SUM_TOL and split_error(no_chunk) > gs.TRAIN_SUM_TOL
