"""The MNLE gradient kernels row by row against float64 autograd of the CPU spec away from kinks, and their sums against
single-row calls of the same kernel (oracle/mnle_grad_spec.py).

* Potential gradient (``loglik_sum_and_grad``, kernel "tc" = reverse mode on tcgen05, "simt" = fp32 forward mode):
  calls with T = 1 make every output one (trial, chain) row's value and d/d theta.  Rows clear of every ReLU kink,
  spline knot, tail bound and probability clamp by ``DELTA`` are compared entry by entry with float64
  (``check_rows``: in units of the column's RMS, within k x the fp32 CPU spec's own error plus an absolute term).
* Sums: a call over T trials against the float64 sum of its T single-trial calls.  A row's arithmetic does not depend
  on where it sits, so only fp32 summation may separate them, kinks or not.
* Training step with the tcgen05 forward on minibatches of kink-free rows against float64 autograd, and the gradient of
  R rows against the sum of the gradients of the pieces the minibatch splits into.

The bounds are in ``oracle.mnle_grad_spec`` with the numbers they were set from; ``tests/test_mnle_grad_spec.py``
shows on the CPU that the same checks reject mutated gradients (a dropped plane, swapped columns, a trial missing
from a sum, a tensor off by 1 %, ...)."""
import os

import numpy as np
import pytest
import torch

from oracle import ddm_oracle as orc
from oracle import mnle_grad_spec as gs
from oracle import mnle_spec as ms
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE, unpack_params
from sbi_for_diffusion_models_b200.mnle_train import MNLETrainer

pytestmark = pytest.mark.gpu

TRAINED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mnle_trained.npz")


def _session(T, seed=7):
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(123)), 0, T, 80, 0.75))
    x, _ = orc.sim_rng_c(np.repeat(np.array([[0.45, 0.6, 1.3, 14.0, 0.25]], np.float32), T, 0), pulses.numpy(), seed)
    return torch.from_numpy(x), pulses


def _tail_session(p32, K):
    """Observations in the spline tails and on the tail bound, each with every choice in [0, K) (as in
    tests/test_gpu_mnle.py): rt in {1e-6, 3e-5, 1e-3, 8, 50, 1e4}, the float32 rt nearest to exp(mu_y +- 10 sigma_y)
    and its two neighbours, and u = +-10 +- 1e-6."""
    mu, sg = float(p32["flow.mu_y"]), float(p32["flow.sigma_y"])
    rts = [1e-6, 3e-5, 1e-3, 8.0, 50.0, 1e4]
    for edge in (10.0, -10.0):
        r = np.float32(np.exp(mu + sg * edge))
        rts += [r, np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(0.0))]
        rts += [np.exp(mu + sg * (edge + d)) for d in (1e-6, -1e-6)]
    rt = np.repeat(np.array(rts, np.float32), K)
    choice = np.tile(np.arange(K), len(rts)).astype(np.float32)
    x = torch.from_numpy(np.stack([rt, choice], 1))
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(77)), 0, x.shape[0], 80, 0.75))
    return x, pulses


def _net(kind):
    """(fp32 spec params, estimator): "init", "init-K2", "init-K8" default-init nets, "trained" the committed one."""
    if kind == "trained":
        d = np.load(TRAINED)
        packed = PackedMNLE(d["packed"], int(d["n_choices"]))
        p = {k: v.clone() for k, v in unpack_params(torch.from_numpy(d["packed"].copy()), packed.n_choices).items()}
        p["cond_mean"], p["cond_std"] = torch.zeros(85), torch.ones(85)
        return p, DeviceMNLE(packed)
    p = ms.init_params(0, n_choices=int(kind[len("init-K"):]) if "-K" in kind else 3)
    return p, DeviceMNLE(PackedMNLE.from_params(p))


def _observations(p32, K):
    """Eight observed trials: four of a simulated session (choices folded into [0, K)) and four of the tail session --
    deep in the left tail, far in the right one, the float32 rt nearest to the upper tail bound, and u = -10 + 1e-6."""
    xs, ps = _session(32)
    xs[:, 1] = xs[:, 1] % K
    xt, pt = _tail_session(p32, K)
    pick = [0 * K + 0, 5 * K + K - 1, 6 * K + 1 % K, 14 * K + 0]
    return torch.cat([xs[[3, 11, 19, 27]], xt[pick]]), torch.cat([ps[[3, 11, 19, 27]], pt[pick]])


@pytest.fixture(scope="module", params=["init", "trained", "init-K2", "init-K8"])
def rows_case(request):
    """Everything the row tests compare, computed once per net: 8 trials x 512 prior thetas as eight T = 1 calls per
    kernel, the float64 and fp32 spec's values and gradients of the same 4 096 rows, and their kink margins."""
    kind = request.param
    p32, est = _net(kind)
    K = est.packed.n_choices
    theta = orc.prior_sample(512, seed=51)
    x, pulses = _observations(p32, K)
    lp64, pl64 = gs.theta_grad_by_plane(ms.cast_params(p32, torch.float64), theta, x, pulses)
    lp32, pl32 = gs.theta_grad_by_plane(p32, theta, x, pulses)
    xr, cond = ms.potential_rows(theta, x, pulses)
    got = {}
    for kernel in ("tc", "simt"):
        vg = [est.loglik_sum_and_grad(theta, x[t:t + 1], pulses[t:t + 1], kernel=kernel) for t in range(x.shape[0])]
        got[kernel] = (torch.stack([v for v, _ in vg]).reshape(-1, 1), torch.stack([g for _, g in vg]).reshape(-1, 5))
    return dict(kind=kind, got=got, margins=gs.kink_margins(p32, xr, cond),
                ref=(lp64.reshape(-1, 1), pl64.sum(2).reshape(-1, 5)), floor=(lp32.reshape(-1, 1), pl32.sum(2).reshape(-1, 5)))


@pytest.mark.parametrize("kernel", ["tc", "simt"])
def test_potential_gradient_rows_match_float64_away_from_kinks(rows_case, kernel):
    kind, m = rows_case["kind"], rows_case["margins"]
    kept = gs.kept_rows(m, gs.DELTA)
    labels = np.array(gs.kink_kind(m, gs.DELTA))
    (v, g), (v64, g64), (v32, g32) = rows_case["got"][kernel], rows_case["ref"], rows_case["floor"]
    ok_v, st_v = gs.check_rows(v, v64, v32, kept, **gs.ROW_BOUNDS[(kind, kernel, "value")])
    ok_g, st_g = gs.check_rows(g, g64, g32, kept, **gs.ROW_BOUNDS[(kind, kernel, "grad")])
    # worst error of the excluded rows, by the kind of kink that excluded them (same units as the kept rows')
    scale = g64.double()[kept].pow(2).mean(0).sqrt()
    e_all = ((g.double() - g64.double()).abs() / scale).max(dim=1).values
    worst = {k: float(e_all[torch.from_numpy(labels == k)].max()) for k in gs.KINDS if (labels == k).any()}
    print(f"\n{kind} {kernel}: kept {float(kept.float().mean()):.3f} of {kept.numel()} rows "
          f"(excluded by {', '.join(f'{k} {int((labels == k).sum())}' for k in gs.KINDS)}); kept rows: value {st_v}, "
          f"gradient {st_g}; worst gradient error of the excluded rows by kink: {worst}")
    assert float(kept.float().mean()) >= 0.5
    assert ok_v, st_v
    assert ok_g, st_g
    # the excluded rows still meet the bounds the chain sums had before (tests/test_gpu_mnle.py), entry by entry
    # relative to |ref| + 1e-2 max |ref|
    out = ~kept
    e = ((g - g64).double().abs() / (g64.double().abs() + 1e-2 * g64.double().abs().max(dim=0).values))[out]
    assert float(e.median()) < 5e-3 and float(e.mean()) < 5e-2 and float(e.max()) < 5.0, \
        (float(e.median()), float(e.mean()), float(e.max()))


def _seq_sum_f32(parts):
    """The fp32 sum 0 + parts[0] + parts[1] + ... in this order (the trial loops of the tc kernels)."""
    acc = torch.zeros_like(parts[0])
    for q in parts:
        acc = acc + q
    return acc


@pytest.fixture(scope="module", params=["init", "trained"])
def sum_net(request):
    return _net(request.param)


@pytest.mark.parametrize("T,C", [(50, 1024), (7, 1), (23, 130), (65, 7), (3, 300), (50, 129)])
def test_potential_sums_equal_single_trial_calls(sum_net, T, C):
    """configs[3] = 400 row tiles (two-tile and one-tile CTAs), chain blocks of 128 with ragged ends, r = t*C + c."""
    p32, est = sum_net
    theta = orc.prior_sample(C, seed=T + C)
    x, pulses = _session(T)
    x[:, 1] = x[:, 1] % est.packed.n_choices
    one = [(x[t:t + 1], pulses[t:t + 1]) for t in range(T)]
    for kernel in ("tc", "simt"):
        v, g = est.loglik_sum_and_grad(theta, x, pulses, kernel=kernel)
        vg = [est.loglik_sum_and_grad(theta, xo, po, kernel=kernel) for xo, po in one]
        ok_v, e_v = gs.check_sum(v, [a for a, _ in vg], tol=gs.SUM_TOL)
        ok_g, e_g = gs.check_sum(g, [b for _, b in vg], tol=gs.SUM_TOL)
        print(f"\nT={T} C={C} {kernel}: value {e_v:.3g}, gradient {e_g:.3g} of the parts' L1")
        assert ok_v and ok_g, (kernel, e_v, e_g)
        if kernel == "tc":
            # potential_grad_final_kernel adds the trials' log-probabilities in trial order: same rows, same bits
            assert torch.equal(v, _seq_sum_f32([a for a, _ in vg])), kernel
    # the forward-only tcgen05 path hoists the pulses' part of the first layers per trial, so a row's arithmetic does not
    # depend on T either, and its last tile adds the trials in order
    f = est.loglik_sum(theta, x, pulses, kernel="tc")
    parts = [est.loglik_sum(theta, xo, po, kernel="tc") for xo, po in one]
    ok, e = gs.check_sum(f, parts, tol=gs.SUM_TOL)
    assert ok, e
    assert torch.equal(f, _seq_sum_f32(parts))


# ---- training step -------------------------------------------------------------------------------------------------

def _data(R, seed, K=3):
    theta = orc.prior_sample(R, seed=seed + 2)
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(seed + 1)), 0, R, 80, 0.75))
    cond = torch.cat([theta, pulses], dim=1)
    rs = np.random.RandomState(seed)
    x = torch.from_numpy(np.stack([np.exp(rs.uniform(-3, 2.1, R)), rs.randint(0, K, R)], 1).astype(np.float32))
    x[:5, 0] = torch.tensor([1e-6, 8.0, 7.999999, 1e-3, 3e-5])      # linear tails of the spline
    return x, cond


def _trainer(p):
    return MNLETrainer(int(p["cat.Wo"].shape[0]), cond_mean=p["cond_mean"], cond_std=p["cond_std"],
                       mu_y=float(p["flow.mu_y"]), sigma_y=float(p["flow.sigma_y"]), init=p)


@pytest.fixture(scope="module", params=[3, 2, 8], ids=["K3", "K2", "K8"])
def train_pool(request):
    """A pool of rows clear of every kink under the net's own parameters."""
    K = request.param
    p = ms.init_params(1) if K == 3 else ms.init_params(20 + K, n_choices=K)
    N = 20000 if K == 3 else 1000
    x, cond = _data(N, K, K)
    m = gs.kink_margins(p, x, cond)
    kept = gs.kept_rows(m, gs.DELTA)
    print(f"\nK={K}: {float(kept.float().mean()):.3f} of {N} pool rows clear of the kinks")
    return K, p, x[kept].contiguous(), cond[kept].contiguous(), x, cond


def _sizes(K):
    return (300, 4096, 64 * 130 + 5) if K == 3 else (333,)


def test_training_gradient_on_kink_free_rows_matches_float64(train_pool):
    K, p, x, cond, _, _ = train_pool
    tr = _trainer(p)
    for R in _sizes(K):
        assert x.shape[0] >= R
        want_loss, want = gs.nll_grads(ms.cast_params(p, torch.float64), x[:R], cond[:R])
        stats = tr.nll(x[:R].cuda(), tr.standardise(cond[:R]), forward="tc").cpu()
        got = tr.named_grads()
        ok, errs = gs.check_named(got, want, tol=gs.TRAIN_TOL)
        worst = max(errs, key=errs.get)
        e_loss = abs(float(stats[0]) - want_loss) / abs(want_loss)
        print(f"\nK={K} R={R}: loss {e_loss:.3g} relative; worst tensor {worst} {errs[worst]:.3g} of its largest entry, "
              f"median tensor {float(np.median(list(errs.values()))):.3g}")
        assert e_loss <= gs.TRAIN_LOSS_TOL, e_loss
        assert ok, {k: v for k, v in errs.items() if v > gs.TRAIN_TOL}


def _splits(R):
    cuts = sorted({c for c in (1, 63, 64, 127, 129, R - 257) if 0 < c < R})
    return list(zip([0] + cuts, cuts + [R]))


def test_training_gradient_of_a_minibatch_is_the_sum_over_its_pieces(train_pool):
    """R g_R = sum_k R_k g_(R_k) for pieces of 1, 62, 1, 63, 2, ... rows: row splits of the weight gradients, 64-row
    chunks, ragged tails and train_reduce_kernel, with the rows read in place and gathered through an index vector."""
    K, p, _, _, x_all, cond_all = train_pool
    tr = _trainer(p)
    xd, cd = x_all.cuda(), tr.standardise(cond_all)
    perm = torch.randperm(x_all.shape[0], generator=torch.Generator().manual_seed(K)).cuda()

    def run(a, b, gathered):
        if gathered:
            s = tr.nll(xd, cd, perm[a:b].contiguous(), forward="tc")
        else:
            s = tr.nll(xd[a:b].contiguous(), cd[a:b].contiguous(), forward="tc")
        return float(s[0]) * (b - a), {k: v.double() * (b - a) for k, v in tr.named_grads().items()}

    for R in _sizes(K):
        for gathered in (False, True):
            loss, total = run(0, R, gathered)
            pieces = [run(a, b, gathered) for a, b in _splits(R)]
            worst = max((gs.sum_error(total[k], [q[k] for _, q in pieces], gs.TRAIN_SUM_FLOOR), k)
                        for k in total if k not in ("flow.mu_y", "flow.sigma_y"))
            e_loss = gs.sum_error(torch.tensor([loss]), [torch.tensor([l]) for l, _ in pieces])
            print(f"\nK={K} R={R} {'index' if gathered else 'in place'}: loss {e_loss:.3g}, worst tensor {worst[1]} "
                  f"{worst[0]:.3g} of the parts' L1")
            assert e_loss <= gs.TRAIN_SUM_TOL and worst[0] <= gs.TRAIN_SUM_TOL, (e_loss, worst)
