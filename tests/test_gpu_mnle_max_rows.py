"""The largest calls the C ABI admits, 8e6 rows, on the trained net of ``tests/golden/mnle_trained.npz``.

At 8e6 rows every byte offset into the workspaces is past 2^31 (the expanded condition matrix is 2.7 GB, the context
images 3.1 GB) and the offsets into the spline-parameter block (23 GB) are past 2^32.  A 32-bit product anywhere in
those paths corrupts only the far end of a large call, so rows are checked across the whole range: against the float64
spec, and bit for bit against small calls on the same rows (rows are independent, and the per-chain sums over the
trials run in a fixed order that does not depend on the other chains).

Each test needs one large workspace (sample and tc64 potential ~27 GiB each at 8e6 rows, the reverse-mode gradient
~6.2 KB per row: ~46 GiB at 8e6 rows; it also runs at 4e6 rows, ~23 GiB, where the byte offsets into its buffers are
still past 2^32) and frees it before the next; a test skips, naming the amount, when the device has less free memory
than that."""
import gc
import os

import numpy as np
import pytest
import torch

from oracle import ddm_oracle as orc
from oracle import mnle_sample_spec as mss
from oracle import mnle_spec as ms
from sbi_for_diffusion_models_b200 import _native
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE, unpack_params

pytestmark = pytest.mark.gpu

TRAINED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mnle_trained.npz")
ROWS = 8_000_000          # rows per call admitted by mnle_sample_tc_f32, mnle_loglik_sum_tc64_f32, ..._grad_tc_f32
T, C = 50, 160_000        # a potential call of exactly ROWS rows


@pytest.fixture(scope="module")
def trained():
    d = np.load(TRAINED)
    packed, K = d["packed"], int(d["n_choices"])
    p = {k: v.clone() for k, v in unpack_params(torch.from_numpy(packed.copy()), K).items()}
    p["cond_mean"], p["cond_std"] = torch.zeros(85), torch.ones(85)
    return p, ms.cast_params(p, torch.float64), DeviceMNLE(PackedMNLE(packed, K))


@pytest.fixture(autouse=True)
def release_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _need(ws_floats):
    """Skip unless the device has room for the workspace plus 4 GiB for inputs, outputs and the spec."""
    torch.cuda.empty_cache()
    need = ws_floats * 4 + 4 * 2**30
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _session(T, seed=7):
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(123)), 0, T, 80, 0.75))
    x, _ = orc.sim_rng_c(np.repeat(np.array([[0.45, 0.6, 1.3, 14.0, 0.25]], np.float32), T, 0), pulses.numpy(), seed)
    return torch.from_numpy(x), pulses


def _spread(n, count, seed, extra):
    """count indices spread over [0, n) plus the given ones, sorted and unique."""
    rng = np.random.default_rng(seed)
    return torch.from_numpy(np.unique(np.concatenate([rng.integers(0, n, count), np.asarray(extra)])))


def test_sample_at_the_row_limit(trained, monkeypatch):
    """B = 4000 conditions x S = 2000 samples with injected draws: rows over the whole range (the first tile, past 2^22
    and 6 * 2^20, the last two tiles) against the float64 spec with the bounds of tests/test_gpu_mnle_sample.py; the
    same request split over two calls gives the same bits, and so does a small call on just the checked rows."""
    p32, p64, est = trained
    B, S = 4000, 2000
    R = B * S
    assert R == ROWS
    _need(_native.lib().mnle_sample_tc_workspace_floats(est.packed.n_choices, B, S))
    theta = orc.prior_sample(B, seed=51)
    pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(52)), 0, B, 80, 0.75))
    cond = torch.cat([theta, pulses], dim=1).cuda()
    rng = np.random.default_rng(53)
    uc = ((rng.integers(0, 2**32, R) + 0.5) * 2.0**-32).astype(np.float32)
    draws = torch.from_numpy(np.stack([uc, rng.standard_normal(R).astype(np.float32)], 1)).cuda()
    got = est.sample((S,), condition=cond, draws=draws).reshape(R, 2)
    idx = _spread(R, 4096, 54, [*range(128), *range(2**22 - 64, 2**22 + 64), *range(6 * 2**20 - 64, 6 * 2**20 + 64),
                                *range(R - 256, R)]).cuda()
    g, rows, d = got[idx].double().cpu(), cond[idx % B].double(), draws[idx].double()
    # against the float64 spec: the choice except within 1e-4 of a CDF boundary, log rt by the bounds of the trained net
    p64c = {k: v.cuda() for k, v in p64.items()}
    want = mss.sample(p64c, rows, d[:, 0], d[:, 1]).cpu()
    cdf = torch.cumsum(torch.softmax(mss.choice_logits(p64c, rows), dim=-1), dim=-1).cpu()
    near = ((d[:, 0].cpu()[:, None] - cdf[:, :-1]).abs() < 1e-4).any(dim=1)
    differ = g[:, 1] != want[:, 1]
    assert not bool((differ & ~near).any()), idx[(differ & ~near).cuda()][:8].tolist()
    w32 = mss.sample({k: v.cuda() for k, v in p32.items()}, rows.float(), d[:, 0], d[:, 1]).cpu().double()
    both = ~differ & (w32[:, 1] == want[:, 1])
    dy = (torch.log(g[both, 0]) - torch.log(want[both, 0])).abs()
    floor = (torch.log(w32[both, 0]) - torch.log(want[both, 0])).abs()
    print(f"\n8e6-row sample, {idx.numel()} rows: choice differs on {int(differ.sum())} ({int(near.sum())} near a boundary); "
          f"|d log rt| max {float(dy.max()):.3g} mean {float(dy.mean()):.3g} median {float(dy.median()):.3g}; "
          f"fp32 spec mean {float(floor.mean()):.3g}")
    assert float(dy.median()) <= 1e-4 and float(dy.mean()) <= 4.0 * float(floor.mean()), (float(dy.median()), float(dy.mean()))
    assert bool(torch.isfinite(got).all()) and bool((got[:, 0] > 0).all())
    # rows are independent: a small call on the checked rows alone
    assert torch.equal(est.sample((), condition=cond[idx % B], draws=draws[idx]), got[idx])
    # the same request in two calls of 1000 samples each
    monkeypatch.setattr(est, "SAMPLE_MAX_ROWS", R // 2)
    assert torch.equal(est.sample((S,), condition=cond, draws=draws).reshape(R, 2), got)


def _chains(C=C):
    return _spread(C, 56, 61, range(C - 8, C))


def test_tc64_potential_at_the_row_limit(trained):
    """T = 50 trials x C = 160 000 chains: 64 chains spread over C, the last eight included, have exactly the values
    of a small call on just those chains, and are within the tc64 bound of test_potential_sum_matches_spec of the
    float64 spec."""
    p32, p64, est = trained
    _need(_native.lib().mnle_loglik_tc64_workspace_floats(est.packed.n_choices, T, C))
    theta = orc.prior_sample(C, seed=62)
    x, pulses = _session(T)
    big = est.loglik_sum(theta.cuda(), x.cuda(), pulses.cuda(), kernel="tc64").cpu()
    assert bool(torch.isfinite(big).all())
    ch = _chains()
    small = est.loglik_sum(theta[ch].cuda(), x.cuda(), pulses.cuda(), kernel="tc64").cpu()
    assert torch.equal(big[ch], small), (big[ch] - small).abs().max()
    xr, cond = ms.potential_rows(theta[ch], x, pulses)
    want_rows = ms.log_prob(p64, xr, cond).reshape(T, -1)
    want = want_rows.sum(0)
    e = (big[ch].double() - want).abs() / torch.maximum(want.abs(), want_rows.abs().sum(0) / 10)
    print(f"\n8e6-row tc64 potential: {float(e.max()):.3g} of scale from the float64 spec")
    assert float(e.max()) < 5e-4, float(e.max())


@pytest.mark.parametrize("C", [C, C // 2], ids=["8e6-rows", "4e6-rows"])
def test_reverse_mode_gradient_at_the_row_limit(trained, C):
    """loglik_sum_and_grad(kernel="tc") at T = 50 x C: 64 chains spread over C, the last eight included, have exactly the
    values and gradients of a small call on just those chains (the backward pass is per row, and the sums over trials
    and planes run in a fixed order per chain), and are within the reverse-mode bounds of
    test_potential_gradient_matches_autograd_of_the_spec of the float64 spec and autograd of it."""
    p32, p64, est = trained
    _need(_native.lib().mnle_loglik_grad_tc_workspace_floats(est.packed.n_choices, T, C))
    theta = orc.prior_sample(C, seed=63)
    x, pulses = _session(T)
    val, grad = est.loglik_sum_and_grad(theta.cuda(), x.cuda(), pulses.cuda(), kernel="tc")
    val, grad = val.cpu(), grad.cpu()
    assert bool(torch.isfinite(val).all()) and bool(torch.isfinite(grad).all())
    ch = _chains(C)
    v_s, g_s = est.loglik_sum_and_grad(theta[ch].cuda(), x.cuda(), pulses.cuda(), kernel="tc")
    assert torch.equal(val[ch], v_s.cpu()) and torch.equal(grad[ch], g_s.cpu())
    th64 = theta[ch].double().requires_grad_(True)
    want = ms.loglik_sum(p64, th64, x, pulses)
    (want_grad,) = torch.autograd.grad(want.sum(), th64)
    want = want.detach()
    err_v = (val[ch].double() - want).abs()
    eg = (grad[ch].double() - want_grad).abs() / (want_grad.abs() + 1e-2 * want_grad.abs().max())
    print(f"\n{T * C}-row reverse mode: value {float((err_v / want.abs()).max()):.3g} relative; gradient median "
          f"{float(eg.median()):.3g} mean {float(eg.mean()):.3g} max {float(eg.max()):.3g}")
    assert bool((err_v <= 1e-3 * want.abs() + 2e-2).all())
    assert float(eg.median()) < 5e-3 and float(eg.mean()) < 5e-2 and float(eg.max()) < 5.0
