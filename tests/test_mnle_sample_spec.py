"""The CPU specification of ``estimator.sample`` (``oracle/mnle_sample_spec.py``): the inverse spline pinned against the
nflows-derived VITS spline, its round trip with the forward spline, the law of ``sample`` at one condition, and the
argument checks of ``mnle_sample_tc_f32`` that need no device."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import ddm_oracle as orc
from oracle import mnle_sample_spec as mss
from oracle import mnle_spec as ms
from sbi_for_diffusion_models_b200 import _native
from sbi_for_diffusion_models_b200.build import build_native


def _params(R, scale, dtype, g):
    return (torch.randn(R, 3 * ms.NUM_BINS - 1, generator=g) * scale).to(dtype)


def test_inverse_spline_matches_the_nflows_derived_implementation_shipped_in_transformers():
    vits = pytest.importorskip("transformers.models.vits.modeling_vits")
    ref = vits._unconstrained_rational_quadratic_spline
    K = ms.NUM_BINS
    g = torch.Generator().manual_seed(11)
    for dtype, tol in ((torch.float64, 1e-12), (torch.float32, 2e-6)):
        for scale in (1.0, 30.0, 120.0):      # 120 / sqrt(128) ~ 10: the sharp bins of a trained net
            R = 4000
            q = _params(R, scale, dtype, g)
            y = (torch.rand(R, generator=g) * 24.0 - 12.0).to(dtype)
            y[:8] = torch.tensor([-ms.TAIL_BOUND, ms.TAIL_BOUND, 0.0, -12.0, 12.0, 9.999999, -9.999999, 1e-30], dtype=dtype)
            got_u, got_lad = mss.rqs_inverse(y, q)
            want_u, want_lad = ref(y.clone(), q[:, :K] / math.sqrt(ms.HIDDEN), q[:, K:2 * K] / math.sqrt(ms.HIDDEN),
                                   q[:, 2 * K:].clone(), reverse=True, tail_bound=ms.TAIL_BOUND, min_bin_width=ms.MIN_BIN,
                                   min_bin_height=ms.MIN_BIN, min_derivative=ms.MIN_DERIV)
            assert torch.allclose(got_u, want_u, rtol=tol, atol=tol * 10), (dtype, scale, float((got_u - want_u).abs().max()))
            assert torch.allclose(got_lad, want_lad, rtol=tol, atol=tol * 100), (dtype, scale, float((got_lad - want_lad).abs().max()))
            outside = (y < -ms.TAIL_BOUND) | (y > ms.TAIL_BOUND)
            assert torch.equal(got_u[outside], y[outside]) and float(got_lad[outside].abs().max()) == 0.0


def test_inverse_spline_on_the_height_knots():
    """Inputs exactly on the interior height knots go to the matching width knots."""
    g = torch.Generator().manual_seed(3)
    q = _params(50, 30.0, torch.float64, g)
    K = ms.NUM_BINS
    h = ms.MIN_BIN + (1.0 - ms.MIN_BIN * K) * torch.softmax(q[:, K:2 * K] / math.sqrt(ms.HIDDEN), dim=-1)
    w = ms.MIN_BIN + (1.0 - ms.MIN_BIN * K) * torch.softmax(q[:, :K] / math.sqrt(ms.HIDDEN), dim=-1)
    ch = 2 * ms.TAIL_BOUND * torch.cumsum(h, -1) - ms.TAIL_BOUND
    cw = 2 * ms.TAIL_BOUND * torch.cumsum(w, -1) - ms.TAIL_BOUND
    for j in (0, 5, 11, 22):
        u, _ = mss.rqs_inverse(ch[:, j].clone(), q)
        assert float((u - cw[:, j]).abs().max()) < 1e-12


def test_inverse_round_trip_and_logdets_cancel():
    """float64 round trip y -> u -> y.  The error in y is the rounding of u times the forward slope, which grows with the
    sharpness of the bins: measured 2e-15 / 6e-11 / 2e-8 at scales 1 / 30 / 120 (120 / sqrt(128) ~ 10 logits: slopes
    of several hundred)."""
    g = torch.Generator().manual_seed(4)
    for scale, tol in ((1.0, 1e-9), (30.0, 1e-9), (120.0, 1e-7)):
        R = 20000
        q = _params(R, scale, torch.float64, g)
        y = (torch.rand(R, generator=g, dtype=torch.float64) * 24.0 - 12.0)
        u, lad_inv = mss.rqs_inverse(y, q)
        back, lad_fwd = ms.rqs_forward(u, q)
        assert float((back - y).abs().max()) <= tol, (scale, float((back - y).abs().max()))
        assert float((lad_inv + lad_fwd).abs().max()) <= 1e-9, (scale, float((lad_inv + lad_fwd).abs().max()))


@pytest.mark.parametrize("scale", [1.0, 1.6])
def test_spec_sample_has_the_estimators_law(scale):
    """At one condition, 2e5 numpy-drawn (u_choice, n): choice counts against softmax(logits) (chi^2), and per choice
    the forward flow maps the sampled rt back to N(0,1) (KS, alpha = 1e-3 with Bonferroni over the choices)."""
    p = ms.cast_params(ms.init_params(2, scale=scale), torch.float64)
    cond1 = torch.cat([orc.prior_sample(1, seed=5)[0].double(), torch.ones(80, dtype=torch.float64)])[None, :]
    N = 200_000
    rng = np.random.default_rng(9)
    uc = torch.from_numpy((rng.integers(0, 2**32, N) + 0.5) * 2.0**-32)
    n = torch.from_numpy(rng.standard_normal(N))
    cond = cond1.expand(N, 85)
    x = mss.sample(p, cond, uc, n)
    assert x.shape == (N, 2) and bool((x[:, 0] > 0).all())
    probs = torch.softmax(mss.choice_logits(p, cond1), dim=-1)[0].numpy()
    counts = np.bincount(x[:, 1].long().numpy(), minlength=3)
    assert stats.chisquare(counts, probs * N).pvalue > 1e-3, (counts, probs * N)
    z = mss.flow_forward(p, x, cond)
    assert float((z - n).abs().max()) < 1e-8          # the forward chain undoes the inverse one row by row
    for c in range(3):
        zc = z[x[:, 1] == c].numpy()
        assert stats.kstest(zc, "norm").pvalue > 1e-3 / 3, c


def test_choice_draw_edges():
    logits = torch.tensor([[0.0, 0.0, 0.0]] * 4, dtype=torch.float64)
    u = torch.tensor([1e-12, 1 / 3 - 1e-9, 1 / 3 + 1e-9, 1 - 1e-16], dtype=torch.float64)
    assert mss.choice_from_uniform(logits, u).tolist() == [0, 0, 1, 2]
    assert mss.choice_from_uniform(logits[:1], torch.tensor([1.0], dtype=torch.float64)).tolist() == [2]   # at the total


@pytest.fixture(scope="module")
def L():
    build_native()
    return _native.lib()


def test_sample_arguments_are_rejected_before_cuda(L):
    ws = ctypes.create_string_buffer(1024)
    buf = (ctypes.addressof(ws) + 255) & ~255
    args = dict(handle=None, cond=buf, ld=85, B=4, S=3, draws=None, out=buf, ws=buf)

    def call(**kw):
        a = dict(args, **kw)
        return L.mnle_sample_tc_f32(a["handle"], a["cond"], a["ld"], a["B"], a["S"], 1, 0, a["draws"], a["out"], a["ws"], None)

    assert call() == _native.DDM_ERR_STATE                      # null handle, every other argument fine
    assert b"bad handle" in L.ddm_last_error()
    assert call(B=-1) == _native.DDM_ERR_INVALID
    assert call(S=-1) == _native.DDM_ERR_INVALID
    assert call(ld=84) == _native.DDM_ERR_INVALID and b"ld_cond=84" in L.ddm_last_error()
    assert call(cond=None) == _native.DDM_ERR_INVALID
    assert call(out=None) == _native.DDM_ERR_INVALID
    assert call(ws=None) == _native.DDM_ERR_INVALID
    assert call(ws=buf + 4) == _native.DDM_ERR_INVALID and b"256-byte" in L.ddm_last_error()
    assert call(B=4000, S=2001) == _native.DDM_ERR_INVALID and b"8e6" in L.ddm_last_error()
    assert call(B=2, S=2**62) == _native.DDM_ERR_INVALID
    assert L.mnle_sample_tc_workspace_floats(3, 4000, 2001) == 0
    assert L.mnle_sample_tc_workspace_floats(3, 0, 5) == 0
    assert L.mnle_sample_tc_workspace_floats(9, 4, 5) == 0
    assert L.mnle_sample_tc_workspace_floats(3, 4000, 2000) > 0
