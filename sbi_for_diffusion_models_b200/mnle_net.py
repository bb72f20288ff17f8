"""Packed MNLE parameters and the device-side estimator (``mnle_*`` entry points).

The reference never touches MNLE weights itself: it asks sbi for an estimator
(mnle.py:31-48) and calls ``estimator.log_prob(x, condition=...)`` (potentials.py:113).  To run
that call on the GPU the weights are packed once into one fp32 buffer (layout documented in
``include/ddm_b200.h``) with the per-dimension z-scoring of the condition folded into each
first layer, copied to the device lazily per (process, device) -- the object pickles as the
CPU buffer only, so it survives pyro's ``spawn`` chain workers (potentials.py:61).
"""
from __future__ import annotations

import ctypes
import os
import weakref
from typing import Dict, Optional

import numpy as np
import torch

from . import _native
from .simulator import compute_device

HIDDEN, NUM_BINS, NUM_TRANSFORMS, COND_DIM = 128, 24, 10, 85
CTX_DIM, SPLINE_OUT = COND_DIM + 1, 3 * NUM_BINS - 1


def packed_sections(n_choices: int):
    """(name, shape) of every tensor in the packed buffer, in order (names of ``oracle/mnle_spec.py``)."""
    out = [("cat.W0", (HIDDEN, COND_DIM)), ("cat.b0", (HIDDEN,)), ("cat.W1", (HIDDEN, HIDDEN)), ("cat.b1", (HIDDEN,)),
           ("cat.W2", (HIDDEN, HIDDEN)), ("cat.b2", (HIDDEN,)), ("cat.Wo", (n_choices, HIDDEN)), ("cat.bo", (n_choices,))]
    for k in range(NUM_TRANSFORMS):
        out += [(f"flow.{k}.W1", (HIDDEN, CTX_DIM)), (f"flow.{k}.b1", (HIDDEN,)), (f"flow.{k}.W2", (HIDDEN, HIDDEN)),
                (f"flow.{k}.b2", (HIDDEN,)), (f"flow.{k}.W3", (SPLINE_OUT, HIDDEN)), (f"flow.{k}.b3", (SPLINE_OUT,))]
    out += [("flow.mu_y", ()), ("flow.sigma_y", ())]
    return out


def unpack_params(packed: torch.Tensor, n_choices: int) -> Dict[str, torch.Tensor]:
    """Views of a packed buffer (any device) by name.  No un-folding: first layers come out as
    stored (the trainer keeps them raw, its condition is standardised beforehand)."""
    out, o = {}, 0
    for name, shape in packed_sections(n_choices):
        n = int(np.prod(shape)) if shape else 1
        out[name] = packed[o:o + n].reshape(shape)
        o += n
    if o != packed.numel():
        raise ValueError(f"packed MNLE buffer has {packed.numel()} floats, layout needs {o}")
    return out


def session_offsets(lengths) -> np.ndarray:
    """Trial offsets (D+1,) int64 of ragged sessions: session d owns flat trials [offsets[d], offsets[d+1]).
    ``lengths``: a sequence or 1-D CPU integer tensor of D non-negative session lengths."""
    if isinstance(lengths, torch.Tensor):
        if lengths.device.type != "cpu" or lengths.ndim != 1 or lengths.is_floating_point() or lengths.is_complex():
            raise ValueError(f"lengths must be a 1-D CPU integer tensor, got {lengths.dtype} {tuple(lengths.shape)} "
                             f"on {lengths.device}")
        arr = lengths.to(torch.int64).numpy()
    else:
        arr = np.asarray(list(lengths))
        if arr.size == 0:
            arr = arr.astype(np.int64)
        if arr.ndim != 1 or not np.issubdtype(arr.dtype, np.integer):
            raise ValueError(f"lengths must be a sequence of ints, got {arr.dtype} {arr.shape}")
    arr = arr.astype(np.int64)
    if arr.size and int(arr.min()) < 0:
        raise ValueError(f"session lengths must be non-negative, got {int(arr.min())} for session {int(arr.argmin())}")
    return np.concatenate([np.zeros(1, np.int64), np.cumsum(arr)])


def split_sessions(offsets: np.ndarray, max_trials: int, max_sessions: int) -> list:
    """Consecutive session ranges [d0, d1) covering all D sessions, each with at most ``max_trials`` trials and
    ``max_sessions`` sessions: the launches of one ragged potential call.  A single session longer than
    ``max_trials`` raises ValueError."""
    D = len(offsets) - 1
    chunks, d0 = [], 0
    for d in range(D):
        if offsets[d + 1] - offsets[d] > max_trials:
            raise ValueError(f"session {d} has {int(offsets[d + 1] - offsets[d])} trials, more than the {max_trials} "
                             "one launch can take")
        if d > d0 and (offsets[d + 1] - offsets[d0] > max_trials or d - d0 >= max_sessions):
            chunks.append((d0, d))
            d0 = d
    if D:
        chunks.append((d0, D))
    return chunks


class SessionPlan:
    """D ragged sessions laid out for ``DeviceMNLE.loglik_sum_sessions`` with C chains each and one kernel: the trial
    offsets (checked on the host), their split into launches at session boundaries, and each launch's offsets on the
    device.  Built once (``DeviceMNLE.session_plan``); a call through it copies nothing between host and device, so
    a CUDA graph can record it."""

    def __init__(self, lengths, C: int, kernel: str, device: torch.device, max_trials: int, max_sessions: int):
        self.offsets = session_offsets(lengths)
        self.lengths = np.diff(self.offsets)
        self.D, self.N, self.C, self.kernel, self.device = len(self.offsets) - 1, int(self.offsets[-1]), int(C), kernel, device
        self.chunks = []
        for d0, d1 in split_sessions(self.offsets, max_trials, max_sessions):
            n0, n1 = int(self.offsets[d0]), int(self.offsets[d1])
            off = torch.from_numpy(self.offsets[d0:d1 + 1] - n0).to(device)
            self.chunks.append((d0, d1, n0, n1, off))


class PackedMNLE:
    """CPU-resident packed parameters + lazily created device handles."""

    def __init__(self, packed: np.ndarray, n_choices: int):
        packed = np.ascontiguousarray(packed, dtype=np.float32)
        need = self.packed_floats(n_choices)
        if packed.shape != (need,):
            raise ValueError(f"packed MNLE buffer has shape {packed.shape}, expected ({need},)")
        self.packed, self.n_choices = packed, int(n_choices)
        self._handles: Dict[tuple, int] = {}
        # device copies (cudaMalloc'd by mnle_create) are released when the object is collected
        self._finalizer = weakref.finalize(self, PackedMNLE._release, self._handles)

    @staticmethod
    def _release(handles: Dict[tuple, int]) -> None:
        for (pid, _), h in list(handles.items()):
            if pid == os.getpid():           # a forked child does not own its parent's device memory
                try:
                    _native.lib().mnle_destroy(h)
                except Exception:
                    pass
        handles.clear()

    @staticmethod
    def packed_floats(n_choices: int) -> int:
        return (HIDDEN * COND_DIM + HIDDEN + 2 * (HIDDEN * HIDDEN + HIDDEN) + n_choices * HIDDEN + n_choices
                + NUM_TRANSFORMS * (HIDDEN * CTX_DIM + HIDDEN + HIDDEN * HIDDEN + HIDDEN + SPLINE_OUT * HIDDEN + SPLINE_OUT)
                + 2)

    # ---- construction -----------------------------------------------------------------
    @classmethod
    def from_params(cls, p: Dict[str, torch.Tensor]) -> "PackedMNLE":
        """From a dict with the names of ``oracle/mnle_spec.py`` (also what ``from_state_dict``
        produces).  z-scoring is folded in float64: W' = W / std, b' = b - W (mean / std)."""
        f64 = lambda t: np.asarray(t.detach().cpu().to(torch.float64).numpy())
        mean, std = f64(p["cond_mean"]), np.maximum(f64(p["cond_std"]), 1e-7)
        if mean.shape != (COND_DIM,) or std.shape != (COND_DIM,):
            raise ValueError("condition mean/std must have 85 entries")

        # optional: a flow that standardises ALL 86 context columns itself (choice column included)
        ctx_mean = f64(p["flow.ctx_mean"]) if "flow.ctx_mean" in p else None
        ctx_std = np.maximum(f64(p["flow.ctx_std"]), 1e-7) if "flow.ctx_std" in p else None
        if (ctx_mean is None) != (ctx_std is None) or (ctx_mean is not None and ctx_mean.shape != (CTX_DIM,)):
            raise ValueError("flow.ctx_mean / flow.ctx_std must both be given with 86 entries")

        def fold(W, b, flow=False):
            W, b = f64(W), f64(b)
            Wf = W.copy()
            if flow and ctx_mean is not None:   # z-scoring of the 86-wide context owned by the flow
                return W / ctx_std[None, :], b - W @ (ctx_mean / ctx_std)
            Wf[:, :COND_DIM] = W[:, :COND_DIM] / std[None, :]
            return Wf, b - W[:, :COND_DIM] @ (mean / std)

        def shape(t, s, what):
            if tuple(t.shape) != s:
                raise ValueError(f"{what}: shape {tuple(t.shape)}, expected {s}")
            return t

        n_choices = int(p["cat.Wo"].shape[0])
        parts = []
        W0, b0 = fold(shape(p["cat.W0"], (HIDDEN, COND_DIM), "cat.W0"), p["cat.b0"])
        parts += [W0, b0, f64(shape(p["cat.W1"], (HIDDEN, HIDDEN), "cat.W1")), f64(p["cat.b1"]),
                  f64(shape(p["cat.W2"], (HIDDEN, HIDDEN), "cat.W2")), f64(p["cat.b2"]),
                  f64(shape(p["cat.Wo"], (n_choices, HIDDEN), "cat.Wo")), f64(p["cat.bo"])]
        for k in range(NUM_TRANSFORMS):
            W1, b1 = fold(shape(p[f"flow.{k}.W1"], (HIDDEN, CTX_DIM), f"flow.{k}.W1"), p[f"flow.{k}.b1"], flow=True)
            parts += [W1, b1, f64(shape(p[f"flow.{k}.W2"], (HIDDEN, HIDDEN), f"flow.{k}.W2")), f64(p[f"flow.{k}.b2"]),
                      f64(shape(p[f"flow.{k}.W3"], (SPLINE_OUT, HIDDEN), f"flow.{k}.W3")), f64(p[f"flow.{k}.b3"])]
        parts += [f64(p["flow.mu_y"]).reshape(1), f64(p["flow.sigma_y"]).reshape(1)]
        packed = np.concatenate([a.reshape(-1) for a in parts]).astype(np.float32)
        return cls(packed, n_choices)

    @classmethod
    def from_state_dict(cls, sd: Dict[str, torch.Tensor]) -> "PackedMNLE":
        """Import of an sbi MNLE ``state_dict`` (the only way weights leave sbi, reference mnle.py:247-259).

        UNVERIFIED against a real sbi 0.25.0 checkpoint (sbi is not installable in this repository's build
        environment; ``tools/compare_with_sbi.py`` is the check to run where it is).  Key names are sbi / nflows
        internals, so layers are recognised by SHAPE in registration order -- exactly one categorical net
        ``(128,85) (128,128) (128,128) (K,128)`` and exactly ten conditioners ``(128,86) (128,128) (71,128)`` --
        and the standardisation buffers by name AND width:

        * ``*mean*`` / ``*std*`` pairs (sbi ``Standardize``: (x - mean) / std) or ``*_shift`` / ``*_scale`` pairs
          (nflows ``AffineTransform``: x * scale + shift, i.e. mean = -shift / scale, std = 1 / scale);
        * one 85-wide pair = z-scoring of the condition, shared by both nets;
        * optionally one 86-wide pair = the flow's own z-scoring of [condition, choice]; it is folded into the
          conditioners' first layers (then the 85-wide pair feeds the categorical net only);
        * exactly one 1-wide pair = z-scoring of log rt.

        Anything else -- extra or missing layers, more than one candidate for a buffer, widths that do not fit --
        raises ``ValueError`` naming what was found; nothing is guessed."""
        layers, stats = [], []
        items = list(sd.items())
        i = 0
        while i < len(items):
            k, v = items[i]
            if v.ndim == 2 and i + 1 < len(items) and items[i + 1][1].ndim == 1 \
                    and items[i + 1][1].shape[0] == v.shape[0]:
                layers.append((k, v, items[i + 1][1]))
                i += 2
                continue
            if v.ndim <= 1 and v.numel() in (1, COND_DIM, CTX_DIM) and v.dtype.is_floating_point:
                stats.append((k, v.reshape(-1)))
            i += 1
        shapes = [tuple(w.shape) for _, w, _ in layers]

        def find_run(first, rest):
            return [j for j, s in enumerate(shapes) if s == first and
                    all(j + 1 + m < len(shapes) and (shapes[j + 1 + m] == r or (r is None and shapes[j + 1 + m][1] == HIDDEN))
                        for m, r in enumerate(rest))]

        cat = find_run((HIDDEN, COND_DIM), [(HIDDEN, HIDDEN), (HIDDEN, HIDDEN), None])
        flows = find_run((HIDDEN, CTX_DIM), [(HIDDEN, HIDDEN), (SPLINE_OUT, HIDDEN)])
        if len(cat) != 1 or len(flows) != NUM_TRANSFORMS or len(layers) != 4 + 3 * NUM_TRANSFORMS:
            raise ValueError(f"state_dict does not look like the reference's MNLE: found {len(cat)} categorical "
                             f"nets, {len(flows)} spline conditioners and {len(layers)} linear layers (expected 1, "
                             f"{NUM_TRANSFORMS} and {4 + 3 * NUM_TRANSFORMS}); layer shapes {shapes}")

        def pair(width):
            """(mean, std) of the one standardisation of this width, or None if there is none."""
            def named(*tags):
                return [(k, v) for k, v in stats if v.numel() == width and any(t in k.lower() for t in tags)]
            means, stds = named("mean"), named("std")
            shifts, scales = named("shift"), named("scale")
            if len(means) == 1 and len(stds) == 1 and not shifts and not scales:
                return means[0][1].double(), stds[0][1].double()
            if len(shifts) == 1 and len(scales) == 1 and not means and not stds:
                scale = scales[0][1].double()
                return -shifts[0][1].double() / scale, 1.0 / scale
            if not (means or stds or shifts or scales):
                return None
            raise ValueError(f"ambiguous standardisation buffers of width {width}: "
                             f"{[k for k, _ in means + stds + shifts + scales]}")

        cond, ctx, y = pair(COND_DIM), pair(CTX_DIM), pair(1)
        if y is None or (cond is None and ctx is None):
            raise ValueError("state_dict lacks the standardisation buffers of the reference's MNLE "
                             f"(condition: 85- or 86-wide, log rt: 1-wide); candidates seen: {[k for k, _ in stats]}")
        p: Dict[str, torch.Tensor] = {"flow.mu_y": y[0][0], "flow.sigma_y": y[1][0]}
        if cond is not None:
            p["cond_mean"], p["cond_std"] = cond
        else:   # only the flow standardises; the categorical net then sees the first 85 columns' statistics
            p["cond_mean"], p["cond_std"] = ctx[0][:COND_DIM], ctx[1][:COND_DIM]
        if ctx is not None:
            p["flow.ctx_mean"], p["flow.ctx_std"] = ctx
        j = cat[0]
        for n, name in enumerate(("0", "1", "2", "o")):
            p[f"cat.W{name}"], p[f"cat.b{name}"] = layers[j + n][1], layers[j + n][2]
        for k, j in enumerate(flows):
            for n in range(3):
                p[f"flow.{k}.W{n + 1}"], p[f"flow.{k}.b{n + 1}"] = layers[j + n][1], layers[j + n][2]
        return cls.from_params(p)

    # ---- device handle ------------------------------------------------------------------
    def handle(self, dev: torch.device) -> int:
        key = (os.getpid(), dev.index)
        h = self._handles.get(key)
        if h is None:
            out = ctypes.c_void_p()
            with torch.cuda.device(dev):
                rc = _native.lib().mnle_create(self.packed.ctypes.data, self.packed.size, self.n_choices,
                                               ctypes.byref(out))
            _native.check(rc, "mnle_create")
            h = self._handles[key] = out.value
        return h

    def close(self) -> None:
        PackedMNLE._release(self._handles)

    def __getstate__(self):
        return {"packed": self.packed, "n_choices": self.n_choices}

    def __setstate__(self, st):
        self.packed, self.n_choices, self._handles = st["packed"], st["n_choices"], {}
        self._finalizer = weakref.finalize(self, PackedMNLE._release, self._handles)


class DeviceMNLE(torch.nn.Module):
    """Estimator object with the call shape the reference uses (potentials.py:113) plus the
    fused potential.  Inputs may live on the CPU; results are returned on the input's device."""

    def __init__(self, packed: PackedMNLE, device=None):
        super().__init__()
        self.packed = packed
        self._device = device
        # the reference checkpoints an estimator as {"state_dict": est.state_dict(), "config": cfg}
        # (mnle.py:241-259): the packed parameters are the state (z-scoring already folded in)
        self.register_buffer("packed_params", torch.from_numpy(packed.packed.copy()))
        self.register_buffer("n_choices", torch.tensor(packed.n_choices, dtype=torch.int64))

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        key_p, key_k = prefix + "packed_params", prefix + "n_choices"
        if key_p in state_dict and key_k in state_dict:
            K = int(state_dict[key_k])
            new = PackedMNLE(state_dict[key_p].detach().cpu().numpy().astype(np.float32, copy=True), K)   # validates the size
            if self.packed_params.numel() != new.packed.size:   # a different number of choice categories
                self.packed_params = torch.empty(new.packed.size, dtype=torch.float32, device=self.packed_params.device)
            self.packed.close()
            self.packed = new
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    def __getstate__(self):
        return {"packed": self.packed, "device": self._device}

    def __setstate__(self, st):
        self.__init__(st["packed"], st["device"])

    def _dev(self, t: Optional[torch.Tensor] = None) -> torch.device:
        return compute_device(self._device if self._device is not None else (t.device if t is not None and t.is_cuda else None))

    def log_prob(self, x: torch.Tensor, condition: torch.Tensor, *, kernel: str = "auto") -> torch.Tensor:
        """x (1,R,2) or (R,2) = [rt seconds, choice], condition (R,85) -> (1,R).
        ``kernel``: "tc" / "auto" tensor cores (tcgen05), "simt" fp32 CUDA cores, "precise" fp32 networks with
        the spline chain in fp64 (accuracy anchor for trained estimators)."""
        if kernel not in ("auto", "tc", "simt", "precise"):
            raise ValueError(f"unknown kernel {kernel!r}")
        dev = self._dev(condition)
        xr = x.reshape(-1, 2).to(device=dev, dtype=torch.float32).contiguous()
        cond = condition.to(device=dev, dtype=torch.float32)
        if cond.ndim != 2 or cond.shape[1] != COND_DIM or cond.shape[0] != xr.shape[0]:
            raise ValueError(f"condition must be (R,{COND_DIM}) with R={xr.shape[0]}, got {tuple(cond.shape)}")
        if cond.stride(1) != 1 or cond.stride(0) < COND_DIM:    # (a broadcast row has row stride 0)
            cond = cond.contiguous()
        R = xr.shape[0]
        with torch.cuda.device(dev):
            out = torch.empty((R,), dtype=torch.float32, device=dev)
            L = _native.lib()
            fn = {"simt": L.mnle_log_prob_rows_f32, "precise": L.mnle_log_prob_rows_precise_f32}.get(
                kernel, L.mnle_log_prob_rows_tc_f32)
            rc = fn(self.packed.handle(dev), xr.data_ptr(), cond.data_ptr(), cond.stride(0) if R > 1 else COND_DIM, R,
                    out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "mnle_log_prob_rows")
        return out.to(condition.device).unsqueeze(0)

    SAMPLE_MAX_ROWS = 8_000_000   # rows of one mnle_sample_tc_f32 call

    def sample(self, sample_shape=torch.Size(), condition: Optional[torch.Tensor] = None, *, seed: Optional[int] = None,
               draws: Optional[torch.Tensor] = None) -> torch.Tensor:
        """estimator.sample(sample_shape, condition): condition (B,85) -> x (*sample_shape, B, 2) = [rt seconds, choice]
        on the condition's device.  The choice is drawn from the categorical net, then log rt from the spline flow
        conditioned on it (the ten splines run in inverse, in fp64, on tensor-core network outputs).  rt is not clamped
        to the simulator's window: the estimator is a continuous density, and sbi does not clamp its samples either.

        [UNVERIFIED against sbi] the order "choice first, then the flow given the choice" and the output shape of sbi
        >= 0.23's ConditionalDensityEstimator.sample follow sbi's MixedDensityEstimator; sbi is not installable where
        this package is built, so they have not been checked against it (the inverse spline itself is pinned against
        nflows' formulas, tests/test_mnle_sample_spec.py).

        ``seed``: Philox key of the draws; None draws one from torch's global generator, so ``torch.manual_seed``
        makes runs reproducible.  Sample s of condition b uses the Philox block of (s, b) (include/ddm_b200.h), so the
        result does not depend on how large requests are split over calls.  ``draws``: (S*B, 2) or (*sample_shape, B,
        2) of [u_choice in (0,1), standard normal] used instead of Philox (row s*B + b)."""
        if condition is None:
            raise ValueError("sample needs a condition (B,85)")
        shape = torch.Size(sample_shape)
        S = int(np.prod(shape)) if len(shape) else 1
        dev = self._dev(condition)
        cond = condition.to(device=dev, dtype=torch.float32)
        if cond.ndim != 2 or cond.shape[1] != COND_DIM:
            raise ValueError(f"condition must be (B,{COND_DIM}), got {tuple(cond.shape)}")
        if cond.stride(1) != 1 or cond.stride(0) < COND_DIM:    # (a broadcast row has row stride 0)
            cond = cond.contiguous()
        B = cond.shape[0]
        if B > self.SAMPLE_MAX_ROWS:
            raise ValueError(f"at most {self.SAMPLE_MAX_ROWS} conditions per call, got {B}")
        if draws is not None:
            if draws.numel() != S * B * 2:
                raise ValueError(f"draws must hold (S*B, 2) = ({S * B}, 2) values, got {tuple(draws.shape)}")
            draws = draws.reshape(S * B, 2).to(device=dev, dtype=torch.float32).contiguous()
            seed = 0
        elif seed is None:
            from .simulator import next_seed
            seed = next_seed()
        L = _native.lib()
        out = torch.empty((S * B, 2), dtype=torch.float32, device=dev)
        if S * B > 0:
            step = max(1, self.SAMPLE_MAX_ROWS // B)
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream(dev).cuda_stream
                ws = None
                for s0 in range(0, S, step):
                    sc = min(step, S - s0)
                    n_ws = L.mnle_sample_tc_workspace_floats(self.packed.n_choices, B, sc)
                    if ws is None or ws.numel() < n_ws:
                        ws = torch.empty((n_ws,), dtype=torch.float32, device=dev)   # torch allocations are 512-byte aligned
                    d = draws[s0 * B:(s0 + sc) * B] if draws is not None else None
                    rc = L.mnle_sample_tc_f32(self.packed.handle(dev), cond.data_ptr(), cond.stride(0) if B > 1 else COND_DIM,
                                              B, sc, ctypes.c_uint64(seed & (2**64 - 1)), ctypes.c_uint64(s0),
                                              d.data_ptr() if d is not None else None, out[s0 * B:].data_ptr(), ws.data_ptr(),
                                              stream)
                    _native.check(rc, "mnle_sample_tc_f32")
        return out.reshape(*shape, B, 2).to(condition.device)

    def loglik_sum(self, theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor, *, kernel: str = "auto"
                   ) -> torch.Tensor:
        """out[c] = sum_t log p(x_o[t] | [theta[c], pulses[t]]): theta (C,5), x_o (T,2), pulses (T,>=80)."""
        L = _native.lib()
        dev = self._dev(theta)
        th = theta.to(device=dev, dtype=torch.float32)
        xo = x_o.reshape(-1, 2).to(device=dev, dtype=torch.float32).contiguous()
        pl = pulses.to(device=dev, dtype=torch.float32)
        if th.ndim != 2 or th.shape[1] != 5:
            raise ValueError(f"theta must be (C,5), got {tuple(th.shape)}")
        if pl.ndim != 2 or pl.shape[0] != xo.shape[0] or pl.shape[1] < COND_DIM - 5:
            raise ValueError(f"pulses must be (T,>=80) with T={xo.shape[0]}, got {tuple(pl.shape)}")
        if th.stride(1) != 1:
            th = th.contiguous()
        if pl.stride(1) != 1:
            pl = pl.contiguous()
        C, T = th.shape[0], xo.shape[0]
        with torch.cuda.device(dev):
            out = torch.empty((C,), dtype=torch.float32, device=dev)
            fn, ws_floats = self._pick_kernel(kernel, T)
            n_ws = ws_floats(T, C) if ws_floats is not None else L.mnle_loglik_tc64_workspace_floats(self.packed.n_choices, T, C)
            ws = torch.empty((max(n_ws, 1),), dtype=torch.float32, device=dev)
            rc = fn(self.packed.handle(dev), th.data_ptr(), th.stride(0) if C > 1 else 5, xo.data_ptr(), pl.data_ptr(),
                    pl.stride(0) if T > 1 else pl.shape[1], T, C, out.data_ptr(), ws.data_ptr(),
                    torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "mnle_loglik_sum")
        return out.to(theta.device)

    # "auto" takes the reverse-mode tensor-core path from this many rows on.  Measured (tools/time_grad_sizes.py, trained
    # estimator, eager calls): T=50 x C=2 (the reference's NUM_CHAINS) 0.14 ms against 0.39 ms for the forward-mode
    # fp32 kernel, T=1 x C=1 0.10 against 0.38, T=50 x C=1024 1.27 against 9.97 -- reverse mode wins at every size.
    # kernel="simt" remains for callers who want every gradient entry within fp32 rounding of float64 (the tensor-core
    # path can put a ReLU unit that sits within 1e-5 of its kink on the other side, see tests/test_gpu_mnle.py).
    GRAD_TC_MIN_ROWS = 0

    def loglik_sum_and_grad(self, theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor, *, kernel: str = "auto"):
        """(out (C,), grad (C,5)) with grad[c] = d out[c] / d theta[c].
        ``kernel``: "tc" reverse mode on the tensor cores (the training step's tcgen05 forward / backward-data
        kernels over the T*C expanded rows), "simt" forward mode on the CUDA cores (five tangents per row, fp32),
        "auto" picks by the number of rows."""
        if kernel not in ("auto", "tc", "simt"):
            raise ValueError(f"unknown kernel {kernel!r}")
        L = _native.lib()
        dev = self._dev(theta)
        th = theta.detach().to(device=dev, dtype=torch.float32).contiguous()
        xo = x_o.reshape(-1, 2).to(device=dev, dtype=torch.float32).contiguous()
        pl = pulses.to(device=dev, dtype=torch.float32).contiguous()
        if th.ndim != 2 or th.shape[1] != 5:
            raise ValueError(f"theta must be (C,5), got {tuple(th.shape)}")
        if pl.ndim != 2 or pl.shape[0] != xo.shape[0] or pl.shape[1] < COND_DIM - 5:
            raise ValueError(f"pulses must be (T,>=80) with T={xo.shape[0]}, got {tuple(pl.shape)}")
        C, T = th.shape[0], xo.shape[0]
        if kernel == "auto":
            kernel = "tc" if self.GRAD_TC_MIN_ROWS <= T * C <= 8_000_000 else "simt"
        with torch.cuda.device(dev):
            out = torch.empty((C,), dtype=torch.float32, device=dev)
            grad = torch.empty((C, 5), dtype=torch.float32, device=dev)
            if kernel == "tc":
                ws = torch.empty((max(L.mnle_loglik_grad_tc_workspace_floats(self.packed.n_choices, T, C), 1),),
                                 dtype=torch.float32, device=dev)
                rc = L.mnle_loglik_sum_grad_tc_f32(self.packed.handle(dev), th.data_ptr(), 5, xo.data_ptr(), pl.data_ptr(),
                                                   pl.shape[1], T, C, out.data_ptr(), grad.data_ptr(), ws.data_ptr(),
                                                   torch.cuda.current_stream(dev).cuda_stream)
                _native.check(rc, "mnle_loglik_sum_grad_tc_f32")
            else:
                ws = torch.empty((max(L.mnle_loglik_grad_workspace_floats(T, C), 1),), dtype=torch.float32, device=dev)
                rc = L.mnle_loglik_sum_grad_f32(self.packed.handle(dev), th.data_ptr(), 5, xo.data_ptr(), pl.data_ptr(),
                                                pl.shape[1], T, C, out.data_ptr(), grad.data_ptr(), ws.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream)
                _native.check(rc, "mnle_loglik_sum_grad_f32")
        return out.to(theta.device), grad.to(theta.device)

    def loglik_sum_batched(self, theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor) -> torch.Tensor:
        """D independent datasets in one launch (the SBC loop evaluates one potential per dataset,
        reference mnle.py:183-218): theta (D,C,5), x_o (D,T,2), pulses (D,T,>=80) -> (D,C) with
        out[d,c] = sum_t log p(x_o[d,t] | [theta[d,c], pulses[d,t]]).  Tensor-core kernel only."""
        L = _native.lib()
        dev = self._dev(theta)
        if theta.ndim != 3 or theta.shape[2] != 5:
            raise ValueError(f"theta must be (D,C,5), got {tuple(theta.shape)}")
        D, C = theta.shape[0], theta.shape[1]
        if x_o.ndim != 3 or x_o.shape[0] != D or x_o.shape[2] != 2:
            raise ValueError(f"x_o must be (D,T,2) with D={D}, got {tuple(x_o.shape)}")
        T = x_o.shape[1]
        if pulses.ndim != 3 or pulses.shape[0] != D or pulses.shape[1] != T or pulses.shape[2] < COND_DIM - 5:
            raise ValueError(f"pulses must be (D,T,>=80) with D={D}, T={T}, got {tuple(pulses.shape)}")
        th = theta.to(device=dev, dtype=torch.float32).contiguous()
        xo = x_o.to(device=dev, dtype=torch.float32).contiguous()
        pl = pulses.to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            out = torch.empty((D, C), dtype=torch.float32, device=dev)
            ws = torch.empty((max(L.mnle_loglik_batched_tc_workspace_floats(D, T, C), 1),), dtype=torch.float32, device=dev)
            rc = L.mnle_loglik_sum_batched_tc_f32(self.packed.handle(dev), th.data_ptr(), 5, xo.data_ptr(), pl.data_ptr(),
                                                  pl.shape[2], D, T, C, out.data_ptr(), ws.data_ptr(),
                                                  torch.cuda.current_stream(dev).cuda_stream)
            _native.check(rc, "mnle_loglik_sum_batched_tc_f32")
        return out.to(theta.device)

    SESSIONS_MAX_TRIALS = 524_280        # trials of one mnle_loglik_sum_sessions_tc_f32 launch (its hoist grid)
    SESSIONS_TC64_MAX_ROWS = 8_000_000   # (trial, chain) rows of one mnle_loglik_sum_sessions_tc64_f32 launch
    SESSIONS_TC64_MAX_SESSIONS = 65_535  # sessions of one tc64 launch (its final sum's grid)

    def session_plan(self, lengths, C: int, *, kernel: str = "tc", device=None) -> SessionPlan:
        """The layout ``loglik_sum_sessions`` needs for sessions of these lengths with C chains each, built once: pass
        it as ``lengths`` to calls that must not touch the host (a sampler's CUDA graph)."""
        if kernel not in ("tc", "tc64"):
            raise ValueError(f"unknown kernel {kernel!r} for sessions (tc or tc64)")
        if kernel == "tc":
            max_trials, max_sessions = self.SESSIONS_MAX_TRIALS, 2**31 - 1
        else:
            max_trials, max_sessions = self.SESSIONS_TC64_MAX_ROWS // max(int(C), 1), self.SESSIONS_TC64_MAX_SESSIONS
        return SessionPlan(lengths, C, kernel, self._dev() if device is None else torch.device(device), max_trials, max_sessions)

    def loglik_sum_sessions(self, theta: torch.Tensor, x_o: torch.Tensor, pulses: torch.Tensor, lengths, *,
                            kernel: str = "tc") -> torch.Tensor:
        """D observed sessions of different lengths in one call: theta (D,C,5), x_o (N,2), pulses (N,>=80) with the
        sessions' trials one after the other, ``lengths`` the D session lengths (sequence or CPU tensor, sum N) or a
        ``SessionPlan`` of them -> (D,C), out[d,c] = sum over session d's trials t of log p(x_o[t] | [theta[d,c],
        pulses[t]]), 0 for an empty session.  Each output has the bits of ``loglik_sum(theta[d], x_d, pulses_d,
        kernel=kernel)``.  ``kernel``: "tc" (tcgen05) or "tc64" (tensor-core networks, fp64 spline chain).  Requests
        over one launch's limit are split at session boundaries; shapes and lengths are checked before any launch."""
        if kernel not in ("tc", "tc64"):
            raise ValueError(f"unknown kernel {kernel!r} for sessions (tc or tc64)")
        if theta.ndim != 3 or theta.shape[2] != 5:
            raise ValueError(f"theta must be (D,C,5), got {tuple(theta.shape)}")
        D, C = theta.shape[0], theta.shape[1]
        dev = self._dev(theta)
        plan = lengths if isinstance(lengths, SessionPlan) else self.session_plan(lengths, C, kernel=kernel, device=dev)
        if (plan.D, plan.C, plan.kernel, plan.device) != (D, C, kernel, dev):
            raise ValueError(f"the session plan is for D={plan.D}, C={plan.C}, kernel {plan.kernel!r} on {plan.device}; "
                             f"the call has D={D}, C={C}, kernel {kernel!r} on {dev}")
        if x_o.ndim != 2 or tuple(x_o.shape) != (plan.N, 2):
            raise ValueError(f"x_o must be (N,2) with N={plan.N} (the sum of the lengths), got {tuple(x_o.shape)}")
        if pulses.ndim != 2 or pulses.shape[0] != plan.N or pulses.shape[1] < COND_DIM - 5:
            raise ValueError(f"pulses must be (N,>=80) with N={plan.N}, got {tuple(pulses.shape)}")
        th = theta.to(device=dev, dtype=torch.float32).contiguous()
        xo = x_o.to(device=dev, dtype=torch.float32).contiguous()
        pl = pulses.to(device=dev, dtype=torch.float32)
        if pl.stride(1) != 1 or (pl.shape[0] > 1 and pl.stride(0) < COND_DIM - 5):
            pl = pl.contiguous()
        ld_pulses = pl.stride(0) if pl.shape[0] > 1 else pl.shape[1]
        out = torch.empty((D, C), dtype=torch.float32, device=dev)
        if D == 0 or C == 0:
            return out.to(theta.device)
        L = _native.lib()
        if kernel == "tc":
            fn, ws_floats = L.mnle_loglik_sum_sessions_tc_f32, L.mnle_loglik_sessions_tc_workspace_floats
        else:
            fn = L.mnle_loglik_sum_sessions_tc64_f32
            ws_floats = lambda d, n, c: L.mnle_loglik_sessions_tc64_workspace_floats(self.packed.n_choices, d, n, c)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            n_ws = max(ws_floats(d1 - d0, n1 - n0, C) for d0, d1, n0, n1, _ in plan.chunks)
            ws = torch.empty((max(n_ws, 1),), dtype=torch.float32, device=dev)   # torch allocations are 512-byte aligned
            for d0, d1, n0, n1, off in plan.chunks:
                rc = fn(self.packed.handle(dev), th[d0].data_ptr(), 5, xo[n0:].data_ptr(), pl[n0:].data_ptr(), ld_pulses,
                        off.data_ptr(), d1 - d0, n1 - n0, C, out[d0].data_ptr(), ws.data_ptr(), stream)
                _native.check(rc, "mnle_loglik_sum_sessions")
        return out.to(theta.device)

    @staticmethod
    def _pick_kernel(kernel: str, T: int):
        """"tc": tcgen05 tensor-core kernel; "simt": fp32 CUDA-core kernel; "precise": fp32 networks + fp64
        spline chain (accuracy anchor); "tc64": tensor-core networks + fp64 spline chain; "auto": tensor cores
        whenever the shape is covered."""
        L = _native.lib()
        if kernel == "auto":
            kernel = "tc" if T <= 524280 else "simt"
        if kernel == "tc":
            return L.mnle_loglik_sum_tc_f32, L.mnle_loglik_tc_workspace_floats
        if kernel == "simt":
            return L.mnle_loglik_sum_simt_f32, L.mnle_loglik_workspace_floats
        if kernel == "precise":
            return L.mnle_loglik_sum_precise_f32, L.mnle_loglik_workspace_floats
        if kernel == "tc64":
            return L.mnle_loglik_sum_tc64_f32, None
        raise ValueError(f"unknown kernel {kernel!r}")
