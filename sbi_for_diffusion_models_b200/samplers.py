"""Many-chain slice sampler that keeps every chain on the device (SURVEY 8 (f3)).

The reference samples the posterior with sbi's ``MCMCPosterior`` (mnle.py:77-93; NUTS through
pyro, one process per chain, CPU) and its notebook uses sbi's ``slice_np_vectorized``.  Both are
third-party and host-bound.  Here the same job -- draw from exp(potential) -- is done by a
coordinate-wise slice sampler (Neal 2003: stepping out + shrinkage) whose N chains advance in
lock-step as one (N, D) tensor, so each step is ONE call of the potential over all chains: exactly
the (trials x chains) shape the fused MNLE kernel is built for.  Gradient free.

Pure torch: runs on whatever device ``init`` lives on (tests use the CPU, the product the GPU).
"""
from __future__ import annotations

from typing import Callable, Optional

import torch


class GraphedLogProb:
    """``fn``: (N, D) -> (N,) captured once into a CUDA graph and replayed on static buffers.

    A slice-sampler step is one potential evaluation followed by a handful of tiny elementwise
    ops; at the sizes of one observed session the Python / launch path of the potential (prior,
    workspace allocation, two kernel launches) costs several times the kernels themselves, so the
    whole evaluation is recorded once and replayed.  Falls back to calling ``fn`` for inputs that
    are not CUDA tensors of the captured shape."""

    def __init__(self, fn: Callable[[torch.Tensor], torch.Tensor], example: torch.Tensor, warmup: int = 2):
        self.fn = fn
        self.graph = None
        if not example.is_cuda:
            return
        self.x = example.clone()
        side = torch.cuda.Stream(example.device)
        side.wait_stream(torch.cuda.current_stream(example.device))
        try:
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    fn(self.x)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    self.y = fn(self.x)
            self.graph = graph
        except Exception:       # fn synchronises or leaves the device (e.g. a CPU-only prior): call it directly
            self.graph = None
            torch.cuda.synchronize(example.device)
        torch.cuda.current_stream(example.device).wait_stream(side)

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        if self.graph is None or x.shape != self.x.shape or x.device != self.x.device or x.dtype != self.x.dtype:
            return self.fn(x)
        self.x.copy_(x)
        self.graph.replay()
        return self.y.clone()


class PhiloxUniforms:
    """Counter-based uniforms for chains [first_row, first_row + n_rows): draw k of global chain g is
    Philox4x32-10(key = seed + k // block, counter = (g, k % block)), whichever process owns the chain
    and whatever other chains run beside it -- so a sampler run sharded over GPUs reproduces the
    single-GPU run bit for bit.  Uses the simulator's device generator (``ddm_philox_words_u32``)."""

    def __init__(self, seed: int, first_row: int, n_rows: int, device, block: int = 256):
        self.seed, self.first, self.n, self.device, self.block = int(seed), int(first_row), int(n_rows), device, int(block)
        self._buf, self._blk = None, -1

    def __call__(self, k: int) -> torch.Tensor:
        """Draw number ``k`` of every chain: (n_rows,) fp32 in (0, 1)."""
        from .simulator import philox_words
        blk, j = divmod(int(k), self.block)
        if blk != self._blk:
            words = philox_words(self.seed + blk, self.n, self.block, trial_offset=self.first, device=self.device)
            # top 24 bits -> (0, 1): ((w >> 8) + 0.5) * 2^-24, exact in fp32
            self._buf = ((words >> 8) & 0xFFFFFF).to(torch.float32).add_(0.5).mul_(2.0 ** -24)
            self._blk = blk
        return self._buf[j]


class VectorizedSliceSampler:
    """Coordinate-wise slice sampler (Neal 2003: stepping out with a limit + shrinkage) over N chains, **every chain
    on its own clock**.  ``log_prob_fn``: (N, D) -> (N,), ``-inf`` outside the support.  ``init``: (N, D) starting
    points with finite log-probability.

    One potential call evaluates, for each chain, whatever point THAT chain needs next -- the left or right end of
    its bracket while stepping out, a shrinkage proposal afterwards -- for whatever coordinate it is working on.
    (A lock-step version, where all chains step out, then all shrink, runs every phase until its slowest chain is
    done: with 16 000 chains ~30 calls per coordinate update instead of the ~9 a single chain needs.)  Chains are
    fully independent: own uniforms (counter-based: draw 4 * it + j of chain g), own slice widths (running mean of
    the final bracket while tuning, as sbi's slice samplers do), own sweep count -- so a run sharded over GPUs, or
    batched with other datasets, reproduces the unsharded one bit for bit.  On a CUDA device one iteration (the
    potential plus ~60 elementwise ops of bookkeeping) is captured once into a CUDA graph and replayed.
    """

    MAX_FUSED_DIM = 64      # the largest D the kernels of csrc/mnle_sampler.cu accept

    def __init__(self, log_prob_fn: Callable[[torch.Tensor], torch.Tensor], init: torch.Tensor, *,
                 init_width: float = 0.1, max_step_out: int = 8, max_shrink: int = 64,
                 generator: Optional[torch.Generator] = None, uniforms: Optional[Callable[[int], torch.Tensor]] = None,
                 chain_groups: int = 1, use_graph: bool = True, fused: Optional[bool] = None):
        if init.ndim != 2:
            raise ValueError(f"init must be (num_chains, dim), got {tuple(init.shape)}")
        # a GraphedLogProb cannot be replayed inside another capture: use the function it wraps
        self.f = log_prob_fn.fn if isinstance(log_prob_fn, GraphedLogProb) else log_prob_fn
        self.x = init.clone()
        self.gen, self.uniforms = generator, uniforms
        self.N, self.D = init.shape
        if init.shape[0] % int(chain_groups):
            raise ValueError("the number of chains must be a multiple of chain_groups")
        self.n_evals = 0
        self.lp = self._eval(self.x)
        if not bool(torch.isfinite(self.lp).all()):
            raise ValueError("every chain must start at a point of finite log-probability")
        # starting widths: a tenth of the typical magnitude of the coordinate within the chain's group (SBC: its
        # dataset), then tuned per chain
        G, per = int(chain_groups), self.N // int(chain_groups)
        w0 = float(init_width) * init.abs().view(G, per, self.D).mean(dim=1).clamp_min(1e-3)
        self.width = w0.repeat_interleave(per, dim=0).contiguous()                        # (N, D)
        self.max_step_out, self.max_shrink = int(max_step_out), int(max_shrink)
        self._use_graph = bool(use_graph) and init.is_cuda
        # the bookkeeping of an iteration as two CUDA kernels around the potential (csrc/mnle_sampler.cu) instead of
        # ~80 elementwise torch launches; same arithmetic in the same order, same bits (float32 chains on a GPU, at
        # most MAX_FUSED_DIM coordinates; by default larger D runs the torch implementation, fused=True refuses it)
        fusable = init.is_cuda and init.dtype == torch.float32 and self.D <= self.MAX_FUSED_DIM
        self._fused = fusable if fused is None else bool(fused)
        if self._fused and not fusable:
            raise ValueError(f"the fused sampler kernels need float32 chains on a CUDA device and at most "
                             f"{self.MAX_FUSED_DIM} coordinates, got {init.dtype} on {init.device}, D = {self.D}")
        self._graph = None
        self._it = 0

    # ------------------------------------------------------------------------------------
    def _eval(self, x: torch.Tensor) -> torch.Tensor:
        lp = self.f(x)
        self.n_evals = getattr(self, "n_evals", 0) + 1
        return torch.nan_to_num(lp, nan=-float("inf"), posinf=float("inf"), neginf=-float("inf"))

    def _draw4(self, it: int) -> torch.Tensor:
        """The four uniforms every chain may consume in iteration ``it``: (4, N) in (0, 1)."""
        if self.uniforms is not None:
            return torch.stack([self.uniforms(4 * it + j) for j in range(4)]).to(self.x.dtype)
        return torch.rand((4, self.N), dtype=self.x.dtype, device=self.x.device, generator=self.gen).clamp_(1e-12, 1 - 1e-12)

    def _begin(self, mask: torch.Tensor, u: torch.Tensor) -> None:
        """Chains in ``mask`` start the slice update of their current coordinate ``self.d`` (uniforms u[1..3])."""
        m = self.max_step_out
        idx = self._idx
        w = self.width[idx, self.d]
        x0 = self.x[idx, self.d]
        lo = x0 - w * u[2]
        J = torch.floor(m * u[3]).clamp_(0, m - 1)
        K = (m - 1) - J
        phase = torch.where(J > 0, 1, torch.where(K > 0, 2, 3)).to(self.phase.dtype)
        self.log_y.copy_(torch.where(mask, self.lp + torch.log(u[1]), self.log_y))
        self.lo.copy_(torch.where(mask, lo, self.lo))
        self.hi.copy_(torch.where(mask, lo + w, self.hi))
        self.x0.copy_(torch.where(mask, x0, self.x0))
        self.J.copy_(torch.where(mask, J, self.J))
        self.K.copy_(torch.where(mask, K, self.K))
        self.phase.copy_(torch.where(mask, phase, self.phase))
        self.nshr.copy_(torch.where(mask, torch.zeros_like(self.nshr), self.nshr))

    def _step_fused(self) -> None:
        import ctypes
        from . import _native
        L = _native.lib()
        stream = torch.cuda.current_stream(self.x.device).cuda_stream
        _native.check(L.ddm_slice_propose_f32(self._ptrs, self._ints, self._u.data_ptr(), self._q.data_ptr(), stream),
                      "ddm_slice_propose_f32")
        f = self.f(self._q)
        self.n_evals += 1
        f = f.to(torch.float32).contiguous()
        _native.check(L.ddm_slice_update_f32(self._ptrs, self._ints, self._u.data_ptr(), f.data_ptr(), stream),
                      "ddm_slice_update_f32")

    def _step(self) -> None:
        """One potential call for all chains, and each chain's move through its own state machine."""
        if self._fused:
            return self._step_fused()
        u, idx, D = self._u, self._idx, self.D
        ph, lo, hi = self.phase, self.lo, self.hi
        w = self.width[idx, self.d]
        q_val = torch.where(ph == 1, lo, torch.where(ph == 2, hi, lo + (hi - lo) * u[0]))
        q = self.x.clone()
        q[idx, self.d] = q_val
        f = self._eval(q)
        inside = f > self.log_y
        live = self.sweeps < self._total
        # stepping out, left end then right end, at most J resp. K expansions
        g1 = (ph == 1) & inside
        g2 = (ph == 2) & inside
        J = self.J - g1.to(self.J.dtype)
        K = self.K - g2.to(self.K.dtype)
        leave1 = (ph == 1) & ~(g1 & (J > 0))
        leave2 = (ph == 2) & ~(g2 & (K > 0))
        lo = torch.where(g1, lo - w, lo)
        hi = torch.where(g2, hi + w, hi)
        # shrinkage
        nshr = self.nshr + (ph == 3).to(self.nshr.dtype)
        give_up = (ph == 3) & ~inside & (nshr >= self.max_shrink)      # (never seen; the chain keeps its point)
        acc = (ph == 3) & inside & live
        rej = (ph == 3) & ~inside & ~give_up
        left = q_val < self.x0
        lo = torch.where(rej & left, q_val, lo)
        hi = torch.where(rej & ~left, q_val, hi)
        self.x[idx, self.d] = torch.where(acc, q_val, self.x[idx, self.d])
        self.lp.copy_(torch.where(acc, f, self.lp))
        ph = torch.where(leave1, torch.where(K > 0, 2, 3).to(ph.dtype), ph)
        ph = torch.where(leave2, torch.full_like(ph, 3), ph)
        self.lo.copy_(lo)
        self.hi.copy_(hi)
        self.J.copy_(J)
        self.K.copy_(K)
        self.nshr.copy_(nshr)
        self.phase.copy_(ph)
        # a finished update: tune the width, move to the next coordinate, count sweeps, record a draw
        fin = (acc | (give_up & live))
        tune = fin & (self.sweeps < self._warmup)
        cnt = self.tuned[idx, self.d]
        self.width[idx, self.d] = torch.where(tune, (w + ((hi - lo) - w) / (cnt + 1.0)).clamp_min(1e-6), w)
        self.tuned[idx, self.d] = cnt + tune.to(cnt.dtype)
        sweep_end = fin & (self.d == D - 1)
        self.d.copy_(torch.where(fin, (self.d + 1) % D, self.d))
        self.sweeps.add_(sweep_end.to(self.sweeps.dtype))
        past = self.sweeps - self._warmup
        rec = sweep_end & (past > 0) & (past % self._thin == 0) & (self.taken < self._S)
        slot = self.taken.clamp(max=self._S - 1)
        cur = self.out[slot, idx]
        self.out[slot, idx] = torch.where(rec[:, None], self.x, cur)
        self.taken.add_(rec.to(self.taken.dtype))
        self._begin(fin & (self.sweeps < self._total), u)

    @torch.no_grad()
    def run(self, num_samples_per_chain: int, *, warmup: int = 100, thin: int = 1) -> torch.Tensor:
        """-> (num_samples_per_chain, N, D): every chain's state after each of its post-warm-up sweeps (every
        ``thin``-th), ``warmup`` tuning sweeps first."""
        dev, N, D = self.x.device, self.N, self.D
        S, thin, warmup = int(num_samples_per_chain), max(int(thin), 1), int(warmup)
        long_, fl = dict(dtype=torch.int64, device=dev), dict(dtype=self.x.dtype, device=dev)
        self._S, self._thin, self._warmup, self._total = S, thin, warmup, warmup + S * thin
        self._idx = torch.arange(N, device=dev)
        self.out = torch.empty((max(S, 1), N, D), **fl)
        self.d, self.sweeps, self.taken = torch.zeros(N, **long_), torch.zeros(N, **long_), torch.zeros(N, **long_)
        self.phase, self.nshr = torch.zeros(N, **long_), torch.zeros(N, **long_)
        self.tuned = torch.zeros((N, D), **fl)
        self.lo, self.hi, self.x0, self.log_y = (torch.zeros(N, **fl) for _ in range(4))
        self.J, self.K = torch.zeros(N, **fl), torch.zeros(N, **fl)
        self._u = self._draw4(self._it).contiguous()
        self._it += 1
        self._graph = None
        if self._fused:
            import ctypes
            self.x, self.lp, self.width = self.x.contiguous(), self.lp.to(torch.float32).contiguous(), self.width.contiguous()
            self._q = torch.empty_like(self.x)
            order = (self.x, self.lp, self.width, self.tuned, self.lo, self.hi, self.x0, self.log_y, self.J, self.K, self.d,
                     self.sweeps, self.taken, self.phase, self.nshr, self.out)
            self._ptrs = (ctypes.c_void_p * 16)(*[t.data_ptr() for t in order])
            self._ints = (ctypes.c_int64 * 8)(N, D, max(S, 1), thin, warmup, self._total, self.max_step_out, self.max_shrink)
        if self._total == 0:
            return self.out[:S]
        self._begin(torch.ones(N, dtype=torch.bool, device=dev), self._u)
        check_every = 16
        while True:
            for _ in range(check_every):
                self._u.copy_(self._draw4(self._it))
                self._it += 1
                self._iterate()
            if not bool((self.sweeps < self._total).any()):
                break
        return self.out[:S].clone()

    def _iterate(self) -> None:
        if not self._use_graph:
            self._step()
            return
        if self._graph is None:
            dev = self.x.device
            snap = {k: v.clone() for k, v in self._state().items()}      # the warm-up calls below must not count
            evals = self.n_evals
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            try:
                with torch.cuda.stream(side):
                    self._step()
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, stream=side):
                        self._step()
                self._graph = graph
            except Exception:        # the potential synchronises or leaves the device: run eagerly
                self._use_graph = False
                torch.cuda.synchronize(dev)
            torch.cuda.current_stream(dev).wait_stream(side)
            for k, v in self._state().items():
                v.copy_(snap[k])
            self.n_evals = evals
            if not self._use_graph:
                self._step()
                return
        self._graph.replay()
        self.n_evals += 1

    def _state(self):
        return {k: getattr(self, k) for k in ("x", "lp", "width", "tuned", "d", "sweeps", "taken", "phase", "nshr", "lo", "hi",
                                               "x0", "log_y", "J", "K", "out")}
