#!/usr/bin/env python
"""Benchmark of the B200 pulse-DDM hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU algorithm

Workload (BASELINE.json configs[1]): a 1e8-trial MNLE training set drawn from
ExtendedProposal (pipeline prior for theta, PulseSequenceProposal(P=80, p=0.75, seed=0) for the
pulses) with the default schedule (n_max=16000, steps_per_pulse=200), resident in HBM as
z (1e8, 85) fp32 = 34 GB.  A "step" is one pass of the simulator over all of it (one
``ddm_sim_f32`` launch; new Philox key every step).  With N>1 every rank owns its own 1e8-trial
shard of one global trial index space (weak scaling); the all-gather of x -- the only exchange the
path has -- is fused into the simulator kernel: every finished trial's 8 bytes are stored into all ranks'
gathered array over NVLink peer memory (``ddm_sim_gather_f32``, ``sharding.PeerGather``), with a stream barrier
per step; NCCL ``all_gather_into_tensor`` is the fallback when symmetric memory cannot be set up.

Besides the headline line the N > 1 arm checks on the device that the gathered x equals a single-rank
recomputation of another rank's rows (``sharded_equals_single``) and measures BASELINE configs[2] (long
schedule, 1.25e8 trials per GPU), configs[3] with the chains split over the ranks and configs[4] (run_sbc, 125
datasets per GPU = 1000 on 8 GPUs), each with its own sharded-equals-single check.

Metric: useful Euler steps per second (sum over trials of the first-passage / censoring step,
the count the reference's loop would have had to execute for those trials), whole job.

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "simulated DDM Euler steps/sec"
UNIT = "steps/s"
W_ALG = 7             # fp32 lane-ops per useful step in the reference's unfused form (SURVEY 8d)
BYTES_PER_TRIAL = 348  # 340 B of z in + 8 B of x out
P = 80
DUMP_ROWS = 1 << 21    # --dump-outputs: 16 MB of the 800 MB x of a 1e8-trial step


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--trials", type=int, default=int(os.environ.get("DDM_BENCH_TRIALS", 100_000_000)),
                    help="trials per GPU per step (default: the 1e8-trial config)")
    ap.add_argument("--e2e-trials", type=int, default=int(os.environ.get("DDM_BENCH_E2E_TRIALS", 1 << 24)),
                    help="trials per end-to-end step (default 2^24 = 5.7 GB of pinned host z per rank: four batches of the "
                         "streaming pipeline per call; the headline's 1e8 would pin 34 GB per rank, 272 GB on 8 GPUs)")
    ap.add_argument("--cpu-trials", type=int, default=int(os.environ.get("DDM_BENCH_CPU_TRIALS", 65536)),
                    help="trials per CPU step: the lock-step reference algorithm only amortises its ~19 tensor-op "
                         "dispatches per Euler step at large batches (2x the per-trial rate of the 4096 batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--long-trials", type=int, default=int(os.environ.get("DDM_BENCH_LONG_TRIALS", 125_000_000)),
                    help="configs[2]: trials per GPU on the long schedule dt=1e-4 (1e9 on 8 GPUs); 0 skips it")
    ap.add_argument("--sbc-datasets", type=int, default=int(os.environ.get("DDM_BENCH_SBC_DATASETS", 125)),
                    help="configs[4]: SBC datasets per GPU (1000 on 8 GPUs); 0 skips it")
    ap.add_argument("--train-set-trials", type=int, default=int(os.environ.get("DDM_BENCH_TRAINSET_TRIALS", 10_000_000)),
                    help="end-to-end simulate_training_set_with_conditions leg (N=1 only); 0 skips it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write x of the last timed step to DIR/x.npy (float32, (rows, 2)) so that two builds can be "
                         f"compared: every row when there are at most {DUMP_ROWS}, else {DUMP_ROWS} rows drawn without "
                         "replacement by numpy default_rng(0), in ascending row order")
    return ap.parse_args()


# ------------------------------------------------------------------------------- clocks ---

class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML, 100 ms)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no NVML samples"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "power_w_max": max(self.power), "samples": len(self.samples)}


# -------------------------------------------------------------------------- reference arm ---

def cpu_sample(n_trials: int, seed: int):
    """A bounded sample of the workload on the host: same prior family, same pulse stream."""
    import numpy as np
    import torch
    from oracle import ddm_oracle as orc
    theta = orc.prior_sample(n_trials, seed=seed)
    st, inc = orc.pcg64_state(np.random.default_rng(0))
    pulses = torch.from_numpy(orc.pulses_pcg64_c(st, inc, 0, n_trials, P, 0.75))
    return theta, pulses


def time_cpu_port(n_trials: int, repeats: int, warmup: int):
    """The reference's own CPU algorithm (lock-step torch ops + torch.randn, restated in
    oracle/ddm_oracle.py) on all host threads torch uses.  Returns (steps/s, seconds, steps)."""
    import torch
    from oracle import ddm_oracle as orc
    theta, pulses = cpu_sample(n_trials, seed=1)
    torch.manual_seed(0)
    for _ in range(warmup):
        orc.sim_lockstep_torch(theta[:256], pulses[:256])
    times, steps = [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        _, when, _ = orc.sim_lockstep_torch(theta, pulses)
        times.append(time.perf_counter() - t0)
        steps.append(int(when.sum()))
    return sum(steps) / sum(times), times, steps


def time_cpu_port_cfg1():
    """configs[0] as the reference runs it (README default: NUM_SIMULATIONS = 10 000 in batches of
    TRAIN_BATCH_SIZE = 4096, data_simulator.py:46-58): the lock-step port over 4096 + 4096 + 1808 trials."""
    import torch
    from oracle import ddm_oracle as orc
    theta, pulses = cpu_sample(10_000, seed=2)
    torch.manual_seed(0)
    t0 = time.perf_counter()
    steps = 0
    for a in range(0, 10_000, 4096):
        _, when, _ = orc.sim_lockstep_torch(theta[a:a + 4096], pulses[a:a + 4096])
        steps += int(when.sum())
    dt = time.perf_counter() - t0
    return {"trials": 10_000, "batch": 4096, "seconds": dt, "steps_per_s": steps / dt, "trials_per_s": 10_000 / dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host core it can
    try:
        torch.set_num_threads(len(os.sched_getaffinity(0)))
    except Exception:
        torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    rate, times, steps = time_cpu_port(args.cpu_trials, args.steps, args.warmup)
    ms = 1e3 * sum(times) / len(times)
    sample = (f"{args.cpu_trials} trials per step of the same workload (pipeline prior, PCG64 pulse stream seed 0, "
              f"default schedule), lock-step torch port of rt_choice_model.py:112-221 with torch.randn")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1] sample: ExtendedProposal training set, default schedule "
                               "(n_max=16000, steps_per_pulse=200, P=80)", "trials_per_step": args.cpu_trials,
                   "host_threads": cores, "os_cpu_count": os.cpu_count()},
        "trials_per_s": args.cpu_trials * len(times) / sum(times),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- native arm ---

def build_workload(n: int, rank: int, device):
    """z (n, 85) on the device: theta ~ pipeline prior (rt_choice_model_pipeline.py:38-46),
    pulses = rows [rank*n, (rank+1)*n) of PulseSequenceProposal(P=80, p=0.75, seed=0)'s stream."""
    import numpy as np
    import torch
    from torch.distributions import Beta, LogNormal
    from sbi_for_diffusion_models_b200.pulses import pcg64_state, pulses_from_state

    z = torch.empty((n, 5 + P), dtype=torch.float32, device=device)
    gen_seed = 1000 + rank
    torch.manual_seed(gen_seed)
    one = lambda v: torch.tensor(v, device=device)
    chunk = 1 << 24
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        m = b - a
        z[a:b, 0] = Beta(one(2.0), one(2.0)).sample((m,))
        z[a:b, 1] = LogNormal(one(-1.0), one(1.0)).sample((m,))
        z[a:b, 2] = LogNormal(one(0.0), one(1.0)).sample((m,))
        z[a:b, 3] = LogNormal(one(2.75), one(0.5)).sample((m,))
        z[a:b, 4] = Beta(one(2.0), one(2.0)).sample((m,))
    state, inc = pcg64_state(np.random.default_rng(0))
    pulses_from_state(state, inc, rank * n, n, P, 0.75, out=z[:, 5:])
    return z


def dump_outputs(out_dir: str, x) -> None:
    """x (device, (n, 2) float32) as out_dir/x.npy: all rows, or DUMP_ROWS of them sampled with a fixed seed."""
    import numpy as np
    import torch
    n = x.shape[0]
    if n > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
        x = x[torch.from_numpy(rows).to(x.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), x.cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------- MNLE potential (cfg-4) ---

def random_mnle_params(seed: int = 0):
    """Seeded random MNLE parameters with the reference's architecture (no trained checkpoint
    exists offline); same family as the test nets."""
    import numpy as np
    import torch
    rs = np.random.RandomState(seed)

    def lin(n_out, n_in, s=1.0):
        b = s / np.sqrt(n_in)
        return (torch.from_numpy(rs.uniform(-b, b, (n_out, n_in)).astype(np.float32)),
                torch.from_numpy(rs.uniform(-b, b, (n_out,)).astype(np.float32)))

    p = {"cond_mean": torch.cat([torch.tensor([0.5, 0.6, 1.6, 17.7, 0.5]), torch.zeros(80)]),
         "cond_std": torch.cat([torch.tensor([0.22, 0.8, 2.1, 9.4, 0.22]), torch.ones(80)]),
         "flow.mu_y": torch.tensor(0.35), "flow.sigma_y": torch.tensor(1.1)}
    p["cat.W0"], p["cat.b0"] = lin(128, 85)
    p["cat.W1"], p["cat.b1"] = lin(128, 128)
    p["cat.W2"], p["cat.b2"] = lin(128, 128)
    p["cat.Wo"], p["cat.bo"] = lin(3, 128)
    for k in range(10):
        p[f"flow.{k}.W1"], p[f"flow.{k}.b1"] = lin(128, 86)
        p[f"flow.{k}.W2"], p[f"flow.{k}.b2"] = lin(128, 128)
        p[f"flow.{k}.W3"], p[f"flow.{k}.b3"] = lin(71, 128, 4.0)
    return p


def trained_mnle():
    """(DeviceMNLE, spec parameter dict) of the committed TRAINED estimator (tests/golden/mnle_trained.npz,
    made by tools/train_reference_net.py with this repository's simulator and trainer): the reference only ever
    evaluates a trained net (mnle.py:41-48).  The packed buffer has the z-scoring folded in, so the spec gets
    identity z-scoring and the very same fp32 numbers."""
    import numpy as np
    import torch
    from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE, unpack_params
    d = np.load(os.path.join(ROOT, "tests", "golden", "mnle_trained.npz"))
    packed, K = d["packed"], int(d["n_choices"])
    p = {k: v.clone() for k, v in unpack_params(torch.from_numpy(packed.copy()), K).items()}
    p["cond_mean"], p["cond_std"] = torch.zeros(85), torch.ones(85)
    return DeviceMNLE(PackedMNLE(packed, K)), p


def potential_inputs(dev, T=50, C=1024):
    import torch
    from sbi_for_diffusion_models_b200.data_simulator import simulate_observed_session
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    x_o, pulses_o = simulate_observed_session(torch.tensor([0.45, 0.6, 1.3, 14.0, 0.25]), T, "cpu", mu_sensory=1.0,
                                              p_success=0.75, P=P, seed=123, log_rt=False, noise_seed=1)
    torch.manual_seed(0)
    theta = build_prior_theta().sample((C,)).to(torch.float32)
    return theta, x_o, pulses_o


def _time_graph(fn, reps=20, replays=5):
    """ms per call of ``fn`` captured in a CUDA graph (device time without the Python / ctypes launch path)."""
    import torch
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                fn()
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (replays * reps)


def mnle_bench(dev, with_cpu: bool):
    """configs[3]: MNLE log-likelihood sum over T=50 trials x C=1024 chains on the TRAINED estimator,
    device-resident; the potential's gradient (row f2) at C=1024 and at the reference's NUM_CHAINS=2."""
    import torch
    T, C = 50, 1024
    est, params = trained_mnle()
    theta, x_o, pulses_o = potential_inputs(dev, T, C)
    th, xo, pl = theta.to(dev), x_o.to(dev), pulses_o.to(dev)
    out = {"workload": f"configs[3]: MNLE log_prob sum over T={T} trials x C={C} chains, trained estimator "
                       "(tests/golden/mnle_trained.npz)", "rows": T * C, "dense_mflop_per_row": 0.818}
    lls = {}
    for kernel in ("tc", "simt", "precise", "tc64"):
        for _ in range(3):
            est.loglik_sum(th, xo, pl, kernel=kernel)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            ll = est.loglik_sum(th, xo, pl, kernel=kernel)
        e1.record()
        torch.cuda.synchronize()
        ms_call = e0.elapsed_time(e1) / reps
        lls[kernel] = ll
        ms_graph = _time_graph(lambda: est.loglik_sum(th, xo, pl, kernel=kernel))
        out[kernel] = {"ms_per_call": ms_call, "ms_per_call_graph": ms_graph, "rows_per_s": T * C / (ms_graph * 1e-3),
                       "dense_tflops": 0.818e6 * T * C / (ms_graph * 1e-3) / 1e12}
    # tensor-core work actually issued: hi/lo split = 3 bf16 MMAs per product, N padded (71 -> 80, K -> 16)
    tc_flop_row = 2.0 * (11 * 128 * 32 + 3 * (12 * 128 * 128 + 10 * 80 * 128 + 16 * 128))
    out["tc"]["bf16_mma_tflops"] = tc_flop_row * T * C / (out["tc"]["ms_per_call_graph"] * 1e-3) / 1e12
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
        src = "MEASURED_PEAKS.json bf16_tflops (burst: the kernel is timed alone)"
    except Exception:
        peak, src = 1590.0, "fallback"
    out["tc"]["roofline"] = {"bound": "tensor", "achieved": out["tc"]["bf16_mma_tflops"], "peak": peak, "unit": "TFLOP/s",
                             "frac": out["tc"]["bf16_mma_tflops"] / peak, "peak_source": src,
                             "flop_per_row": tc_flop_row,
                             "frac_algorithmic": 0.818e6 * T * C / (out["tc"]["ms_per_call_graph"] * 1e-3) / 1e12 / peak,
                             "note": "bf16 MMA flops issued per (trial, chain) row: 3 passes (hi*hi, hi*lo, lo*hi) over "
                                     "the 128x128 / 128x80 layers + the K=32 theta stage; frac_algorithmic counts the "
                                     "0.818 MFLOP of fp32 dense work per row of SURVEY 8d instead"}
    # row f2: value + d/d theta (what NUTS asks the potential for, potentials.py:112) at C = 1024 and C = 2
    grad = {}
    for Cg in (C, 2):
        thg = th[:Cg].contiguous()
        for _ in range(3):
            est.loglik_sum_and_grad(thg, xo, pl)
        grad[f"C{Cg}"] = {"ms_per_call_graph": _time_graph(lambda: est.loglik_sum_and_grad(thg, xo, pl), reps=5),
                          "ms_reverse_mode_tcgen05": _time_graph(lambda: est.loglik_sum_and_grad(thg, xo, pl, kernel="tc"), reps=5),
                          "ms_forward_mode_fp32": _time_graph(lambda: est.loglik_sum_and_grad(thg, xo, pl, kernel="simt"), reps=5),
                          "ms_forward_only_graph": _time_graph(lambda: est.loglik_sum(thg, xo, pl), reps=5)}
    out["grad"] = grad
    if with_cpu:
        from oracle import mnle_spec
        t0 = time.perf_counter()
        ref32 = mnle_spec.loglik_sum(params, theta, x_o, pulses_o).double()
        out["cpu_spec_fp32"] = {"ms_per_call": (time.perf_counter() - t0) * 1e3, "cores": torch.get_num_threads(),
                                "kind": "port (oracle/mnle_spec.py; sbi itself is not installable offline)"}
        # float64 spec, row by row: the sums (C,) and the L1 norm of each sum's T summands.  |sum| can be arbitrarily
        # close to zero (50 log-densities of either sign), so the error is reported three ways: relative to |sum|
        # (rel_err: ill-conditioned, its maximum is whichever chain's sum happens to sit nearest zero), absolute
        # (abs_err: what an MCMC acceptance ratio sees), and relative to the L1 norm of the summands (rel_l1)
        xr, cond = mnle_spec.potential_rows(theta, x_o, pulses_o)
        rows64 = mnle_spec.log_prob(mnle_spec.cast_params(params, torch.float64), xr.double(), cond.double()).reshape(T, C)
        ref64, l1 = rows64.sum(0), rows64.abs().sum(0)

        def errs(v):
            e = (v.double().cpu() - ref64).abs()
            return {"rel_err_vs_float64": {"max": float((e / ref64.abs()).max()), "median": float((e / ref64.abs()).median())},
                    "abs_err_vs_float64": {"max": float(e.max()), "median": float(e.median())},
                    "rel_l1_vs_float64": {"max": float((e / l1).max()), "median": float((e / l1).median())}}
        out["cpu_spec_fp32"].update(errs(ref32))
        out["sum_magnitudes"] = {"abs_sum_min": float(ref64.abs().min()), "abs_sum_median": float(ref64.abs().median()),
                                 "l1_median": float(l1.median())}
        for kernel, ll in lls.items():
            out[kernel].update(errs(ll))
    return out


def configs0_bench(dev):
    """configs[0] through the public API on the GPU: simulate_training_set_with_conditions(ExtendedProposal,
    NUM_SIMULATIONS = 10 000, TRAIN_BATCH_SIZE = 4096) -> CPU (z, x), proposal sampling included."""
    import contextlib
    import io
    import torch
    from sbi_for_diffusion_models_b200 import data_simulator as ds
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.proposals import ExtendedProposal, PulseSequenceProposal

    # as in the reference's pipeline (rt_choice_model_pipeline.py:38-75) the prior is built once, outside the call
    priors = {None: build_prior_theta(None), dev: build_prior_theta(dev)}

    def once(seed, prior_dev=None):
        prop = ExtendedProposal(priors[prior_dev], PulseSequenceProposal(P, 0.75, seed=seed, device=dev), device=dev)
        with contextlib.redirect_stdout(io.StringIO()):
            return ds.simulate_training_set_with_conditions(prop, 10_000, 4096, dev, mu_sensory=1.0, p_success=0.75, P=P,
                                                            log_rt=False, seed=seed)

    def timed(prior_dev):
        for i in range(3):
            once(100 + i, prior_dev)
        torch.cuda.synchronize()
        ts = []
        for i in range(9):
            t0 = time.perf_counter()
            z, x = once(1 + i, prior_dev)
            ts.append(time.perf_counter() - t0)
        return sorted(ts)[4], z, x
    dt, z, x = timed(None)
    dt_dev, _, _ = timed(dev)
    steps = float(torch.round((x[:, 0] - z[:, 4].clamp(0.0, 7.999999)) / 5e-4).sum())
    # simulate_observed_session (data_simulator.py:74-99) at NUM_TRIALS_OBS = 50: what run_sbc calls once per dataset
    theta_true = torch.tensor([0.45, 0.6, 1.3, 14.0, 0.25])
    sess = lambda seed: ds.simulate_observed_session(theta_true, 50, dev, mu_sensory=1.0, p_success=0.75, P=P, seed=seed, log_rt=False)
    for i in range(3):
        sess(i)
    ts = []
    for i in range(9):
        t0 = time.perf_counter()
        sess(10 + i)
        ts.append(time.perf_counter() - t0)
    return {"workload": "configs[0]: simulate_training_set_with_conditions, 10 000 trials in batches of 4096, CPU (z, x) out",
            "seconds": dt, "trials_per_s": 10_000 / dt, "steps_per_s": steps / dt, "seconds_with_cuda_prior": dt_dev,
            "observed_session_T50_seconds": sorted(ts)[4],
            "note": "median of 9 calls, prior object built once outside the call as in the reference's pipeline.  seconds: the "
                    "reference's CPU prior object -- most of it is torch's CPU Beta sampler (tools/time_configs0.py); "
                    "seconds_with_cuda_prior: the same call with the prior's parameters on the GPU; observed_session_T50_seconds: "
                    "simulate_observed_session(theta, 50 trials) -> CPU (x_o, pulses_o), one launch of the small-batch kernel "
                    "(floor: 16 000 serial Euler steps = 0.38 ms)"}


def long_schedule_bench(args, z, rank, world, dev, gather):
    """BASELINE configs[2]: the long pulse schedule (dt = 1e-4: n_max = 80 000, steps_per_pulse = 1000, P = 80),
    ``--long-trials`` trials per GPU (1.25e8: 1e9 on 8 GPUs), gather of x included.  One warm-up + two timed
    launches, device time, max over ranks."""
    import torch
    import torch.distributed as dist
    from sbi_for_diffusion_models_b200.simulator import Schedule, simulate_trials
    n = min(args.long_trials, z.shape[0])
    sched = Schedule.from_constants(1.0, dt=1e-4)
    zz = z[:n]
    pg = gather(n)
    x = pg.local if pg is not None else torch.empty((n, 2), dtype=torch.float32, device=dev)
    x_all = None if pg is not None or world == 1 else torch.empty((world * n, 2), dtype=torch.float32, device=dev)

    def launch(seed):
        simulate_trials(zz[:, :5], zz[:, 5:], seed=seed, trial_offset=rank * n, out=x, schedule=sched,
                        peer_blocks=pg.peers if pg is not None else None)
        if pg is not None:
            pg.barrier()
        elif world > 1:
            dist.all_gather_into_tensor(x_all, x)

    launch(900)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    e0.record()
    for i in range(reps):
        launch(901 + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    useful = 0
    for i in range(reps):       # exact useful-step totals of the timed keys (untimed, plain launch)
        _, st = simulate_trials(zz[:, :5], zz[:, 5:], seed=901 + i, trial_offset=rank * n, schedule=sched, return_stats=True)
        useful += st.useful_steps
    t = torch.tensor([ms, float(useful)], dtype=torch.float64, device=dev)
    if world > 1:
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, useful = float(tm[0]), float(t[1])
    else:
        useful = float(useful)
    return {"workload": f"configs[2]: {world} x {n} trials, long schedule dt=1e-4 (n_max={sched.n_max}, "
                        f"steps_per_pulse={sched.steps_per_pulse}, P={sched.n_pulses}), gather of x included",
            "trials_total": world * n, "ms_per_launch": ms, "useful_steps_per_s": useful / reps / (ms * 1e-3),
            "trials_per_s": world * n / (ms * 1e-3), "mean_steps_per_trial": useful / reps / (world * n),
            "exchange": "fused peer stores" if pg is not None else ("all_gather(x)" if world > 1 else "none")}


def sbc_bench(args, rank, world, dev):
    """BASELINE configs[4]: run_sbc (reference mnle.py:128-237) over ``--sbc-datasets`` datasets per GPU (125: 1000
    on 8 GPUs) with the reference's own settings -- NUM_TRIALS_OBS = 50, WARMUP_STEPS = 100, SBC_POST_SAMPLES = 1500 --
    on the trained estimator: per dataset a prior draw, a simulated session, a posterior sample (128 chains of the
    device slice sampler in lock-step over all datasets of the rank) and the ranks; datasets sharded over the
    GPUs, ranks and samples all-gathered.  Then the check: every rank recomputes three datasets of ANOTHER rank's
    shard on its own and must find the very same ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from sbi_for_diffusion_models_b200 import mnle
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    from sbi_for_diffusion_models_b200.sbc import draw_sbc_datasets
    from sbi_for_diffusion_models_b200.sharding import shard_bounds
    est, _ = trained_mnle()
    cfg = RunConfig()
    prior = build_prior_theta()
    D, S, chains, seed = args.sbc_datasets * world, int(cfg.SBC_POST_SAMPLES), 128, 0
    small = RunConfig(WARMUP_STEPS=2)
    mnle.run_sbc(small, prior_theta=prior, density_estimator=est, num_datasets=2 * world, posterior_samples_per_dataset=128,
                 save=False)                                                   # warm-up: allocator, graphs
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    out = mnle.run_sbc(cfg, prior_theta=prior, density_estimator=est, num_datasets=D, posterior_samples_per_dataset=S,
                       seed=seed, chains_per_dataset=chains, save=False)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    ok = True
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        # datasets [lo, lo + 3) of the next rank's shard, recomputed here without any other dataset around
        thetas_true, ds_seeds = draw_sbc_datasets(prior, D, seed)
        init_all = prior.sample((D * chains,)).to(torch.float32)
        lo, _ = shard_bounds(D, (rank + 1) % world, world)
        ranks_again, _ = mnle.sbc_shard(cfg, prior, est, thetas_true, ds_seeds, init_all, lo, lo + 3, S, seed, dev)
        ok = bool(np.array_equal(ranks_again.numpy(), out["ranks"][lo:lo + 3]))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    dt = float(tt.item())
    ranks = out["ranks"].astype(np.float64) / S
    return {"workload": f"configs[4]: run_sbc, {D} datasets over {world} GPU(s), T={cfg.NUM_TRIALS_OBS} trials each, "
                        f"{chains} chains x ({cfg.WARMUP_STEPS} warm-up sweeps + {-(-S // chains)} draws), {S} posterior "
                        "samples per dataset, trained estimator",
            "datasets": D, "seconds": dt, "datasets_per_s": D / dt,
            "rank_mean_over_S": ranks.mean(0).tolist(), "rank_std_over_S": ranks.std(0).tolist(),
            "sharded_equals_single": ok if world > 1 else None,
            "note": "uniform ranks have mean 0.5 and std 0.289; the estimator was trained on 1e6 simulated trials"}


def mcmc_bench(dev):
    """run_inference_mcmc (reference mnle.py:52-95) with the reference's run_config: one observed session of
    NUM_TRIALS_OBS = 50 trials, WARMUP_STEPS = 100, POSTERIOR_SAMPLES = 1000, on the trained estimator.  The reference
    runs pyro NUTS with NUM_CHAINS = 2 CPU processes; here 128 slice-sampling chains advance per potential launch."""
    import torch
    from sbi_for_diffusion_models_b200 import mnle, samplers
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    est, _ = trained_mnle()
    cfg, prior = RunConfig(), build_prior_theta()
    _, x_o, pulses_o = potential_inputs(dev)
    calls = {"n": 0}
    orig = samplers.VectorizedSliceSampler.run

    def counting(self, *a, **kw):
        out = orig(self, *a, **kw)
        calls["n"] += self.n_evals
        return out
    samplers.VectorizedSliceSampler.run = counting
    try:
        mnle.run_inference_mcmc(RunConfig(WARMUP_STEPS=2, POSTERIOR_SAMPLES=128), prior, est, x_o, pulses_o)   # warm-up
        torch.cuda.synchronize()
        calls["n"] = 0
        t0 = time.perf_counter()
        samples = mnle.run_inference_mcmc(cfg, prior, est, x_o, pulses_o)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        samplers.VectorizedSliceSampler.run = orig
    return {"workload": f"run_inference_mcmc: T={cfg.NUM_TRIALS_OBS} trials, 128 chains, {cfg.WARMUP_STEPS} warm-up sweeps, "
                        f"{cfg.POSTERIOR_SAMPLES} posterior samples, trained estimator",
            "seconds": dt, "potential_calls": calls["n"], "ms_per_call": dt / max(calls["n"], 1) * 1e3,
            "posterior_mean": samples.mean(0).tolist(), "theta_true": [0.45, 0.6, 1.3, 14.0, 0.25]}


def potential_sharded_bench(rank, world, dev):
    """configs[3] with the chains split over the ranks (SURVEY 8e): weights replicated, every rank sums its own
    chains, one all-gather of C floats; must equal the single-GPU call bit for bit."""
    import torch
    import torch.distributed as dist
    from sbi_for_diffusion_models_b200.sharding import loglik_sum_sharded
    est, _ = trained_mnle()
    theta, x_o, pulses_o = potential_inputs(dev)
    th, xo, pl = theta.to(dev), x_o.to(dev), pulses_o.to(dev)
    fn = lambda t: est.loglik_sum(t, xo, pl)
    for _ in range(3):
        got = loglik_sum_sharded(fn, th)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        got = loglik_sum_sharded(fn, th)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    flag = torch.tensor([1 if torch.equal(got, fn(th)) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"workload": f"configs[3]: T=50 x C=1024 chains split over {world} GPUs, all-gather of the C sums",
            "ms_per_call": float(t.item()), "rows_per_s": 51200 / (float(t.item()) * 1e-3),
            "sharded_equals_single": bool(flag.item())}


def training_set_e2e_bench(args, dev):
    """The entry point north_star names, end to end at size: simulate_training_set_with_conditions(ExtendedProposal
    on the device, N trials, batch 2^18) -> CPU (z (N,85), x (N,2)) -- proposal draws, simulation and the
    device->host copy of z and x (348 B per trial) all inside the timed region."""
    import contextlib
    import io
    import torch
    from sbi_for_diffusion_models_b200 import data_simulator as ds
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.proposals import ExtendedProposal, PulseSequenceProposal
    N = args.train_set_trials

    def once(seed, n):
        prop = ExtendedProposal(build_prior_theta(dev), PulseSequenceProposal(P, 0.75, seed=seed, device=dev), device=dev)
        with contextlib.redirect_stdout(io.StringIO()):
            return ds.simulate_training_set_with_conditions(prop, n, 1 << 18, dev, mu_sensory=1.0, p_success=0.75, P=P,
                                                            log_rt=False, seed=seed)
    once(0, 1 << 20)
    torch.cuda.synchronize()
    ts, steps = [], 0.0
    for i in range(2):
        t0 = time.perf_counter()
        z, x = once(1 + i, N)
        ts.append(time.perf_counter() - t0)
        steps = float(torch.round((x[:, 0].double() - z[:, 4].double().clamp(0.0, 7.999999)) / 5e-4).sum())
        del z, x
    dt = min(ts)
    return {"api": "data_simulator.simulate_training_set_with_conditions(ExtendedProposal on cuda) -> CPU (z, x)",
            "trials": N, "seconds": dt, "trials_per_s": N / dt, "value": steps / dt, "unit": UNIT,
            "d2h_bytes": N * 40, "h2d_bytes": 0, "host_bytes_out": N * BYTES_PER_TRIAL,
            "note": "z comes home as 32-byte records (theta bits + pulse sign masks, packed by the GPU) and is rebuilt to "
                    "fp32 rows by the host cores while the next block is simulated; x as it is (8 B per trial)"}


def mnle_train_bench(dev, with_cpu: bool, rows: int = 4096):
    """Row f4: one MNLE training step (TRAIN_BATCH_SIZE = 4096 rows, run_config.py:12) = loss + gradient +
    Adam on the device; the same step through the CPU spec under torch autograd beside it."""
    import numpy as np
    import torch
    from sbi_for_diffusion_models_b200.mnle_train import MNLETrainer
    N = 1 << 18
    p = random_mnle_params(0)
    z = build_workload(N, 0, dev)
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.stack([torch.exp(torch.rand(N, device=dev, generator=g) * 5.1 - 3.0),
                     torch.randint(0, 3, (N,), device=dev, generator=g).float()], 1).contiguous()
    tr = MNLETrainer(3, cond_mean=p["cond_mean"], cond_std=p["cond_std"], mu_y=0.35, sigma_y=1.1, init=p, device=dev)
    cd = tr.standardise(z)
    idx = [torch.randperm(N, device=dev, generator=g)[:rows].contiguous() for _ in range(8)]
    for i in range(5):
        tr.nll(x, cd, idx[i % 8])
        tr.adam()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 50
    e0.record()
    for i in range(steps):
        tr.nll(x, cd, idx[i % 8])
        tr.adam()
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / steps
    e0.record()
    for i in range(steps):
        tr.nll(x, cd, idx[i % 8], grad=False)
    e1.record()
    torch.cuda.synchronize()
    ms_fwd = e0.elapsed_time(e1) / steps
    out = {"workload": f"row f4: MNLE training step, {rows}-row minibatch gathered from {N} resident rows, "
                       "loss + gradient of all 412 489 parameters + clip + Adam",
           "rows": rows, "ms_per_step": ms_step, "ms_loss_only": ms_fwd, "rows_per_s": rows / (ms_step * 1e-3),
           "dense_tflops": 3 * 0.818e6 * rows / (ms_step * 1e-3) / 1e12,
           "note": "dense work = forward + backward-data + weight-gradient products, 3 x 0.818 MFLOP per row, all on "
                   "tcgen05 (bf16 hi/lo operands, 3 MMAs per product)",
           "loss_after": float(tr.stats[0])}
    if with_cpu:
        from oracle import mnle_spec
        frozen = ("cond_mean", "cond_std", "flow.mu_y", "flow.sigma_y")
        pc = {k: v.clone().requires_grad_(k not in frozen) for k, v in p.items()}
        opt = torch.optim.Adam([v for k, v in pc.items() if k not in frozen], lr=5e-4)
        xs, cs = x[:rows].cpu(), z[:rows].cpu()
        ts = []
        for _ in range(4):
            t0 = time.perf_counter()
            opt.zero_grad()
            loss = -mnle_spec.log_prob(pc, xs, cs).mean()
            loss.backward()
            torch.nn.utils.clip_grad_norm_([v for k, v in pc.items() if k not in frozen], 5.0)
            opt.step()
            ts.append(time.perf_counter() - t0)
        out["cpu_spec_autograd_fp32"] = {"ms_per_step": 1e3 * float(np.median(ts[1:])), "cores": torch.get_num_threads(),
                                         "kind": "port (oracle/mnle_spec.py under torch autograd; sbi is not installable offline)"}
    return out


def run_native(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sbi_for_diffusion_models_b200 import _native
    from sbi_for_diffusion_models_b200 import data_simulator as ds
    from sbi_for_diffusion_models_b200.simulator import Schedule, simulate_trials

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _native.lib()

    n = args.trials
    sched = Schedule.from_constants(1.0)
    z_big = build_workload(max(n, args.long_trials), rank, dev)   # configs[2] re-uses (and extends) the same z
    z = z_big[:n]
    torch.cuda.synchronize()

    # ---- the exchange: fused into the kernel over peer memory, NCCL as the fallback --------------------
    gather_note = "none"
    peer_ok = world > 1 and os.environ.get("DDM_BENCH_EXCHANGE", "peer") == "peer"

    def make_gather(rows):
        """PeerGather over `rows` trials per rank, or None (single GPU / symmetric memory unavailable)."""
        nonlocal peer_ok
        if not peer_ok:
            return None
        try:
            from sbi_for_diffusion_models_b200.sharding import PeerGather
            return PeerGather(rows)
        except Exception as e:   # every rank must take the same branch: agree below
            print(f"[rank {rank}] symmetric memory unavailable, falling back to NCCL all_gather: {e!r}", file=sys.stderr)
            return None

    pg = make_gather(n)
    if world > 1:
        agree = torch.tensor([1 if pg is not None else 0], device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if int(agree.item()) == 0:
            pg, peer_ok = None, False
    if pg is not None:
        x, x_all = pg.local, pg.x_all
        gather_note = ("fused into the kernel: 8-byte peer stores over NVLink into every rank's gathered x "
                       "(ddm_sim_gather_f32), one stream barrier per step")
    else:
        x = torch.empty((n, 2), dtype=torch.float32, device=dev)
        x_all = torch.empty((world * n, 2), dtype=torch.float32, device=dev) if world > 1 else None
        if world > 1:
            gather_note = "NCCL all_gather_into_tensor(x) after each launch"
    torch.cuda.synchronize()

    base_seed = 20261018

    def step(i, events=None):
        if events is not None:
            events[0].record()
        simulate_trials(z[:, :5], z[:, 5:], seed=base_seed + i, trial_offset=rank * n, out=x, schedule=sched,
                        peer_blocks=pg.peers if pg is not None else None)
        if events is not None:
            events[1].record()
        if pg is not None:
            pg.barrier()
        elif world > 1:
            dist.all_gather_into_tensor(x_all, x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # useful steps of a step depend on its key: recount each timed key afterwards (outside timing)
    for i in range(args.warmup):
        step(-1 - i)
    barrier()

    clocks = ClockSampler(local)
    kernel_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                     for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.start()
    barrier()
    t_start.record()
    for i in range(args.steps):
        step(i, kernel_events[i])
    t_end.record()
    barrier()
    clock_info = clocks.stop()
    elapsed_ms = t_start.elapsed_time(t_end)
    kernel_ms = [a.elapsed_time(b) for a, b in kernel_events]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x_all if x_all is not None else x)

    # ---- N > 1: the gathered x of the last timed step equals a single-rank recomputation -------------
    # Every rank takes 65 536 rows of the NEXT rank's z (all-gathered), simulates them alone with that
    # rank's global trial offsets and compares with what the exchange delivered here.
    sharded_equals_single = None
    if world > 1:
        m = min(65536, n)
        z_heads = torch.empty((world * m, 5 + P), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(z_heads, z[:m].contiguous())
        nb = (rank + 1) % world
        zn = z_heads[nb * m:(nb + 1) * m]
        again = simulate_trials(zn[:, :5], zn[:, 5:], seed=base_seed + args.steps - 1, trial_offset=nb * n, schedule=sched)
        flag = torch.tensor([1 if torch.equal(again, x_all[nb * n:nb * n + m]) else 0], device=dev)
        mine = torch.tensor([1 if torch.equal(x_all[rank * n:(rank + 1) * n], x) else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.all_reduce(mine, op=dist.ReduceOp.MIN)
        sharded_equals_single = bool(flag.item()) and bool(mine.item())
        del z_heads

    # recount useful steps per timed key (same launches, untimed) to get exact totals
    useful, lane = 0, 0
    for i in range(args.steps):
        _, st = simulate_trials(z[:, :5], z[:, 5:], seed=base_seed + i, trial_offset=rank * n, out=x,
                                schedule=sched, return_stats=True)
        useful += st.useful_steps
        lane += st.lane_steps
    choice_frac = (torch.bincount(x[:, 1].to(torch.int64), minlength=3).float() / n).tolist()

    tot = torch.tensor([float(useful), float(lane)], dtype=torch.float64, device=dev)
    tmax = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    useful_all, lane_all = tot.tolist()
    elapsed_ms = float(tmax.item())
    value = useful_all / (elapsed_ms * 1e-3)

    # ---- end to end through the public API with HOST buffers (pinned), copies timed --------
    n_e2e = min(args.e2e_trials, n)
    z_host = torch.empty((n_e2e, 5 + P), dtype=torch.float32, pin_memory=True)
    z_host.copy_(z[:n_e2e])
    torch.cuda.synchronize()
    xo = None
    for i in range(max(args.warmup, 5)):   # (5: the ingest tries packed records and fp32 rows twice each, then keeps the faster)
        xo = ds.sim_wrapper(z_host, mu_sensory=1.0, p_success=0.75, P=P, log_rt=False, seed=base_seed - 1 - i,
                            trial_offset=rank * n)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    link0 = ds.host_pipeline_counters()["h2d_bytes"]
    e0.record()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        # each step: host z -> device, simulate, x back on the host.  The previous step's result is
        # dropped, as a caller consuming x batch by batch would (its pinned block is reused).
        xo = ds.sim_wrapper(z_host, mu_sensory=1.0, p_success=0.75, P=P, log_rt=False, seed=base_seed + i,
                            trial_offset=rank * n)
    e1.record()
    torch.cuda.synchronize()
    wall_e2e = time.perf_counter() - wall0
    link_bytes_per_step = (ds.host_pipeline_counters()["h2d_bytes"] - link0) // args.steps
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), wall_e2e * 1e3)
    # useful steps of the timed calls: the same keys again, untimed (results are deterministic)
    t_nd = z_host[:, 4].clamp(0.0, sched.t_nd_hi)
    e2e_steps = 0
    for i in range(args.steps):
        xi = ds.sim_wrapper(z_host, mu_sensory=1.0, p_success=0.75, P=P, log_rt=False, seed=base_seed + i,
                            trial_offset=rank * n)
        if i == args.steps - 1:
            assert torch.equal(xi, xo), "end-to-end path is not reproducible"
        e2e_steps += int(torch.round((xi[:, 0] - t_nd) / sched.dt).to(torch.int64).sum())
        del xi
    e2e_tot = torch.tensor([float(e2e_steps)], dtype=torch.float64, device=dev)
    e2e_t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = float(e2e_tot.item()) / (float(e2e_t.item()) * 1e-3)

    # ---- the other BASELINE configs, on every rank (they contain collectives) ---------------------------
    # A watchdog makes sure the headline line is printed even if one of these legs should hang on some box.
    extras, headline = {}, {}

    def bail():
        if rank == 0 and headline:
            headline["line"]["extras_timeout"] = True
            headline["line"].update(extras)
            print(json.dumps(headline["line"]), flush=True)
        os._exit(0)

    def leg(name, fn):
        try:
            extras[name] = fn()
        except Exception as e:   # the headline metric must still print
            extras[name] = {"error": repr(e)}

    def run_extras():
        if args.long_trials > 0:
            leg("long_schedule", lambda: long_schedule_bench(args, z_big, rank, world, dev, make_gather))
        if world > 1:
            leg("mnle_potential_sharded", lambda: potential_sharded_bench(rank, world, dev))
        if args.sbc_datasets > 0:
            leg("sbc", lambda: sbc_bench(args, rank, world, dev))

    if rank != 0:
        watchdog = threading.Timer(float(os.environ.get("DDM_BENCH_EXTRAS_TIMEOUT", 900)), bail)
        watchdog.daemon = True
        watchdog.start()
        run_extras()
        watchdog.cancel()

    if rank == 0:
        sms, khz = np.zeros(1, np.int32), np.zeros(1, np.int32)
        _native.lib().ddm_device_info(local, sms.ctypes.data, khz.ctypes.data, None, None)
        peaks, peak_src = {}, "fallback"
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peak_src = "MEASURED_PEAKS.json"
        except Exception:
            pass
        sm_max_mhz = float(peaks.get("sm_max_mhz") or clock_info.get("sm_max_mhz") or khz[0] / 1e3)
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        lane_peak = int(sms[0]) * 128 * sm_max_mhz * 1e6           # fp32 lane-ops / s at max clock
        k_ms = sum(kernel_ms) / len(kernel_ms)
        per_launch_steps = useful / args.steps
        achieved = per_launch_steps * W_ALG / (k_ms * 1e-3)
        roofline = {
            "bound": "fp32_issue", "kernel": "ddm::sim_kernel (MASKW=3, Philox, aligned rows, resident z)",
            "achieved": achieved / 1e12, "peak": lane_peak / 1e12, "unit": "TFLOP/s (fp32 lane-ops, FMA=1)",
            "frac": achieved / lane_peak,
            "peak_source": f"{int(sms[0])} SMs x 128 fp32 lanes x sm_max_mhz={sm_max_mhz:.0f} ({peak_src}); "
                           "HBM and bf16 peaks do not bound this kernel (SURVEY 8d)",
            "algorithmic_ops_per_step": W_ALG, "kernel_ms": k_ms,
            "lane_efficiency": useful / lane if lane else None,
            "hbm": {"achieved": BYTES_PER_TRIAL * n / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": BYTES_PER_TRIAL * n / (k_ms * 1e-3) / 1e9 / hbm_peak,
                    "algorithmic_bytes_per_trial": BYTES_PER_TRIAL},
            "traffic": None,
        }
        # evidence from the committed ncu --set full capture of this kernel (profiles/): issue-slot
        # utilisation (what BASELINE's ">= 60 % of FP32 issue" refers to) and DRAM bytes per trial
        try:
            prof_file = json.load(open(os.path.join(ROOT, "profiles", "r02_sim_kernel_ncu_full.json")))
            prof, cap = prof_file["launches"][0], prof_file["capture"]
            trials_prof = int(cap["trials_per_launch"])
            dram = 0.0
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[prof[key]["unit"]]
                dram += prof[key]["value"] * scale
            roofline["traffic"] = dram / trials_prof * n
            roofline["traffic_note"] = (f"ncu dram bytes per trial ({dram / trials_prof:.0f} B at {trials_prof} trials per launch, "
                                        "profiles/r02_sim_kernel_ncu_full.json) x trials per launch; a constant of that capture, not "
                                        "measured in this run")
            roofline["ncu_issue_active_pct"] = prof["sm__issue_active.avg.pct_of_peak_sustained_elapsed"]["value"]   # (of that capture)
            # issue-slot view of the same launch: warp-instructions per useful Euler step from that capture
            # (all of them: RNG, physics, bookkeeping) x the live step rate, against one instruction per
            # lane per clock
            inst_per_step = prof["smsp__inst_executed.sum"]["value"] * 32.0 / (trials_prof * float(cap["useful_steps_per_trial"]))
            roofline["issue"] = {"lane_inst_per_useful_step": inst_per_step,
                                 "achieved": per_launch_steps * inst_per_step / (k_ms * 1e-3) / 1e12, "peak": lane_peak / 1e12,
                                 "unit": "T lane-instructions/s",
                                 "frac": per_launch_steps * inst_per_step / (k_ms * 1e-3) / lane_peak,
                                 "note": "instructions per step from profiles/r02_sim_kernel_ncu_full.json (8388608 trials, "
                                         f"{float(cap['useful_steps_per_trial']):.2f} useful steps per trial: a constant of that capture), step rate measured live"}
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: 1e8-trial MNLE training set from ExtendedProposal, default "
                                   "schedule (n_max=16000, steps_per_pulse=200, P=80)" if n == 100_000_000 else
                                   f"configs[1] shape at {n} trials per GPU (default schedule, P=80)",
                       "trials_per_gpu_per_step": n, "z_bytes_per_gpu": n * 340,
                       "l2": "inputs (z) larger than L2; new Philox key each step", "rng": "Philox4x32-10, six 21-bit Box-Muller fields per block",
                       "exchange": gather_note},
            "trials_per_s": world * n * args.steps / (elapsed_ms * 1e-3),
            "mean_steps_per_trial": useful_all / (world * n * args.steps),
            "choice_frac": choice_frac,
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": link_bytes_per_step,
                    "d2h_bytes_per_step": n_e2e * 8, "host_z_bytes_per_step": n_e2e * 340,
                    "ingest": ("z rows (340 B/trial, pinned host) are packed to 32-byte records by the host cores "
                               "(ddm_pack_z_host) chunk by chunk while the streaming kernel runs; the link carries the records"
                               if link_bytes_per_step < n_e2e * 340 else
                               "fp32 z rows over the link (measured faster than packing on this host at this rank count: "
                               "HostPipeline.choose_packed)"),
                    "trials_per_step_per_gpu": n_e2e, "api": "data_simulator.sim_wrapper(z pinned host) -> x host",
                    "ms_per_step": float(e2e_t.item()) / args.steps},
            "gpu_launches": args.steps * world,
            "clocks": clock_info,
        }
        if sharded_equals_single is not None:
            line["sharded_equals_single"] = sharded_equals_single
        headline["line"] = line
        watchdog = threading.Timer(float(os.environ.get("DDM_BENCH_EXTRAS_TIMEOUT", 900)), bail)
        watchdog.daemon = True
        watchdog.start()
        run_extras()
        watchdog.cancel()
        line.update(extras)
        if world == 1 and args.train_set_trials > 0:
            try:
                line["e2e_training_set"] = training_set_e2e_bench(args, dev)
            except Exception as e:
                line["e2e_training_set"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            import torch as _t
            rate, times, _ = time_cpu_port(args.cpu_trials, 1, 1)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": _t.get_num_threads(), "kind": "port",
                "sample": f"1 x {args.cpu_trials} trials of the same workload through the lock-step torch port "
                          f"(oracle.sim_lockstep_torch = rt_choice_model.py:112-221 restated, torch.randn), "
                          f"{sum(times):.1f} s",
                "configs0": time_cpu_port_cfg1(),
            }
        if world == 1:
            try:
                line["mnle_potential"] = mnle_bench(dev, with_cpu=not args.no_cpu_baseline)
            except Exception as e:  # the headline metric must still print
                line["mnle_potential"] = {"error": repr(e)}
            try:
                line["mcmc"] = mcmc_bench(dev)
            except Exception as e:
                line["mcmc"] = {"error": repr(e)}
            try:
                line["configs0_api"] = configs0_bench(dev)
            except Exception as e:
                line["configs0_api"] = {"error": repr(e)}
            try:
                line["mnle_train_step"] = mnle_train_bench(dev, with_cpu=not args.no_cpu_baseline)
            except Exception as e:
                line["mnle_train_step"] = {"error": repr(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
