#!/usr/bin/env python
"""Timings of the ragged-session potential and driver on the trained estimator (tests/golden/mnle_trained.npz):
100 sessions with T_i drawn from the integers [20, 500] (seed 2026), C = 128 chains per session.

  (a) one ragged potential call (tc, tc64) against a Python loop of per-session ``loglik_sum`` calls;
  (b) ``run_inference_sessions`` at the reference's settings (WARMUP_STEPS=100, POSTERIOR_SAMPLES=1000) against a loop
      of ``run_inference_mcmc`` over the same sessions;
  (c) with --parent-root DIR (a checkout of another revision with its library built): the uniform path
      (configs[3]: one session T=50 x C=1024; the SBC shape: 125 datasets x T=50 x C=128) timed in this tree and in DIR,
      alternating, in separate processes; each process also reports digests of its outputs and of a short run_sbc /
      run_inference_mcmc, which must agree between the two trees.

    python tools/time_sessions.py [--parent-root DIR] [--skip-b] [--out FILE.json]

Device times are CUDA events around back-to-back calls after warm-up; loops are host clocks around work that ends in
a synchronise.  The GPU name and power limit are printed with the numbers.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name()} | nvidia-smi: {q}"


def event_ms(fn, reps, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_s(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def digest(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()[:16]


def trained(root):
    import numpy as np
    from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE
    d = np.load(os.path.join(root, "tests", "golden", "mnle_trained.npz"))
    return DeviceMNLE(PackedMNLE(d["packed"], int(d["n_choices"])))


def uniform(root):
    """(c), run in one process per tree: the uniform path's times and output digests."""
    import torch
    from sbi_for_diffusion_models_b200.mnle import run_inference_mcmc, run_sbc
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    from sbi_for_diffusion_models_b200.sbc import draw_sbc_datasets, simulate_sbc_sessions
    torch.cuda.set_device(0)
    est, prior = trained(ROOT), build_prior_theta()
    res = {"root": root}
    thetas, seeds = draw_sbc_datasets(prior, 125, seed=1)
    x, pulses = simulate_sbc_sessions(thetas, seeds, 50, mu_sensory=1.0, p_success=0.75, noise_seed=2)
    torch.manual_seed(0)
    th1 = prior.sample((1024,)).cuda()
    th125 = prior.sample((125 * 128,)).view(125, 128, 5).cuda()
    one = lambda: est.loglik_sum(th1, x[0], pulses[0], kernel="tc")
    sbc = lambda: est.loglik_sum_batched(th125, x, pulses)
    res["configs3_ms"] = [event_ms(one, 200) for _ in range(5)]
    res["sbc_shape_ms"] = [event_ms(sbc, 50) for _ in range(5)]
    res["digest_configs3"], res["digest_sbc_shape"] = digest(one()), digest(sbc())
    cfg = RunConfig(WARMUP_STEPS=20, NUM_TRIALS_OBS=50)
    out = run_sbc(cfg, prior_theta=prior, density_estimator=est, num_datasets=25, posterior_samples_per_dataset=200, seed=0,
                  save=False)
    res["digest_sbc_ranks"] = digest(torch.from_numpy(out["ranks"]))
    res["digest_sbc_samples"] = digest(torch.stack(out["all_samples"]))
    g = torch.Generator(device="cuda").manual_seed(0)
    torch.manual_seed(0)
    res["digest_mcmc"] = digest(run_inference_mcmc(RunConfig(WARMUP_STEPS=20, POSTERIOR_SAMPLES=500), prior, est, x[0].cpu(),
                                                   pulses[0].cpu(), generator=g))
    print("UNIFORM " + json.dumps(res), flush=True)


def sessions_data(n=100, tmin=20, tmax=500, seed=2026):
    import numpy as np
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.sbc import draw_sbc_datasets, simulate_sbc_sessions
    lengths = np.random.default_rng(seed).integers(tmin, tmax + 1, n).tolist()
    thetas, seeds = draw_sbc_datasets(build_prior_theta(), n, seed=seed)
    x, pulses = simulate_sbc_sessions(thetas, seeds, tmax, mu_sensory=1.0, p_success=0.75, noise_seed=seed)
    return lengths, [x[i, :T] for i, T in enumerate(lengths)], [pulses[i, :T] for i, T in enumerate(lengths)]


def spread(ts):
    return {"median": statistics.median(ts), "min": min(ts), "max": max(ts), "runs": ts}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root", default=None)
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--skip-b", action="store_true")
    ap.add_argument("--out", default=None)
    ap.add_argument("--uniform-only", default=None, help=argparse.SUPPRESS)   # (c) worker: the tree to import from
    args = ap.parse_args()
    if args.uniform_only is not None:
        sys.path.insert(0, os.path.abspath(args.uniform_only))
        uniform(args.uniform_only)
        return
    sys.path.insert(0, ROOT)
    import torch
    from sbi_for_diffusion_models_b200.mnle import run_inference_mcmc, run_inference_sessions
    from sbi_for_diffusion_models_b200.priors import build_prior_theta
    from sbi_for_diffusion_models_b200.run_config import RunConfig
    torch.cuda.set_device(0)
    report = {"gpu": gpu_info()}
    print("GPU:", report["gpu"], flush=True)
    est, prior = trained(ROOT), build_prior_theta()
    lengths, xs, pls = sessions_data()
    D, C, N = len(lengths), 128, sum(lengths)
    x, pl = torch.cat(xs), torch.cat(pls)
    torch.manual_seed(0)
    th = prior.sample((D * C,)).view(D, C, 5).cuda()
    report["sessions"] = {"D": D, "C": C, "N": N, "rows": N * C, "T_min": min(lengths), "T_max": max(lengths)}
    print(f"sessions: D={D}, T in [{min(lengths)}, {max(lengths)}], N={N} trials, C={C}: {N * C} rows", flush=True)

    # (a) one ragged call against the per-session loop, both kernels; the outputs must have the same bits
    report["a"] = {}
    for kernel in ("tc", "tc64"):
        plan = est.session_plan(lengths, C, kernel=kernel)
        ragged = lambda: est.loglik_sum_sessions(th, x, pl, plan, kernel=kernel)
        loop = lambda: [est.loglik_sum(th[d], xs[d], pls[d], kernel=kernel) for d in range(D)]
        same = torch.equal(ragged(), torch.stack(loop()))
        t_ragged = event_ms(ragged, 20)
        t_loop = statistics.median(host_s(loop) for _ in range(5)) * 1e3
        report["a"][kernel] = {"ragged_ms": t_ragged, "loop_ms": t_loop, "speedup": t_loop / t_ragged, "same_bits": same}
        print(f"(a) {kernel}: one ragged call {t_ragged:.3f} ms | loop of {D} loglik_sum calls {t_loop:.3f} ms | "
              f"{t_loop / t_ragged:.1f}x | same bits: {same}", flush=True)

    # (b) the driver against a loop of run_inference_mcmc, the reference's settings
    if not args.skip_b:
        cfg = RunConfig(WARMUP_STEPS=100, POSTERIOR_SAMPLES=1000)
        sessions = [(xs[i].cpu(), pls[i].cpu()) for i in range(D)]
        run_inference_sessions(RunConfig(WARMUP_STEPS=2, POSTERIOR_SAMPLES=128), prior, est, sessions, seed=0)   # warm-up
        t_sessions = host_s(lambda: run_inference_sessions(cfg, prior, est, sessions, seed=0))
        g = torch.Generator(device="cuda").manual_seed(0)
        run_inference_mcmc(RunConfig(WARMUP_STEPS=2, POSTERIOR_SAMPLES=128), prior, est, *sessions[0], generator=g)
        t_loop = host_s(lambda: [run_inference_mcmc(cfg, prior, est, s[0], s[1], generator=g) for s in sessions])
        report["b"] = {"run_inference_sessions_s": t_sessions, "run_inference_mcmc_loop_s": t_loop,
                       "speedup": t_loop / t_sessions}
        print(f"(b) run_inference_sessions over {D} sessions {t_sessions:.2f} s | loop of {D} run_inference_mcmc "
              f"{t_loop:.2f} s | {t_loop / t_sessions:.1f}x", flush=True)

    # (c) the uniform path in this tree and in the parent tree, alternating, one process each
    if args.parent_root:
        runs = {"this": [], "parent": []}
        for _ in range(args.pairs):
            for name, root in (("parent", os.path.abspath(args.parent_root)), ("this", ROOT)):
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--uniform-only", root], capture_output=True,
                                   text=True, timeout=1200)
                line = [ln for ln in r.stdout.splitlines() if ln.startswith("UNIFORM ")]
                if r.returncode != 0 or not line:
                    raise RuntimeError(f"uniform worker in {root} failed:\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}")
                runs[name].append(json.loads(line[0][len("UNIFORM "):]))
        c = {}
        for key in ("configs3_ms", "sbc_shape_ms"):
            c[key] = {name: spread([t for r in rs for t in r[key]]) for name, rs in runs.items()}
            print(f"(c) {key}: parent median {c[key]['parent']['median']:.4f} ms [{c[key]['parent']['min']:.4f}, "
                  f"{c[key]['parent']['max']:.4f}] | this median {c[key]['this']['median']:.4f} ms "
                  f"[{c[key]['this']['min']:.4f}, {c[key]['this']['max']:.4f}]", flush=True)
        for key in ("digest_configs3", "digest_sbc_shape", "digest_sbc_ranks", "digest_sbc_samples", "digest_mcmc"):
            vals = {r[key] for rs in runs.values() for r in rs}
            c[key + "_identical"] = len(vals) == 1
            print(f"(c) {key} identical in both trees and every run: {len(vals) == 1}", flush=True)
        report["c"] = c
    report["gpu_after"] = gpu_info()
    print("GPU:", report["gpu_after"], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
