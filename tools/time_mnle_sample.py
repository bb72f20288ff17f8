"""Time ``DeviceMNLE.sample`` on cuda:0 at 51 200 rows (configs[3]: T=50 x C=1024) and at 2^20 rows, next to
``loglik_sum(kernel="tc64")`` over the same number of rows (the same tensor-core forward plus an fp64 spline chain)
and the CPU specification's ``sample`` in float64 and float32 on the host threads (51 200 rows).  Trained estimator of
tests/golden/mnle_trained.npz.  Prints one JSON object; ``--out FILE`` also writes it there.

    python tools/time_mnle_sample.py [--out FILE]

eager: wall time of the first call of a shape (host clock around call + synchronise: workspace allocation, module
loading).  steady: CUDA events around 20 back-to-back calls after 3 warm-up calls, per call."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle import ddm_oracle as orc  # noqa: E402
from oracle import mnle_sample_spec as mss  # noqa: E402
from oracle import mnle_spec as ms  # noqa: E402
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE, unpack_params  # noqa: E402


def timed(fn, reps=20, warm=3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    eager = (time.perf_counter() - t0) * 1e3
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return eager, e0.elapsed_time(e1) / reps


def main():
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    d = np.load(os.path.join(ROOT, "tests", "golden", "mnle_trained.npz"))
    packed, K = d["packed"], int(d["n_choices"])
    est = DeviceMNLE(PackedMNLE(packed, K))
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        power = f"unavailable ({e})"
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "rows": {}}
    for T, C in ((50, 1024), (1024, 1024)):
        R = T * C
        theta = orc.prior_sample(C, seed=1).to(dev)
        pulses = torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(2)), 0, T, 80, 0.75)).to(dev)
        x_o = est.sample((), condition=torch.cat([theta[:1].expand(T, 5), pulses], 1), seed=3)
        cond = torch.cat([theta.repeat(T, 1), pulses.repeat_interleave(C, 0)], 1).contiguous()   # the potential's rows
        s_eager, s_ms = timed(lambda: est.sample((), condition=cond, seed=11))
        p_eager, p_ms = timed(lambda: est.loglik_sum(theta, x_o, pulses, kernel="tc64"))
        res["rows"][R] = {"sample_eager_ms": round(s_eager, 3), "sample_ms": round(s_ms, 4),
                          "sample_rows_per_s": float(f"{R / s_ms * 1e3:.4g}"),
                          "tc64_eager_ms": round(p_eager, 3), "tc64_ms": round(p_ms, 4),
                          "tc64_rows_per_s": float(f"{R / p_ms * 1e3:.4g}"), "sample_over_tc64": round(s_ms / p_ms, 3)}
        print(json.dumps({R: res["rows"][R]}), flush=True)
    # CPU specification on the host threads, 51 200 rows
    p32 = dict(unpack_params(torch.from_numpy(packed.copy()), K))
    p32["cond_mean"], p32["cond_std"] = torch.zeros(85), torch.ones(85)
    R = 51200
    cond = torch.cat([orc.prior_sample(R, seed=4),
                      torch.from_numpy(orc.pulses_pcg64_c(*orc.pcg64_state(np.random.default_rng(5)), 0, R, 80, 0.75))], 1)
    rng = np.random.default_rng(6)
    uc, n = torch.from_numpy(rng.random(R)), torch.from_numpy(rng.standard_normal(R))
    res["cpu_spec"] = {"threads": torch.get_num_threads(), "rows": R}
    for name, dt in (("float64", torch.float64), ("float32", torch.float32)):
        p = ms.cast_params(p32, dt)
        t0 = time.perf_counter()
        mss.sample(p, cond.to(dt), uc, n)
        t = time.perf_counter() - t0
        res["cpu_spec"][name] = {"ms": round(t * 1e3, 1), "rows_per_s": float(f"{R / t:.4g}")}
    print(json.dumps(res, indent=1))
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
