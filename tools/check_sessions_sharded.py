#!/usr/bin/env python
"""Run under torchrun on >= 2 GPUs: run_inference_sessions with the sessions sharded over the ranks equals the
same run on one rank, bit for bit.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29531 tools/check_sessions_sharded.py
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import mnle_spec as ms  # noqa: E402
from sbi_for_diffusion_models_b200.mnle import run_inference_sessions  # noqa: E402
from sbi_for_diffusion_models_b200.mnle_net import DeviceMNLE, PackedMNLE  # noqa: E402
from sbi_for_diffusion_models_b200.priors import build_prior_theta  # noqa: E402
from sbi_for_diffusion_models_b200.run_config import RunConfig  # noqa: E402
from sbi_for_diffusion_models_b200.sbc import draw_sbc_datasets, simulate_sbc_sessions  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    est = DeviceMNLE(PackedMNLE.from_params(ms.init_params(0)))
    lengths = [17, 0, 40, 5, 33, 21, 9]
    thetas, seeds = draw_sbc_datasets(build_prior_theta(), len(lengths), seed=11)
    x, pulses = simulate_sbc_sessions(thetas, seeds, max(lengths), mu_sensory=1.0, p_success=0.75, noise_seed=12)
    sessions = [(x[i, :T].cpu(), pulses[i, :T].cpu()) for i, T in enumerate(lengths)]
    cfg = RunConfig(WARMUP_STEPS=3, POSTERIOR_SAMPLES=130)
    solo = dist.new_group([0])
    out = run_inference_sessions(cfg, build_prior_theta(), est, sessions, seed=5)
    if rank == 0:
        one = run_inference_sessions(cfg, build_prior_theta(), est, sessions, seed=5, group=solo)
        ok = len(out) == len(one) == len(lengths) and all(torch.equal(a, b) for a, b in zip(out, one))
        print(f"sessions sharded over {dist.get_world_size()} GPUs == single GPU: {ok}", flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
