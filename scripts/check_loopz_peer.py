#!/usr/bin/env python
"""Multi-GPU check of the data-parallel loopz learner (run under torchrun, one rank per GPU, wrapped in `timeout`):
  timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 scripts/check_loopz_peer.py
K rollout + update cycles of scripts/train_loopz.py on the classic task (no batch-wide quirks, so sharding changes nothing) with N envs
per rank and in-order minibatches: (1) the ranks' parameters and Adam state are bit-identical (all-gathered exact checksum);
(2) rank 0 then runs one rank over all W x N envs from the same start and compares parameters; (3) seconds per update and frames/s at
W ranks and at one rank, with the card name and power limit read in this run.  Needs >= 2 GPUs."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
from omniisaacgymenvs_loop_b200.rl.a2c import ranks_hold_identical
from scripts.train_loopz import LoopzRunner, build_learner, make_env

world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
if world < 2:
    sys.exit("check_loopz_peer.py needs >= 2 ranks (torchrun --nproc-per-node W, one GPU each)")
dev = f"cuda:{local}"
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=torch.device(dev))
log = (lambda *a: print(*a, flush=True)) if rank == 0 else (lambda *a: None)
N, K, HORIZON = int(os.environ.get("LOOPZ_PEER_ENVS", 8192)), int(os.environ.get("LOOPZ_PEER_UPDATES", 20)), 16


def run(num_envs, r, w, updates):
    """(learner, start parameters, seconds per update over the last updates - 3 cycles)."""
    torch.manual_seed(3)
    env = make_env(UsvEnvConfig(num_envs=num_envs, max_episode_length=200).to_task_cfg(), dev, seed=3, env_id_offset=r * num_envs)
    ppo = build_learner(env, dev, HORIZON, seed=3, rank=r, world_size=w)
    start = ppo.params.clone()
    runner = LoopzRunner(env, ppo, HORIZON)
    for u in range(updates):
        if u == 3:
            torch.cuda.synchronize()
            if w > 1:
                dist.barrier()
            t0 = time.perf_counter()
        runner.cycle(u)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / (updates - 3)
    ppo.check_peers()
    return ppo, start, dt


ppo, start, dt_w = run(N, rank, world, K)
assert ranks_hold_identical([ppo.params, ppo.exp_avg, ppo.exp_avg_sq, ppo.adam_step], world), "ranks diverged"
assert torch.isfinite(ppo.params).all()
log(f"[loopz-peer] world={world} envs/gpu={N}: ranks bit-identical after {K} updates")
if rank == 0:
    one, start1, dt_1 = run(world * N, 0, 1, K)
    assert torch.equal(start, start1)
    err = float((one.params - ppo.params).abs().max())
    scale = float(one.params.abs().max())
    gpu = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    log(f"[loopz-peer] one rank over {world * N} envs vs {world} ranks x {N}: max |dparam| = {err:.3e} (param scale {scale:.3e}; "
        f"summation order, compounded over {K} updates of a chaotic rollout)")
    log(f"[loopz-peer] {gpu}: {world} ranks x {N} envs: {dt_w * 1e3:.2f} ms/update = {world * N * HORIZON / dt_w:.3e} frames/s; "
        f"1 rank x {world * N} envs: {dt_1 * 1e3:.2f} ms/update = {world * N * HORIZON / dt_1:.3e} frames/s (speed-up {dt_1 / dt_w:.2f})")
dist.barrier()
dist.destroy_process_group()
