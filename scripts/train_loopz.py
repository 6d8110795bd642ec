#!/usr/bin/env python
"""The loopz training loop on the GPU learner [ref: OIGE/scripts/rlgames_train_loopz.py:700-1440]: MLPEncode actor / critic with a
squashed Gaussian, horizon-length rollouts, reward scale 0.01, 4 epochs x 4 in-order minibatches, lr 5e-4, std floor 0.05 after
every update.  python scripts/train_loopz.py --num-envs 4096 --updates 200 [--classic]
Data-parallel on one node: torchrun --nproc-per-node 8 scripts/train_loopz.py --num-envs 4096 (4096 envs per GPU; NCCL only at
start-up and for the log lines, the gradient exchange runs over NVLink peer memory inside the update graph; rank 0 prints and saves)."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes

import torch
import torch.distributed as dist

from omniisaacgymenvs_loop_b200 import _lib
from omniisaacgymenvs_loop_b200.algo.ppo import PPO, module as ppo_module
from omniisaacgymenvs_loop_b200.config import live_default_config, live_task_cfg, load_task_yaml
from omniisaacgymenvs_loop_b200.envs.usv_raisim_vecenv import USVRaisimVecEnv
from omniisaacgymenvs_loop_b200.envs.vec_env_rlgames import VecEnvRLGames
from omniisaacgymenvs_loop_b200.rl.a2c import reduce_episode_stats
from omniisaacgymenvs_loop_b200.tasks.USV_Virtual import SimConfig, USVVirtual


def make_env(task_cfg: dict, device: str, seed: int, env_id_offset: int = 0):
    env = VecEnvRLGames(headless=True)
    sim = SimConfig({"sim_device": device, "rl_device": device, "seed": seed, "env_id_offset": env_id_offset, "task": task_cfg})
    env.set_task(USVVirtual("USVVirtual", sim, env, collect_stats=False), backend="torch")
    return USVRaisimVecEnv(env)


def build_learner(env, device, horizon, seed, mass_dim=8, sampling="in_order", use_cuda_graph=True, rank=0, world_size=1):
    """rlgames_train_loopz.py:784-842"""
    arch = dict(speed_dim=3, mass_dim=mass_dim, mass_latent_dim=8, mass_encoder_shape=[64, 16])
    actor = ppo_module.Actor(ppo_module.MLPEncode_wrap([128, 128], "LeakyReLU", env.num_obs, env.num_acts, "Tanh", False, **arch),
                             ppo_module.SquashedGaussianDiagonalCovariance(env.num_acts, 0.3, action_scale=1.0), device, seed=seed)
    critic = ppo_module.Critic(ppo_module.MLPEncode_wrap([128, 128], "LeakyReLU", env.num_obs, 1, **arch), device)
    return PPO(actor=actor, critic=critic, num_envs=env.num_envs, num_transitions_per_env=horizon, num_learning_epochs=4, gamma=0.997,
               lam=0.95, num_mini_batches=4, device=device, mini_batch_sampling=sampling, learning_rate=5e-4, use_cuda_graph=use_cuda_graph,
               rank=rank, world_size=world_size)


class LoopzRunner:
    """The rollout / update cycle of the loopz script.  The rollout phase (horizon x {observe, env.step, ppo.step, episode-return
    bookkeeping}) only touches static buffers and device-side counters, so after two eager cycles it is captured into a CUDA graph and
    replayed (the env kernels and the sampling kernel take device-side step / counter offsets); graphs are keyed by the host-side
    parameters they bake in (`FusedUsvEnv.graph_key`), a window that straddles a change runs eagerly."""

    def __init__(self, env, ppo, horizon=16, reward_scale=0.01, use_cuda_graph=True):
        self.env, self.ppo, self.T, self.reward_scale = env, ppo, int(horizon), float(reward_scale)
        dev = ppo.device
        self.task = env._task
        self.engine = getattr(self.task, "engine", None)
        self.use_cuda_graph = bool(use_cuda_graph) and self.engine is not None
        self.ep_ret = torch.zeros(env.num_envs, device=dev)
        self.ep_len = torch.zeros(env.num_envs, device=dev)
        self.fin = torch.zeros(3, dtype=torch.float64, device=dev)        # finished episodes: sum of returns, sum of lengths, count
        self.meter = torch.zeros(4, device=dev)                           # windowed (100) mean return / size, mean length / size
        self.min_std = torch.full((env.num_acts,), 0.05, device=dev)
        env.reset()
        self.obs = env.observe(as_numpy=False).clone()                     # static: graph replays read / write it in place
        self.cycles = 0
        self._graph, self._graph_key = None, None

    def _rollout(self):
        env, ppo = self.env, self.ppo
        obs = self.obs
        for _ in range(self.T):
            action = ppo.observe(obs)
            reward, dones = env.step(action)
            # reward scaling into the storage, uint8 dones, running returns / lengths and the finished-episode sums: one launch
            st, m = ppo.storage, self.meter
            _lib.check(_lib.lib().ppo_rollout_bookkeep_f32(
                _lib.ptr(reward.contiguous(), torch.float32), _lib.ptr(dones.contiguous(), torch.int64), ctypes.c_float(self.reward_scale),
                _lib.ptr(st.rewards[st.step]), _lib.ptr(st.dones[st.step]), _lib.ptr(self.ep_ret), _lib.ptr(self.ep_len), _lib.ptr(self.fin),
                ctypes.c_void_p(m.data_ptr()), ctypes.c_void_p(m.data_ptr() + 4), ctypes.c_void_p(m.data_ptr() + 8),
                ctypes.c_void_p(m.data_ptr() + 12), ctypes.c_float(100.0), ctypes.c_int64(env.num_envs), _lib.stream()),
                "ppo_rollout_bookkeep_f32")
            ppo.step(value_obs=obs, rews=None, dones=None, infos=[], prewritten=True)
            obs = env.observe(as_numpy=False)
        self.obs.copy_(obs)

    def rollout(self):
        eng, task, ppo, T = self.engine, self.task, self.ppo, self.T
        key = eng.graph_key(T) if self.use_cuda_graph else None
        if key is None or self.cycles < 2 or eng.cfg.spawn_curriculum:
            self._rollout()
            return
        if key != self._graph_key:
            self._graph, self._graph_key = None, key
        if self._graph is None:
            task._nan_probe = False                                         # no host sync inside the capture: check_finite() at log time
            saved = (eng.step_counter, eng.first_call, task.step, task._calls, ppo._store.counter, ppo.storage.step)
            torch.cuda.synchronize(ppo.device)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._rollout()
                eng.advance_step_offset(T)
                ppo._store.advance_counter_offset(T)
            # the capture ran the host code once without executing anything: rewind the host-side counters
            eng.step_counter, eng.first_call, task.step, task._calls, ppo._store.counter, ppo.storage.step = saved
        self._graph.replay()
        eng.note_graph_replay(T)
        ppo._store.note_graph_replay(T)
        task.step += T / task.cfg.horizon_length
        task._calls += T
        ppo.storage.step = T

    def cycle(self, update: int = 0):
        self.rollout()
        self.ppo.update(actor_obs=self.obs, value_obs=self.obs, log_this_iteration=False, update=update)
        self.ppo.actor.distribution.enforce_minimum_std(self.min_std)       # rlgames_train_loopz.py:1380-1384
        self.cycles += 1

    def pop_episode_stats(self):
        """(mean return, count) of the episodes that finished since the last call on any rank (one host read; one all-reduce on
        `world` ranks)."""
        mean_ret, _, c = reduce_episode_stats(self.fin, self.ppo.world)
        self.fin.zero_()
        return mean_ret, c


def train(env, ppo, updates, horizon=16, reward_scale=0.01, log_every=10, quiet=False, use_cuda_graph=True, runner=None):
    """-> list of (update, mean return of the episodes finished since the previous log line, frames/s)."""
    run = runner if runner is not None else LoopzRunner(env, ppo, horizon, reward_scale, use_cuda_graph)
    hist = []
    t0, n0 = time.time(), 0
    for update in range(updates):
        run.cycle(update)
        if log_every and (update % log_every == 0 or update == updates - 1):
            torch.cuda.synchronize(ppo.device)
            if run.engine is not None:
                run.engine.check_finite()
            ppo.check_peers()
            dt = time.time() - t0
            fps = horizon * env.num_envs * ppo.world * (update + 1 - n0) / max(dt, 1e-9)
            t0, n0 = time.time(), update + 1
            mean_ret, n_ep = run.pop_episode_stats()
            hist.append((update, mean_ret, fps))
            if not quiet:
                print(f"update {update:5d}  return {mean_ret:9.3f} ({n_ep} episodes)  std {ppo.actor.distribution.std.tolist()}  "
                      f"v_loss {ppo.last_stats['mean_value_loss']:.4f}  fps {fps:,.0f}", flush=True)
    return hist


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--task-yaml", default=None)
    ap.add_argument("--num-envs", type=int, default=4096)
    ap.add_argument("--updates", type=int, default=200)
    ap.add_argument("--horizon", type=int, default=16)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--save", default=None)
    ap.add_argument("--checkpoint", default=None)
    args = ap.parse_args()
    world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
    device = f"cuda:{local}"
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    task_cfg = load_task_yaml(args.task_yaml, num_envs=args.num_envs) if args.task_yaml else live_task_cfg(live_default_config(num_envs=args.num_envs))
    env = make_env(task_cfg, device, args.seed, env_id_offset=rank * args.num_envs)
    ppo = build_learner(env, device, args.horizon, args.seed, rank=rank, world_size=world)
    start = 0
    if args.checkpoint:
        start = ppo.load_state_dict(torch.load(args.checkpoint, map_location=device, weights_only=False))
        if rank == 0:
            print(f"[loopz] resumed from {args.checkpoint} (start_update={start})")
    train(env, ppo, args.updates, args.horizon, quiet=rank != 0)
    if args.save and rank == 0:
        torch.save(ppo.state_dict(start + args.updates - 1), args.save)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
