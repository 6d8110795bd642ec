#!/usr/bin/env python
"""USV SysID distillation loop [ref: omniisaacgymenvs/scripts/dagger_usv_sysid_loopz.py:140-420]: the frozen loopz teacher's mass encoder
labels every step with z* = mass_encoder(privileged tail), the student (StateHistoryEncoder over the last 50 non-privileged observations)
drives the boat through the frozen action head and is regressed onto z* every `horizon` steps.  Everything stays on the device: fused live
env step, history window, student inference, teacher labels, MSE / backward / Adam kernels; one host read per update (the metrics).
The script runs the fused loop (build_fused / run_fused): one collect launch per control step, each frame stored once, windows rebuilt
inside the training kernels (USVSysIDDistiller).  build / run are the unfused loop on USVSysIDVecEnv it reproduces bit for bit.

    python scripts/dagger_usv_sysid_loopz.py --envs 4096 --updates 50 [--checkpoint teacher.pt] [--save student.pt]

--save writes one file with the trainer's state, the teacher it was distilled from and the shapes (algo/ppo/dagger.student_checkpoint);
scripts/play_loopz.py --student plays it.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from omniisaacgymenvs_loop_b200.algo.ppo.dagger import (USVSysIDAgent, USVSysIDDistiller, USVSysIDStudentPolicy, USVSysIDTrainer,
                                                        student_checkpoint)
from omniisaacgymenvs_loop_b200.algo.ppo.module import StateHistoryEncoder
from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config, live_task_cfg
from omniisaacgymenvs_loop_b200.envs.usv_raisim_vecenv import USVSysIDVecEnv
from scripts.train_loopz import build_learner, make_env


def _parts(envs, device, seed, history_len, priv_dim, horizon, checkpoint, max_episode_length):
    """-> (live env, USVSysIDTrainer, teacher PPO): the teacher policy (random unless a checkpoint is given), the student and its trainer"""
    over = {} if max_episode_length is None else {"max_episode_length": max_episode_length}
    cfg = live_default_config(num_envs=envs, **over)
    base = make_env(live_task_cfg(cfg, UsvLiveConfig(priv_dim=priv_dim)), device, seed=seed)
    ppo = build_learner(base, device, horizon, seed=seed, mass_dim=priv_dim)
    if checkpoint:
        ppo.load_state_dict(torch.load(checkpoint, map_location=device, weights_only=False))
    arch = ppo.actor.architecture.architecture
    D = base.num_obs - priv_dim
    student = StateHistoryEncoder("LeakyReLU", D, history_len, 8, device, seed=seed)
    agent = USVSysIDAgent(teacher_mass_encoder=arch.mass_encoder, id_encoder=student, frozen_action_head=arch.action_mlp,
                          history_len=history_len, obs_nonpriv_dim=D, device=device)
    trainer = USVSysIDTrainer(actor=agent, num_envs=base.num_envs, num_transitions_per_env=horizon, history_dim=history_len * D,
                              latent_dim=8, num_learning_epochs=4, num_mini_batches=4, device=device, learning_rate=5e-4)
    return base, trainer, ppo


def build_with_teacher(envs: int, device: str, seed: int, history_len: int = 50, priv_dim: int = 8, horizon: int = 16, checkpoint=None,
                       fill_history_on_reset: str = "zeros", max_episode_length=None):
    """-> (USVSysIDVecEnv, trainer, teacher PPO): the unfused loop's pieces"""
    base, trainer, ppo = _parts(envs, device, seed, history_len, priv_dim, horizon, checkpoint, max_episode_length)
    env = USVSysIDVecEnv(base._env, history_len=history_len, priv_dim=priv_dim, fill_history_on_reset=fill_history_on_reset, device=device)
    return env, trainer, ppo


def build(envs: int, device: str, seed: int, history_len: int = 50, priv_dim: int = 8, horizon: int = 16, checkpoint=None):
    env, trainer, _ = build_with_teacher(envs, device, seed, history_len, priv_dim, horizon, checkpoint)
    return env, trainer


def build_fused(envs: int, device: str, seed: int, history_len: int = 50, priv_dim: int = 8, horizon: int = 16, checkpoint=None,
                fill_history_on_reset: str = "zeros", max_episode_length=None):
    """-> (live USVRaisimVecEnv, USVSysIDDistiller, teacher PPO): the same teacher, student and trainer as build_with_teacher, collected
    by the fused student step on the plain live env (no history wrapper)"""
    base, trainer, ppo = _parts(envs, device, seed, history_len, priv_dim, horizon, checkpoint, max_episode_length)
    agent = trainer.actor
    policy = USVSysIDStudentPolicy(id_encoder=agent.id_encoder, frozen_action_head=agent.frozen_action_head, history_len=history_len,
                                   obs_nonpriv_dim=agent.obs_nonpriv_dim, fill_history_on_reset=fill_history_on_reset)
    return base, USVSysIDDistiller(trainer, policy), ppo


def write_student(path: str, trainer, ppo, seed: int, *, priv_dim: int, fill_history_on_reset: str) -> None:
    """The student file: trainer state + the teacher's PPO state + meta (USVSysIDStudentPolicy.from_checkpoint reads it)."""
    ckpt = student_checkpoint(trainer.state_dict(), ppo.state_dict(), history_len=trainer.actor.history_len, priv_dim=priv_dim,
                              obs_nonpriv_dim=trainer.actor.obs_nonpriv_dim, latent_dim=trainer.latent_dim,
                              fill_history_on_reset=fill_history_on_reset, seed=seed)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    torch.save(ckpt, path)


def save_student(path: str, env, trainer, ppo, seed: int) -> None:
    """write_student for the unfused loop's pieces."""
    write_student(path, trainer, ppo, seed, priv_dim=env.priv_dim, fill_history_on_reset=env._fill_history_on_reset)


def run(env, trainer, updates: int, horizon: int = 16, log_every: int = 10, quiet: bool = False):
    env.reset()
    out = []
    for upd in range(updates):
        for _ in range(horizon):
            sysid_obs = env.observe_sysid_obs(as_numpy=False)
            trainer.step(sysid_obs, env.get_priv_tail())
            env.step(trainer.observe(sysid_obs))
        m = trainer.update()
        out.append(m)
        if not quiet and (upd % log_every == 0 or upd == updates - 1):
            print(f"[sysid] update {upd}: mse {m['mse']:.5f} r2_total {m['r2_total']:.4f} zstar_var {m['zstar_var_mean']:.4f} zhat_var {m['zhat_var_mean']:.4f}",
                  flush=True)
    return out


def run_fused(env, distiller, updates: int, horizon: int = 16, log_every: int = 10, quiet: bool = False):
    """run() on the fused collect step: one dagger_sysid_collect_f32 launch per control step feeds env.step the head output
    get_student_action returns in run(); the same updates and metrics, bit for bit."""
    env.reset()
    out = []
    dones = None
    for upd in range(updates):
        for t in range(horizon):
            obs = env.observe(as_numpy=False)
            mu = distiller.reset(obs) if upd == 0 and t == 0 else distiller.act(obs, dones)
            _, dones = env.step(mu)
        m = distiller.update()
        out.append(m)
        if not quiet and (upd % log_every == 0 or upd == updates - 1):
            print(f"[sysid] update {upd}: mse {m['mse']:.5f} r2_total {m['r2_total']:.4f} zstar_var {m['zstar_var_mean']:.4f} zhat_var {m['zhat_var_mean']:.4f}",
                  flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--updates", type=int, default=50)
    ap.add_argument("--horizon", type=int, default=16)
    ap.add_argument("--history-len", type=int, default=50)
    ap.add_argument("--priv-dim", type=int, default=8)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--save", default=None, help="write the distilled student (with its teacher) to this file")
    ap.add_argument("--device", default="cuda:0")
    a = ap.parse_args()
    torch.cuda.set_device(a.device)
    torch.manual_seed(a.seed)
    env, distiller, ppo = build_fused(a.envs, a.device, a.seed, a.history_len, a.priv_dim, a.horizon, a.checkpoint)
    run_fused(env, distiller, 2, a.horizon, quiet=True)              # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ms = run_fused(env, distiller, a.updates, a.horizon)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(f"[sysid] {a.envs} envs x horizon {a.horizon}: {a.updates} updates in {dt:.2f} s = {a.updates * a.horizon * a.envs / dt:.3e} frames/s "
          f"({dt / a.updates * 1e3:.1f} ms per collect + update); final r2_total {ms[-1]['r2_total']:.4f}")
    if a.save:
        write_student(a.save, distiller.trainer, ppo, a.seed, priv_dim=a.priv_dim, fill_history_on_reset=distiller.policy.fill_history_on_reset)
        print(f"[sysid] wrote the student to {a.save}")
