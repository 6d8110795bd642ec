#!/usr/bin/env python
"""Batched evaluation of a loopz actor with the reference's per-episode CSV [ref: OIGE/scripts/rlgames_play_loopz.py:860-1439]:
deterministic actions `tanh(mu) * action_scale` (:1219-1222), every env of the fused live task evaluated in parallel, one CSV row per
finished episode (columns and definitions: `utils/episode_metrics.py`), bootstrap summary at the end.
  python scripts/play_loopz.py --checkpoint full_100.pt --num-envs 1024 --episodes 2000 --csv runs/play.csv
The distilled SysID student (scripts/dagger_usv_sysid_loopz.py --save) plays the same way from its non-privileged history alone:
  python scripts/play_loopz.py --student student.pt [--policy student|teacher|both] --episodes 2000 --csv runs/student.csv
(`both` plays the embedded teacher, then the student on a fresh env with the same seed; run_id tells the rows apart.)"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config, live_task_cfg, load_task_yaml
import numpy as np

from omniisaacgymenvs_loop_b200.utils.episode_metrics import EpisodeRecorder, apply_mass_mode_to_obs
from scripts.train_loopz import build_learner, make_env


def play(env, actor, episodes: int, reward_scale: float = 0.01, max_steps: int = 1_000_000, mass_mode: str = "normal", **meta) -> EpisodeRecorder:
    """Runs until `episodes` episodes have finished (all envs in parallel; the last step may overshoot); returns the recorder.
    `mass_mode`: the control-side intervention on the mass / CoM columns the policy sees (LOOPZ_PLAY_MASS_MODE, :1212-1218)."""
    rng = np.random.default_rng(int(meta.get("seed", 0)))
    rec = EpisodeRecorder(env._task.engine, reward_scale=reward_scale, action_scale=float(actor.distribution.action_scale.reshape(-1)[0]), **meta)
    # reset() flags every env and runs the zero-action reset step (VecEnvRLGames.reset): feed it to the recorder as the start snapshot
    env.reset()
    n = env.num_envs
    zero = torch.zeros((n, env.num_acts), device=actor.device)
    rec.record(zero, torch.zeros(n, device=actor.device), env._task.reset_buf)
    scale = actor.distribution.action_scale.to(actor.device)
    for _ in range(max_steps):
        if len(rec.rows) >= episodes:
            break
        obs = apply_mass_mode_to_obs(env.observe(as_numpy=False), mass_mode, rng)
        action = torch.tanh(actor.noiseless_action(obs)) * scale
        reward, dones = env.step(action)
        rec.record(action, reward, dones)
    return rec


def play_student(env, student, episodes: int, reward_scale: float = 0.01, max_steps: int = 1_000_000, **meta) -> EpisodeRecorder:
    """play() for the SysID student: `student.reset(obs)` fills the history from the first observation, `student.act(obs, dones)` appends
    each step's observation (dones of that step: "repeat" refills finished envs); action = tanh(mu) * student.action_scale, as for the
    teacher.  `student` is a USVSysIDStudentPolicy or anything with the same reset / act / action_scale."""
    scale = student.action_scale
    rec = EpisodeRecorder(env._task.engine, reward_scale=reward_scale, action_scale=float(scale.reshape(-1)[0]), **meta)
    env.reset()
    n, dev = env.num_envs, scale.device
    rec.record(torch.zeros((n, env.num_acts), device=dev), torch.zeros(n, device=dev), env._task.reset_buf)
    mu = student.reset(env.observe(as_numpy=False))
    for _ in range(max_steps):
        if len(rec.rows) >= episodes:
            break
        action = torch.tanh(mu) * scale
        reward, dones = env.step(action)
        rec.record(action, reward, dones)
        mu = student.act(env.observe(as_numpy=False), dones)
    return rec


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--task-yaml", default=None)
    ap.add_argument("--num-envs", type=int, default=1024)
    ap.add_argument("--episodes", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--checkpoint", default=None, help="teacher (loopz PPO) checkpoint")
    ap.add_argument("--student", default=None, help="student file of scripts/dagger_usv_sysid_loopz.py --save (embeds its teacher)")
    ap.add_argument("--policy", default=None, choices=["student", "teacher", "both"],
                    help="what to play (default: student with --student, else teacher); both = teacher, then student, same seed")
    ap.add_argument("--csv", default=None)
    ap.add_argument("--mass-mode", default=os.getenv("LOOPZ_PLAY_MASS_MODE", "normal"), help="normal | zero | shuffle | swap (policy-side only)")
    ap.add_argument("--obs-source", default="sim", choices=["sim", "base", "both"],
                    help="privileged-tail source (mass.masscom_obs_source); both = the reference's two-mode comparison (eval.modes)")
    args = ap.parse_args(argv)
    if args.policy is None:
        args.policy = "student" if args.student else "teacher"
    if args.policy in ("student", "both"):
        if not args.student:
            ap.error(f"--policy {args.policy} needs --student")
        if args.mass_mode != "normal" or args.obs_source != "sim":
            ap.error("--mass-mode and --obs-source change the privileged tail, which the student never reads: play the student with "
                     "--mass-mode normal --obs-source sim (or --policy teacher)")
    return args


def main(argv=None):
    args = parse_args(argv)
    device = "cuda:0"
    torch.cuda.set_device(device)
    student, teacher_sd, priv = None, None, 8
    if args.student:
        from omniisaacgymenvs_loop_b200.algo.ppo.dagger import USVSysIDStudentPolicy
        student = USVSysIDStudentPolicy.from_checkpoint(args.student, device)
        priv = student.meta["priv_dim"]
        teacher_sd = torch.load(args.student, map_location=device, weights_only=False)["teacher"]
    if args.checkpoint:
        teacher_sd = torch.load(args.checkpoint, map_location=device, weights_only=False)

    def new_env():
        if args.task_yaml:
            return make_env(load_task_yaml(args.task_yaml, num_envs=args.num_envs), device, args.seed)
        live = live_default_config(num_envs=args.num_envs)
        return make_env(live_task_cfg(live, UsvLiveConfig(priv_dim=priv)) if student else live_task_cfg(live), device, args.seed)

    rows = []
    rec = None
    if args.policy in ("teacher", "both"):
        env = new_env()
        ppo = build_learner(env, device, 16, args.seed, mass_dim=priv, use_cuda_graph=False)
        if teacher_sd is not None:
            ppo.load_state_dict(teacher_sd)
        for mode in (["sim", "base"] if args.obs_source == "both" else [args.obs_source]):
            env._task._masscom_obs_source = mode                    # rlgames_play_loopz.py:1100-1110 (_set_obs_source)
            rec = play(env, ppo.actor, args.episodes, run_id="play", ckpt=str(args.checkpoint or args.student), seed=args.seed, obs_source=mode,
                       mass_mode=args.mass_mode)
            print(f"[loopz-play][EVAL] policy=teacher mode={mode}")
            rec.summarize(seed=args.seed)
            rows += rec.rows
    if args.policy in ("student", "both"):
        env = new_env()
        if env.num_obs - priv != student.obs_nonpriv_dim:
            raise SystemExit(f"the task's observation ({env.num_obs} wide, priv_dim {priv}) does not carry the student's "
                             f"{student.obs_nonpriv_dim} non-privileged columns")
        rec = play_student(env, student, args.episodes, run_id="student", ckpt=str(args.student), seed=args.seed, obs_source="sim")
        print("[loopz-play][EVAL] policy=student mode=sim")
        rec.summarize(seed=args.seed)
        rows += rec.rows
    if args.csv:
        os.makedirs(os.path.dirname(os.path.abspath(args.csv)), exist_ok=True)
        rec.rows = rows
        rec.write_csv(args.csv)
        print(f"[loopz-play][EVAL] wrote {len(rows)} rows to {args.csv}")

if __name__ == "__main__":
    main()
