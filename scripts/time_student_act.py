#!/usr/bin/env python
"""The deployed student's control step: USVSysIDStudentPolicy.act (one dagger_student_act_f32 launch: history ring, encoder, action head)
against the unfused composition it replaces (USVSysIDVecEnv's torch.roll + frame write of the (N, T, D) history, then
USVSysIDAgent.get_student_action: cat, encoder, cat, head), device-timed with CUDA events over K steps after W warm-up steps.
Each (arm, env count) runs in its own subprocess and the arms alternate, round after round:
    python scripts/time_student_act.py --rounds 3 > student_act.jsonl
The env step is not part of either arm: the observations are 8 random buffers in turn.  Both arms see the same inputs, and each
worker reports a hash of its last mu, which must agree between the arms.  One JSON line per (round, arm, env count), with the card it
ran on; then one line per env count with the min / median / max per arm over rounds."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARMS = ("fused", "unfused")


def worker(args):
    sys.path.insert(0, ROOT)
    import torch

    from omniisaacgymenvs_loop_b200.algo.ppo.dagger import USVSysIDAgent, USVSysIDStudentPolicy
    from omniisaacgymenvs_loop_b200.algo.ppo.module import E1, E2, H, MLPEncode, StateHistoryEncoder
    from scripts.time_step_residency import card

    if not torch.cuda.is_available():
        raise SystemExit("time_student_act.py times CUDA kernels: no GPU found")
    dev = torch.device("cuda:0")
    n, T, D, priv, lat = args.envs, args.history_len, 25, 8, 8
    torch.manual_seed(1234)
    arch = MLPEncode([H, H], "LeakyReLU", D + priv, 2, "Tanh", speed_dim=3, mass_dim=priv, mass_latent_dim=lat, mass_encoder_shape=[E1, E2])
    arch.flat = arch.flat.to(dev)
    enc = StateHistoryEncoder("LeakyReLU", D, T, lat, dev, seed=1234)
    g = torch.Generator(device=dev).manual_seed(1234)
    obs = [torch.randn((n, D + priv), device=dev, generator=g) for _ in range(8)]
    if args.arm == "fused":
        pol = USVSysIDStudentPolicy(id_encoder=enc, frozen_action_head=arch.action_mlp, history_len=T, obs_nonpriv_dim=D)
        pol.reset(obs[0])
        step = lambda o: pol.act(o)                                                   # noqa: E731
    else:
        agent = USVSysIDAgent(teacher_mass_encoder=None, id_encoder=enc, frozen_action_head=arch.action_mlp, history_len=T,
                              obs_nonpriv_dim=D, device=dev)
        hist = torch.zeros((n, T, D), device=dev)
        hist[:, -1, :] = obs[0][:, :D]
        state = {"hist": hist}

        def step(o):                                                                  # usv_raisim_vecenv.py:137-139 + dagger.py:45-50
            cur = o[:, :D]
            h = torch.roll(state["hist"], shifts=-1, dims=1)
            h[:, -1, :] = cur
            state["hist"] = h
            return agent.get_student_action(torch.cat([h.reshape(n, -1), cur], dim=1))
    for w in range(args.warmup):
        step(obs[(w + 1) % 8])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        mu = step(obs[(args.warmup + k + 1) % 8])
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / args.steps
    print(json.dumps({"envs": n, "history_len": T, "steps": args.steps, "us_per_step": us, "env_steps_per_s": n / (us * 1e-6),
                      "mu_sha1": hashlib.sha1(mu.cpu().numpy().tobytes()).hexdigest(), "gpu": card()}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--history-len", type=int, default=50, choices=[50, 20, 10])
    ap.add_argument("--arm", choices=ARMS, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.rounds < 1:
        ap.error("--steps and --rounds must be at least 1, --warmup at least 0")
    if args.arm:
        args.envs = args.envs[0]
        worker(args)
        return
    runs = {}
    for rnd in range(args.rounds):
        for n in args.envs:
            for arm in (ARMS if rnd % 2 == 0 else ARMS[::-1]):
                cmd = [sys.executable, os.path.abspath(__file__), "--arm", arm, "--envs", str(n), "--steps", str(args.steps),
                       "--warmup", str(args.warmup), "--history-len", str(args.history_len)]
                r = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, check=True)
                line = {"round": rnd, "arm": arm, **json.loads(r.stdout.strip().splitlines()[-1])}
                runs.setdefault(n, {}).setdefault(arm, []).append(line)
                print(json.dumps(line), flush=True)
    for n, by_arm in runs.items():
        out = {"summary": True, "envs": n, "history_len": args.history_len, "rounds": args.rounds}
        for arm, lines in by_arm.items():
            us = [x["us_per_step"] for x in lines]
            out.update({f"{arm}_us_min": min(us), f"{arm}_us_median": statistics.median(us), f"{arm}_us_max": max(us)})
        out["speedup_median"] = out["unfused_us_median"] / out["fused_us_median"]
        out["same_mu"] = len({x["mu_sha1"] for lines in by_arm.values() for x in lines}) == 1
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
