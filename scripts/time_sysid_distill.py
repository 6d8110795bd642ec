#!/usr/bin/env python
"""SysID distillation, collect and update timed apart: the fused loop (USVSysIDDistiller: one dagger_sysid_collect_f32 launch per control
step into a frame store, windows rebuilt inside the training kernels) against the unfused loop it replaces (USVSysIDVecEnv's roll + cat,
USVSysIDTrainer.step / observe / update on ObsStorage), both on the live env (scripts/dagger_usv_sysid_loopz.py build_fused / build).
Each (arm, env count) runs in its own subprocess and the arms alternate, round after round:
    python scripts/time_sysid_distill.py --rounds 3 > sysid_distill.jsonl
Per update, CUDA events time the collect phase (horizon x {observe, student step, env step}) and the update phase (4 epochs x 4
minibatches + the metrics, which end in host reads) after W warm-up updates.  torch.cuda.max_memory_allocated is taken over the timed
updates only (the peak statistics are reset after the build and the warm-up).  Both arms start from one seed and must end with the same
encoder parameters (params_sha1).  One JSON line per (round, arm, env count), with the card it ran on; then one summary line per env
count with the median per arm over rounds."""
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

    from scripts.dagger_usv_sysid_loopz import build_fused, build_with_teacher
    from scripts.time_step_residency import card

    if not torch.cuda.is_available():
        raise SystemExit("time_sysid_distill.py times CUDA kernels: no GPU found")
    dev, n, T, H, seed = "cuda:0", args.envs, args.history_len, args.horizon, 1234
    torch.cuda.set_device(dev)
    torch.manual_seed(seed)
    if args.arm == "fused":
        env, dist, _ = build_fused(n, dev, seed, history_len=T, priv_dim=8, horizon=H)
        trainer, state = dist.trainer, {"dones": None}

        def collect():                                                        # dagger_usv_sysid_loopz.run_fused
            for _ in range(H):
                obs = env.observe(as_numpy=False)
                mu = dist.reset(obs) if state["dones"] is None else dist.act(obs, state["dones"])
                _, state["dones"] = env.step(mu)

        update = dist.update
        D = dist.D
        sample_bytes = dist.store.numel() * 4 + dist.refill.numel() * 4
    else:
        env, trainer, _ = build_with_teacher(n, dev, seed, history_len=T, priv_dim=8, horizon=H)

        def collect():                                                        # dagger_usv_sysid_loopz.run
            for _ in range(H):
                sysid_obs = env.observe_sysid_obs(as_numpy=False)
                trainer.step(sysid_obs, env.get_priv_tail())
                env.step(trainer.observe(sysid_obs))

        update = trainer.update
        D = env.obs_nonpriv_dim
        sample_bytes = trainer.storage.obs.numel() * 4
    env.reset()
    for _ in range(args.warmup):
        collect()
        update()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.updates)]
    for u in range(args.updates):
        ev[u][0].record()
        collect()
        ev[u][1].record()
        update()
        ev[u][2].record()
    torch.cuda.synchronize()
    col = sum(e[0].elapsed_time(e[1]) for e in ev) / args.updates
    upd = sum(e[1].elapsed_time(e[2]) for e in ev) / args.updates
    frames = H * n
    print(json.dumps({"envs": n, "history_len": T, "horizon": H, "obs_nonpriv_dim": D, "updates": args.updates, "collect_ms": col,
                      "update_ms": upd, "total_ms": col + upd, "collect_frames_per_s": frames / (col * 1e-3),
                      "frames_per_s": frames / ((col + upd) * 1e-3), "sample_bytes": sample_bytes,
                      "max_memory_allocated": torch.cuda.max_memory_allocated(),
                      "params_sha1": hashlib.sha1(trainer.actor.id_encoder.flat.cpu().numpy().tobytes()).hexdigest(), "gpu": card()}),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--updates", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--history-len", type=int, default=50, choices=[50, 20, 10])
    ap.add_argument("--horizon", type=int, default=16)
    ap.add_argument("--arm", choices=ARMS, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.updates < 1 or args.warmup < 0 or args.rounds < 1 or args.horizon < 1:
        ap.error("--updates, --rounds and --horizon must be at least 1, --warmup at least 0")
    if args.arm:
        args.envs = args.envs[0]
        worker(args)
        return
    runs = {}
    for rnd in range(args.rounds):
        for n in args.envs:
            for arm in (ARMS if rnd % 2 == 0 else ARMS[::-1]):
                cmd = [sys.executable, os.path.abspath(__file__), "--arm", arm, "--envs", str(n), "--updates", str(args.updates),
                       "--warmup", str(args.warmup), "--history-len", str(args.history_len), "--horizon", str(args.horizon)]
                r = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, check=True)
                line = {"round": rnd, "arm": arm, **json.loads(r.stdout.strip().splitlines()[-1])}
                runs.setdefault(n, {}).setdefault(arm, []).append(line)
                print(json.dumps(line), flush=True)
    for n, by_arm in runs.items():
        out = {"summary": True, "envs": n, "history_len": args.history_len, "rounds": args.rounds}
        for arm, lines in by_arm.items():
            for key in ("collect_ms", "update_ms", "total_ms", "frames_per_s"):
                out[f"{arm}_{key}_median"] = statistics.median(x[key] for x in lines)
            out[f"{arm}_sample_bytes"] = lines[0]["sample_bytes"]
            out[f"{arm}_max_memory_allocated"] = max(x["max_memory_allocated"] for x in lines)
        out["same_params"] = len({x["params_sha1"] for lines in by_arm.values() for x in lines}) == 1
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
