#!/usr/bin/env python
"""L2 residency of the fused step across env counts: the classic full-DR step kernel, device-timed with CUDA events over K steps
after W warm-up steps, at 2^18 .. 2^21 envs.  Each arm (a build of libusv_b200.so) runs in its own subprocess and the arms
alternate, round after round, so that two builds are compared on the same GPU:
    python scripts/time_step_residency.py --lib parent=/path/to/parent/libusv_b200.so --rounds 3 > residency.jsonl
The arm `this` is the library of this tree.  One JSON line per (round, arm, env count), with the card it ran on; then one summary
line per (arm, env count) with the min / median / max over rounds.

Byte model per env-step (DESIGN.md, "L2 residency"): env state 52 B + reset_buf 8 B are read and written every step and are the
only bytes the next step reads again (resident); per-episode constants 96 B + actions 8 B read, obs 52 B + reward 4 B written are
one-pass (streamed).  --stats adds the 15 episode-sum words (60 B read + 60 B written), reported on their own."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RESIDENT_B, STREAMED_B, STATS_B = 52 + 8, 96 + 8 + 52 + 4, 2 * 60


def card():
    """name, power limit and max SM clock of cuda:0 (read-only nvidia-smi query, matched by UUID)."""
    import torch

    uuid = str(torch.cuda.get_device_properties(0).uuid)
    r = subprocess.run(["nvidia-smi", "-i", "GPU-" + uuid, "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else None


def worker(args):
    sys.path.insert(0, ROOT)
    import torch

    from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
    from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv

    if not torch.cuda.is_available():
        raise SystemExit("time_step_residency.py times the CUDA kernel: no GPU found")
    dev = torch.device("cuda:0")
    gpu = card()
    for lg in args.log2_envs:
        n = 1 << lg
        env = FusedUsvEnv(UsvEnvConfig().full_dr(), n, dev, collect_stats=args.stats)
        g = torch.Generator(device=dev).manual_seed(1234)
        acts = [torch.rand((n, 2), device=dev, generator=g) * 2 - 1 for _ in range(8)]      # as bench.py: 8 action buffers in turn
        for w in range(args.warmup):
            env.step(acts[w % 8])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.steps):
            env.step(acts[k % 8])
        e1.record()
        torch.cuda.synchronize()
        env.check_finite()
        us = e0.elapsed_time(e1) * 1e3 / args.steps
        line = {"envs": n, "stats": args.stats, "steps": args.steps, "us_per_step": us, "env_steps_per_s": n / (us * 1e-6),
                "resident_mb_per_step": RESIDENT_B * n / 1e6, "streamed_mb_per_step": STREAMED_B * n / 1e6, "gpu": gpu}
        if args.stats:
            line["stats_mb_per_step"] = STATS_B * n / 1e6
        print(json.dumps(line), flush=True)
        del env, acts
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH", help="another build to alternate with this tree's")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--log2-envs", type=int, nargs="+", default=[18, 19, 20, 21])
    ap.add_argument("--stats", action="store_true", help="collect the episode sums (the <kDisturb, true> kernel)")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.rounds < 1:
        ap.error("--steps and --rounds must be at least 1, --warmup at least 0")
    if args.worker:
        worker(args)
        return
    arms = [("this", None)]
    for spec in args.lib:
        name, sep, path = spec.partition("=")
        if not sep or not os.path.isfile(path):
            ap.error(f"--lib wants NAME=PATH to an existing library, got {spec!r}")
        arms.append((name, os.path.abspath(path)))
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(args.steps), "--warmup", str(args.warmup),
           "--log2-envs", *map(str, args.log2_envs)] + (["--stats"] if args.stats else [])
    runs = {}
    for rnd in range(args.rounds):
        for name, path in arms:
            env = dict(os.environ)
            env.pop("USV_B200_LIB", None)
            if path:
                env["USV_B200_LIB"] = path
            r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, text=True, check=True)
            for s in r.stdout.splitlines():
                line = {"round": rnd, "arm": name, **json.loads(s)}
                runs.setdefault((name, line["envs"]), []).append(line["us_per_step"])
                print(json.dumps(line), flush=True)
    for (name, n), us in runs.items():
        print(json.dumps({"summary": True, "arm": name, "envs": n, "stats": args.stats, "rounds": len(us), "us_per_step_min": min(us),
                          "us_per_step_median": statistics.median(us), "us_per_step_max": max(us),
                          "env_steps_per_s_median": n / (statistics.median(us) * 1e-6)}), flush=True)


if __name__ == "__main__":
    main()
