#!/usr/bin/env python
"""Overlap of consecutive fused steps (programmatic dependent launch): the classic full-DR step kernel at 2^19 .. 2^21 envs, device-timed
with CUDA events over K steps after W warm-up steps.  Each arm (a build of libusv_b200.so) runs in its own subprocess and the arms
alternate, round after round, so that two builds are compared on the same GPU:
    python scripts/time_step_overlap.py --lib parent=/path/to/parent/libusv_b200.so --rounds 3 > overlap.jsonl
The arm `this` is the library of this tree.  One JSON line per (round, arm, env count), with the card it ran on and the median SM clock
of the timed window; then one summary line per (arm, env count) with the min / median / max over rounds.

With --profile-steps P, one more process per arm records P steps per env count under torch.profiler (a run of its own: no event timing
in it) and reports, per step, the kernel's own duration, the start-to-start period and the gap from one step kernel's end to the next
one's start.  A negative gap means the next launch was already resident (waiting in griddepcontrol.wait) when this one ended; its
duration then includes that wait."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RESIDENT_B = 52 + 8            # env state + reset_buf: the bytes the next step reads again (see step_fused_kernel)
RESIDENT_L2_SHARE = 0.75       # kResidentL2Share of csrc/usv_step.cu: above it the launch picks the plain-access instance


def setup(n):
    import torch

    from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
    from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv

    dev = torch.device("cuda:0")
    env = FusedUsvEnv(UsvEnvConfig().full_dr(), n, dev)
    g = torch.Generator(device=dev).manual_seed(1234)
    acts = [torch.rand((n, 2), device=dev, generator=g) * 2 - 1 for _ in range(8)]      # as bench.py: 8 action buffers in turn
    return env, acts


def instance(n):
    import torch

    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    return "stream" if RESIDENT_B * n <= RESIDENT_L2_SHARE * l2 else "plain"


def time_events(env, acts, steps, warmup):
    import torch

    from bench import ClockSampler

    for w in range(warmup):
        env.step(acts[w % 8])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        env.step(acts[k % 8])
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    env.check_finite()
    return e0.elapsed_time(e1) * 1e3 / steps, clocks


def profile_steps(env, acts, steps, warmup):
    """Start, duration (us) of every step kernel of `steps` steps recorded by torch.profiler (CUDA activities only)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    for w in range(warmup):
        env.step(acts[w % 8])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(steps):
            env.step(acts[k % 8])
        torch.cuda.synchronize()
    env.check_finite()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return sorted((float(e["ts"]), float(e["dur"])) for e in events
                  if e.get("cat") == "kernel" and "step_fused_kernel" in e.get("name", ""))


def worker(args):
    sys.path.insert(0, ROOT)
    import torch

    from scripts.time_step_residency import card

    if not torch.cuda.is_available():
        raise SystemExit("time_step_overlap.py times the CUDA kernel: no GPU found")
    gpu = card()
    for lg in args.log2_envs:
        n = 1 << lg
        env, acts = setup(n)
        line = {"envs": n, "instance": instance(n), "gpu": gpu}
        if args.profile_steps:
            ks = profile_steps(env, acts, args.profile_steps, args.warmup)
            dur = [d for _, d in ks]
            period = [b[0] - a[0] for a, b in zip(ks, ks[1:])]
            gap = [b[0] - (a[0] + a[1]) for a, b in zip(ks, ks[1:])]
            line.update({"profiled_steps": len(ks), "kernel_us_median": statistics.median(dur), "period_us_median": statistics.median(period),
                         "gap_us_median": statistics.median(gap), "gap_us_min": min(gap), "gap_us_max": max(gap)})
        else:
            us, clocks = time_events(env, acts, args.steps, args.warmup)
            line.update({"steps": args.steps, "us_per_step": us, "env_steps_per_s": n / (us * 1e-6), "sm_mhz_median": clocks["sm_mhz"],
                         "clock_reasons": clocks["reasons"]})
        print(json.dumps(line), flush=True)
        del env, acts
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH", help="another build to alternate with this tree's")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--log2-envs", type=int, nargs="+", default=[19, 20, 21])
    ap.add_argument("--profile-steps", type=int, default=0, help="after the timed rounds, one torch.profiler run of this many steps per arm")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.rounds < 1 or args.profile_steps < 0:
        ap.error("--steps and --rounds must be at least 1, --warmup and --profile-steps at least 0")
    if args.worker:
        worker(args)
        return
    arms = [("this", None)]
    for spec in args.lib:
        name, sep, path = spec.partition("=")
        if not sep or not os.path.isfile(path):
            ap.error(f"--lib wants NAME=PATH to an existing library, got {spec!r}")
        arms.append((name, os.path.abspath(path)))
    base = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(args.steps), "--warmup", str(args.warmup),
            "--log2-envs", *map(str, args.log2_envs)]

    def run(name, path, extra):
        env = dict(os.environ)
        env.pop("USV_B200_LIB", None)
        if path:
            env["USV_B200_LIB"] = path
        r = subprocess.run(base + extra, env=env, stdout=subprocess.PIPE, text=True, check=True)
        return [json.loads(s) for s in r.stdout.splitlines()]

    runs = {}
    for rnd in range(args.rounds):
        for name, path in arms:
            for res in run(name, path, []):
                line = {"round": rnd, "arm": name, **res}
                runs.setdefault((name, line["envs"]), []).append(line["us_per_step"])
                print(json.dumps(line), flush=True)
    for (name, n), us in runs.items():
        print(json.dumps({"summary": True, "arm": name, "envs": n, "rounds": len(us), "us_per_step_min": min(us),
                          "us_per_step_median": statistics.median(us), "us_per_step_max": max(us),
                          "env_steps_per_s_median": n / (statistics.median(us) * 1e-6)}), flush=True)
    if args.profile_steps:
        for name, path in arms:
            for res in run(name, path, ["--profile-steps", str(args.profile_steps)]):
                print(json.dumps({"profile": True, "arm": name, **res}), flush=True)


if __name__ == "__main__":
    main()
