#!/usr/bin/env python
"""bench.py -- headline benchmark of the fused ASV env step (BASELINE.json metric: ASV env-steps/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host cores (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write obs / reward / done of the last timed step as DIR/*.npy

A "step" is one control step of every env of the batch (one launch of step_fused_kernel):
reset-if-flagged + 5 physics sub-steps + CaptureXY obs + reward + penalties + done, full per-env
domain randomisation ("A, full DR": 268 algorithmic bytes per env-step, SURVEY 8(d) / DESIGN.md).
Workload: CaptureXY SysID (classic snapshot constants), --envs per GPU (default 2^20, the top point of
BASELINE's env-count sweep: the SoA working set is ~2.2x the 126 MB L2, so every step streams from HBM);
the 4096-env point of BASELINE config[1] is launch-latency bound and is reported beside it under "c2_4096".

One JSON line on stdout (rank 0); everything else goes to stderr.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

BYTES_PER_ENV_STEP = 268          # "A, full DR, stats off" (SURVEY 8(d)): 156 B read + 112 B written
METRIC, UNIT = "ASV env-steps/sec", "env-steps/s"
DUMP_LIMIT_BYTES = 64_000_000     # --dump-outputs: all files together (2^20 envs x (13 + 1 + 1) float32 = 62.9 MB fits whole)
NPY_HEADER_BYTES = 128


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            log("clock sampling unavailable:", e)
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = get(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
def pick_threads(make_env, n_probe=65536):
    """The CPU port may use every host thread: time EVERY candidate thread count on a probe of the workload's own scale (65 536 envs per
    step; the r01 probe of 4096 envs sat in launch overhead and picked 1 or 8 threads at random, a 4.5x swing of the reference arm) and
    keep the fastest.  Returns (threads, {threads: env-steps/s})."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64, ncpu // 2, ncpu) if 1 <= c <= ncpu})
    env = make_env(n_probe)
    act = torch.zeros((n_probe, 2))
    env.step(act)
    rates = {}
    for nt in cands:
        torch.set_num_threads(nt)
        env.step(act)
        t = time.perf_counter()
        for _ in range(3):
            env.step(act)
        rates[nt] = 3 * n_probe / (time.perf_counter() - t)
        log(f"  cpu probe ({n_probe} envs): {nt} threads -> {rates[nt]:.3g} env-steps/s")
    best = max(rates, key=rates.get)
    torch.set_num_threads(best)
    return best, rates


def cpu_port(budget_s: float, steps: int | None = None, warmup: int = 1, envs: int | None = None):
    """Times the oracle port (the reference's torch algorithm, CPU) on a bounded sample of the workload."""
    from oracle import usv_oracle as O

    cfg = O.EnvConfig().full_dr()
    mk = lambda n: O.ClassicEnvOracle(cfg, n)
    threads, probe_rates = pick_threads(mk)
    if envs is None or steps is None:
        # size the sample: n envs per step so that `steps` steps fit the budget
        probe = mk(16384)
        act = torch.zeros((16384, 2))
        probe.step(act)
        t = time.perf_counter()
        probe.step(act)
        rate = 16384 / (time.perf_counter() - t)
        auto_steps = steps is None
        steps = steps or 8
        envs = envs or int(min(1 << 20, max(4096, rate * budget_s / (steps + warmup))))
        envs = 1 << (envs.bit_length() - 1)
        if auto_steps:          # the env count is capped at the workload's: spend the rest of the budget on more control steps
            steps = int(max(8, min(64, rate * budget_s / envs - warmup)))
    env = mk(envs)
    g = torch.Generator().manual_seed(0)
    acts = [torch.rand((envs, 2), generator=g) * 2 - 1 for _ in range(4)]
    for w in range(warmup):
        env.step(acts[w % 4])
    t = time.perf_counter()
    for k in range(steps):
        env.step(acts[k % 4])
    dt = time.perf_counter() - t
    return {"value": envs * steps / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{envs} envs x {steps} control steps (oracle/usv_oracle.ClassicEnvOracle, torch CPU fp32, "
                      f"{threads} of {os.cpu_count()} host threads: the fastest of {sorted(probe_rates)} on a 65 536-env probe), full DR, 5 sub-steps",
            "thread_probe": {str(k): round(v) for k, v in probe_rates.items()}}, dt / steps


def run_reference(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = 150.0
    # exactly --warmup + --steps control steps; only the env count is sized to the budget
    cb, s_per_step = cpu_port(budget, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.envs, note="reference arm: the oracle port of the reference's torch path on host cores "
                                      "(the Python reference needs Isaac Sim); the env count is sized so that warm-up + timed steps "
                                      f"fit a {budget:.0f} s budget"),
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_config(envs, note=None):
    c = {"workload": f"CaptureXY SysID classic (13-dim obs), fused reset+dynamics+obs+reward+done step, {envs} envs/GPU, "
                     f"full per-env DR, 5 sub-steps/control step",
         "envs_per_gpu": envs, "substeps": 5, "obs_dim": 13, "bytes_per_env_step": BYTES_PER_ENV_STEP,
         "l2": "inputs larger than L2 (SoA working set = envs*~280 B; 2^20 envs = 294 MB vs 126 MB L2), no flush needed"}
    if note:
        c["note"] = note
    return c


def dump_outputs(out_dir, arrays):
    """Writes per-env arrays (first dim = env) as <out_dir>/<name>.npy in float32, so that two builds can be compared output for output.
    Above DUMP_LIMIT_BYTES in all, every array keeps the same fixed, seeded sample of env rows; env_index.npy (float64) lists them."""
    import numpy as np

    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(4 * a[0].numel() for a in arrays.values())
    keep = None
    if n * row_bytes + NPY_HEADER_BYTES * len(arrays) > DUMP_LIMIT_BYTES:
        m = (DUMP_LIMIT_BYTES - NPY_HEADER_BYTES * (len(arrays) + 1)) // (row_bytes + 8)
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:m].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach()
        if keep is not None:
            a = a[keep.to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.to(torch.float32).cpu().numpy())
    if keep is not None:
        np.save(os.path.join(out_dir, "env_index.npy"), keep.to(torch.float64).numpy())
    log(f"  outputs of the last timed step -> {out_dir}: {', '.join(arrays)}"
        + (f" ({len(keep)} of {n} envs, env_index.npy)" if keep is not None else f" ({n} envs)"))


# ------------------------------------------------------------------------------------------------
def time_steps(env, acts, steps, warmup, dist_on, device):
    """Device-timed: W warm-up steps, then exactly K steps between CUDA events on the launching stream."""
    import torch.distributed as dist

    for w in range(warmup):
        env.step(acts[w % len(acts)])
    torch.cuda.synchronize(device)
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        env.step(acts[k % len(acts)])
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms


def gpu_local_cpus(device):
    """CPUs on the NUMA node of `device`'s PCIe slot (sysfs local_cpulist), or None."""
    try:
        pr = torch.cuda.get_device_properties(device)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        return cpus or None
    except Exception:
        return None


def time_e2e(env, steps, warmup, dist_on, device):
    """The same metric through the public host-buffer call (engine.HostStepper.submit): per step the actions come from pinned host
    memory and obs + reward + done go back to pinned host memory; every copy is inside the timed region, the copies of neighbouring
    steps overlap the kernel (3 streams, 2 staging slots).  The final synchronize() is inside the timed region too."""
    import torch.distributed as dist
    from omniisaacgymenvs_loop_b200.engine import HostStepper

    n = env.num_envs
    # multi-rank: allocate (first-touch) the pinned staging buffers from the CPUs next to this rank's GPU, otherwise every rank's
    # copies cross the socket interconnect and share one memory controller (8 ranks: 1.55e9 env-steps/s whatever the rank count)
    saved_aff = None
    if dist_on:
        cpus = gpu_local_cpus(device)
        if cpus:
            saved_aff = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus)
            log(f"  e2e: rank pinned to {len(cpus)} CPUs local to {device}")
    g = torch.Generator().manual_seed(1)
    h_act = [(torch.rand((n, 2), generator=g) * 2 - 1).pin_memory() for _ in range(2)]
    h_obs = [torch.empty((n, 13), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_rew = [torch.empty(n, dtype=torch.float32).pin_memory() for _ in range(2)]
    h_done = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(2)]
    hs = HostStepper(env, depth=2)

    def one(k):
        hs.submit(h_act[k & 1], h_obs[k & 1], h_rew[k & 1], h_done[k & 1])

    for w in range(warmup):
        one(w)
    hs.synchronize()
    torch.cuda.synchronize(device)
    if dist_on:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        one(k)
    hs.synchronize()
    torch.cuda.synchronize(device)
    ms = (time.perf_counter() - t0) * 1e3          # three streams: wall clock around a fully synchronised region
    if dist_on:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    h2d = n * 2 * 4
    d2h = n * 13 * 4 + n * 4 + n * 1
    if saved_aff is not None:
        os.sched_setaffinity(0, saved_aff)
    return ms, h2d, d2h, float(h_rew[0].mean())


def ppo_cpu_port(envs=2048, epochs=2, horizon=16, minibatch=8192, mini_epochs=8):
    """The PPO half of the metric on the host cores: the oracle port of the whole rl_games epoch (rollout through the CPU env oracle +
    policy inference, GAE, prepare_dataset, mini_epochs x minibatches of loss / autograd backward / clip / Adam / adaptive lr) on a
    bounded sample (`envs` envs; the per-frame cost does not depend on the env count once a minibatch is 8192 rows)."""
    from oracle import ppo_oracle as P
    from oracle import usv_oracle as O

    D = 13
    threads = torch.get_num_threads()
    env = O.ClassicEnvOracle(O.EnvConfig(), envs)
    lay = P.param_layout(D)
    g = torch.Generator().manual_seed(0)
    params = torch.zeros(lay["P"])
    for name in ("w1", "w2", "wv", "wmu"):
        a, b = lay[name]
        fan = D if name == "w1" else 128
        params[a:b] = (torch.rand(b - a, generator=g) * 2 - 1) / fan ** 0.5
    m, v, step, lr = torch.zeros_like(params), torch.zeros_like(params), 0, 1e-4
    obs_rms, val_rms = P.RunningMeanStd((D,)), P.RunningMeanStd((1,))
    obs, _, done = env.step(torch.zeros((envs, 2)))
    times = []
    for ep in range(epochs + 1):
        t0 = time.perf_counter()
        roll = {k: [] for k in ("obses", "actions", "neglogpacs", "values", "mus", "sigmas", "rewards", "dones")}
        with torch.no_grad():
            for t in range(horizon):
                r = P.policy_inference(params, obs, D, obs_rms, val_rms, eps=torch.randn((envs, 2), generator=g))
                roll["obses"].append(obs.clone()); roll["dones"].append(done.to(torch.uint8))
                for k, src in (("actions", "actions"), ("neglogpacs", "neglogpacs"), ("values", "values"), ("mus", "mus"), ("sigmas", "sigmas")):
                    roll[k].append(r[src])
                obs, rew, done = env.step(torch.clamp(r["actions"], -1.0, 1.0))
                roll["rewards"].append(rew * 0.01)
            roll = {k: torch.stack(x) for k, x in roll.items()}
            last_v = P.policy_inference(params, obs, D, obs_rms, val_rms)["values"][:, 0]
            adv = P.discount_values(done.float(), last_v, roll["dones"].float(), roll["values"][..., 0], roll["rewards"])
            ds = P.prepare_dataset(roll, (adv + roll["values"][..., 0]).unsqueeze(-1), val_rms)
        params, m, v, step, lr = P.train_epoch(params, m, v, step, lr, ds, D, obs_rms, minibatch_size=min(minibatch, horizon * envs),
                                               mini_epochs=mini_epochs)
        if ep > 0:
            times.append(time.perf_counter() - t0)
    s_per_epoch = sum(times) / len(times)
    return {"value": horizon * envs / s_per_epoch, "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"{envs} envs x horizon {horizon}, {mini_epochs} mini-epochs x {horizon * envs // min(minibatch, horizon * envs)} minibatches of "
                      f"{min(minibatch, horizon * envs)} rows, {epochs} epochs (oracle/ppo_oracle + oracle/usv_oracle, torch CPU + autograd, {threads} threads)",
            "s_per_epoch": s_per_epoch}


def memcpy_probe(device, h2d_bytes, d2h_bytes, iters=30):
    """Plain pinned cudaMemcpyAsync bandwidth of this rank with every rank copying at the same time: the ceiling of the e2e leg.
    One H2D and one D2H stream, the e2e step's own byte counts per iteration; returns GB/s (both directions summed) of this rank."""
    h_in, h_out = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory(), torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    d_in, d_out = torch.empty(h2d_bytes, dtype=torch.uint8, device=device), torch.empty(d2h_bytes, dtype=torch.uint8, device=device)
    s1, s2 = torch.cuda.Stream(device), torch.cuda.Stream(device)
    def run(n):
        for _ in range(n):
            with torch.cuda.stream(s1):
                d_in.copy_(h_in, non_blocking=True)
            with torch.cuda.stream(s2):
                h_out.copy_(d_out, non_blocking=True)
        s1.synchronize(); s2.synchronize()
    run(3)
    t0 = time.perf_counter()
    run(iters)
    dt = time.perf_counter() - t0
    return (h2d_bytes + d2h_bytes) * iters / dt / 1e9


def bench_ppo(args, rank, world, device, dist_on):
    """BASELINE config[2]: CaptureXY + USV_PPOcontinuous_MLP, 16384 envs/GPU, env-sharded; gradient all-reduce = one kernel over NVLink
    peer memory per minibatch (rl/peer.py), update phase replayed as one CUDA graph per rank.
    PPO frames/s = horizon * envs * world / epoch time (rollout + GAE + dataset + 8 mini-epochs x 32 minibatches)."""
    import torch.distributed as dist
    from omniisaacgymenvs_loop_b200 import _lib
    from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
    from omniisaacgymenvs_loop_b200.rl.a2c import A2CAgent, PPOConfig
    from scripts.train_usv import make_env

    n = args.ppo_envs
    cfg = UsvEnvConfig(num_envs=n)
    env = make_env(cfg.to_task_cfg(), str(device), seed=1234, env_id_offset=rank * n, collect_stats=False)
    env.env._task._nan_probe = False
    agent = A2CAgent(env, PPOConfig(seed=1234), device, rank, world)
    ar_err = None
    if dist_on and agent.peer is not None:          # warm-up: one result of the NVLink peer all-reduce against NCCL's
        x = torch.randn(agent.policy.grads.numel(), device=device, generator=torch.Generator(device=device).manual_seed(77 + rank))
        want = x.clone()
        dist.all_reduce(want)
        got = agent.peer(x.clone())
        ar_err = float((got - want).abs().max())
    for _ in range(3):
        agent.train_epoch()
    torch.cuda.synchronize(device)
    if dist_on:
        dist.barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    play = upd = 0.0
    e0.record()
    for _ in range(args.ppo_epochs):
        p, u = agent.train_epoch()
        play += p
        upd += u
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    frames = agent.batch_size * world * args.ppo_epochs
    st = agent.policy.stats()
    agent.check_peers()
    identical = agent.ranks_identical()             # all-gather of an exact checksum of parameters, Adam moments, lr and step count
    launches = (_lib.launch_count() - l0) / args.ppo_epochs + sum(agent.graph_launches.values())
    fused = agent.peer_step is not None and agent.fused_step
    detail = {"horizon": agent.T, "minibatch": agent.minibatch_size, "mini_epochs": agent.cfg.mini_epochs, "epochs_timed": args.ppo_epochs,
              "host_play_s": play, "host_update_s": upd, "rollout_in_cuda_graph": agent._graph_play is not None,
              "update_in_cuda_graph": agent._graph is not None, "update_graph_launches": agent.graph_launches["update"],
              "mlp": ("tcgen05 TF32 UMMA + TMEM (csrc/ppo_mlp_tc.cu)" if agent.policy.tensor_cores else "fp32 SIMT fused kernels (csrc/ppo_mlp.cu)"),
              "kl": st["kl"], "lr": st["lr"]}
    short = {"metric": "PPO frames/sec", "value": frames / (ms * 1e-3), "unit": "frames/s", "envs_per_gpu": n, "ms_per_epoch": ms / args.ppo_epochs,
             "collective": ("none" if world == 1 else ("peer packets fused into the minibatch tail kernel (NVLink P2P)" if fused else agent.collective)),
             "launches_per_epoch": launches, "ranks_identical": bool(identical), "allreduce_vs_nccl_max_abs_err": ar_err}
    return short, detail


def bench_gae_mlp(device):
    """Secondary kernels of the north_star's ncu evidence: GAE (HBM-bound) and the policy MLP (tensor pipe)."""
    import ctypes
    from omniisaacgymenvs_loop_b200 import _lib
    from omniisaacgymenvs_loop_b200.rl.a2c import gae
    from omniisaacgymenvs_loop_b200.rl.policy import PolicyMLP

    out = {}
    T, n = 16, 1 << 22                                      # 4M envs x 16: 1.16 GB touched per launch (>> L2)
    g = torch.Generator(device=device).manual_seed(0)
    rew, val = torch.randn((T, n), device=device, generator=g), torch.randn((T, n), device=device, generator=g)
    dones = (torch.rand((T, n), device=device, generator=g) < 0.1).to(torch.uint8)
    lv, ld = torch.randn(n, device=device, generator=g), torch.zeros(n, dtype=torch.uint8, device=device)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    for _ in range(3):
        gae(rew, val, dones, lv, ld, 0.99, 0.95, adv, ret)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        gae(rew, val, dones, lv, ld, 0.99, 0.95, adv, ret)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / 20
    peak, _ = measured_peak()
    gbs = 277.0 * n / (ms * 1e-3) / 1e9                     # 149 B read + 128 B written per env per rollout (SURVEY 8(d))
    out["gae"] = {"kernel": "usv::gae_kernel<4>", "envs": n, "horizon": T, "ms": ms, "achieved_gbs": gbs, "frac_of_measured_hbm": gbs / peak,
                  "bytes_per_env_rollout": 277}
    del rew, val, dones, adv, ret
    M = 1 << 20
    pol = PolicyMLP(13, device)
    obs = torch.randn((M, 13), device=device, generator=g)
    o = pol.act(obs)
    for _ in range(3):
        pol.act(obs, o)
    e0.record()
    for _ in range(10):
        pol.act(obs, o)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / 10
    flops = 2.0 * (13 * 128 + 128 * 128 + 128 * 3) * M     # algorithmic (un-padded) forward FLOPs
    out["mlp_forward"] = {"kernel": "ppotc::forward_tc_kernel (tcgen05 kind::tf32, TMEM accumulators)", "rows": M, "ms": ms,
                          "rows_per_s": M / (ms * 1e-3), "algorithmic_tflops": flops / (ms * 1e-3) / 1e12,
                          "note": "tiny-K/N GEMMs: bounded by the tanh/TMEM epilogue and operand staging, not by the tensor pipe"}
    return out


def bench_loopz(device, envs=16384, updates=10):
    """SURVEY 8(f) row 4: the loopz learner (MLPEncode actor / critic, squashed Gaussian) on the live CaptureXY task, 16 384 envs, horizon 16,
    4 epochs x 4 in-order minibatches of 65 536 rows: frames/s of the whole loop, the update phase alone, and the kernels."""
    from omniisaacgymenvs_loop_b200.config import live_default_config, live_task_cfg
    from scripts.train_loopz import LoopzRunner, build_learner, make_env, train

    torch.manual_seed(1234)
    env = make_env(live_task_cfg(live_default_config(num_envs=envs)), str(device), seed=1234)
    ppo = build_learner(env, str(device), 16, seed=1234)
    run = LoopzRunner(env, ppo, 16)
    train(env, ppo, 4, 16, log_every=0, quiet=True, runner=run)          # warm-up: kernels, rollout / update graph capture
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    train(env, ppo, updates, 16, log_every=0, quiet=True, runner=run)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / updates
    # update phase alone on the last rollout (storage contents are still there; advantages recomputed)
    obs = env.observe(as_numpy=False)
    ppo.storage.step = 16
    e0.record()
    for _ in range(5):
        ppo.storage.compute_returns(ppo.critic.predict(obs), ppo.gamma, ppo.lam)
        ppo._train_step()
    e1.record()
    torch.cuda.synchronize(device)
    ums = e0.elapsed_time(e1) / 5
    M = envs * 16 // 4
    e0.record()
    for _ in range(4):
        ppo._minibatch(0, M)
    e1.record()
    torch.cuda.synchronize(device)
    mms = e0.elapsed_time(e1) / 4
    flops = 3 * 2.0 * (22874 + 22745) * M                                 # fwd + 2x bwd, both networks, algorithmic
    # the optional tcgen05 path of the same minibatch step (TF32 trunk, off by default)
    ppo.tensor_cores = True
    for _ in range(2):
        ppo._minibatch(0, M)
    e0.record()
    for _ in range(4):
        ppo._minibatch(0, M)
    e1.record()
    torch.cuda.synchronize(device)
    tms = e0.elapsed_time(e1) / 4
    ppo.tensor_cores = False
    # the same minibatch step by the CPU oracle (plain torch + autograd, the reference's algorithm) on a bounded sample
    from oracle import loopz_oracle as Z
    cm = 8192
    g = torch.Generator().manual_seed(0)
    rows = [torch.randn((cm, 33), generator=g), None, torch.tanh(torch.randn((cm, 2), generator=g)), torch.randn((cm, 1), generator=g),
            torch.randn((cm, 1), generator=g), torch.randn((cm, 1), generator=g), torch.randn((cm, 1), generator=g) - 1.0]
    rows[1] = rows[0]
    flat = ppo.params.detach().cpu().clone()
    opt = Z.Adam(flat.numel(), 5e-4)
    Z.minibatch_grad(flat, Z.LoopzCfg(), *rows)
    t0 = time.perf_counter()
    for _ in range(3):
        gr, *_ = Z.minibatch_grad(flat, Z.LoopzCfg(), *rows)
        opt.step(flat, gr, 0.5)
    cpu_s = (time.perf_counter() - t0) / 3
    return {"metric": "PPO frames/sec (loopz learner)", "value": envs * 16 / (ms * 1e-3), "unit": "frames/s", "envs_per_gpu": envs, "horizon": 16,
            "ms_per_update": ms, "update_phase_ms": ums, "minibatch_rows": M, "minibatch_step_ms": mms,
            "minibatch_algorithmic_tflops": flops / (mms * 1e-3) / 1e12, "minibatch_step_ms_tcgen05_tf32": tms,
            "update_in_cuda_graph": ppo._graph is not None, "rollout_in_cuda_graph": run._graph is not None,
            "kernels": "loopz::train_kernel + reduce + adam (fp32 SIMT, csrc/ppo_loopz.cu)", "params": ppo.P,
            "cpu_oracle": {"minibatch_rows": cm, "minibatch_step_ms": cpu_s * 1e3, "rows_per_s": cm / cpu_s, "threads": torch.get_num_threads(),
                           "kind": "port", "gpu_rows_per_s": M / (mms * 1e-3)}}


def bench_variant_b(device, envs=16384, steps=400, warmup=50):
    """SURVEY rows B1-B6 (live CaptureXY, 16 obstacles, potential field): the fused live step alone, the steady state with the
    scene rebuilds of the envs that reset (episodes of <= 200 steps), and the scene builder on a dense batch; the CPU oracle's
    step / field build beside them (bounded samples)."""
    import time

    from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config
    from omniisaacgymenvs_loop_b200.engine import FusedUsvLiveEnv

    cfg = live_default_config(num_envs=envs)
    env = FusedUsvLiveEnv(cfg, UsvLiveConfig(), envs, device)
    g = torch.Generator(device=device).manual_seed(99)
    acts = [torch.rand((envs, 2), device=device, generator=g) * 2 - 1 for _ in range(8)]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # steady state: step + scene rebuild; the first step resets (and builds) every env, so warm up past the first episodes
    for w in range(max(warmup, 210)):
        env.step(acts[w % 8])
    torch.cuda.synchronize(device)
    r0 = 0
    e0, e1 = ev(), ev()
    e0.record()
    for k in range(steps):
        env.step(acts[k % 8])
    e1.record()
    torch.cuda.synchronize(device)
    full_ms = e0.elapsed_time(e1) / steps
    resets = float(env.reset_buf.float().mean())
    # step kernel alone (scene rebuild skipped: the fields of resetting envs go stale, which does not change the kernel's work)
    e0, e1 = ev(), ev()
    e0.record()
    for k in range(steps):
        env.step(acts[k % 8], rebuild_scene=False)
    e1.record()
    torch.cuda.synchronize(device)
    step_ms = e0.elapsed_time(e1) / steps
    env.check_finite()
    # scene builder on a dense batch of 8 waves of CTAs
    m = 1184
    ob, tg = env.obstacles[:m].contiguous(), torch.zeros((m, 2), device=device)
    env.build_fields(ob, tg)
    torch.cuda.synchronize(device)
    e0, e1 = ev(), ev()
    e0.record()
    env.build_fields(ob, tg)
    e1.record()
    torch.cuda.synchronize(device)
    build_ms = e0.elapsed_time(e1)
    out = {"envs_per_gpu": envs, "obs_dim": 33, "substeps": cfg.n_substeps, "step_kernel_us": step_ms * 1e3,
           "step_kernel_env_steps_per_s": envs / (step_ms * 1e-3), "steady_state_us_per_step": full_ms * 1e3,
           "steady_state_env_steps_per_s": envs / (full_ms * 1e-3), "reset_fraction_per_step": resets,
           "scene_build": {"batch": m, "ms": build_ms, "us_per_env": build_ms * 1e3 / m},
           "bytes_per_env_step": 610, "step_kernel_gbps": 610 * envs / (step_ms * 1e-3) / 1e9,
           "note": "steady state = usv_live_reset_scene_f32 (obstacle placement + 150x150 wavefront + potential field for the envs "
                   "that reset) + usv_step_live_f32 per control step; random actions, episodes <= 200 steps"}
    try:
        from oracle import usv_oracle_b as B
        from tests.test_gpu_live import oracle_live, oracle_task
        from tests.util import oracle_cfg
        torch.set_num_threads(min(8, os.cpu_count() or 1))
        nb = 32
        orc = B.LiveEnvOracle(oracle_cfg(cfg), oracle_task(cfg), oracle_live(UsvLiveConfig()), nb)
        t0 = time.perf_counter()
        orc.step(torch.zeros((nb, 2)))                       # first step: resets + builds all 32 scenes
        t_reset = time.perf_counter() - t0
        t0 = time.perf_counter()
        for _ in range(5):
            orc.step(torch.rand((nb, 2)) * 2 - 1)
        t_step = (time.perf_counter() - t0) / 5
        out["cpu_oracle"] = {"envs": nb, "threads": torch.get_num_threads(), "step_ms": t_step * 1e3, "env_steps_per_s": nb / t_step,
                             "first_step_with_32_scene_builds_s": t_reset, "kind": "port"}
    except Exception as ex:   # the oracle is optional for this leg
        out["cpu_oracle"] = {"error": repr(ex)}
    return out


def main():
    # exactly ONE line on stdout: libraries (NCCL's version banner, ...) write to fd 1 too, so park fd 1 on stderr while we
    # run and print the JSON line to the real stdout at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line: dict):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the 4096-env and e2e legs (profiling runs)")
    ap.add_argument("--no-ppo", action="store_true", help="skip the PPO frames/s leg")
    ap.add_argument("--no-variant-b", action="store_true", help="skip the live-task (Variant B) leg")
    ap.add_argument("--no-loopz", action="store_true", help="skip the loopz-learner leg")
    ap.add_argument("--ppo-envs", type=int, default=16384, help="envs per GPU of the PPO leg (BASELINE config[2])")
    ap.add_argument("--ppo-epochs", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write obs / reward / done of the last one (rank 0's envs) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the timed CUDA path: use it with --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference(args, emit)
        return

    import torch.distributed as dist
    from omniisaacgymenvs_loop_b200 import _lib
    from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
    from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    if dist_on:
        dist.init_process_group("nccl", device_id=device)
    n = args.envs
    cfg = UsvEnvConfig().full_dr()
    # envs are sharded across ranks: rank r owns global env ids [r*n, (r+1)*n) -- same Philox streams as one big env
    env = FusedUsvEnv(cfg, n, device, env_id_offset=rank * n)
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    acts = [torch.rand((n, 2), device=device, generator=g) * 2 - 1 for _ in range(8)]

    sampler = ClockSampler(local)
    launches0 = _lib.launch_count()
    sampler.start()
    ms = time_steps(env, acts, args.steps, args.warmup, dist_on, device)
    clocks = sampler.stop()
    launches = _lib.launch_count() - launches0 - args.warmup
    env.check_finite()
    if args.dump_outputs and rank == 0:
        # env.step returns the env's own buffers: until the next step they hold what the last timed step returned
        dump_outputs(args.dump_outputs, {"obs": env.obs, "reward": env.rew, "done": env.reset_buf})
    value = world * n * args.steps / (ms * 1e-3)
    ms_per_step = ms / args.steps
    peak, peak_src = measured_peak()
    achieved = BYTES_PER_ENV_STEP * n / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": "usv::step_fused_kernel<2,false> (kDisturb = 2: all disturbance kinds on, stats off)", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * n}
    # dram bytes/launch come from the committed ncu --set full capture of this kernel at this env count (a profiler cannot run inside
    # the timed run); `traffic_source` says so
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            with open(tr) as f:
                t = json.load(f)
            if int(t.get("envs", -1)) == n:
                roofline["traffic"] = t["dram_bytes_per_launch"]
                roofline["traffic_source"] = "profiles/traffic.json: ncu --set full capture of this kernel at this env count (" + str(t.get("source", "r01")) + "), not measured in this run"
        except Exception:
            pass

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(n), "roofline": roofline, "clocks": clocks,
            "gpu_launches": int(launches), "substeps_per_s": value * cfg.n_substeps}

    if not args.no_extra and args.steps < 2000:
        # the driver's K steps are ~1 ms of device time: the same measurement over 2000 steps beside it (one clock sample covers neither)
        sampler2 = ClockSampler(local)
        sampler2.start()
        lms = time_steps(env, acts, 2000, 3, dist_on, device)
        line["value_2000_steps"] = {"value": world * n * 2000 / (lms * 1e-3), "ms_per_step": lms / 2000, "steps": 2000,
                                    "frac": BYTES_PER_ENV_STEP * n / (lms / 2000 * 1e-3) / 1e9 / peak, "clocks": sampler2.stop()}
    if not args.no_extra:
        e2e_steps = max(3, min(args.steps, 200))
        ems, h2d, d2h, _ = time_e2e(env, e2e_steps, 3, dist_on, device)
        if dist_on:
            dist.barrier()
        link = memcpy_probe(device, h2d, d2h)           # every rank copies at once: the host side of the box is shared
        if dist_on:
            t = torch.tensor([link], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            link = float(t.item())
        e2e_gbs = (h2d + d2h) * e2e_steps / (ems * 1e-3) / 1e9
        line["e2e"] = {"value": world * n * e2e_steps / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                       "roofline": {"bound": "pcie", "achieved": e2e_gbs, "peak": link, "unit": "GB/s per rank (H2D + D2H)", "frac": e2e_gbs / link,
                                    "peak_source": f"plain pinned cudaMemcpyAsync of the same byte counts, both directions at once, all {world} ranks "
                                                   "copying together (slowest rank), measured in this run"},
                       "path": "engine.HostStepper.submit -> usv_step_fused_f32 (C ABI): pinned host actions -> device, obs + reward + uint8 "
                               "done -> pinned host every step; copy-in / compute / copy-out on 3 streams, 2 staging slots"}
        # BASELINE config[1]: 4096 envs/GPU -- launch-latency bound (working set ~1 MB, L2 resident): reported, not the headline
        small = FusedUsvEnv(cfg, 4096, device, env_id_offset=rank * 4096)
        sacts = [a[:4096].contiguous() for a in acts]
        sms = time_steps(small, sacts, max(args.steps, 2000), 20, dist_on, device)
        T = 512
        roll_act = torch.rand((T, 4096, 2), device=device, generator=g) * 2 - 1
        small.rollout(roll_act)
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            small.rollout(roll_act)
        e1.record()
        torch.cuda.synchronize(device)
        rms = e0.elapsed_time(e1)
        # the same launch-per-step kernel replayed from a CUDA graph of 256 control steps (device-side Philox step offset)
        gact = torch.rand((256, 4096, 2), device=device, generator=g) * 2 - 1
        replay = small.capture_steps(gact)
        for _ in range(3):
            replay()
        torch.cuda.synchronize(device)
        e0.record()
        for _ in range(16):
            replay()
        e1.record()
        torch.cuda.synchronize(device)
        gms = e0.elapsed_time(e1)
        small.check_finite()
        line["c2_4096"] = {"envs_per_gpu": 4096, "step_kernel_env_steps_per_s": world * 4096 * max(args.steps, 2000) / (sms * 1e-3),
                           "us_per_step": sms * 1e3 / max(args.steps, 2000),
                           "graph_replay_env_steps_per_s": world * 4096 * 256 * 16 / (gms * 1e-3), "graph_replay_us_per_step": gms * 1e3 / (256 * 16),
                           "rollout_kernel_env_steps_per_s": world * 4096 * T * 4 / (rms * 1e-3),
                           "note": "one launch per control step vs one launch per 512 control steps (state in registers); "
                                   "latency-bound, working set L2-resident -> no HBM roofline claimed"}
    ppo_short = None
    if not args.no_extra and not args.no_ppo:
        ppo_short, line["ppo_detail"] = bench_ppo(args, rank, world, device, dist_on)
    # single-GPU legs: on a multi-rank launch they would only hold the other ranks at a barrier (the N=1 run carries them)
    if not args.no_extra and world == 1:
        line["secondary_kernels"] = bench_gae_mlp(device)
        if not args.no_variant_b:
            line["variant_b"] = bench_variant_b(device)
        if not args.no_loopz:
            line["loopz_ppo"] = bench_loopz(device)
    if dist_on:
        dist.barrier()
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cb, _ = cpu_port(20.0)
        line["cpu_baseline"] = cb
        if ppo_short is not None:
            ncpu = os.cpu_count() or 1
            best = None
            for nt in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):      # every candidate, keep the fastest (as for the env step)
                torch.set_num_threads(nt)
                r = ppo_cpu_port(epochs=1)
                log(f"  ppo cpu port: {nt} threads -> {r['value']:.3g} frames/s")
                if best is None or r["value"] > best["value"]:
                    best = r
            torch.set_num_threads(best["cores"])
            ppo_short["cpu_baseline"] = ppo_cpu_port(epochs=3)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()
    if ppo_short is not None:
        line["ppo"] = ppo_short         # LAST key: a truncated tail of the line (the driver keeps 1500 characters) still carries it
    if rank == 0:
        emit(line)


if __name__ == "__main__":
    main()
