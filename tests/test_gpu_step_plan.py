"""The full-DR step plan (csrc/usv_step_core.cuh, PlanFullDr): usv_step_fused_f32 launches a step_fused_kernel instance whose discrete
parameters are fixed at compile time when the configuration is UsvEnvConfig().full_dr() with stats off, and the generic instances
otherwise.  The plan instance must compute what the generic instance computes, bit for bit.  A zero-velocity water current sends the
same configuration to the generic kDisturb == 1 instance with the same arithmetic (the current subtracts an exact zero)."""
import ctypes
import dataclasses

import pytest
import torch

from omniisaacgymenvs_loop_b200 import _lib
from omniisaacgymenvs_loop_b200.config import PEN_NEG_ABS, PenaltyTerm, UsvEnvConfig
from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv

DEV = "cuda:0"
PLAN = _lib.ENUMS["USV_STEP_PLAN_FULL_DR"]
GENERIC = _lib.ENUMS["USV_STEP_PLAN_GENERIC"]


def _plan(cfg, stats=False):
    return _lib.lib().usv_step_fused_plan(ctypes.byref(cfg.to_params()), ctypes.c_int32(int(stats)))


def _zero_current(cfg):
    return dataclasses.replace(cfg, use_water_current=True, flow_vel_xy=(0.0, 0.0))


def test_plan_is_chosen_for_full_dr_only():
    cfg = UsvEnvConfig().full_dr()
    assert _plan(cfg) == PLAN
    assert _plan(dataclasses.replace(cfg, seed=99, dt=0.01, kill_dist=5.0, max_episode_length=7)) == PLAN   # continuous values
    assert _plan(cfg, stats=True) == GENERIC
    assert _plan(dataclasses.replace(cfg, pen_linear_vel=PenaltyTerm(PEN_NEG_ABS, 0.01))) == GENERIC
    assert _plan(dataclasses.replace(cfg, n_substeps=4)) == GENERIC
    assert _plan(dataclasses.replace(cfg, envs_per_row=64)) == GENERIC
    assert _plan(dataclasses.replace(cfg, noise_pos=False)) == GENERIC
    assert _plan(dataclasses.replace(cfg, reward_mode=2)) == GENERIC
    assert _plan(dataclasses.replace(cfg, thr_separate=True, kdrag_rand=True, mass_rand=False)) == PLAN   # reset switches: run-time
    assert _plan(dataclasses.replace(cfg, use_sin_torque=False)) == GENERIC
    assert _plan(_zero_current(cfg)) == GENERIC
    assert _plan(UsvEnvConfig()) == GENERIC
    assert _lib.lib().usv_step_fused_plan(None, ctypes.c_int32(0)) == _lib.ENUMS["USV_E_NULL"]


def _run(cfg, n, acts, steps):
    env = FusedUsvEnv(cfg, n, DEV)
    out = []
    for k in range(steps):
        if k == 150:
            env.first_call = True                        # Penalties.prev_state is None again: both variations are zero
        if k % 25 == 7:
            env.reset_buf[k::97].fill_(1)                # scattered envs
        if k % 40 == 13:
            w = (k * 7919) % (n // 32)
            env.reset_buf[32 * w: 32 * (w + 3)].fill_(1)  # three whole warps
        obs, rew, done = env.step(acts[k % len(acts)])
        if k % 10 == 0 or k == 150 or k % 25 == 7 or k % 40 == 13:
            out.append((k, obs.clone(), rew.clone(), done.clone()))
    torch.cuda.synchronize()
    env.check_finite()
    return out, env.state.clone(), env.consts.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4099, (1 << 20) + 37])
def test_plan_instance_equals_generic_instance(n):
    cfg = UsvEnvConfig(max_episode_length=90).full_dr()
    assert _plan(cfg) == PLAN and _plan(_zero_current(cfg)) == GENERIC
    g = torch.Generator(device=DEV).manual_seed(5)
    acts = [torch.rand((n, 2), device=DEV, generator=g) * 2.4 - 1.2 for _ in range(8)]
    steps = 300
    got, got_state, got_consts = _run(cfg, n, acts, steps)
    want, want_state, want_consts = _run(_zero_current(cfg), n, acts, steps)
    resets = 0
    for (k, *a), (_, *b) in zip(got, want):
        for name, x, y in zip(("obs", "reward", "done"), a, b):
            assert torch.equal(x, y), (name, k)
        resets += int(a[2].sum())
    assert resets > 0
    assert torch.equal(got_state, want_state) and torch.equal(got_consts, want_consts)


@pytest.mark.gpu
def test_plan_instance_sees_reset_buf_written_by_torch_on_the_stream():
    n = 4099
    cfg = UsvEnvConfig().full_dr()
    assert _plan(cfg) == PLAN
    env = FusedUsvEnv(cfg, n, DEV)
    a = torch.zeros((n, 2), device=DEV)
    for _ in range(5):
        env.step(a)
    ids = torch.arange(3, n, 211, device=DEV)
    mass_before = env.field("USV_C_MASS").clone()
    progress_before = env.progress_buf.clone()
    env.reset_buf.zero_()
    env.reset_buf[ids] = 1                               # torch kernels on the same stream, no synchronisation before the step
    env.step(a)
    progress = env.progress_buf
    assert torch.equal(progress[ids].cpu(), torch.ones(len(ids), dtype=torch.long))
    others = torch.ones(n, dtype=torch.bool, device=DEV)
    others[ids] = False
    assert torch.equal(progress[others], progress_before[others] + 1)
    mass = env.field("USV_C_MASS")
    assert bool((mass[ids] != mass_before[ids]).all()) and torch.equal(mass[others], mass_before[others])
