"""TEST INFRASTRUCTURE ONLY -- the CPU oracle of the ASV hot path (never on the product path).

A torch-on-CPU restatement of the reference's algorithm for SURVEY rows A1-A19 (force layer,
env orchestration, classic CaptureXY task), one function per reference function, each citing the
reference file:line it follows.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module.

Pinning: this restatement is checked against outputs of the *reference modules themselves*
(imported from a reference checkout through oracle/ref_shim.py) frozen in tests/golden/*.npz by
oracle/make_golden.py.  The reference's own tests hold no vectors for
this path (SURVEY 4.2).  The PhysX step is NOT in the reference tree: its stand-in (planar
semi-implicit Euler, DESIGN.md) is "parity unpinned" and is checked against the float64 host
integration in oracle/integrator64.py instead.

Abbreviations:  OIGE = omniisaacgymenvs/, SNAP = 811_3.5*(classic snapshot)/.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np
import torch

from . import philox

F32 = torch.float32


# --------------------------------------------------------------------------------------------
# third-party boundary: pytorch3d.transforms.quaternion_to_matrix (public formula, real-first)
# call sites: OIGE/envs/USV/Utils.py:5-7, Hydrodynamics.py:210
def quaternion_to_matrix(q: torch.Tensor) -> torch.Tensor:
    r, i, j, k = torch.unbind(q, -1)
    two_s = 2.0 / (q * q).sum(-1)
    o = torch.stack(
        (
            1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
            two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
            two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j),
        ),
        -1,
    )
    return o.reshape(q.shape[:-1] + (3, 3))


def _rot_t(R: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    # getLocalLinearVelocities(world, R.mT): bmm(R^T, v)  [OIGE/envs/USV/Utils.py:10-22]
    return torch.bmm(R.mT, v.unsqueeze(1).mT).mT.squeeze(1)


# --------------------------------------------------------------------------------------------
# A1  [OIGE/envs/USV/Hydrostatics.py:63-133]
def hydrostatics_local(vol, rpy, quat, *, water_density, gravity, metacentric_width, metacentric_length,
                       average_hydrostatics_force_value, amplify_torque):
    n = vol.shape[0]
    fg = torch.zeros((n, 3), dtype=F32)
    tg = torch.zeros((n, 3), dtype=F32)
    roll, pitch = rpy[:, 0], rpy[:, 1]
    fg[:, 2] = -water_density * gravity * vol                                     # :67-69
    # :72-81 is overwritten by :83-92 -> the constant average force is what survives
    tg[:, 0] = -1 * metacentric_width * (torch.sin(roll) * average_hydrostatics_force_value)
    tg[:, 1] = -1 * metacentric_length * (torch.sin(pitch) * average_hydrostatics_force_value)
    R = quaternion_to_matrix(quat)                                                # :105
    f_local = _rot_t(R, fg)                                                       # :110-115
    t_local = tg                                                                  # :123 (not rotated)
    return torch.hstack([f_local, t_local * amplify_torque]), fg, tg              # :127-132


# A2  [OIGE/envs/USV/Hydrodynamics.py:176-245]
def hydrodynamics(quat, world_vel, linear_damping, quadratic_damping, drag_scale, *,
                  linear_damping_forward_speed, offset_linear_damping, offset_lin_forward_damping_speed,
                  offset_nonlin_damping, scaling_damping, use_drag_scale, use_water_current=False,
                  flow_vel=(0.0, 0.0, 0.0)):
    R = quaternion_to_matrix(quat)                                                # :210
    lin = _rot_t(R, world_vel[:, :3])                                             # :213-215
    ang = _rot_t(R, world_vel[:, 3:])                                             # :216-218
    if use_water_current:                                                         # :224-237
        fv = torch.tensor(flow_vel, dtype=F32)
        if fv.dim() == 1:
            fv = fv.unsqueeze(0).expand_as(world_vel[:, :3])
        lin = lin - _rot_t(R, fv.contiguous())
    vel = torch.hstack([lin, ang])
    fwd = torch.as_tensor(linear_damping_forward_speed, dtype=F32)
    lin_damp = linear_damping + offset_linear_damping - (fwd + offset_lin_forward_damping_speed)   # :186-193
    quad_damp = ((quadratic_damping + offset_nonlin_damping).mT * torch.abs(vel.mT)).mT            # :195-197
    D = (lin_damp + quad_damp) * scaling_damping                                                  # :200
    if use_drag_scale:
        D = D * drag_scale                                                                        # :203-204
    return -1 * D * vel, vel                                                                      # :243


# thruster LUT  [OIGE/envs/USV/ThrusterDynamics.py:152-177]
def build_lut(points, n_out: int) -> torch.Tensor:
    pts = torch.as_tensor(points, dtype=F32)
    return torch.nn.functional.interpolate(pts.unsqueeze(0).unsqueeze(0), size=n_out, mode="linear",
                                           align_corners=True).squeeze(0).squeeze(0)


def build_lut_restated(points, n_out: int) -> np.ndarray:
    """The same LUT without calling ATen: upsample_linear1d(align_corners=True) in explicit fp32."""
    pts = np.asarray(points, dtype=np.float32)
    n_in = len(pts)
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    out = np.empty(n_out, np.float32)
    for i in range(n_out):
        src = np.float32(scale * np.float32(i))
        i0 = min(int(math.floor(src)), n_in - 1)
        l1 = np.float32(min(max(np.float32(src - np.float32(i0)), 0.0), 1.0))
        l0 = np.float32(np.float32(1.0) - l1)
        i1 = i0 + (1 if i0 < n_in - 1 else 0)
        # ATen's CPU kernel contracts w0*x0 + w1*x1 into fma(w0, x0, w1*x1) (pinned against the reference LUTs)
        out[i] = np.float32(np.float64(l0) * np.float64(pts[i0]) + np.float64(np.float32(l1 * pts[i1])))
    return out


# A4  [OIGE/envs/USV/ThrusterDynamics.py:179-213]
def thruster_target(cmd, lut_left, lut_right, mult_left=None, mult_right=None):
    n = lut_left.shape[0]
    il = torch.round(((cmd[:, 0] + 1) / 2) * (n - 1)).to(torch.long)              # :187
    ir = torch.round(((cmd[:, 1] + 1) / 2) * (n - 1)).to(torch.long)              # :188
    il = torch.clamp(il, 0, n - 1)
    ir = torch.clamp(ir, 0, n - 1)
    before = torch.stack([lut_left[il], lut_right[ir]], dim=1)                    # :194-197
    after = before.clone()
    if mult_left is not None:
        after[:, 0] = before[:, 0] * mult_left.reshape(-1)                        # :201-213
    if mult_right is not None:
        after[:, 1] = before[:, 1] * mult_right.reshape(-1)
    return before, after


# A5  [OIGE/envs/USV/ThrusterDynamics.py:129-141]
def lag_alpha(dt: float, tau: float) -> torch.Tensor:
    return torch.exp(torch.tensor(-dt / tau))


def thruster_lag(cur, target, alpha):
    return cur * alpha + (1.0 - alpha) * target


# --------------------------------------------------------------------------------------------
# closed set of penalty lambdas (SURVEY A9); mirrors UsvPenaltyTerm in include/usv_b200.h
PEN_OFF, PEN_NEG_SUM, PEN_EXP_NEG_SUMSQ, PEN_NEG_ABS, PEN_NEG_DEADZONE, PEN_EXP_NEG_ABS = range(6)


@dataclass
class PenaltyTerm:
    form: int = PEN_OFF
    c1: float = 0.0
    c2: float = 0.0
    k: float = 0.0

    def scalar(self, x):
        if self.form == PEN_NEG_ABS:
            return -torch.abs(x) * self.c1 + self.c2
        if self.form == PEN_NEG_DEADZONE:
            return -torch.clamp(torch.abs(x) - self.k, min=0.0) * self.c1
        if self.form == PEN_EXP_NEG_ABS:
            return (torch.exp(-self.k * torch.abs(x)) - 1.0) * self.c1
        return torch.zeros_like(x)

    def vector(self, x):
        if self.form == PEN_NEG_SUM:
            return -torch.sum(x, dim=-1) * self.c1 + self.c2
        if self.form == PEN_EXP_NEG_SUMSQ:
            return (torch.exp(-torch.sum(x ** 2, dim=-1)) - 1.0) * self.c1
        if self.form == PEN_NEG_ABS:  # -norm(x)*c1
            return -torch.norm(x, dim=-1) * self.c1 + self.c2
        return torch.zeros(x.shape[0], dtype=F32)


@dataclass
class EnvConfig:
    """Everything UsvStepParams carries (include/usv_b200.h), with the classic snapshot's YAML values
    as defaults  [SNAP/USV_Virtual_CaptureXY_SysID-TEST.yaml]."""
    seed: int = 1234
    dt: float = 0.02
    n_substeps: int = 5
    max_episode_length: int = 3000
    clip_actions: float = 1.0
    clip_obs: float = 12.0
    izz: float = 10.0                      # URDF placeholder izz (heron.urdf:69); parity unpinned
    thr_y_left: float = 0.377654           # heron.urdf:242 (left = +y, REP-103)
    thr_y_right: float = -0.377654         # heron.urdf:167
    time_constant: float = 0.05
    env_spacing: float = 15.0
    envs_per_row: int = 0
    grid_row_offset: float = 0.0
    grid_col_offset: float = 0.0
    lin_fwd: tuple = (0.0, 0.0, 0.0)
    offset_linear_damping: float = 0.0
    offset_lin_forward_damping_speed: float = 0.0
    offset_nonlin_damping: float = 0.0
    scaling_damping: float = 1.0
    use_drag_scale: bool = False
    n_lut: int = 1000
    lut_points_left: tuple = (-3.8, -3.8, -3.6, -3.6, -1.6, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0,
                              4.0, 10.0, 15.0, 21.0, 23.0, 22.0)
    lut_points_right: tuple = (-5.0, -5.0, -5.0, -4.6, -2.2, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0,
                               4.6, 10.0, 17.0, 24.0, 24.0, 23.0)
    action_affine: bool = False
    action_noise: bool = True
    action_noise_min: float = -0.05
    action_noise_max: float = 0.05
    action_bias: float = 0.0
    action_bias_steps: int = 0      # the bias is applied while the control-step counter is below this [OIGE/tasks/USV_Virtual.py:1070-1077]
    penalties_use_u: bool = False
    noise_pos: bool = False
    pos_noise_min: float = -0.03
    pos_noise_max: float = 0.03
    noise_vel: bool = True
    vel_noise_min: float = -0.03
    vel_noise_max: float = 0.03
    noise_heading: bool = True
    heading_noise_min: float = -0.025
    heading_noise_max: float = 0.025
    use_force_disturbance: bool = False
    use_const_force: bool = False
    use_sin_force: bool = False
    use_torque_disturbance: bool = False
    use_const_torque: bool = False
    use_sin_torque: bool = False
    position_tolerance: float = 0.1
    kill_after_n_steps_in_tolerance: int = 1
    kill_dist: float = 20.0
    boundary_cost: float = 25.0
    goal_reward: float = 30.0
    time_reward: float = -0.2
    goal_speed_gate: float = 0.05
    reward_mode: int = 0                   # 0 linear, 1 square, 2 exponential
    position_scale: float = 1.0
    exponential_reward_coeff: float = 0.25
    align_la1: float = 0.02
    align_la2: float = -10.0
    align_la3: float = -0.1
    pen_linear_vel: PenaltyTerm = field(default_factory=PenaltyTerm)
    pen_angular_vel: PenaltyTerm = field(default_factory=PenaltyTerm)
    pen_angular_vel_variation: PenaltyTerm = field(default_factory=lambda: PenaltyTerm(PEN_EXP_NEG_ABS, 1.0, 0.0, 0.033))
    pen_energy: PenaltyTerm = field(default_factory=lambda: PenaltyTerm(PEN_EXP_NEG_SUMSQ, 0.01))
    pen_action_variation: PenaltyTerm = field(default_factory=PenaltyTerm)
    goal_random_position: float = 0.0
    retarget_on_reset: bool = False
    spawn_min_dist: float = 0.3
    spawn_max_dist: float = 12.0
    spawn_curriculum: bool = False
    spawn_curriculum_min_dist: float = 0.2
    spawn_curriculum_max_dist: float = 3.0
    spawn_curriculum_kill_dist: float = 30.0
    spawn_curriculum_warmup: int = 250
    spawn_curriculum_end: int = 1000
    horizon_length: int = 16
    spawn_about_origin: bool = False
    retarget_after_spawn: bool = False
    reset_pose_external: bool = False
    spawn_vel_range: float = 1.5
    mass_rand: bool = False
    mass_min: float = 34.96
    mass_max: float = 36.96
    mass_base: float = 35.96
    drag_rand: bool = False
    lin_base: tuple = (0.0, 99.99, 0.82985084)          # u, v, r of linear_damping
    quad_base: tuple = (17.257603, 99.99, 17.33600724)  # u, v, r of quadratic_damping
    lin_rand_frac: tuple = (0.1, 0.1, 0.1)
    quad_rand_frac: tuple = (0.1, 0.1, 0.1)
    kdrag_rand: bool = False
    kdrag_min: float = 1.0
    kdrag_max: float = 1.0
    kdrag_log: bool = False
    thr_rand: bool = False
    thr_separate: bool = False
    thr_rand_frac: float = 0.5
    thr_left_frac: float = 0.5
    thr_right_frac: float = 0.5
    mass_coupling: bool = False
    couple_mass_max: float = 54.96
    couple_thr_a: float = 0.5
    couple_kiz_min: float = 1.0
    couple_kiz_max: float = 1.5
    couple_targets: int = 7            # bits: 1 drag_scale, 2 thruster, 4 yaw_inertia  [OIGE/tasks/USV_Virtual.py:393-411]
    kiz_rand: bool = False             # independent k_Iz draw in [couple_kiz_min, couple_kiz_max]  [:153-170,1532-1533]
    kiz_log: bool = False
    use_water_current: bool = False    # [OIGE/tasks/USV_Virtual.py:444-445 ; Hydrodynamics.py:224-237]
    flow_vel_xy: tuple = (0.0, 0.0)
    force_const_min: float = 0.0
    force_const_max: float = 2.5
    force_sin_min: float = 0.0
    force_sin_max: float = 2.5
    force_min_freq: float = 0.25
    force_max_freq: float = 3.0
    force_min_shift: float = 0.0
    force_max_shift: float = 100.0
    torque_const_min: float = 0.0
    torque_const_max: float = 1.0
    torque_sin_min: float = 0.0
    torque_sin_max: float = 1.0
    torque_min_freq: float = 0.25
    torque_max_freq: float = 3.0
    torque_min_shift: float = 0.0
    torque_max_shift: float = 100.0

    @property
    def lin_rand(self):
        # _linear_rand = frac * base  [OIGE/envs/USV/Hydrodynamics.py:41-62]
        return tuple(f * b for f, b in zip(self.lin_rand_frac, self.lin_base))

    @property
    def quad_rand(self):
        return tuple(f * b for f, b in zip(self.quad_rand_frac, self.quad_base))

    @property
    def force_ranges(self):
        # ForceDisturbance.__init__ rescales the per-axis amplitudes by 1/sqrt(2)  [USV_disturbances.py:281-289]
        s = lambda v: math.sqrt(v ** 2 / 2)
        return s(self.force_const_min), s(self.force_const_max), s(self.force_sin_min), s(self.force_sin_max)

    def full_dr(self) -> "EnvConfig":
        """The DR50 flag set: every per-env randomisation on (BASELINE config C4 / 'A, full DR')."""
        import dataclasses
        return dataclasses.replace(
            self, use_force_disturbance=True, use_const_force=True, use_sin_force=True,
            use_torque_disturbance=True, use_const_torque=True, use_sin_torque=True, noise_pos=True,
            mass_rand=True, drag_rand=True, thr_rand=True, thr_rand_frac=0.5, envs_per_row=0)


def curriculum(c: "EnvConfig", step: float):
    """(rmin, rmax, kill_dist) at curriculum step `step`  [SNAP/USV_capture_xy.py:238-258 (kill), :346-380 (spawn)]."""
    if not c.spawn_curriculum:
        return c.spawn_min_dist, c.spawn_max_dist, c.kill_dist
    if step < c.spawn_curriculum_warmup:
        return c.spawn_curriculum_min_dist, c.spawn_curriculum_max_dist, c.spawn_curriculum_kill_dist
    if step > c.spawn_curriculum_end:
        return c.spawn_min_dist, c.spawn_max_dist, c.kill_dist
    r = (step - c.spawn_curriculum_warmup) / (c.spawn_curriculum_end - c.spawn_curriculum_warmup)
    return (r * (c.spawn_min_dist - c.spawn_curriculum_min_dist) + c.spawn_curriculum_min_dist,
            r * (c.spawn_max_dist - c.spawn_curriculum_max_dist) + c.spawn_curriculum_max_dist,
            r * (c.kill_dist - c.spawn_curriculum_kill_dist) + c.spawn_curriculum_kill_dist)


def sample_k_iz(u: torch.Tensor, kmin: float, kmax: float, log_space: bool) -> torch.Tensor:
    """USVVirtual._sample_k_iz on given uniforms  [OIGE/tasks/USV_Virtual.py:153-170]."""
    if log_space:
        log_min = torch.log(torch.tensor(kmin, dtype=F32))
        log_max = torch.log(torch.tensor(kmax, dtype=F32))
        return torch.exp(log_min + u * (log_max - log_min))
    return kmin + u * (kmax - kmin)


def com_disc(base, u_r: torch.Tensor, u_theta: torch.Tensor, max_disp: float) -> torch.Tensor:
    """MDD._randomize_com, legacy branch: a disc in the XY plane around base_com, z untouched  [OIGE/tasks/USV/USV_disturbances.py:108-124]."""
    r = u_r * max_disp
    theta = u_theta * math.pi * 2.0
    com = torch.tensor(base, dtype=F32).unsqueeze(0).repeat(u_r.shape[0], 1)
    com[:, 0] = com[:, 0] + torch.cos(theta) * r
    com[:, 1] = com[:, 1] + torch.sin(theta) * r
    return com


def mass_coupling(c: "EnvConfig", mass: torch.Tensor):
    """_apply_mass_driven_coupling  [OIGE/tasks/USV_Virtual.py:988-1040]: mass -> r in [0,1] -> (k_drag, thruster scale, k_Iz)."""
    denom = max(c.couple_mass_max - c.mass_base, 1e-6)
    rr = torch.clamp((mass - c.mass_base) / denom, 0.0, 1.0)
    kd = c.kdrag_min + rr * (c.kdrag_max - c.kdrag_min)
    sthr = torch.clamp(1.0 - rr * c.couple_thr_a, 1.0 - c.couple_thr_a, 1.0)
    kiz = c.couple_kiz_min + rr * (c.couple_kiz_max - c.couple_kiz_min)
    return kd, sthr, kiz


def _u(u, lo, hi):
    return u * (hi - lo) + lo


class ClassicEnvOracle:
    """VecEnvRLGames.step over the classic USVVirtual + CaptureXYTask with the planar integrator
    standing in for world.step().  AoS (N,k) fp32 torch tensors, eager op chains -- i.e. the shape
    of the reference's own CPU path.  Randomness comes from oracle.philox with the same keys the
    CUDA kernel uses, so both sides see identical uniforms."""

    def __init__(self, cfg: EnvConfig, num_envs: int, env_id_offset: int = 0):
        self.cfg = cfg
        self.n = n = num_envs
        self.env_ids = np.arange(n, dtype=np.uint64) + np.uint64(env_id_offset)
        z = lambda *s: torch.zeros(s, dtype=F32)
        # PhysX-side state (planar)
        self.pos = z(n, 2); self.psi = z(n); self.vel = z(n, 2); self.r = z(n)
        # DynamicsFirstOrder
        self.current_forces = z(n, 2)
        self.lut_left = build_lut(cfg.lut_points_left, cfg.n_lut)
        self.lut_right = build_lut(cfg.lut_points_right, cfg.n_lut)
        self.alpha = lag_alpha(cfg.dt, cfg.time_constant)
        self.thr_mult_left = torch.ones(n, dtype=F32); self.thr_mult_right = torch.ones(n, dtype=F32)
        # HydrodynamicsObject (6-DOF tensors; w,p,q rows are inert in the planar stand-in)
        lb, qb = cfg.lin_base, cfg.quad_base
        self.linear_damping = torch.tensor([[lb[0], lb[1], 99.99, 13.0, 13.0, lb[2]]] * n, dtype=F32)
        self.quadratic_damping = torch.tensor([[qb[0], qb[1], 10.0, 5.0, 5.0, qb[2]]] * n, dtype=F32)
        self.drag_scale = torch.ones((n, 1), dtype=F32)
        self.k_iz = torch.ones(n, dtype=F32)
        self.mass = torch.full((n,), cfg.mass_base, dtype=F32)
        # disturbances
        self.f_const = z(n, 2); self.f_freq = z(n, 2); self.f_shift = z(n, 2); self.f_amp = z(n)
        self.t_const = z(n); self.t_freq = z(n); self.t_shift = z(n); self.t_amp = z(n)
        # task
        self.target = z(n, 2)
        self.goal_reached = torch.zeros(n, dtype=torch.int32)
        self.prev_d = z(n); self.prev_w = z(n); self.prev_asum = z(n)
        self.reset_buf = torch.ones(n, dtype=torch.long)       # [SNAP/USV_Virtual.py:342-344]
        self.progress_buf = torch.zeros(n, dtype=torch.long)
        self.step_counter = 0
        self.curriculum_step = 0.0           # task `step` = control steps / horizon_length
        self.first_call = True
        self.stats = {}
        if cfg.envs_per_row > 0:
            ids = torch.arange(n)
            self.origin = torch.stack([cfg.grid_row_offset - (ids // cfg.envs_per_row).float() * cfg.env_spacing,
                                       (ids % cfg.envs_per_row).float() * cfg.env_spacing - cfg.grid_col_offset], 1)
        else:
            self.origin = z(n, 2)

    # ---- reset_idx  [SNAP/USV_Virtual.py:750-817] ------------------------------------------
    def reset_idx(self, ids: torch.Tensor, step: int):
        c = self.cfg
        if ids.numel() == 0:
            return
        R = [torch.from_numpy(philox.uniform4(c.seed, self.env_ids[ids.numpy()], step, s)) for s in philox.RS_RESET]
        r0, r1, r2, r3, r4, r5, r6, r7, r8 = R
        self.goal_reached[ids] = 0                                          # task.reset
        fcmin, fcmax, fsmin, fsmax = c.force_ranges
        if c.use_force_disturbance:                                         # UF.generate_force
            if c.use_sin_force:
                self.f_freq[ids, 0] = _u(r5[:, 2], c.force_min_freq, c.force_max_freq)
                self.f_freq[ids, 1] = _u(r5[:, 3], c.force_min_freq, c.force_max_freq)
                self.f_shift[ids, 0] = _u(r6[:, 0], c.force_min_shift, c.force_max_shift)
                self.f_shift[ids, 1] = _u(r6[:, 1], c.force_min_shift, c.force_max_shift)
                self.f_amp[ids] = _u(r6[:, 2], fsmin, fsmax)
            if c.use_const_force:
                rr = _u(r6[:, 3], fcmin, fcmax)
                th = r7[:, 0] * math.pi * 2
                self.f_const[ids, 0] = torch.cos(th) * rr
                self.f_const[ids, 1] = torch.sin(th) * rr
        if c.use_torque_disturbance:                                        # TD.generate_torque
            if c.use_sin_torque:
                self.t_freq[ids] = _u(r7[:, 1], c.torque_min_freq, c.torque_max_freq)
                self.t_shift[ids] = _u(r7[:, 2], c.torque_min_shift, c.torque_max_shift)
                self.t_amp[ids] = _u(r7[:, 3], c.torque_sin_min, c.torque_sin_max)
            if c.use_const_torque:
                rr = _u(r8[:, 0], c.torque_const_min, c.torque_const_max)
                rr[r8[:, 1] > 0.5] *= -1
                self.t_const[ids] = rr
        # MDD.randomize_masses  [USV_disturbances.py:127-151]
        self.mass[ids] = _u(r1[:, 3], c.mass_min, c.mass_max) if c.mass_rand else r1[:, 3] * 0 + c.mass_base
        # _apply_yaw_inertia_randomization, unless the coupling owns k_Iz  [OIGE/tasks/USV_Virtual.py:1532-1533]
        if c.kiz_rand and not (c.mass_coupling and (c.couple_targets & 4)):
            self.k_iz[ids] = sample_k_iz(r5[:, 1], c.couple_kiz_min, c.couple_kiz_max, c.kiz_log)
        # hydrodynamics.reset_coefficients  [Hydrodynamics.py:136-174]
        if c.drag_rand:
            lr, qr = c.lin_rand, c.quad_rand
            for col, j in ((0, 0), (1, 1), (5, 2)):
                self.linear_damping[ids, col] = c.lin_base[j] + (r3[:, j] * 2 - 1) * lr[j]
                self.quadratic_damping[ids, col] = c.quad_base[j] + (r4[:, j] * 2 - 1) * qr[j]
        if c.kdrag_rand:
            if c.kdrag_log:
                l0, l1 = torch.log(torch.tensor(c.kdrag_min)), torch.log(torch.tensor(c.kdrag_max))
                self.drag_scale[ids, 0] = torch.exp(l0 + r2[:, 3] * (l1 - l0))
            else:
                self.drag_scale[ids, 0] = c.kdrag_min + r2[:, 3] * (c.kdrag_max - c.kdrag_min)
        # thrusters.reset_thruster_randomization  [ThrusterDynamics.py:112-127]
        if c.thr_rand:
            if c.thr_separate:
                self.thr_mult_left[ids] = r4[:, 3] * 2 * c.thr_left_frac + (1 - c.thr_left_frac)
                self.thr_mult_right[ids] = r5[:, 0] * 2 * c.thr_right_frac + (1 - c.thr_right_frac)
            else:
                m = r3[:, 3] * 2 * c.thr_rand_frac + (1 - c.thr_rand_frac)
                self.thr_mult_left[ids] = m
                self.thr_mult_right[ids] = m
        if c.mass_coupling:                                                 # _apply_mass_driven_coupling: only the listed targets
            kd, sthr, kiz = mass_coupling(c, self.mass[ids])
            if c.couple_targets & 1:
                self.drag_scale[ids, 0] = kd
            if c.couple_targets & 2:
                self.thr_mult_left[ids] = sthr
                self.thr_mult_right[ids] = sthr
            if c.couple_targets & 4:
                self.k_iz[ids] = kiz
        if not c.reset_pose_external:
            rmin, rmax, _ = curriculum(c, self.curriculum_step)
            # the kernel receives rmin / rmax as fp32 parameters and forms (rmax - rmin) in fp32
            rmin32, rmax32 = torch.tensor(rmin, dtype=F32), torch.tensor(rmax, dtype=F32)
            sr = r0[:, 2] * (rmax32 - rmin32) + rmin32
            th = r0[:, 3] * 2 * math.pi

            def spawn():                                                        # get_spawns  [SNAP/USV_capture_xy.py:330-394]
                if c.spawn_about_origin:                                        # live CaptureXY: USV_capture_xy_static_obs.py:955-956
                    self.pos[ids, 0] = sr * torch.cos(th)
                    self.pos[ids, 1] = sr * torch.sin(th)
                else:
                    self.pos[ids, 0] = sr * torch.cos(th) + self.target[ids, 0]
                    self.pos[ids, 1] = sr * torch.sin(th) + self.target[ids, 1]

            if c.retarget_after_spawn:                                          # live reset_idx: get_spawns first, set_targets last
                spawn()
            if c.retarget_on_reset:                                             # get_goals [SNAP/USV_capture_xy.py:312-326]
                self.target[ids, 0] = r0[:, 0] * c.goal_random_position * 2 - c.goal_random_position
                self.target[ids, 1] = r0[:, 1] * c.goal_random_position * 2 - c.goal_random_position
            if not c.retarget_after_spawn:
                spawn()
            self.psi[ids] = r1[:, 0] * math.pi
            # [SNAP/USV_Virtual.py:786-794]
            self.vel[ids, 0] = r1[:, 1] * (2 * c.spawn_vel_range) - c.spawn_vel_range
            self.vel[ids, 1] = r1[:, 2] * (2 * c.spawn_vel_range) - c.spawn_vel_range
            self.r[ids] = 0
        self.reset_buf[ids] = 0
        self.progress_buf[ids] = 0

    # ---- one physics sub-step: apply_forces + world.step stand-in ---------------------------
    def planar_wrench(self):
        c = self.cfg
        n = self.n
        half = self.psi * 0.5
        quat = torch.stack([torch.cos(half), torch.zeros(n), torch.zeros(n), torch.sin(half)], 1)
        vel6 = torch.zeros((n, 6), dtype=F32)
        vel6[:, 0:2] = self.vel
        vel6[:, 5] = self.r
        fwd6 = (c.lin_fwd[0], c.lin_fwd[1], 0.0, 0.0, 0.0, c.lin_fwd[2])
        drag, _ = hydrodynamics(quat, vel6, self.linear_damping, self.quadratic_damping, self.drag_scale,
                                linear_damping_forward_speed=fwd6, offset_linear_damping=c.offset_linear_damping,
                                offset_lin_forward_damping_speed=c.offset_lin_forward_damping_speed,
                                offset_nonlin_damping=c.offset_nonlin_damping, scaling_damping=c.scaling_damping,
                                use_drag_scale=c.use_drag_scale, use_water_current=c.use_water_current,
                                flow_vel=(c.flow_vel_xy[0], c.flow_vel_xy[1], 0.0))
        # disturbances from WORLD position, applied in the body frame [USV_disturbances.py:386-410,510-530]
        wpos = self.pos + self.origin
        fd = torch.zeros((n, 2), dtype=F32)
        td = torch.zeros(n, dtype=F32)
        if c.use_const_force:
            fd = self.f_const.clone()
        if c.use_sin_force:
            fd = self.f_const + torch.sin(wpos * self.f_freq + self.f_shift) * self.f_amp.unsqueeze(1)
        if c.use_const_torque:
            td = self.t_const.clone()
        if c.use_sin_torque:
            td = self.t_const + torch.sin((wpos[:, 0] + wpos[:, 1]) * self.t_freq + self.t_shift) * self.t_amp
        thrL, thrR = self.current_forces[:, 0], self.current_forces[:, 1]
        Fx = fd[:, 0] + drag[:, 0] + thrL + thrR
        Fy = fd[:, 1] + drag[:, 1]
        Tz = td + drag[:, 5] - c.thr_y_left * thrL - c.thr_y_right * thrR
        cs, sn = torch.cos(self.psi), torch.sin(self.psi)
        inv_m = 1.0 / self.mass
        ax = (cs * Fx - sn * Fy) * inv_m
        ay = (sn * Fx + cs * Fy) * inv_m
        rdot = Tz / (c.izz * self.k_iz)
        return drag, Fx, Fy, Tz, ax, ay, rdot

    def substep(self, target):
        c = self.cfg
        self.current_forces = thruster_lag(self.current_forces, target, self.alpha)   # update_forces
        _, _, _, _, ax, ay, rdot = self.planar_wrench()
        self.vel[:, 0] = self.vel[:, 0] + c.dt * ax
        self.vel[:, 1] = self.vel[:, 1] + c.dt * ay
        self.r = self.r + c.dt * rdot
        self.pos = self.pos + c.dt * self.vel
        self.psi = self.psi + c.dt * self.r

    # ---- VecEnvRLGames.step  [OIGE/envs/vec_env_rlgames.py:120-217] --------------------------
    def dynamics(self, actions: torch.Tensor):
        """pre_physics_step + the physics sub-steps + update_state; shared by the classic and the live (Variant B) task."""
        c = self.cfg
        n = self.n
        step = self.step_counter
        # one Philox call per env-step: 8 x 16-bit uniforms (act0, act1, vel_x, vel_y, vel_r, heading, pos_x, pos_y)
        nz = torch.from_numpy(philox.uniform8x16(c.seed, self.env_ids, step, philox.RS_STEP_A))
        actions = torch.clamp(actions, -c.clip_actions, c.clip_actions).clone()
        # pre_physics_step  [SNAP/USV_Virtual.py:571-617]
        reset_ids = self.reset_buf.nonzero(as_tuple=False).squeeze(-1)
        self.reset_idx(reset_ids, step)
        raw_actions = actions.clone()
        if not c.action_affine:
            if c.action_noise:
                actions = actions + _u(nz[:, 0:2], c.action_noise_min, c.action_noise_max)
            pen_actions = actions
            cmd = torch.clamp(actions, -1.0, 1.0)
            before_rect = cmd.clone()
        else:                                                               # [OIGE/tasks/USV_Virtual.py:1064-1097]
            t = actions + (c.action_bias if self.step_counter < c.action_bias_steps else 0.0)
            if c.action_noise:
                t = t + _u(nz[:, 0:2], c.action_noise_min, c.action_noise_max)
            t = torch.clamp(t, -1.0, 1.0)
            before_rect = t.clone()
            cmd = torch.clamp(0.5 * (t + 1.0), 0.0, 1.0)
            pen_actions = cmd.clone() if c.penalties_use_u else actions
        unit = cmd.clone()
        cmd[reset_ids] = 0
        _, target = thruster_target(cmd, self.lut_left, self.lut_right, self.thr_mult_left, self.thr_mult_right)
        for _ in range(c.n_substeps):
            self.substep(target)
        # yaw read-back branch of atan2 on the quaternion: (-pi, pi]
        self.psi = _wrap_pi(self.psi)
        # post_physics_step  [OIGE/tasks/base/rl_task.py:283-303]
        self.progress_buf += 1
        # update_state  [SNAP/USV_Virtual.py:476-530]
        pos = self.pos.clone(); vel = self.vel.clone(); w = self.r.clone(); yaw = self.psi.clone()
        if c.noise_pos:
            pos = pos + _u(nz[:, 6:8], c.pos_noise_min, c.pos_noise_max)
        if c.noise_vel:
            vel = vel + _u(nz[:, 2:4], c.vel_noise_min, c.vel_noise_max)
            w = w + _u(nz[:, 4], c.vel_noise_min, c.vel_noise_max)
        if c.noise_heading:
            yaw = yaw + _u(nz[:, 5], c.heading_noise_min, c.heading_noise_max)
        heading = torch.stack([torch.cos(yaw), torch.sin(yaw)], 1)
        state = {"position": pos, "orientation": heading, "linear_velocity": vel, "angular_velocity": w}
        return state, {"pen_actions": pen_actions, "reset_ids": reset_ids, "raw_actions": raw_actions, "before_rect": before_rect,
                       "unit": unit, "target": target}

    def step(self, actions: torch.Tensor):
        c = self.cfg
        state, dyn = self.dynamics(actions)
        pen_actions, reset_ids, w = dyn["pen_actions"], dyn["reset_ids"], state["angular_velocity"]
        obs, aux = capture_xy_observation(state, self.target)
        out = capture_xy_reward(c, aux, state, self.goal_reached, self.prev_d, reset_ids)
        self.prev_d = aux["d"]
        pen = penalties(c, state, pen_actions, self.prev_w, self.prev_asum, self.first_call)
        self.prev_w = w
        self.prev_asum = pen["asum"]
        self.first_call = False
        rew = out["reward"] + pen["total"]
        kill_dist = curriculum(c, self.curriculum_step + 1.0 / c.horizon_length)[2]      # update_kills(step) after `step += 1/horizon`
        die = capture_xy_kills(c, aux["d"], out["speed"], self.goal_reached, kill_dist)
        self.curriculum_step += 1.0 / c.horizon_length
        ones = torch.ones_like(self.reset_buf)
        self.reset_buf = torch.where(self.progress_buf >= c.max_episode_length - 1, ones, die)   # is_done
        obs = torch.clamp(obs, -c.clip_obs, c.clip_obs)                     # _process_data
        self.step_counter += 1
        self.last = {**out, **pen, **aux, "reset_ids": reset_ids}
        return obs, rew, self.reset_buf.clone()


def _wrap_pi(a: torch.Tensor) -> torch.Tensor:
    two_pi = torch.tensor(2 * math.pi, dtype=F32)
    pi = torch.tensor(math.pi, dtype=F32)
    out = a.clone()
    m = (a > pi) | (a <= -pi)
    w = a - two_pi * torch.round(a * (1.0 / two_pi))
    w = torch.where(w > pi, w - two_pi, w)
    w = torch.where(w <= -pi, w + two_pi, w)
    out[m] = w[m]
    return out


# A16  [SNAP/USV_capture_xy.py:80-97 ; SNAP/USV_core.py:31-55 ("local" frame)]
def capture_xy_observation(state: Dict[str, torch.Tensor], target: torch.Tensor):
    n = target.shape[0]
    err = target - state["position"]
    theta = torch.atan2(state["orientation"][:, 1], state["orientation"][:, 0])
    beta = torch.atan2(err[:, 1], err[:, 0])
    alpha = torch.fmod(beta - theta + math.pi, 2 * math.pi) - math.pi
    herr = torch.abs(alpha)
    td = torch.zeros((n, 6), dtype=F32)
    td[:, 0] = torch.cos(alpha)
    td[:, 1] = torch.sin(alpha)
    td[:, 2] = torch.norm(err, dim=1)
    td[:, 3:5] = state["linear_velocity"]
    obs = torch.zeros((n, 13), dtype=F32)
    ct, st = state["orientation"][:, 0], state["orientation"][:, 1]
    v = state["linear_velocity"]
    obs[:, 0] = ct * v[:, 0] + st * v[:, 1]
    obs[:, 1] = -st * v[:, 0] + ct * v[:, 1]
    obs[:, 2] = state["angular_velocity"]
    obs[:, 3:9] = td
    obs[:, 9:11] = v
    d = torch.sqrt(torch.square(err).sum(-1))          # position_dist as compute_reward sees it (:108)
    return obs, {"err": err, "herr": herr, "d": d, "alpha": alpha}


# A17  [SNAP/USV_capture_xy.py:101-227 ; SNAP/USV_task_rewards.py:40-76]
def capture_xy_reward(c: EnvConfig, aux, state, goal_reached, prev_d, just_reset_ids):
    d, herr = aux["d"], aux["herr"]
    speed = torch.norm(state["linear_velocity"], dim=-1)
    goal = ((d < c.position_tolerance) & (speed < c.goal_speed_gate)).int()
    goal_reached *= goal
    goal_reached += goal
    if c.reward_mode == 0:
        dist = c.position_scale * (prev_d - d)
    elif c.reward_mode == 1:
        dist = c.position_scale * (prev_d.pow(2) - d.pow(2))
    else:
        dist = c.position_scale * (torch.exp(-d / c.exponential_reward_coeff) - torch.exp(-prev_d / c.exponential_reward_coeff))
    align = c.align_la1 * (torch.exp(c.align_la2 * herr.pow(4)) + torch.exp(c.align_la3 * herr.pow(2)))
    dist = dist.clone()
    dist[just_reset_ids] = 0
    sr = torch.zeros_like(d)
    far = d > 3.5
    in_range = (speed[far] >= 0.8) & (speed[far] <= 1.5)
    sr[far] = torch.where(in_range, torch.ones_like(speed[far]) * 0.1, torch.exp(-((speed[far] - 1.15) ** 2) / 0.2) * 0.1)
    m = (d <= 3.5) & (d > 2.5)
    sr[m] = (1.0 - torch.clamp(speed[m] / 1.0, 0.0, 1.0)) * 0.15
    m = (d <= 2.5) & (d > 1.5)
    sr[m] = (1.0 - torch.clamp(speed[m] / 1.0, 0.0, 1.0)) * 0.25
    m = d <= 1.5
    sr[m] = (1.0 - torch.clamp(speed[m] / 1.0, 0.0, 1.0)) * 0.35
    goal_reward = (goal_reached * c.goal_reward).float()
    reward = dist + align + sr + goal_reward + c.time_reward
    bdist = d - c.kill_dist
    bpen = -torch.exp(-bdist / 0.25) * c.boundary_cost
    return {"reward": reward, "distance_reward": dist, "alignment_reward": align, "speed_reward": sr,
            "speed": speed, "boundary_dist": bdist, "boundary_penalty": bpen}


# A9  [SNAP/USV_task_rewards.py:422-506]
def penalties(c: EnvConfig, state, actions, prev_w, prev_asum, first_call: bool):
    n = actions.shape[0]
    w = state["angular_velocity"]
    asum = torch.sum(actions, dim=-1)
    dw = torch.zeros(n, dtype=F32) if first_call else (w - prev_w)
    dasum = torch.zeros(n, dtype=F32) if first_call else (asum - prev_asum)
    speed = torch.norm(state["linear_velocity"], dim=-1)
    lin = c.pen_linear_vel.scalar(speed) if c.pen_linear_vel.form != PEN_OFF else torch.zeros(n, dtype=F32)
    ang = c.pen_angular_vel.scalar(w) if c.pen_angular_vel.form != PEN_OFF else torch.zeros(n, dtype=F32)
    angvar = c.pen_angular_vel_variation.scalar(dw) if c.pen_angular_vel_variation.form != PEN_OFF else torch.zeros(n, dtype=F32)
    energy = c.pen_energy.vector(actions)
    actvar = c.pen_action_variation.scalar(dasum) if c.pen_action_variation.form != PEN_OFF else torch.zeros(n, dtype=F32)
    return {"total": lin + ang + angvar + energy + actvar, "pen_lin": lin, "pen_ang": ang, "pen_angvar": angvar,
            "pen_energy": energy, "pen_actvar": actvar, "asum": asum}


# A18  [SNAP/USV_capture_xy.py:231-275]
def capture_xy_kills(c: EnvConfig, d, speed, goal_reached, kill_dist=None):
    die = torch.zeros_like(goal_reached, dtype=torch.long)
    ones = torch.ones_like(goal_reached, dtype=torch.long)
    die = torch.where(d > (c.kill_dist if kill_dist is None else kill_dist), ones, die)
    die = torch.where((goal_reached >= c.kill_after_n_steps_in_tolerance) & (speed < c.goal_speed_gate), ones, die)
    return die
