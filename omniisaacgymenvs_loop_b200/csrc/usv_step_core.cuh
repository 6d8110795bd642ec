// Shared device code of the fused ASV step kernels (Variant A classic / Variant B live): AoSoA state access, branch-free
// trigonometry, per-episode reset randomisation, the planar force model and the action->physics part of a control step; plus the
// host-side argument checks both step entry points share.
#pragma once
#include <math_constants.h>
#include "philox.cuh"
#include "usv_common.cuh"

namespace usv {

constexpr int kObs = 13;
// python: math.pi / 2*math.pi are doubles that meet fp32 tensors -> rounded to fp32
#define USV_PI_F 3.14159274101257324f
#define USV_2PI_F 6.28318548202514648f

struct EnvState {
  float x, y, psi, vx, vy, r, thrL, thrR, prev_d, prev_w, prev_asum;
  int goal_cnt, progress;
};
struct EnvConst {
  float tx, ty, mass, linu, linv, linr, quadu, quadv, quadr, kdrag, mL, mR, kiz;
  float fcx, fcy, fxf, fyf, fxs, fys, famp, tc, tf, ts, tamp;
};
struct StepOut {
  float obs[kObs];
  float rew, task_rew, penalty;
  int done, die;
  bool finite;
  // diagnostics for stats
  float dist_rew, align_rew, speed_rew, d, speed, bpen, bdist;
  float pen_lin, pen_ang, pen_angvar, pen_energy, pen_actvar, absw, asum;
};

// AoSoA: envs are grouped in tiles of 32 (one warp); inside a tile the fields are consecutive 128 B lines:
//   field f of env i lives at base[((i >> 5) * COUNT + f) * 32 + (i & 31)].
// A warp reads/writes one full line per field, and every field of an env is an IMMEDIATE offset from one
// per-thread base pointer (plain field-major SoA with a runtime stride cost two 64-bit adds per access,
// ~100 of the 1678 instructions per env-step in the r01 profile).
constexpr int kTile = 32;
__device__ __forceinline__ int64_t tile_base(int64_t i, int count) { return (i >> 5) * (int64_t)(count * kTile) + (i & 31); }

// L2 policy of a global access.  kStream (ld/st.global.cs: evict-first in L2) marks data that one launch of the per-step kernel
// touches once and the next launch does not read again, so that the L2 victimises those lines before the ones that it does re-read
// (env state, reset flags).  kNormal is a plain access and leaves the code of every other caller unchanged.
enum class Cache { kNormal, kStream };
template <Cache C, class T>
__device__ __forceinline__ T ld(const T* p) {
  if constexpr (C == Cache::kStream) return __ldcs(p);
  else return *p;
}
template <Cache C, class T>
__device__ __forceinline__ void st(T* p, T v) {
  if constexpr (C == Cache::kStream) __stcs(p, v);
  else *p = v;
}

__device__ __forceinline__ void load_state(const float* __restrict__ s0, int64_t i0, EnvState& e) {
  const float* __restrict__ s = s0 + tile_base(i0, USV_S_COUNT);
  e.x = s[USV_S_X * kTile];
  e.y = s[USV_S_Y * kTile];
  e.psi = s[USV_S_PSI * kTile];
  e.vx = s[USV_S_VX * kTile];
  e.vy = s[USV_S_VY * kTile];
  e.r = s[USV_S_R * kTile];
  e.thrL = s[USV_S_THR_L * kTile];
  e.thrR = s[USV_S_THR_R * kTile];
  e.prev_d = s[USV_S_PREV_D * kTile];
  e.prev_w = s[USV_S_PREV_W * kTile];
  e.prev_asum = s[USV_S_PREV_ASUM * kTile];
  e.goal_cnt = __float_as_int(s[USV_S_GOAL_CNT * kTile]);
  e.progress = __float_as_int(s[USV_S_PROGRESS * kTile]);
}

__device__ __forceinline__ void store_state(float* __restrict__ s0, int64_t i0, const EnvState& e) {
  float* __restrict__ s = s0 + tile_base(i0, USV_S_COUNT);
  s[USV_S_X * kTile] = e.x;
  s[USV_S_Y * kTile] = e.y;
  s[USV_S_PSI * kTile] = e.psi;
  s[USV_S_VX * kTile] = e.vx;
  s[USV_S_VY * kTile] = e.vy;
  s[USV_S_R * kTile] = e.r;
  s[USV_S_THR_L * kTile] = e.thrL;
  s[USV_S_THR_R * kTile] = e.thrR;
  s[USV_S_PREV_D * kTile] = e.prev_d;
  s[USV_S_PREV_W * kTile] = e.prev_w;
  s[USV_S_PREV_ASUM * kTile] = e.prev_asum;
  s[USV_S_GOAL_CNT * kTile] = __int_as_float(e.goal_cnt);
  s[USV_S_PROGRESS * kTile] = __int_as_float(e.progress);
}

template <int kDisturb, Cache C = Cache::kNormal>
__device__ __forceinline__ void load_consts(const float* __restrict__ c0, int64_t i0, EnvConst& k) {
  const float* __restrict__ c = c0 + tile_base(i0, USV_C_COUNT);
  k.tx = ld<C>(c + USV_C_TX * kTile);
  k.ty = ld<C>(c + USV_C_TY * kTile);
  k.mass = ld<C>(c + USV_C_MASS * kTile);
  k.linu = ld<C>(c + USV_C_LIN_U * kTile);
  k.linv = ld<C>(c + USV_C_LIN_V * kTile);
  k.linr = ld<C>(c + USV_C_LIN_R * kTile);
  k.quadu = ld<C>(c + USV_C_QUAD_U * kTile);
  k.quadv = ld<C>(c + USV_C_QUAD_V * kTile);
  k.quadr = ld<C>(c + USV_C_QUAD_R * kTile);
  k.kdrag = ld<C>(c + USV_C_KDRAG * kTile);
  k.mL = ld<C>(c + USV_C_THR_ML * kTile);
  k.mR = ld<C>(c + USV_C_THR_MR * kTile);
  k.kiz = ld<C>(c + USV_C_KIZ * kTile);
  if (kDisturb) {
    k.fcx = ld<C>(c + USV_C_FCX * kTile);
    k.fcy = ld<C>(c + USV_C_FCY * kTile);
    k.fxf = ld<C>(c + USV_C_FXF * kTile);
    k.fyf = ld<C>(c + USV_C_FYF * kTile);
    k.fxs = ld<C>(c + USV_C_FXS * kTile);
    k.fys = ld<C>(c + USV_C_FYS * kTile);
    k.famp = ld<C>(c + USV_C_FAMP * kTile);
    k.tc = ld<C>(c + USV_C_TC * kTile);
    k.tf = ld<C>(c + USV_C_TF * kTile);
    k.ts = ld<C>(c + USV_C_TS * kTile);
    k.tamp = ld<C>(c + USV_C_TAMP * kTile);
  } else {
    k.fcx = k.fcy = k.fxf = k.fyf = k.fxs = k.fys = k.famp = k.tc = k.tf = k.ts = k.tamp = 0.0f;
  }
}

template <int kDisturb, Cache C = Cache::kNormal>
__device__ __forceinline__ void store_consts(float* __restrict__ c0, int64_t i0, const EnvConst& k) {
  float* __restrict__ c = c0 + tile_base(i0, USV_C_COUNT);
  st<C>(c + USV_C_TX * kTile, k.tx);
  st<C>(c + USV_C_TY * kTile, k.ty);
  st<C>(c + USV_C_MASS * kTile, k.mass);
  st<C>(c + USV_C_LIN_U * kTile, k.linu);
  st<C>(c + USV_C_LIN_V * kTile, k.linv);
  st<C>(c + USV_C_LIN_R * kTile, k.linr);
  st<C>(c + USV_C_QUAD_U * kTile, k.quadu);
  st<C>(c + USV_C_QUAD_V * kTile, k.quadv);
  st<C>(c + USV_C_QUAD_R * kTile, k.quadr);
  st<C>(c + USV_C_KDRAG * kTile, k.kdrag);
  st<C>(c + USV_C_THR_ML * kTile, k.mL);
  st<C>(c + USV_C_THR_MR * kTile, k.mR);
  st<C>(c + USV_C_KIZ * kTile, k.kiz);
  if (kDisturb) {
    st<C>(c + USV_C_FCX * kTile, k.fcx);
    st<C>(c + USV_C_FCY * kTile, k.fcy);
    st<C>(c + USV_C_FXF * kTile, k.fxf);
    st<C>(c + USV_C_FYF * kTile, k.fyf);
    st<C>(c + USV_C_FXS * kTile, k.fxs);
    st<C>(c + USV_C_FYS * kTile, k.fys);
    st<C>(c + USV_C_FAMP * kTile, k.famp);
    st<C>(c + USV_C_TC * kTile, k.tc);
    st<C>(c + USV_C_TF * kTile, k.tf);
    st<C>(c + USV_C_TS * kTile, k.ts);
    st<C>(c + USV_C_TAMP * kTile, k.tamp);
  }
}

__device__ __forceinline__ float urange(float u, float lo, float hi) { return u * (hi - lo) + lo; }

// Branch-free sin/cos for |x| < ~1e5 (every angle in this kernel is bounded: headings, phases x*f+shift):
// 3-term Cody-Waite reduction by pi/2 + the classic single-precision minimax polynomials on [-pi/4, pi/4]
// (~1 ulp).  libdevice's sinf/cosf carry a Payne-Hanek slow path behind a branch + convergence barrier per
// call; 22 calls per env-step made that ~10% of the issued instructions (profiles/r01_step_kernel.md).
__device__ __forceinline__ void trig_reduce(float x, float& r, int& q) {
  const float j = rintf(x * 0.636619772f);
  q = (int)j;
  r = fmaf(j, -1.57079601e+00f, x);
  r = fmaf(j, -3.13916473e-07f, r);
  r = fmaf(j, -5.39030253e-15f, r);
}
__device__ __forceinline__ float poly_sin(float r, float r2) {
  float p = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
  p = fmaf(p, r2, -1.6666654611e-1f);
  return fmaf(p * r2, r, r);
}
__device__ __forceinline__ float poly_cos(float r2) {
  float p = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
  p = fmaf(p, r2, 4.166664568298827e-2f);
  p = fmaf(p, r2, -0.5f);
  return fmaf(p, r2, 1.0f);
}
__device__ __forceinline__ void fsincos(float x, float* sp, float* cp) {
  float r; int q;
  trig_reduce(x, r, q);
  const float r2 = r * r;
  const float s = poly_sin(r, r2), c = poly_cos(r2);
  const float ss = (q & 1) ? c : s;
  const float cc = (q & 1) ? s : c;
  // sign flips as sign-bit XORs: sin negated in quadrants 2,3; cos in quadrants 1,2
  *sp = __int_as_float(__float_as_int(ss) ^ ((q & 2) << 30));
  *cp = __int_as_float(__float_as_int(cc) ^ (((q + 1) & 2) << 30));
}
// sin() for the sinusoidal force/torque disturbances, evaluated 3x per physics sub-step: explicit 2-term
// Cody-Waite reduction to [-pi, pi], then the SFU (MUFU.SIN, abs error <= 2^-21.4 on that interval).  With
// amplitudes <= 1.77 N / 1 Nm the force error is < 1e-6 N against drag/thrust forces of 1..100 N, i.e. far inside
// the 1e-5 parity bar, and it replaces ~17 issue slots by 6 (the loop was 48% of the kernel, r01 profile).
__device__ __forceinline__ float fsin_sfu(float x) {
  const float k = rintf(x * 0.159154943f);
  float r = fmaf(k, -6.28318548e+00f, x);
  r = fmaf(k, 1.74845553e-07f, r);
  return __sinf(r);
}
__device__ __forceinline__ float fsin(float x) {
  float r; int q;
  trig_reduce(x, r, q);
  const float r2 = r * r;
  const float v = (q & 1) ? poly_cos(r2) : poly_sin(r, r2);
  return __int_as_float(__float_as_int(v) ^ ((q & 2) << 30));
}

// atan2 for the goal bearing: octant reduction + degree-15 odd polynomial on [0,1] (max error 1.5e-7 rad, i.e. within
// 1 ulp of pi-scale results) -- ~20 instructions against ~50 for libdevice's atan2f with its special-case ladder.
// atan2(0, 0) = 0 and the (-pi, pi] branch as torch.atan2.
__device__ __forceinline__ float fast_atan2(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  const float t = (mx > 0.0f) ? __fdividef(mn, mx) : 0.0f;
  const float t2 = t * t;
  float p = fmaf(t2, -0.00455979211255908f, 0.023780519142746925f);   // Chebyshev-node fit of atan(t)/t in t^2: 1.5e-7 rad in fp32
  p = fmaf(p, t2, -0.05882975459098816f);
  p = fmaf(p, t2, 0.09868865460157394f);
  p = fmaf(p, t2, -0.14003290235996246f);
  p = fmaf(p, t2, 0.19966961443424225f);
  p = fmaf(p, t2, -0.3333181142807007f);
  p = fmaf(p, t2, 0.9999998807907104f);
  float a = p * t;
  a = (ay > ax) ? 1.57079637f - a : a;
  a = (x < 0.0f) ? 3.14159274f - a : a;
  return (y < 0.0f) ? -a : a;
}

// wrap an angle into (-pi, pi]  (the branch torch.atan2 returns for the yaw read-back)
__device__ __forceinline__ float wrap_pi(float a) {
  // in-range values pass through bit-exactly (rintf gives 0): same as the oracle's masked wrap
  a = a - USV_2PI_F * rintf(a * (1.0f / USV_2PI_F));
  a = (a > USV_PI_F) ? a - USV_2PI_F : a;
  a = (a <= -USV_PI_F) ? a + USV_2PI_F : a;
  return a;
}

// Step plans: the discrete parameters of one step configuration, fixed at compile time so that the kernel neither tests them per
// thread nor loops over a run-time sub-step count.  A field equal to kFromParams is read from UsvStepParams at run time; PlanGeneric
// reads every field so.  Continuous parameters (dt, lag, bounds, scales, noise ranges, penalty coefficients) always come from
// UsvStepParams, so a plan instance runs the same arithmetic as the generic one.
constexpr int kFromParams = -1;
template <int kPlan>
__host__ __device__ __forceinline__ int plan_or(int from_params) { return kPlan == kFromParams ? from_params : kPlan; }

// X(plan field, UsvStepParams member): every discrete field a plan may fix
#define USV_PLAN_FIELDS(X)                                                                                                        \
  X(n_substeps, n_substeps) X(action_affine, action_affine) X(action_noise, action_noise) X(noise_pos, noise_pos)                 \
  X(noise_vel, noise_vel) X(noise_heading, noise_heading) X(envs_per_row, envs_per_row) X(use_drag_scale, use_drag_scale)          \
  X(reward_mode, reward_mode) X(pen_linear_vel, pen_linear_vel.form) X(pen_angular_vel, pen_angular_vel.form)                     \
  X(pen_angular_vel_variation, pen_angular_vel_variation.form) X(pen_energy, pen_energy.form)                                     \
  X(pen_action_variation, pen_action_variation.form) X(use_const_force, use_const_force) X(use_sin_force, use_sin_force)          \
  X(use_const_torque, use_const_torque) X(use_sin_torque, use_sin_torque) X(use_water_current, use_water_current)

struct PlanGeneric {
  static constexpr bool kFixed = false;
#define USV_PLAN_ANY(f, m) static constexpr int f = kFromParams;
  USV_PLAN_FIELDS(USV_PLAN_ANY)
#undef USV_PLAN_ANY
};

// UsvEnvConfig().full_dr(), the configuration training and the benchmark run: classic action path, action / position / velocity /
// heading noise, linear distance reward, the angular-velocity-variation and energy penalties, all four disturbance kinds without a
// water current (the kDisturb == 2 kernel), no env grid.  Fields the plan leaves to UsvStepParams (penalties_use_u) are read only
// behind a switch the plan turns off.  The reset switches (reset_env) stay run-time tests: a reset is rare, and folding them too made
// the step slower on a B200 (47.3 against 43.1 us per step at 2^20 envs, profiles/r05_step_plan.md).
struct PlanFullDr {
  static constexpr bool kFixed = true;
  static constexpr int n_substeps = 5, action_affine = 0, action_noise = 1, noise_pos = 1, noise_vel = 1, noise_heading = 1;
  static constexpr int envs_per_row = 0, use_drag_scale = 0, reward_mode = USV_REWARD_LINEAR;
  static constexpr int pen_linear_vel = USV_PEN_OFF, pen_angular_vel = USV_PEN_OFF, pen_angular_vel_variation = USV_PEN_EXP_NEG_ABS,
                       pen_energy = USV_PEN_EXP_NEG_SUMSQ, pen_action_variation = USV_PEN_OFF;
  static constexpr int use_const_force = 1, use_sin_force = 1, use_const_torque = 1, use_sin_torque = 1, use_water_current = 0;
};

// does `p` have the discrete parameters Plan fixes?
template <class Plan>
inline bool plan_matches(const UsvStepParams& p) {
#define USV_PLAN_EQ(f, m) if (Plan::f != kFromParams && Plan::f != p.m) return false;
  USV_PLAN_FIELDS(USV_PLAN_EQ)
#undef USV_PLAN_EQ
  return true;
}

// The products that end a term are rounded on their own (__fmul_rn): with the form fixed, the compiler could otherwise fuse one into
// the sum of the terms, which the generic kernel (the term behind a run-time switch) never does.
template <int kForm = kFromParams>
__device__ __forceinline__ float penalty_scalar(const UsvPenaltyTerm& t, float x) {
  switch (plan_or<kForm>(t.form)) {
    case USV_PEN_NEG_ABS: return -fabsf(x) * t.c1 + t.c2;
    case USV_PEN_NEG_DEADZONE: return __fmul_rn(-fmaxf(fabsf(x) - t.k, 0.0f), t.c1);
    case USV_PEN_EXP_NEG_ABS: return __fmul_rn(__expf(-t.k * fabsf(x)) - 1.0f, t.c1);
    default: return 0.0f;
  }
}

// get_spawns  [ref SNAP/USV_capture_xy.py:330-394]: annulus around the target (classic) or the env origin (live:
// OIGE/tasks/USV/USV_capture_xy_static_obs.py:955-956).  r0 = philox_uniform4(seed, gid, step, RS_RESET_0); shared with the
// live scene builder, which must see the same spawn point when it places the obstacles.
__device__ __forceinline__ void spawn_xy(const UsvStepParams& p, const Uniform4& r0, float tx, float ty, float& x, float& y) {
  const float sr = r0.c * (p.spawn_max_dist - p.spawn_min_dist) + p.spawn_min_dist;
  const float sth = r0.d * 2.0f * USV_PI_F;
  float ssp, csp;
  fsincos(sth, &ssp, &csp);
  x = p.spawn_about_origin ? sr * csp : sr * csp + tx;
  y = p.spawn_about_origin ? sr * ssp : sr * ssp + ty;
}

// reset_idx for one env  [ref: SNAP/USV_Virtual.py:750-817 ; OIGE/tasks/USV_Virtual.py:1502-1618]
template <int kDisturb>
__device__ __forceinline__ void reset_env(EnvState& e, EnvConst& k, const UsvStepParams& p, uint64_t gid, uint64_t step) {
  const Uniform4 r0 = philox_uniform4(p.seed, gid, step, RS_RESET_0);
  const Uniform4 r1 = philox_uniform4(p.seed, gid, step, RS_RESET_1);
  // task.reset / get_spawns: goal counter cleared  [ref SNAP/USV_capture_xy.py:308-310,342]
  e.goal_cnt = 0;
  if (kDisturb) {
    // UF.generate_force / TD.generate_torque  [ref OIGE/tasks/USV/USV_disturbances.py:327-384,469-508]
    if (p.use_force_disturbance) {
      const Uniform4 r5 = philox_uniform4(p.seed, gid, step, RS_RESET_5);
      const Uniform4 r6 = philox_uniform4(p.seed, gid, step, RS_RESET_6);
      const Uniform4 r7 = philox_uniform4(p.seed, gid, step, RS_RESET_7);
      if (p.use_sin_force) {
        k.fxf = urange(r5.c, p.force_min_freq, p.force_max_freq);
        k.fyf = urange(r5.d, p.force_min_freq, p.force_max_freq);
        k.fxs = urange(r6.a, p.force_min_shift, p.force_max_shift);
        k.fys = urange(r6.b, p.force_min_shift, p.force_max_shift);
        k.famp = urange(r6.c, p.force_sin_min, p.force_sin_max);
      }
      if (p.use_const_force) {
        const float rr = urange(r6.d, p.force_const_min, p.force_const_max);
        const float th = r7.a * USV_PI_F * 2.0f;
        float sth_, cth_;
        fsincos(th, &sth_, &cth_);
        k.fcx = cth_ * rr;
        k.fcy = sth_ * rr;
      }
    }
    if (p.use_torque_disturbance) {
      const Uniform4 r7 = philox_uniform4(p.seed, gid, step, RS_RESET_7);
      const Uniform4 r8 = philox_uniform4(p.seed, gid, step, RS_RESET_8);
      if (p.use_sin_torque) {
        k.tf = urange(r7.b, p.torque_min_freq, p.torque_max_freq);
        k.ts = urange(r7.c, p.torque_min_shift, p.torque_max_shift);
        k.tamp = urange(r7.d, p.torque_sin_min, p.torque_sin_max);
      }
      if (p.use_const_torque) {
        float rr = urange(r8.a, p.torque_const_min, p.torque_const_max);
        if (r8.b > 0.5f) rr *= -1.0f;
        k.tc = rr;
      }
    }
  }
  // MDD.randomize_masses  [ref USV_disturbances.py:127-151]
  k.mass = p.mass_rand ? urange(r1.d, p.mass_min, p.mass_max) : p.mass_base;
  // _apply_yaw_inertia_randomization (skipped when yaw_inertia is a coupling target)  [ref OIGE/tasks/USV_Virtual.py:153-170,1532-1533]
  if (p.kiz_rand && !(p.mass_coupling && (p.couple_targets & 4))) {
    const Uniform4 r5 = philox_uniform4(p.seed, gid, step, RS_RESET_5);
    if (p.kiz_log) {
      const float l0 = logf(p.couple_kiz_min), l1 = logf(p.couple_kiz_max);
      k.kiz = expf(l0 + r5.b * (l1 - l0));
    } else {
      k.kiz = p.couple_kiz_min + r5.b * (p.couple_kiz_max - p.couple_kiz_min);
    }
  }
  // hydrodynamics.reset_coefficients  [ref OIGE/envs/USV/Hydrodynamics.py:136-174]
  if (p.drag_rand) {
    const Uniform4 r3 = philox_uniform4(p.seed, gid, step, RS_RESET_3);
    const Uniform4 r4 = philox_uniform4(p.seed, gid, step, RS_RESET_4);
    k.linu = p.lin_base[0] + (r3.a * 2.0f - 1.0f) * p.lin_rand[0];
    k.linv = p.lin_base[1] + (r3.b * 2.0f - 1.0f) * p.lin_rand[1];
    k.linr = p.lin_base[2] + (r3.c * 2.0f - 1.0f) * p.lin_rand[2];
    k.quadu = p.quad_base[0] + (r4.a * 2.0f - 1.0f) * p.quad_rand[0];
    k.quadv = p.quad_base[1] + (r4.b * 2.0f - 1.0f) * p.quad_rand[1];
    k.quadr = p.quad_base[2] + (r4.c * 2.0f - 1.0f) * p.quad_rand[2];
  }
  if (p.kdrag_rand) {  // _sample_k_drag [ref Hydrodynamics.py:119-134]
    const Uniform4 r2 = philox_uniform4(p.seed, gid, step, RS_RESET_2);
    if (p.kdrag_log) {
      const float l0 = logf(p.kdrag_min), l1 = logf(p.kdrag_max);
      k.kdrag = expf(l0 + r2.d * (l1 - l0));
    } else {
      k.kdrag = p.kdrag_min + r2.d * (p.kdrag_max - p.kdrag_min);
    }
  }
  // thrusters.reset_thruster_randomization  [ref OIGE/envs/USV/ThrusterDynamics.py:112-127]
  if (p.thr_rand) {
    if (p.thr_separate) {
      const Uniform4 r4 = philox_uniform4(p.seed, gid, step, RS_RESET_4);
      const Uniform4 r5 = philox_uniform4(p.seed, gid, step, RS_RESET_5);
      k.mL = r4.d * 2.0f * p.thr_left_frac + (1.0f - p.thr_left_frac);
      k.mR = r5.a * 2.0f * p.thr_right_frac + (1.0f - p.thr_right_frac);
    } else {
      const Uniform4 r3 = philox_uniform4(p.seed, gid, step, RS_RESET_3);
      k.mL = k.mR = r3.d * 2.0f * p.thr_rand_frac + (1.0f - p.thr_rand_frac);
    }
  }
  // _apply_mass_driven_coupling  [ref OIGE/tasks/USV_Virtual.py:988-1040]
  if (p.mass_coupling) {   // every target in p.couple_targets is overridden, the others keep their independent draw
    const float denom = fmaxf(p.couple_mass_max - p.mass_base, 1e-6f);
    const float rr = fminf(fmaxf((k.mass - p.mass_base) / denom, 0.0f), 1.0f);
    if (p.couple_targets & 1) k.kdrag = p.kdrag_min + rr * (p.kdrag_max - p.kdrag_min);
    if (p.couple_targets & 2) {
      const float s = fminf(fmaxf(1.0f - rr * p.couple_thr_a, 1.0f - p.couple_thr_a), 1.0f);
      k.mL = k.mR = s;
    }
    if (p.couple_targets & 4) k.kiz = p.couple_kiz_min + rr * (p.couple_kiz_max - p.couple_kiz_min);
  }
  if (!p.reset_pose_external) {
    // goals [ref SNAP/USV_capture_xy.py:312-326]: the live reset_idx spawns around the OLD target and re-draws the target last
    if (p.retarget_after_spawn) spawn_xy(p, r0, k.tx, k.ty, e.x, e.y);
    if (p.retarget_on_reset) {
      k.tx = r0.a * p.goal_random_position * 2.0f - p.goal_random_position;
      k.ty = r0.b * p.goal_random_position * 2.0f - p.goal_random_position;
    }
    if (!p.retarget_after_spawn) spawn_xy(p, r0, k.tx, k.ty, e.x, e.y);
    // quaternion (cos(a/2),0,0,sin(a/2)) with a ~ U[0,pi)  ->  yaw = a
    e.psi = r1.a * USV_PI_F;
    // root velocities: zero, then vx,vy ~ U(-1.5,1.5) in the world frame  [ref SNAP/USV_Virtual.py:786-794]
    e.vx = r1.b * (2.0f * p.spawn_vel_range) - p.spawn_vel_range;
    e.vy = r1.c * (2.0f * p.spawn_vel_range) - p.spawn_vel_range;
    e.r = 0.0f;
  }
  e.progress = 0;
  // NOTE: thruster lag state (current_forces), prev_d, prev_w and prev_asum are NOT reset
  // (reference quirks 4 and 7, SURVEY appendix C).
}

// ComputeDampingMatrix  [ref Hydrodynamics.py:176-205]:  D = (((lin + off_lin) - (lin_fwd + off_fwd)) + (quad + off_nl)|v|) * scaling [* k_drag]
// is affine in |v| with per-episode coefficients: D = a + b|v|.  a and b are formed once per control step (scaling and k_drag folded
// in: 1e-7 relative against the reference's op order), the sub-step loop spends one FMA per axis.
struct Damp { float au, bu, av, bv, ar, br; };
template <class Plan = PlanGeneric>
__device__ __forceinline__ Damp make_damp(const EnvConst& k, const UsvStepParams& p) {
  const float sc = plan_or<Plan::use_drag_scale>(p.use_drag_scale) ? p.scaling_damping * k.kdrag : p.scaling_damping;
  const float off_fwd = p.offset_lin_forward_damping_speed;
  Damp d;
  d.au = ((k.linu + p.offset_linear_damping) - (p.lin_fwd[0] + off_fwd)) * sc;
  d.av = ((k.linv + p.offset_linear_damping) - (p.lin_fwd[1] + off_fwd)) * sc;
  d.ar = ((k.linr + p.offset_linear_damping) - (p.lin_fwd[2] + off_fwd)) * sc;
  d.bu = (k.quadu + p.offset_nonlin_damping) * sc;
  d.bv = (k.quadv + p.offset_nonlin_damping) * sc;
  d.br = (k.quadr + p.offset_nonlin_damping) * sc;
  return d;
}

// planar force model for one physics sub-step; returns body wrench and world acceleration
template <int kDisturb>
__device__ __forceinline__ void planar_wrench(const EnvState& e, const EnvConst& k, const UsvStepParams& p, const Damp& dm, float ox,
                                              float oy, float inv_m, float inv_iz, float s, float c, float& du, float& dv,
                                              float& dr, float& Fx, float& Fy, float& Tz, float& ax, float& ay,
                                              float& rdot) {
  // R^T v (world -> body)  [ref Hydrodynamics.py:213-222, planar quaternion]
  float u = c * e.vx + s * e.vy;
  float v = -s * e.vx + c * e.vy;
  const float w = e.r;
  // water current: the damping acts on the velocity relative to the flow, both taken to the body frame first
  // [ref Hydrodynamics.py:224-237].  Only the generic variant carries the test (the host routes a config with a current to it).
  if (kDisturb == 1 && p.use_water_current) {
    u -= c * p.flow_vel_xy[0] + s * p.flow_vel_xy[1];
    v -= -s * p.flow_vel_xy[0] + c * p.flow_vel_xy[1];
  }
  du = -fmaf(dm.bu, fabsf(u), dm.au) * u;
  dv = -fmaf(dm.bv, fabsf(v), dm.av) * v;
  dr = -fmaf(dm.br, fabsf(w), dm.ar) * w;
  // disturbances: functions of the WORLD position, applied in the BODY frame (is_global=False)
  // [ref USV_disturbances.py:386-410,510-530 ; SNAP/USV_Virtual.py:621-650]
  float fdx = 0.0f, fdy = 0.0f, td = 0.0f;
  if (kDisturb) {
    // kDisturb == 2: all four disturbance kinds are on (the full-DR configuration): no per-sub-step flag tests
    const bool cf = kDisturb == 2 || p.use_const_force, sf = kDisturb == 2 || p.use_sin_force;
    const bool ct = kDisturb == 2 || p.use_const_torque, stq = kDisturb == 2 || p.use_sin_torque;
    if (cf) { fdx = k.fcx; fdy = k.fcy; }
    if (sf) {
      fdx = k.fcx + fsin_sfu((e.x + ox) * k.fxf + k.fxs) * k.famp;
      fdy = k.fcy + fsin_sfu((e.y + oy) * k.fyf + k.fys) * k.famp;
    }
    if (ct) td = k.tc;
    if (stq) td = k.tc + fsin_sfu(((e.x + ox) + (e.y + oy)) * k.tf + k.ts) * k.tamp;
  }
  // net wrench at the base link; thrusters push along body x at (thr_x, thr_y_*)  (heron.urdf:167,242)
  Fx = fdx + du + e.thrL + e.thrR;
  Fy = fdy + dv;
  Tz = td + dr - p.thr_y_left * e.thrL - p.thr_y_right * e.thrR;
  ax = (c * Fx - s * Fy) * inv_m;
  ay = (s * Fx + c * Fy) * inv_m;
  rdot = Tz * inv_iz;
}

// one physics sub-step: thruster lag, wrench, semi-implicit Euler, heading advance.  (hsn, hcs) = (sin, cos) psi: one full evaluation per
// control step, then advanced by the small per-sub-step yaw increment with a rotation by (cos d, sin d) from short Taylor polynomials
// (|d| = dt*|r| <= 1/16; a full sincos beyond)
template <int kDisturb>
__device__ __forceinline__ void physics_substep(EnvState& e, const EnvConst& k, const UsvStepParams& p, const Damp& dm, float ox, float oy,
                                                float inv_m, float inv_iz, float oma, float tgtL, float tgtR, float& hsn, float& hcs) {
  // apply_forces(): update_forces() advances the lag BEFORE the wrench is applied
  // [ref ThrusterDynamics.py:129-141; SNAP/USV_Virtual.py:640]
  e.thrL = __fadd_rn(__fmul_rn(e.thrL, p.lag_alpha), __fmul_rn(oma, tgtL));
  e.thrR = __fadd_rn(__fmul_rn(e.thrR, p.lag_alpha), __fmul_rn(oma, tgtR));
  float du, dv, dr, Fx, Fy, Tz, ax, ay, rdot;
  planar_wrench<kDisturb>(e, k, p, dm, ox, oy, inv_m, inv_iz, hsn, hcs, du, dv, dr, Fx, Fy, Tz, ax, ay, rdot);
  // world.step(): semi-implicit Euler (velocities first, then positions)
  e.vx += p.dt * ax;
  e.vy += p.dt * ay;
  e.r += p.dt * rdot;
  e.x += p.dt * e.vx;
  e.y += p.dt * e.vy;
  const float dpsi = p.dt * e.r;
  e.psi += dpsi;
  if (fabsf(dpsi) <= 0.0625f) {   // |r| <= 3.1 rad/s at dt = 0.02: sin to d^5 (error d^7/5040 < 8e-13), cos to d^4 (d^6/720 < 9e-11)
    const float d2 = dpsi * dpsi;
    const float sd = dpsi * fmaf(d2, fmaf(d2, 1.0f / 120.0f, -1.0f / 6.0f), 1.0f);
    const float cd = fmaf(d2, fmaf(d2, 1.0f / 24.0f, -0.5f), 1.0f);
    const float nc = hcs * cd - hsn * sd;
    hsn = hsn * cd + hcs * sd;
    hcs = nc;
  } else {
    fsincos(e.psi, &hsn, &hcs);
  }
}

// Sensed state + action bookkeeping handed from the shared dynamics part of a control step to the task-specific part.
struct DynOut {
  float raw0, raw1;              // policy action after the VecEnv clamp (live: prev_thrust_cmds)
  float pa0, pa1;                // what Penalties sees as `actions`
  float t0, t1;                  // live: thrust_cmds_before_rect
  float c0, c1;                  // command that indexed the LUT (live: thrust_cmds_unit, before the reset zeroing)
  float pxn, pyn, vxn, vyn, wn, yawn, hs, hc;  // noisy state the task observes; (hc, hs) = heading
};

// per-step noise draw; a fixed Plan draws it from `keys`, the round keys of p.seed
template <class Plan>
__device__ __forceinline__ Uniform8 step_noise(const UsvStepParams& p, const PhiloxKeys* keys, uint64_t gid, uint64_t step) {
  if constexpr (Plan::kFixed) return philox_uniform8x16(*keys, gid, step, RS_STEP_A);
  else return philox_uniform8x16(p.seed, gid, step, RS_STEP_A);
}

// pre_physics_step + the physics sub-steps + update_state of one control step for one env, state in registers
template <int kDisturb, bool kLutGlobal, class Plan = PlanGeneric>
__device__ __forceinline__ void step_dynamics(EnvState& e, EnvConst& k, const UsvStepParams& p, bool do_reset,
                                             float2 act, uint64_t gid, int64_t lid, uint64_t step,
                                             const float* __restrict__ s_lutL, const float* __restrict__ s_lutR,
                                             DynOut& s, const PhiloxKeys* keys = nullptr) {
  // ---- pre_physics_step ------------------------------------------------------------------
  if (do_reset) reset_env<kDisturb>(e, k, p, gid, step);
  const Uniform8 nz = step_noise<Plan>(p, keys, gid, step);
  const float u_a0 = nz.v[0], u_a1 = nz.v[1], u_vx = nz.v[2], u_vy = nz.v[3], u_w = nz.v[4], u_h = nz.v[5],
              u_px = nz.v[6], u_py = nz.v[7];
  // VecEnvRLGames.step clamps to +-clipActions  [ref vec_env_rlgames.py:136-140]
  float a0 = fminf(fmaxf(act.x, -p.clip_actions), p.clip_actions);
  float a1 = fminf(fmaxf(act.y, -p.clip_actions), p.clip_actions);
  float pa0, pa1;  // what Penalties sees as `actions`
  float c0, c1;    // command that indexes the LUT
  s.raw0 = a0; s.raw1 = a1;
  if (!plan_or<Plan::action_affine>(p.action_affine)) {
    // classic [ref SNAP/USV_Virtual.py:589-615]: AN.add_noise_on_act works IN PLACE on the tensor that
    // self.actions aliases -> penalties see the noisy, unclamped action; resets zero only the thrust.
    if (plan_or<Plan::action_noise>(p.action_noise)) {
      a0 += urange(u_a0, p.action_noise_min, p.action_noise_max);
      a1 += urange(u_a1, p.action_noise_min, p.action_noise_max);
    }
    pa0 = a0; pa1 = a1;
    c0 = fminf(fmaxf(a0, -1.0f), 1.0f);
    c1 = fminf(fmaxf(a1, -1.0f), 1.0f);
    s.t0 = c0; s.t1 = c1;
  } else {
    // live [ref OIGE/tasks/USV_Virtual.py:1064-1097]
    float t0 = a0 + p.action_bias, t1 = a1 + p.action_bias;
    if (plan_or<Plan::action_noise>(p.action_noise)) {
      t0 += urange(u_a0, p.action_noise_min, p.action_noise_max);
      t1 += urange(u_a1, p.action_noise_min, p.action_noise_max);
    }
    t0 = fminf(fmaxf(t0, -1.0f), 1.0f);
    t1 = fminf(fmaxf(t1, -1.0f), 1.0f);
    s.t0 = t0; s.t1 = t1;
    c0 = fminf(fmaxf(0.5f * (t0 + 1.0f), 0.0f), 1.0f);
    c1 = fminf(fmaxf(0.5f * (t1 + 1.0f), 0.0f), 1.0f);
    pa0 = p.penalties_use_u ? c0 : a0;
    pa1 = p.penalties_use_u ? c1 : a1;
  }
  s.pa0 = pa0; s.pa1 = pa1; s.c0 = c0; s.c1 = c1;
  if (do_reset) { c0 = 0.0f; c1 = 0.0f; }
  // set_target_force -> get_cmd_interpolated  [ref ThrusterDynamics.py:179-219]
  const int iL = lut_index(c0, p.n_lut), iR = lut_index(c1, p.n_lut);
  const float tgtL = (kLutGlobal ? __ldg(s_lutL + iL) : s_lutL[iL]) * k.mL;
  const float tgtR = (kLutGlobal ? __ldg(s_lutR + iR) : s_lutR[iR]) * k.mR;

  // ---- physics sub-steps -----------------------------------------------------------------
  float ox = 0.0f, oy = 0.0f;
  if (kDisturb && plan_or<Plan::envs_per_row>(p.envs_per_row) > 0) {
    const int row = (int)(lid / p.envs_per_row), col = (int)(lid % p.envs_per_row);
    ox = p.grid_row_offset - (float)row * p.env_spacing;
    oy = (float)col * p.env_spacing - p.grid_col_offset;
  }
  const float oma = 1.0f - p.lag_alpha;
  // 2-ulp reciprocals (MUFU.RCP): the accelerations they scale are compared at 1e-5
  const float inv_m = __fdividef(1.0f, k.mass), inv_iz = __fdividef(1.0f, p.izz * k.kiz);
  float hsn, hcs;
  fsincos(e.psi, &hsn, &hcs);
  const Damp dm = make_damp<Plan>(k, p);
  if constexpr (Plan::n_substeps != kFromParams) {
#pragma unroll
    for (int ss = 0; ss < Plan::n_substeps; ++ss) physics_substep<kDisturb>(e, k, p, dm, ox, oy, inv_m, inv_iz, oma, tgtL, tgtR, hsn, hcs);
  } else {
    for (int ss = 0; ss < p.n_substeps; ++ss) physics_substep<kDisturb>(e, k, p, dm, ox, oy, inv_m, inv_iz, oma, tgtL, tgtR, hsn, hcs);
  }
  e.psi = wrap_pi(e.psi);

  // ---- post_physics_step ------------------------------------------------------------------
  e.progress += 1;  // [ref rl_task.py:294]
  // update_state: observation noise  [ref SNAP/USV_Virtual.py:476-530 ; USV_disturbances.py:552-601]
  float pxn = e.x, pyn = e.y, vxn = e.vx, vyn = e.vy, wn = e.r, yawn = e.psi;
  if (plan_or<Plan::noise_pos>(p.noise_pos)) { pxn += urange(u_px, p.pos_noise_min, p.pos_noise_max); pyn += urange(u_py, p.pos_noise_min, p.pos_noise_max); }
  if (plan_or<Plan::noise_vel>(p.noise_vel)) {
    vxn += urange(u_vx, p.vel_noise_min, p.vel_noise_max);
    vyn += urange(u_vy, p.vel_noise_min, p.vel_noise_max);
    wn += urange(u_w, p.vel_noise_min, p.vel_noise_max);
  }
  // heading the task observes = (cos, sin)(psi + noise): the loop already tracks (cos psi, sin psi); rotate it by the small noise
  // angle (|dh| <= 0.5: same 5e-9 polynomial error as the per-sub-step update) instead of a third full sincos per control step
  float hs = hsn, hc = hcs;
  if (plan_or<Plan::noise_heading>(p.noise_heading)) {
    const float dh = urange(u_h, p.heading_noise_min, p.heading_noise_max);
    yawn += dh;
    if (fabsf(dh) <= 0.5f) {
      const float d2 = dh * dh;
      const float sd = dh * fmaf(d2, fmaf(d2, fmaf(d2, -1.0f / 5040.0f, 1.0f / 120.0f), -1.0f / 6.0f), 1.0f);
      const float cd = fmaf(d2, fmaf(d2, fmaf(d2, fmaf(d2, 1.0f / 40320.0f, -1.0f / 720.0f), 1.0f / 24.0f), -0.5f), 1.0f);
      hc = hcs * cd - hsn * sd;
      hs = hsn * cd + hcs * sd;
    } else {
      fsincos(yawn, &hs, &hc);
    }
  }
  s.pxn = pxn; s.pyn = pyn; s.vxn = vxn; s.vyn = vyn; s.wn = wn; s.yawn = yawn; s.hs = hs; s.hc = hc;
}

// argument checks shared by the step entry points (classic and live)
inline int check_common(const UsvEnvBuffers* b, int64_t n, const UsvStepParams* p) {
  if (!b || !p) return USV_E_NULL;
  if (n < 0) return USV_E_SIZE;
  if (!b->state || !b->consts || !b->reset_buf || !b->lut_left || !b->lut_right) return USV_E_NULL;
  if (b->state_stride < n || b->consts_stride < n || (b->state_stride & 31) || (b->consts_stride & 31)) return USV_E_SIZE;
  if (b->stats && (b->stats_stride < n || (b->stats_stride & 31))) return USV_E_SIZE;
  if (p->n_lut < 2 || p->n_lut > 8192) return USV_E_PARAM;
  if (p->n_substeps < 0 || p->n_substeps > 1024) return USV_E_PARAM;
  if (!(p->izz > 0.0f)) return USV_E_PARAM;
  if (p->reward_mode < USV_REWARD_LINEAR || p->reward_mode > USV_REWARD_EXPONENTIAL) return USV_E_PARAM;
  return USV_OK;
}

inline bool wants_disturb(const UsvStepParams* p) {
  return p->use_force_disturbance || p->use_torque_disturbance || p->use_const_force || p->use_sin_force ||
         p->use_const_torque || p->use_sin_torque || p->use_water_current;   // a water current rides in the generic variant
}

}  // namespace usv
