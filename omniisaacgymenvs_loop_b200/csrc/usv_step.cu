// Fused ASV env step for sm_100a: reset-if-flagged -> action -> thruster LUT -> n_substeps x
// {first-order thruster lag, hydrodynamic damping, disturbances, planar rigid-body semi-implicit
// Euler} -> CaptureXY observation (13) -> reward + penalties -> kills / done.  One launch replaces
// VecEnvRLGames.step  [ref: OIGE/envs/vec_env_rlgames.py:120-217] and everything below it.
//
// Layout: env state / per-episode constants are structure-of-arrays in HBM (field-major), so a
// warp's 32 envs read each field as one 128 B line; the (n,13) row-major observation rl_games wants
// is staged through shared memory (stride 13 is odd -> conflict-free) and written as float4 lines.
// The thruster LUTs (2 x n_lut floats, gathered at random) are staged once per CTA in shared memory.
// RNG is Philox4x32-10 keyed (seed; env, step, stream): no RNG state in HBM.
//
// Roofline: HBM-bound by design -- algorithmic bytes per env-step are tabulated in DESIGN.md.
// CTA shape of the classic kernels of this file: 128 threads, 7 CTAs per SM = 28 warps per SM at 72 registers (no spill).  The fused step is
// issue-bound and ends in a partial wave: with 256 x 3 (24 warps per SM, 78 registers) 2^20 envs are 9.23 waves and the last 0.23 runs one
// CTA per SM for a whole thread's latency; 28 warps per SM make it 7.9 waves.  Same-box A/B at 2^20 envs, 2000 steps (r02): 256 x 3 1.940e10
// env-steps/s, 160 x 5 1.977, 224 x 4 2.014, 64 x 14 2.016, 128 x 7 2.02-2.05, 32 x 28 2.03; 64 registers (128 x 8, 96 x 10) 1.96-1.97.
// The configuration training and the bench run (full DR, stats off) launches an instance specialised on it (PlanFullDr, usv_step_core.cuh):
// discrete parameters fixed at compile time, five unrolled sub-steps, Philox round keys from the host; same arithmetic, 72 registers, no
// spill.  B200 (1000 W), 2^20 envs: 46.7-46.9 -> 43.2-43.4 us per step; 2^19 -10 %, 2^21 -6 % (profiles/r05_step_plan.md).
#include "usv_step_core.cuh"

namespace usv {

constexpr int kBlock = 128, kMinB = 7;   // threads per CTA, CTAs per SM (see above)
// The fused step streams its one-pass data when the bytes the next step reads again fit in this share of L2 (see step_fused_kernel;
// measured on a B200: gains at 0.5 of L2, losses at 1.0)
constexpr double kResidentL2Share = 0.75;

// Variant A (classic CaptureXY) task part of a control step: observation (13), reward + penalties, kills / done
// `what` (USV_TASK_* bits) selects which of the reference's four calls advance their cross-step state: compute_reward owns the goal
// counter and prev_position_dist, compute_penalty owns prev_state / prev_actions; the fused step passes the literal "all" (folded away)
template <class Plan = PlanGeneric>
__device__ __forceinline__ void post_classic(EnvState& e, const EnvConst& k, const UsvStepParams& p, bool do_reset,
                                             bool first_call, const DynOut& s, StepOut& o, const int what = USV_CXY_ALL) {
  const float pxn = s.pxn, pyn = s.pyn, vxn = s.vxn, vyn = s.vyn, wn = s.wn, yawn = s.yawn, hs = s.hs, hc = s.hc;
  const float pa0 = s.pa0, pa1 = s.pa1;
  // get_state_observations  [ref SNAP/USV_capture_xy.py:80-97]
  const float ex = k.tx - pxn, ey = k.ty - pyn;
  const float theta = wrap_pi(yawn);  // == atan2(sin, cos) up to rounding, same (-pi,pi] branch
  const float beta = fast_atan2(ey, ex);
  // torch.fmod(x, 2pi) has C semantics (sign of the dividend).  beta, theta in [-pi, pi] -> x in [-pi, 3pi]:
  // fmod only acts for x >= 2pi, where x - 2pi is exact; negative x stays unwrapped (reference quirk).
  const float xa = beta - theta + USV_PI_F;
  const float alpha = ((xa >= USV_2PI_F) ? xa - USV_2PI_F : xa) - USV_PI_F;
  const float herr = fabsf(alpha);
  const float d = sqrtf(ex * ex + ey * ey);
  // (cos, sin)(alpha) = (cos, sin)(beta - theta) from the unit vectors e/|e| and (hc, hs): no trigonometric call
  // (shifts by 2pi leave them unchanged); beta = atan2(0, 0) = 0 for a zero error vector
  const float inv_d = (d > 0.0f) ? __fdividef(1.0f, d) : 0.0f;
  const float cb = (d > 0.0f) ? ex * inv_d : 1.0f, sb = ey * inv_d;
  const float ca = cb * hc + sb * hs, sa = sb * hc - cb * hs;
  // Core.update_observation_tensor, "local" frame  [ref SNAP/USV_core.py:41-54]
  o.obs[0] = hc * vxn + hs * vyn;
  o.obs[1] = -hs * vxn + hc * vyn;
  o.obs[2] = wn;
  o.obs[3] = ca;
  o.obs[4] = sa;
  o.obs[5] = d;
  o.obs[6] = vxn;
  o.obs[7] = vyn;
  o.obs[8] = 0.0f;
  o.obs[9] = vxn;
  o.obs[10] = vyn;
  o.obs[11] = 0.0f;
  o.obs[12] = 0.0f;
  // compute_reward  [ref SNAP/USV_capture_xy.py:101-227 ; SNAP/USV_task_rewards.py:40-76]
  const float speed = sqrtf(vxn * vxn + vyn * vyn);
  const int goal = (d < p.position_tolerance) && (speed < p.goal_speed_gate);
  if (what & USV_CXY_REWARD) e.goal_cnt = e.goal_cnt * goal + goal;
  float dist_rew;   // products rounded on their own as in penalty_scalar
  if (plan_or<Plan::reward_mode>(p.reward_mode) == USV_REWARD_LINEAR) {
    dist_rew = __fmul_rn(p.position_scale, e.prev_d - d);
  } else if (plan_or<Plan::reward_mode>(p.reward_mode) == USV_REWARD_SQUARE) {
    dist_rew = __fmul_rn(p.position_scale, e.prev_d * e.prev_d - d * d);
  } else {
    dist_rew = __fmul_rn(p.position_scale, expf(-d / p.exponential_reward_coeff) - expf(-e.prev_d / p.exponential_reward_coeff));
  }
  const float h2 = herr * herr;
  const float align = p.align_la1 * (__expf(p.align_la2 * (h2 * h2)) + __expf(p.align_la3 * h2));
  if (do_reset) dist_rew = 0.0f;  // distance_reward[just_had_been_reset] = 0
  float speed_rew;
  const float sclamp = 1.0f - fminf(fmaxf(speed / 1.0f, 0.0f), 1.0f);
  if (d > 3.5f) {
    const bool in_range = (speed >= 0.8f) && (speed <= 1.5f);
    const float ds = speed - 1.15f;
    speed_rew = in_range ? 0.1f : __expf(-(ds * ds) * 5.0f) * 0.1f;
  } else if (d > 2.5f) {
    speed_rew = sclamp * 0.15f;
  } else if (d > 1.5f) {
    speed_rew = sclamp * 0.25f;
  } else {
    speed_rew = sclamp * 0.35f;
  }
  if (!(d == d)) speed_rew = 0.0f;  // NaN distance matches no mask in the reference -> zeros_like
  const float goal_rew = (float)e.goal_cnt * p.goal_reward;
  const float task_rew = dist_rew + align + speed_rew + goal_rew + p.time_reward;
  if (what & USV_CXY_REWARD) e.prev_d = d;
  // Penalties.compute_penalty  [ref SNAP/USV_task_rewards.py:422-506]
  const float asum = pa0 + pa1;
  const float dw = first_call ? 0.0f : (wn - e.prev_w);
  const float dasum = first_call ? 0.0f : (asum - e.prev_asum);
  float pen_lin = 0.0f, pen_ang = 0.0f, pen_angvar = 0.0f, pen_energy = 0.0f, pen_actvar = 0.0f;
  if (plan_or<Plan::pen_linear_vel>(p.pen_linear_vel.form) != USV_PEN_OFF)
    pen_lin = penalty_scalar<Plan::pen_linear_vel>(p.pen_linear_vel, speed);
  if (plan_or<Plan::pen_angular_vel>(p.pen_angular_vel.form) != USV_PEN_OFF)
    pen_ang = penalty_scalar<Plan::pen_angular_vel>(p.pen_angular_vel, wn);
  if (plan_or<Plan::pen_angular_vel_variation>(p.pen_angular_vel_variation.form) != USV_PEN_OFF)
    pen_angvar = penalty_scalar<Plan::pen_angular_vel_variation>(p.pen_angular_vel_variation, dw);
  if (plan_or<Plan::pen_energy>(p.pen_energy.form) == USV_PEN_NEG_SUM) pen_energy = -(pa0 + pa1) * p.pen_energy.c1 + p.pen_energy.c2;
  else if (plan_or<Plan::pen_energy>(p.pen_energy.form) == USV_PEN_EXP_NEG_SUMSQ) pen_energy = __fmul_rn(__expf(-(pa0 * pa0 + pa1 * pa1)) - 1.0f, p.pen_energy.c1);
  if (plan_or<Plan::pen_action_variation>(p.pen_action_variation.form) != USV_PEN_OFF)
    pen_actvar = penalty_scalar<Plan::pen_action_variation>(p.pen_action_variation, dasum);
  const float penalties = pen_lin + pen_ang + pen_angvar + pen_energy + pen_actvar;
  if (what & USV_CXY_PENALTY) {
    e.prev_w = wn;
    e.prev_asum = asum;
  }
  o.task_rew = task_rew;
  o.penalty = penalties;
  o.rew = task_rew + penalties;  // [ref SNAP/USV_Virtual.py:844]
  // update_kills + is_done  [ref SNAP/USV_capture_xy.py:231-275 ; SNAP/USV_Virtual.py:855-866]
  int die = (d > p.kill_dist) ? 1 : 0;
  if ((e.goal_cnt >= p.kill_after_n_steps_in_tolerance) && (speed < p.goal_speed_gate)) die = 1;
  o.die = die;
  o.done = (e.progress >= p.max_episode_length - 1) ? 1 : die;
  // diagnostics
  o.dist_rew = dist_rew; o.align_rew = align; o.speed_rew = speed_rew; o.d = d; o.speed = speed;
  o.bdist = d - p.kill_dist;
  o.bpen = -expf(-o.bdist / 0.25f) * p.boundary_cost;
  o.pen_lin = pen_lin; o.pen_ang = pen_ang; o.pen_angvar = pen_angvar; o.pen_energy = pen_energy; o.pen_actvar = pen_actvar;
  o.absw = fabsf(wn); o.asum = asum;
  // NaN probe on the un-clamped obs and the reward [ref vec_env_rlgames.py:187-192]: x*0 is 0 for finite x, NaN otherwise
  float chk = o.rew * 0.0f;
#pragma unroll
  for (int j = 0; j < kObs; ++j) chk = fmaf(o.obs[j], 0.0f, chk);
  o.finite = (chk == 0.0f);
  // _process_data: clamp obs to +-clipObservations  [ref vec_env_rlgames.py:82-95]
#pragma unroll
  for (int j = 0; j < kObs; ++j)
    if (j != 8 && j != 11 && j != 12) o.obs[j] = fminf(fmaxf(o.obs[j], -p.clip_obs), p.clip_obs);   // 8, 11, 12 are constant zeros
}

// one full control step for one env, state in registers
template <int kDisturb, bool kLutGlobal, class Plan = PlanGeneric>
__device__ __forceinline__ void control_step(EnvState& e, EnvConst& k, const UsvStepParams& p, bool do_reset,
                                             float2 act, uint64_t gid, int64_t lid, uint64_t step, bool first_call,
                                             const float* __restrict__ s_lutL, const float* __restrict__ s_lutR,
                                             StepOut& o, const PhiloxKeys* keys = nullptr) {
  DynOut s;
  step_dynamics<kDisturb, kLutGlobal, Plan>(e, k, p, do_reset, act, gid, lid, step, s_lutL, s_lutR, s, keys);
  post_classic<Plan>(e, k, p, do_reset, first_call, s, o);
}

__device__ __forceinline__ void accumulate_stats(float* __restrict__ st0, int64_t i0, bool was_reset,
                                                 const StepOut& o, const UsvStepParams& p) {
  float* __restrict__ st = st0 + tile_base(i0, USV_ST_COUNT);
  // episode_sums[k][i] += term  [ref SNAP/USV_capture_xy.py:278-306 ; SNAP/USV_task_rewards.py:526-540 ;
  // SNAP/USV_Virtual.py:819-830]; sums are cleared by the reset that precedes this step.
  const float v[USV_ST_COUNT] = {o.dist_rew, o.align_rew, o.speed_rew, o.d, o.speed, o.bpen, o.bdist,
                                 o.pen_lin, o.pen_ang, o.pen_angvar, o.pen_energy, o.pen_actvar,
                                 o.speed, o.absw, o.asum};
#pragma unroll
  for (int f = 0; f < USV_ST_COUNT; ++f) {
    const float prev = was_reset ? 0.0f : st[f * kTile];
    st[f * kTile] = prev + v[f];
  }
}


// Each WARP stages its own 32 x 13 observation tile in smem (stride 13 is odd -> conflict-free) and writes it
// out as one contiguous 1664 B run of float4 lines: only a __syncwarp, no CTA barrier on the store path.
template <Cache C = Cache::kNormal>
__device__ __forceinline__ void write_obs_tile(float* s_obs, const StepOut& o, bool active, float* __restrict__ obs,
                                               int64_t block_start, int64_t n) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* sw = s_obs + warp * (32 * kObs);
  if (active) {
#pragma unroll
    for (int j = 0; j < kObs; ++j) sw[lane * kObs + j] = o.obs[j];
  }
  __syncwarp();
  const int64_t warp_start = block_start + (int64_t)warp * 32;
  if (warp_start >= n) return;
  const int rows = (int)min((int64_t)32, n - warp_start);
  const int total = rows * kObs;
  float* g = obs + warp_start * kObs;
  if (rows == 32 && (((uintptr_t)g & 15) == 0)) {
    const float4* s4 = reinterpret_cast<const float4*>(sw);
    float4* g4 = reinterpret_cast<float4*>(g);
#pragma unroll
    for (int q = lane; q < (32 * kObs) / 4; q += 32) st<C>(g4 + q, s4[q]);
  } else {
    for (int q = lane; q < total; q += 32) st<C>(g + q, sw[q]);
  }
  __syncwarp();
}

// One control step per launch.  Between launches the env state (52 B), reset_buf (8 B) and, with kStats, the episode sums (60 B) are
// the only bytes the next launch reads again: they always take plain accesses.  kOnePass is the L2 policy of the rest -- per-episode
// constants, actions, obs and reward, read or written once per step.  Evict-first (kStream) keeps those lines from pushing the
// re-read set out of L2, which pays while that set fits; once it does not, evict-first is slower than plain accesses (B200, r03:
// +6 % / +9 % env-steps/s at 2^19 / 2^20 envs, -2 % at 2^21; with stats +27 % at 2^19, -3 % at 2^20), so the launch picks kStream only
// when the re-read set fits in a fraction of L2 (kResidentL2Share).  The thruster LUTs keep the read-only path (L1).
//
// Programmatic dependent launch (launch_pdl): the launch may start while the previous kernel of the stream still runs, so NO
// global-memory read or write may come before pdl_wait() -- that kernel may be the previous step (state, reset_buf), a policy
// forward still reading obs, or a torch op still writing the actions or the state.  Only parameters and index arithmetic come first.
// Each CTA lets the next step launch at entry: its CTAs can then only start once this launch's last wave is resident, so they never
// take slots from this launch's own CTAs; they wait for its completion in place, which hides the launch and CTA ramp-up between steps.
//
// Plan (usv_step_core.cuh) fixes the discrete parameters at compile time; `keys` are the Philox round keys of p.seed, read only by a
// fixed plan.
template <int kDisturb, bool kStats, Cache kOnePass, class Plan = PlanGeneric>
__global__ void __launch_bounds__(kBlock, kMinB) step_fused_kernel(UsvEnvBuffers b, const float2* __restrict__ actions,
                                                            float* __restrict__ obs, float* __restrict__ rew,
                                                            int64_t n, const __grid_constant__ UsvStepParams p,
                                                            const __grid_constant__ PhiloxKeys keys) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float smem[];
  float* s_obs = smem;                       // [kBlock*13]
  // The two 4 KB thruster LUTs are gathered at 2 random indices per env-step.  Staging them per CTA cost 16 LDG+STS
  // per thread plus a CTA barrier in this one-tile-per-CTA kernel (r01 profile); the read-only path keeps the 8 KB
  // resident in L1 instead.  (The multi-step rollout kernel, whose CTAs live for T steps, does stage them in smem.)
  const float* __restrict__ s_lutL = b.lut_left;
  const float* __restrict__ s_lutR = b.lut_right;
  const int64_t block_start = (int64_t)blockIdx.x * kBlock;
  const int64_t i = block_start + threadIdx.x;
  const bool active = i < n;
  EnvState e;
  EnvConst k;
  bool do_reset = false;
  float2 act = make_float2(0.f, 0.f);
  if (active) {
    load_state(b.state, i, e);
    load_consts<kDisturb, kOnePass>(b.consts, i, k);
    do_reset = b.reset_buf[i] != 0;
    act = ld<kOnePass>(actions + i);
  }
  StepOut o;
  if (active) {
    control_step<kDisturb, true, Plan>(e, k, p, do_reset, act, (uint64_t)(p.env_id_offset + i), i,
                                       p.step_counter + (b.step_offset ? *b.step_offset : 0ull), p.first_call != 0, s_lutL, s_lutR, o,
                                       &keys);
    store_state(b.state, i, e);
    if (do_reset) store_consts<kDisturb, kOnePass>(b.consts, i, k);
    if (kStats) accumulate_stats(b.stats, i, do_reset, o, p);
    st<kOnePass>(rew + i, o.rew);
    b.reset_buf[i] = (int64_t)o.done;
    if (b.nonfinite_flag) {
      if (!o.finite) atomicOr(b.nonfinite_flag, 1u);
      // torch.clamp propagates NaN actions and the reference fails fast on them [ref: vec_env_rlgames.py:143];
      // fminf/fmaxf would silently scrub them, so flag them here
      if (!isfinite(act.x) || !isfinite(act.y)) atomicOr(b.nonfinite_flag, 2u);
    }
  }
  write_obs_tile<kOnePass>(s_obs, o, active, obs, block_start, n);
}

// T control steps per launch, state in registers between steps.
template <int kDisturb, bool kStats>
__global__ void __launch_bounds__(kBlock) rollout_fused_kernel(UsvEnvBuffers b, const float2* __restrict__ actions,
                                                               float* __restrict__ obs, float* __restrict__ rew,
                                                               int64_t* __restrict__ done, int T, int64_t n,
                                                               const __grid_constant__ UsvStepParams p) {
  extern __shared__ __align__(16) float smem[];
  float* s_obs = smem;
  float* s_lutL = smem + kBlock * kObs;
  float* s_lutR = s_lutL + p.n_lut;
  for (int t = threadIdx.x; t < p.n_lut; t += kBlock) {
    s_lutL[t] = b.lut_left[t];
    s_lutR[t] = b.lut_right[t];
  }
  const int64_t block_start = (int64_t)blockIdx.x * kBlock;
  const int64_t i = block_start + threadIdx.x;
  const bool active = i < n;
  EnvState e;
  EnvConst k;
  bool do_reset = false;
  bool consts_dirty = false;
  if (active) {
    load_state(b.state, i, e);
    load_consts<kDisturb>(b.consts, i, k);
    do_reset = b.reset_buf[i] != 0;
  }
  __syncthreads();
  bool first_call = p.first_call != 0;
  bool bad = false;
  const uint64_t step0 = p.step_counter + (b.step_offset ? *b.step_offset : 0ull);
  for (int t = 0; t < T; ++t) {
    StepOut o;
    if (active) {
      const float2 act = actions[(int64_t)t * n + i];
      control_step<kDisturb, false>(e, k, p, do_reset, act, (uint64_t)(p.env_id_offset + i), i, step0 + (uint64_t)t,
                             first_call, s_lutL, s_lutR, o);
      consts_dirty |= do_reset;
      if (kStats) accumulate_stats(b.stats, i, do_reset, o, p);
      if (rew) rew[(int64_t)t * n + i] = o.rew;
      if (done) done[(int64_t)t * n + i] = (int64_t)o.done;
      bad |= !o.finite || !isfinite(act.x) || !isfinite(act.y);
      do_reset = o.done != 0;
    }
    first_call = false;
    if (obs) {
      write_obs_tile(s_obs, o, active, obs + (int64_t)t * n * kObs, block_start, n);
    }
  }
  if (active) {
    store_state(b.state, i, e);
    if (consts_dirty) store_consts<kDisturb>(b.consts, i, k);
    b.reset_buf[i] = do_reset ? 1 : 0;
    if (b.nonfinite_flag && bad) atomicOr(b.nonfinite_flag, 1u);
  }
}

template <int kDisturb>
__global__ void __launch_bounds__(kBlock) planar_forces_kernel(UsvEnvBuffers b, float* __restrict__ out, int64_t n,
                                                               const __grid_constant__ UsvStepParams p) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  EnvState e;
  EnvConst k;
  load_state(b.state, i, e);
  load_consts<kDisturb>(b.consts, i, k);
  float ox = 0.0f, oy = 0.0f;
  if (kDisturb && p.envs_per_row > 0) {
    ox = p.grid_row_offset - (float)(int)(i / p.envs_per_row) * p.env_spacing;
    oy = (float)(int)(i % p.envs_per_row) * p.env_spacing - p.grid_col_offset;
  }
  float du, dv, dr, Fx, Fy, Tz, ax, ay, rdot, hsn, hcs;
  fsincos(e.psi, &hsn, &hcs);
  planar_wrench<kDisturb>(e, k, p, make_damp(k, p), ox, oy, 1.0f / k.mass, 1.0f / (p.izz * k.kiz), hsn, hcs, du, dv, dr, Fx, Fy, Tz, ax, ay, rdot);
  float* o = out + i * 8;
  o[0] = du; o[1] = dv; o[2] = dr; o[3] = Fx; o[4] = Fy; o[5] = Tz; o[6] = ax; o[7] = ay;
}

static size_t step_smem(const UsvStepParams* p) { return (size_t)(kBlock * kObs + 2 * p->n_lut) * sizeof(float); }
static size_t step_smem_nolut() { return (size_t)(kBlock * kObs) * sizeof(float); }

// CaptureXYTask.get_state_observations / compute_reward / update_kills and Penalties.compute_penalty on the caller's own state tensors:
// the SAME device code as the task part of the fused step (post_classic), one env per thread, plain row-major inputs.
__global__ void __launch_bounds__(256) capturexy_task_kernel(UsvCaptureXYIO io, int64_t n, UsvStepParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float2 z2 = make_float2(0.f, 0.f);
  const float2 pos = io.position ? reinterpret_cast<const float2*>(io.position)[i] : z2;
  const float2 hd = io.heading ? reinterpret_cast<const float2*>(io.heading)[i] : make_float2(1.f, 0.f);
  const float2 vel = io.linear_velocity ? reinterpret_cast<const float2*>(io.linear_velocity)[i] : z2;
  const float2 act = io.actions ? reinterpret_cast<const float2*>(io.actions)[i] : z2;
  const float2 tgt = io.target ? reinterpret_cast<const float2*>(io.target)[i] : z2;
  DynOut s;
  s.pxn = pos.x; s.pyn = pos.y; s.vxn = vel.x; s.vyn = vel.y;
  s.wn = io.angular_velocity ? io.angular_velocity[i] : 0.f;
  s.hc = hd.x; s.hs = hd.y;
  s.yawn = fast_atan2(hd.y, hd.x);          // theta = atan2(orientation[:,1], orientation[:,0])  [ref SNAP/USV_capture_xy.py:88]
  s.pa0 = act.x; s.pa1 = act.y;
  s.raw0 = s.raw1 = s.t0 = s.t1 = s.c0 = s.c1 = 0.f;
  EnvState e;
  e.x = pos.x; e.y = pos.y; e.psi = s.yawn; e.vx = vel.x; e.vy = vel.y; e.r = s.wn; e.thrL = e.thrR = 0.f;
  e.progress = 0;
  e.goal_cnt = io.goal_reached ? io.goal_reached[i] : 0;
  const bool jr = io.just_reset ? io.just_reset[i] != 0 : false;
  EnvConst k;
  k.tx = tgt.x; k.ty = tgt.y;
  // prev_position_dist is None on the first compute_reward: it becomes the current distance (a zero progress term)
  if (io.first_reward || !io.prev_position_dist) {
    const float ex = tgt.x - pos.x, ey = tgt.y - pos.y;
    e.prev_d = sqrtf(ex * ex + ey * ey);
  } else {
    e.prev_d = io.prev_position_dist[i];
  }
  e.prev_w = io.prev_angular_velocity ? io.prev_angular_velocity[i] : 0.f;
  e.prev_asum = io.prev_action_sum ? io.prev_action_sum[i] : 0.f;
  p.kill_dist = io.kill_dist;                // curriculum-resolved by the caller, like update_kills(step)
  p.max_episode_length = 0x7fffffff;
  StepOut o;
  post_classic(e, k, p, jr, io.first_penalty != 0, s, o, io.what);
  if ((io.what & USV_CXY_OBS) && io.obs) {
#pragma unroll
    for (int j = 0; j < kObs; ++j) io.obs[i * kObs + j] = o.obs[j];
  }
  if (io.what & USV_CXY_REWARD) {
    if (io.reward) io.reward[i] = o.task_rew;
    if (io.reward_terms) { io.reward_terms[i * 3] = o.dist_rew; io.reward_terms[i * 3 + 1] = o.align_rew; io.reward_terms[i * 3 + 2] = o.speed_rew; }
    if (io.goal_reached) io.goal_reached[i] = e.goal_cnt;
    if (io.prev_position_dist) io.prev_position_dist[i] = e.prev_d;
  }
  if (io.what & USV_CXY_PENALTY) {
    if (io.penalty) io.penalty[i] = o.penalty;
    if (io.penalty_terms) {
      io.penalty_terms[i * 5] = o.pen_lin; io.penalty_terms[i * 5 + 1] = o.pen_ang; io.penalty_terms[i * 5 + 2] = o.pen_angvar;
      io.penalty_terms[i * 5 + 3] = o.pen_energy; io.penalty_terms[i * 5 + 4] = o.pen_actvar;
    }
    if (io.prev_angular_velocity) io.prev_angular_velocity[i] = e.prev_w;
    if (io.prev_action_sum) io.prev_action_sum[i] = e.prev_asum;
  }
  if ((io.what & USV_CXY_KILLS) && io.die) io.die[i] = o.die;
}

}  // namespace usv

using namespace usv;

extern "C" {

int usv_capturexy_obs_reward_done_f32(const UsvCaptureXYIO* io, int64_t n, const UsvStepParams* p, void* stream) {
  if (!io || !p) return USV_E_NULL;
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!(io->what & USV_CXY_ALL) || (io->what & ~USV_CXY_ALL)) return USV_E_PARAM;
  if (!io->position || !io->target || !io->linear_velocity) return USV_E_NULL;          // every call needs the distance and the speed
  if ((io->what & USV_CXY_OBS) && (!io->obs || !io->heading || !io->angular_velocity)) return USV_E_NULL;
  if ((io->what & USV_CXY_REWARD) && (!io->reward || !io->heading || !io->goal_reached)) return USV_E_NULL;
  if ((io->what & USV_CXY_PENALTY) && (!io->penalty || !io->actions || !io->angular_velocity)) return USV_E_NULL;
  if ((io->what & USV_CXY_KILLS) && (!io->die || !io->goal_reached)) return USV_E_NULL;
  const uintptr_t al = (uintptr_t)io->position | (uintptr_t)io->target | (uintptr_t)io->linear_velocity | (uintptr_t)io->heading |
                       (uintptr_t)io->actions;
  if (al & 7) return USV_E_ALIGN;
  capturexy_task_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(*io, n, *p);
  return finish_launch();
}

int usv_step_fused_plan(const UsvStepParams* p, int32_t stats) {
  if (!p) return USV_E_NULL;
  return !stats && plan_matches<PlanFullDr>(*p) ? USV_STEP_PLAN_FULL_DR : USV_STEP_PLAN_GENERIC;
}

int usv_step_fused_f32(const UsvEnvBuffers* b, const float* actions, float* obs, float* rew, int64_t n,
                       const UsvStepParams* p, void* stream) {
  int rc = check_common(b, n, p);
  if (rc) return rc;
  if (n == 0) return USV_OK;
  if (!actions || !obs || !rew) return USV_E_NULL;
  if ((uintptr_t)actions & 7) return USV_E_ALIGN;
  const size_t smem = step_smem_nolut();
  const int grid = grid_for(n, kBlock);
  const bool dis = wants_disturb(p), st = b->stats != nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  // bytes per env the next step reads again (state, reset_buf, episode sums): see step_fused_kernel
  const double reread = (double)n * (USV_S_COUNT * 4 + 8 + (st ? USV_ST_COUNT * 4 : 0));
  const bool one_pass_cs = reread <= kResidentL2Share * l2_bytes();
  const PhiloxKeys keys = philox_round_keys(p->seed);
#define USV_LAUNCH_STEP(D, S, P)                                                                                                    \
  do {                                                                                                                              \
    auto* kern = one_pass_cs ? step_fused_kernel<D, S, Cache::kStream, P> : step_fused_kernel<D, S, Cache::kNormal, P>;             \
    ensure_dynamic_smem(kern, smem);                                                                                                \
    launch_pdl(kern, dim3(grid), dim3(kBlock), smem, s, *b, (const float2*)actions, obs, rew, n, *p, keys);                         \
  } while (0)
  const bool all4 = p->use_const_force && p->use_sin_force && p->use_const_torque && p->use_sin_torque && !p->use_water_current;
  if (usv_step_fused_plan(p, st) == USV_STEP_PLAN_FULL_DR) USV_LAUNCH_STEP(2, false, PlanFullDr);
  else if (dis && all4 && !st) USV_LAUNCH_STEP(2, false, PlanGeneric);
  else if (dis && st) USV_LAUNCH_STEP(1, true, PlanGeneric);
  else if (dis) USV_LAUNCH_STEP(1, false, PlanGeneric);
  else if (st) USV_LAUNCH_STEP(0, true, PlanGeneric);
  else USV_LAUNCH_STEP(0, false, PlanGeneric);
#undef USV_LAUNCH_STEP
  return finish_launch();
}

int usv_rollout_fused_f32(const UsvEnvBuffers* b, const float* actions, float* obs, float* rew, int64_t* done,
                          int32_t T, int64_t n, const UsvStepParams* p, void* stream) {
  int rc = check_common(b, n, p);
  if (rc) return rc;
  if (T < 0) return USV_E_SIZE;
  if (n == 0 || T == 0) return USV_OK;
  if (!actions) return USV_E_NULL;
  if ((uintptr_t)actions & 7) return USV_E_ALIGN;
  const size_t smem = step_smem(p);
  const int grid = grid_for(n, kBlock);
  const bool dis = wants_disturb(p), st = b->stats != nullptr;
  cudaStream_t s = (cudaStream_t)stream;
#define USV_LAUNCH_ROLL(D, S)                                                                              \
  do {                                                                                                     \
    ensure_dynamic_smem(rollout_fused_kernel<D, S>, smem);                                                 \
    rollout_fused_kernel<D, S><<<grid, kBlock, smem, s>>>(*b, (const float2*)actions, obs, rew, done, T, n, *p); \
  } while (0)
  if (dis && st) USV_LAUNCH_ROLL(true, true);
  else if (dis) USV_LAUNCH_ROLL(true, false);
  else if (st) USV_LAUNCH_ROLL(false, true);
  else USV_LAUNCH_ROLL(false, false);
#undef USV_LAUNCH_ROLL
  return finish_launch();
}

int usv_planar_forces_f32(const UsvEnvBuffers* b, float* out, int64_t n, const UsvStepParams* p, void* stream) {
  int rc = check_common(b, n, p);
  if (rc) return rc;
  if (n == 0) return USV_OK;
  if (!out) return USV_E_NULL;
  const int grid = grid_for(n, kBlock);
  if (wants_disturb(p))
    planar_forces_kernel<true><<<grid, kBlock, 0, (cudaStream_t)stream>>>(*b, out, n, *p);
  else
    planar_forces_kernel<false><<<grid, kBlock, 0, (cudaStream_t)stream>>>(*b, out, n, *p);
  return finish_launch();
}

}  // extern "C"
