// Fused env step of the LIVE CaptureXY task (Variant B): the same action -> thruster -> n_substeps x {lag, damping,
// disturbances, planar integrator} front half as usv_step.cu, followed by the obstacle task  [ref: OIGE/tasks/USV/
// USV_capture_xy_static_obs.py]: 33-dim observation (goal bearing, the 5 nearest of 16 obstacles in the body frame,
// previous action, privileged tail), bilinear potential-field sample, 10-term shaped reward, collision / goal / distance
// kills and the per-episode outcome latches.  One launch per control step; obstacles + potential fields of the envs that
// reset are rebuilt beforehand by usv_reset_b.cu.
//
// HBM traffic per env-step (stats off, no disturbances): state 13+3 fields r/w (128 B), consts 13+35 fields (192 B), 4 field
// taps (<= 4 x 32 B sectors), obs 132 B, action 8 B, reward 4 B, reset_buf 16 B  ->  ~610 B.
#include "usv_step_core.cuh"

namespace usv {

constexpr int kBlock = 256;   // threads per CTA; CTAs per SM are the kernels' kMinB / __launch_bounds__ arguments
constexpr int kObsB = USV_B_OBS;
constexpr int kGridB = USV_B_GRID;

struct LiveState {
  float prev_h, prev_pot;
  int outcome;
};

struct LiveOut {
  float* sw;     // this lane's row of the warp's shared-memory observation tile (stride 33: conflict-free)
  float chk;     // NaN probe accumulator: x*0 is 0 for finite x, NaN otherwise
  float clip;
  // observations go straight to the staging tile, clamped, as they are produced: holding all 33 in registers until the end
  // cost ~30 registers (113 -> 2 CTAs/SM in the r01 profile)
  __device__ __forceinline__ void put(int j, float v) {
    chk = fmaf(v, 0.0f, chk);
    sw[j] = fminf(fmaxf(v, -clip), clip);
  }
  float rew;
  int done;
  bool finite;
  float st[USV_BST_COUNT];
};

__device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }

// F.grid_sample(field[1,1,H,W], (2*pos/map)[1,1,1,2], bilinear, align_corners=False, padding_mode='border')
// [ref USV_capture_xy_static_obs.py:302-326]; explicit rounding per op: the shaping term multiplies differences of this by 100
__device__ __forceinline__ float sample_potential(const float* __restrict__ f, float px, float py, float map_size) {
  const float W = (float)kGridB;
  const float gx = __fdiv_rn(__fmul_rn(2.0f, px), map_size), gy = __fdiv_rn(__fmul_rn(2.0f, py), map_size);
  float ix = __fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gx, 1.0f), W), 1.0f), 2.0f);
  float iy = __fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gy, 1.0f), W), 1.0f), 2.0f);
  ix = fminf(fmaxf(ix, 0.0f), W - 1.0f);
  iy = fminf(fmaxf(iy, 0.0f), W - 1.0f);
  const float x0f = floorf(ix), y0f = floorf(iy);
  const float wx1 = __fsub_rn(ix, x0f), wy1 = __fsub_rn(iy, y0f);
  const float wx0 = __fsub_rn(1.0f, wx1), wy0 = __fsub_rn(1.0f, wy1);
  const int x0 = (int)x0f, y0 = (int)y0f;
  // the +1 taps fall outside only when ix (iy) sits exactly on the last cell: they contribute 0 there
  const bool xin = x0 + 1 <= kGridB - 1, yin = y0 + 1 <= kGridB - 1;
  const int x1 = xin ? x0 + 1 : x0, y1 = yin ? y0 + 1 : y0;
  const float t00 = __ldg(f + y0 * kGridB + x0);
  const float t01 = xin ? __ldg(f + y0 * kGridB + x1) : 0.0f;
  const float t10 = yin ? __ldg(f + y1 * kGridB + x0) : 0.0f;
  const float t11 = (xin && yin) ? __ldg(f + y1 * kGridB + x1) : 0.0f;
  float acc = __fmul_rn(__fmul_rn(t00, wx0), wy0);
  acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(t01, wx1), wy0));
  acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(t10, wx0), wy1));
  acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(t11, wx1), wy1));
  return acc;
}

__device__ __forceinline__ float priv_encode(const UsvLiveParams& lp, int j, float x) {
  if (lp.priv_mode == USV_PRIV_RAW) return x;
  if (lp.priv_mode == USV_PRIV_CENTERED) return fminf(fmaxf(__fdiv_rn(x - lp.priv_a[j], lp.priv_b[j]), -1.0f), 1.0f);
  if (!lp.priv_active[j]) return 0.0f;
  const float z = __fdiv_rn(x - lp.priv_a[j], lp.priv_b[j]);
  return fminf(fmaxf(__fsub_rn(__fmul_rn(2.0f, z), 1.0f), -1.0f), 1.0f);
}

// Core.update_observation_tensor, "local" frame  [ref OIGE/tasks/USV/USV_core.py:55-125]: obs[0:3] body-frame velocity + yaw rate
__device__ __forceinline__ void obs_head(LiveOut& o, const DynOut& s) {
  o.put(0, s.hc * s.vxn + s.hs * s.vyn);
  o.put(1, -s.hs * s.vxn + s.hc * s.vyn);
  o.put(2, s.wn);
}
// obs[23:25] previous action, obs[25:33] privileged tail
__device__ __forceinline__ void obs_tail(LiveOut& o, const DynOut& s, const EnvConst& k, const float* __restrict__ bc,
                                         const UsvStepParams& p, const UsvLiveParams& lp, bool do_reset) {
  // prev_thrust_cmds: the raw policy command of THIS control step, zero for an env reset in it (USV_Virtual.py:1063-1066)
  o.put(23, do_reset ? 0.0f : s.raw0);
  o.put(24, do_reset ? 0.0f : s.raw1);
  // privileged tail  (USV_Virtual.py:837-984); `base`: the ablation source shows base / neutral values (:840-880)
  const bool base = lp.masscom_obs_base != 0;
  const float m = base ? p.mass_base : k.mass;
  o.put(25, lp.mass_obs_relative ? (base ? 0.0f : __fdiv_rn(m - p.mass_base, fmaxf(fabsf(p.mass_base), 1e-6f))) : m);
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float c = base ? lp.com_base[j] : bc[(USV_BC_COM_X + j) * kTile];
    o.put(26 + j, lp.com_obs_scaled ? __fdiv_rn(c, lp.com_scale_eps[j]) : c);
  }
  o.put(29, priv_encode(lp, 0, base ? lp.priv_neutral[0] : k.kdrag));
  o.put(30, priv_encode(lp, 1, base ? lp.priv_neutral[1] : k.mL));
  o.put(31, priv_encode(lp, 2, base ? lp.priv_neutral[2] : k.mR));
  o.put(32, priv_encode(lp, 3, base ? lp.priv_neutral[3] : k.kiz));
}

// Variant B task part of a control step.  `any_reset`: some env of the batch was reset on entry to this control step
// (reference quirk: CaptureXYTask.reset sets prev_potential = None for EVERY env, :773, :448-452).
template <bool kStats>
__device__ __forceinline__ void post_live(EnvState& e, const EnvConst& k, LiveState& ls, const float* __restrict__ bc,
                                          const float* __restrict__ field, const UsvStepParams& p, const UsvLiveParams& lp,
                                          bool do_reset, bool any_reset, bool first_call, const DynOut& s, LiveOut& o) {
  const float pxn = s.pxn, pyn = s.pyn, vxn = s.vxn, vyn = s.vyn, wn = s.wn, hs = s.hs, hc = s.hc;
  if (do_reset) ls.outcome = 0;  // task.reset(): _done_success / _done_collision cleared  (:768-770)
  // ---- get_state_observations (:193-299) -------------------------------------------------------
  const float ex = k.tx - pxn, ey = k.ty - pyn;
  const float theta = wrap_pi(s.yawn);  // atan2(sin, cos) of the (noisy) heading
  const float beta = atan2f(ey, ex);
  const float xa = beta - theta + USV_PI_F;
  const float alpha = ((xa >= USV_2PI_F) ? xa - USV_2PI_F : xa) - USV_PI_F;  // torch.fmod: sign of the dividend
  const float herr = fabsf(alpha);
  float sa, ca;
  fsincos(alpha, &sa, &ca);
  // position_dist = sqrt(square(err).sum(-1)) for the reward; the observation carries torch.norm(err) = sqrt(fma(y, y, x*x))
  const float d = sqrtf(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
  const float d_obs = sqrtf(__fmaf_rn(ey, ey, __fmul_rn(ex, ex)));
  // 16 obstacle centres: the 5 nearest (ascending centre distance), collision count
  float bd[USV_B_CLOSEST], bx[USV_B_CLOSEST], by[USV_B_CLOSEST];
#pragma unroll
  for (int q = 0; q < USV_B_CLOSEST; ++q) { bd[q] = CUDART_INF_F; bx[q] = 0.0f; by[q] = 0.0f; }
  int ncoll = 0;
#pragma unroll
  for (int j = 0; j < USV_B_OBSTACLES; ++j) {
    const float dx = bc[(USV_BC_OBST + 2 * j) * kTile] - pxn;
    const float dy = bc[(USV_BC_OBST + 2 * j + 1) * kTile] - pyn;
    const float dist = sqrtf(__fmaf_rn(dy, dy, __fmul_rn(dx, dx)));  // torch.norm(rel, dim=-1)
    ncoll += (dist < lp.collision_threshold) ? 1 : 0;
    // insertion into the sorted 5-list; strict '<' keeps the lower index first among equal distances
    float cd = dist, cx = dx, cy = dy;
#pragma unroll
    for (int q = 0; q < USV_B_CLOSEST; ++q) {
      const bool lt = cd < bd[q];
      const float td_ = bd[q], tx_ = bx[q], ty_ = by[q];
      bd[q] = lt ? cd : td_; bx[q] = lt ? cx : tx_; by[q] = lt ? cy : ty_;
      cd = lt ? td_ : cd; cx = lt ? tx_ : cx; cy = lt ? ty_ : cy;
    }
  }
  // Core.update_observation_tensor  [ref OIGE/tasks/USV/USV_core.py:55-125]
  obs_head(o, s);
  o.put(3, ca);
  o.put(4, sa);
  o.put(5, d_obs);
  o.put(6, 0.0f);
  o.put(7, 0.0f);
#pragma unroll
  for (int q = 0; q < USV_B_CLOSEST; ++q) {
    const float xb = bx[q] * hc + by[q] * hs;
    const float yb = -bx[q] * hs + by[q] * hc;
    const float nf = sqrtf(xb * xb + yb * yb + 1e-6f);
    o.put(8 + 3 * q, bd[q] - 0.5f);
    o.put(9 + 3 * q, __fdiv_rn(-xb, nf));
    o.put(10 + 3 * q, __fdiv_rn(-yb, nf));
  }
  obs_tail(o, s, k, bc, p, lp, do_reset);

  // ---- compute_reward (:335-657) ----------------------------------------------------------------
  const int goal = (d < p.position_tolerance) ? 1 : 0;  // no speed gate in the live task
  e.goal_cnt = e.goal_cnt * goal + goal;
  float dist_rew = p.position_scale * (e.prev_d - d);
  const float h2 = herr * herr;
  float align = p.align_la1 * (expf(p.align_la2 * (h2 * h2)) + expf(p.align_la3 * h2));
  if (do_reset) dist_rew = 0.0f;
  const float prev_d = do_reset ? d : e.prev_d;  // prev_position_dist aligned for just-reset envs (:373-380)
  const float pot = sample_potential(field, pxn, pyn, lp.map_size);
  const float pn = clamp01(pot);
  const float xs = clamp01(__fdiv_rn(pn - 0.6f, 0.9f - 0.6f + 1e-6f));
  const float danger = xs * xs * (3.0f - 2.0f * xs);
  align = align * fmaxf(0.3f, 1.0f - danger);
  dist_rew = dist_rew * fmaxf(0.6f, 1.0f - danger * 0.5f);
  const float g = clamp01(ca);  // clamp(cos(heading_error), 0, 1); cos is even
  dist_rew = fminf(dist_rew, 0.0f) + g * fmaxf(dist_rew, 0.0f);
  const float prev_h = do_reset ? herr : ls.prev_h;
  const float h_imp_rew = fminf(fmaxf(prev_h - herr, -0.4f), 0.4f) * 0.05f;
  ls.prev_h = herr;
  const float prev_pot = (do_reset || any_reset) ? pot : ls.prev_pot;
  float praw = (prev_pot - pot) * 100.0f;
  praw = (fabsf(praw) < 0.01f) ? 0.0f : praw;
  const float pa1 = 2.0f * tanhf(__fdiv_rn(praw, 2.0f + 1e-6f));
  const float inv_gd = d + 1e-6f;
  const float gdx = __fdiv_rn(ex, inv_gd), gdy = __fdiv_rn(ey, inv_gd);
  const float v_toward = vxn * gdx + vyn * gdy;
  const float vtp = fmaxf(v_toward, 0.0f);
  const float dd_pos = fmaxf(prev_d - d, 0.0f);
  const float g_v = clamp01(__fdiv_rn(vtp - 0.02f, 0.15f - 0.02f + 1e-6f));
  const float g_d = clamp01(__fdiv_rn(dd_pos, 0.01f + 1e-6f));
  const float g_gate = fmaxf(g_v, g_d) * g;
  const float ppos = fmaxf(pa1, 0.0f), pneg = fminf(pa1, 0.0f);
  const float gate_pos = (ppos < 0.5f) ? 1.0f : g_gate;
  const float shaping = gate_pos * ppos + pneg;
  const bool worsening = shaping < -0.05f;
  const bool turning = fabsf(wn) > 0.2f;
  const float v_fwd = fabsf(vxn * hc + vyn * hs);
  const float speed_factor = clamp01(__fdiv_rn(v_fwd - 0.15f, 0.60f - 0.15f + 1e-6f));
  const float hazard = ((worsening && turning) ? 1.0f : 0.0f) * (-10.0f) * (g * g) * speed_factor;
  ls.prev_pot = pot;
  const float speed_rew = (1.0f - expf(-__fdiv_rn(vtp, 0.8f + 1e-6f))) * 0.05f;
  const float sgn = (alpha > 0.0f) ? 1.0f : ((alpha < 0.0f) ? -1.0f : 0.0f);
  const float tgt_w = (herr > 1.0f) ? sgn * 1.0f : sgn * 0.2f;
  const float dwv = wn - tgt_w;
  const float ang_rew = expf(-__fdiv_rn(dwv * dwv, 0.2f)) * 0.03f;
  const float coll = (float)ncoll * (-100.0f);
  const float goal_rew = ((float)e.goal_cnt * p.goal_reward) * 5.0f;
  e.prev_d = d;
  float total = dist_rew * 0.5f + align * 0.5f;
  total += shaping * 2.0f;
  total += hazard;
  total += goal_rew;
  total += p.time_reward;
  total += coll;
  total += speed_rew;
  total += ang_rew;
  total += h_imp_rew;
  // Penalties.compute_penalty  [ref OIGE/tasks/USV/USV_task_rewards.py Penalties; same closed set as the classic task]
  const float speed = sqrtf(vxn * vxn + vyn * vyn);
  const float pa0_ = s.pa0, pa1_ = s.pa1;
  const float asum = pa0_ + pa1_;
  const float dw = first_call ? 0.0f : (wn - e.prev_w);
  const float dasum = first_call ? 0.0f : (asum - e.prev_asum);
  float pen_lin = 0.0f, pen_ang = 0.0f, pen_angvar = 0.0f, pen_energy = 0.0f, pen_actvar = 0.0f;
  if (p.pen_linear_vel.form != USV_PEN_OFF) pen_lin = penalty_scalar(p.pen_linear_vel, speed);
  if (p.pen_angular_vel.form != USV_PEN_OFF) pen_ang = penalty_scalar(p.pen_angular_vel, wn);
  if (p.pen_angular_vel_variation.form != USV_PEN_OFF) pen_angvar = penalty_scalar(p.pen_angular_vel_variation, dw);
  if (p.pen_energy.form == USV_PEN_NEG_SUM) pen_energy = -(pa0_ + pa1_) * p.pen_energy.c1 + p.pen_energy.c2;
  else if (p.pen_energy.form == USV_PEN_EXP_NEG_SUMSQ) pen_energy = (__expf(-(pa0_ * pa0_ + pa1_ * pa1_)) - 1.0f) * p.pen_energy.c1;
  if (p.pen_action_variation.form != USV_PEN_OFF) pen_actvar = penalty_scalar(p.pen_action_variation, dasum);
  e.prev_w = wn;
  e.prev_asum = asum;
  o.rew = total + (pen_lin + pen_ang + pen_angvar + pen_energy + pen_actvar);  // USV_Virtual.py:1645

  // ---- update_kills (:661-706) + is_done (USV_Virtual.py:1223-1240) ------------------------------
  const bool collision = ncoll > 0;  // min_i |o_i - pos| < threshold
  const bool success = e.goal_cnt >= p.kill_after_n_steps_in_tolerance;
  const bool term = (d > p.kill_dist) || collision || success;
  if (term) ls.outcome = ((success && !collision) ? 1 : 0) | (collision ? 2 : 0);
  const int die = (term && !lp.fixed_horizon_eval) ? 1 : 0;
  o.done = (e.progress >= p.max_episode_length - 1) ? 1 : die;

  if (kStats) {
    const float bover = fminf(fmaxf(d - p.kill_dist, 0.0f) / 0.25f, 20.0f);
    o.st[USV_BST_TOTAL_REWARD] = total;
    o.st[USV_BST_DISTANCE_REWARD] = dist_rew;
    o.st[USV_BST_ALIGNMENT_REWARD] = align;
    o.st[USV_BST_HEADING_IMPROVE_REWARD] = h_imp_rew;
    o.st[USV_BST_POTENTIAL_SHAPING_REWARD] = shaping;
    o.st[USV_BST_SPEED_REWARD] = speed_rew;
    o.st[USV_BST_ANGULAR_REWARD] = ang_rew;
    o.st[USV_BST_TURN_HAZARD_PENALTY] = hazard;
    o.st[USV_BST_GOAL_REWARD] = goal_rew;
    o.st[USV_BST_COLLISION_REWARD] = coll;
    o.st[USV_BST_TIME_REWARD] = p.time_reward;
    o.st[USV_BST_POSITION_ERROR] = d;
    o.st[USV_BST_BOUNDARY_PENALTY] = -expm1f(bover) * p.boundary_cost;
    o.st[USV_BST_DANGER_MEAN] = danger;
    o.st[USV_BST_DANGER_HI_RATE] = (danger > 0.5f) ? 1.0f : 0.0f;
    o.st[USV_BST_G_GATE_MEAN] = gate_pos;
    o.st[USV_BST_LINEAR_VEL_PENALTY] = pen_lin;
    o.st[USV_BST_ANGULAR_VEL_PENALTY] = pen_ang;
    o.st[USV_BST_ANGULAR_VEL_VARIATION_PENALTY] = pen_angvar;
    o.st[USV_BST_ENERGY_PENALTY] = pen_energy;
    o.st[USV_BST_ACTION_VARIATION_PENALTY] = pen_actvar;
    o.st[USV_BST_NORMED_LINEAR_VEL] = speed;
    o.st[USV_BST_NORMED_ANGULAR_VEL] = fabsf(wn);
    o.st[USV_BST_ACTIONS_SUM] = s.raw0 + s.raw1;
    o.st[USV_BST_CMD_NEG_RATE] = 0.5f * ((s.t0 < 0.0f ? 1.0f : 0.0f) + (s.t1 < 0.0f ? 1.0f : 0.0f));
    o.st[USV_BST_THRUSTER_FORCE_NEG_RATE] = 0.5f * ((e.thrL < 0.0f ? 1.0f : 0.0f) + (e.thrR < 0.0f ? 1.0f : 0.0f));
    o.st[USV_BST_U_MEAN] = 0.5f * (s.c0 + s.c1);
    o.st[USV_BST_U_LOW_RATE] = 0.5f * ((s.c0 < 0.05f ? 1.0f : 0.0f) + (s.c1 < 0.05f ? 1.0f : 0.0f));
    o.st[USV_BST_U_SUM] = s.c0 + s.c1;
  }
  // NaN probe on the un-clamped obs and the reward, then _process_data's clamp  [ref vec_env_rlgames.py:82-95,187-192]
  o.finite = (fmaf(o.rew, 0.0f, o.chk) == 0.0f);
}

// each warp stages its 32 x 33 observation tile (stride 33: conflict-free) and writes one contiguous 4224 B run
// obs_w < 33 (the 4-wide privileged tail: 29): the staged rows keep their stride of 33, the global rows are obs_w wide
__device__ __forceinline__ void write_obs_tile_b(float* s_obs, float* __restrict__ obs,
                                                 int64_t block_start, int64_t n, int obs_w = kObsB) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* sw = s_obs + warp * (32 * kObsB);
  __syncwarp();
  const int64_t warp_start = block_start + (int64_t)warp * 32;
  if (warp_start >= n) return;
  const int rows = (int)min((int64_t)32, n - warp_start);
  float* g = obs + warp_start * obs_w;
  if (obs_w != kObsB) {
    for (int q = lane; q < rows * obs_w; q += 32) {
      const int r = q / obs_w;
      g[q] = sw[r * kObsB + (q - r * obs_w)];
    }
  } else if (rows == 32 && (((uintptr_t)g & 15) == 0)) {
    const float4* s4 = reinterpret_cast<const float4*>(sw);
    float4* g4 = reinterpret_cast<float4*>(g);
#pragma unroll
    for (int q = lane; q < (32 * kObsB) / 4; q += 32) g4[q] = s4[q];
  } else {
    for (int q = lane; q < rows * kObsB; q += 32) g[q] = sw[q];
  }
  __syncwarp();
}

// MDD._randomize_com for one resetting env: com_rand 1 = per-axis box around base_com (com_displacement_xyz), 2 = the legacy disc in
// the XY plane (radius U[0, CoM_max_displacement) kept in com_disp[0], angle U[0, 2 pi), z untouched)  [ref USV_disturbances.py:100-124]
__device__ __forceinline__ void redraw_com(const UsvLiveParams& lp, const Uniform4& rc, float* __restrict__ bc) {
  if (lp.com_rand == 2) {
    const float r = rc.a * lp.com_disp[0];
    const float th = rc.b * USV_PI_F * 2.0f;
    float sn, cs;
    fsincos(th, &sn, &cs);
    bc[USV_BC_COM_X * kTile] = lp.com_base[0] + cs * r;
    bc[USV_BC_COM_Y * kTile] = lp.com_base[1] + sn * r;
    bc[USV_BC_COM_Z * kTile] = lp.com_base[2];
  } else {
    bc[USV_BC_COM_X * kTile] = lp.com_base[0] + (rc.a * 2.0f - 1.0f) * lp.com_disp[0];
    bc[USV_BC_COM_Y * kTile] = lp.com_base[1] + (rc.b * 2.0f - 1.0f) * lp.com_disp[1];
    bc[USV_BC_COM_Z * kTile] = lp.com_base[2] + (rc.c * 2.0f - 1.0f) * lp.com_disp[2];
  }
}

// kMinB = CTAs per SM the register allocation aims for: 3 (80 registers, a few spilled words) is the best trade at >= 131 072 envs, where
// the kernel waits on DRAM; up to 2 x 148 CTAs -- one wave either way -- the 2-CTA build (112-128 registers, no spill) is 25-30 % faster
// (14.5 vs 17.4 us at 65 536 envs, 14.8 vs 18.3 at 75 776, r02 A/B).  Above one wave the step time is (number of waves) x (latency of one
// thread's ~2500-instruction chain with that many warps resident: 14.5 us at 16 warps per SM, ~20 us at 24), so 131 072 envs = 1.15 waves
// cost two; a 224-thread x 4-CTA build (28 warps per SM, 72 registers, kB) turns that size into one wave (30 vs 41 us) but loses at
// 262 144 (93 vs 77 us), and 64 registers lose everywhere: not kept, see profiles/r02_live_kernels.md.
template <int kDisturb, bool kStats, bool kStage = true, int kMinB = 3, int kB = kBlock>
__global__ void __launch_bounds__(kB, kMinB) step_live_kernel(UsvEnvBuffers b, UsvLiveBuffers lb, const float2* __restrict__ actions,
                                                              float* __restrict__ obs, float* __restrict__ rew, int64_t n,
                                                              const __grid_constant__ UsvStepParams p,
                                                              const __grid_constant__ UsvLiveParams lp) {
  extern __shared__ __align__(16) float smem[];
  const int64_t block_start = (int64_t)blockIdx.x * kB;
  const int64_t i = block_start + threadIdx.x;
  const bool active = i < n;
  const uint64_t step = p.step_counter + (b.step_offset ? *b.step_offset : 0ull);   // device-side addend: CUDA-graph replays
  const bool any_reset = (lb.reset_epoch[step & 1] == step);
  LiveOut o;
  o.sw = smem + (threadIdx.x >> 5) * (32 * kObsB) + (threadIdx.x & 31) * kObsB;
  o.chk = 0.0f;
  o.clip = p.clip_obs;
  // The task part reads 35 per-episode constants per env (CoM + 16 obstacle centres) ~1500 instructions from here, one dependent
  // load per obstacle (r02 ncu at 262 144 envs: 35 % of the stall samples sat on those loads, long-scoreboard 7.6 cycles per issue).
  // A warp's tile of them is ONE contiguous 4480 B run in the AoSoA buffer: fetch it with cp.async now, wait right before the task part.
  float* s_bc = smem + kB * kObsB + (threadIdx.x >> 5) * (USV_BC_COUNT * kTile);
  if (kStage) {
    const int64_t w0 = block_start + (int64_t)(threadIdx.x & ~31);
    if (w0 < n) {
      const float* src = lb.bconsts + (w0 >> 5) * (int64_t)(USV_BC_COUNT * kTile);
      for (int q = threadIdx.x & 31; q < USV_BC_COUNT * kTile / 4; q += 32) {
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_bc + q * 4);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + q * 4) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  EnvState e;
  EnvConst k;
  LiveState ls;
  DynOut s;
  bool do_reset = false;
  float2 act = make_float2(0.f, 0.f);
  float* __restrict__ bs = lb.bstate + tile_base(active ? i : 0, USV_BS_COUNT);
  float* __restrict__ bc = lb.bconsts + tile_base(active ? i : 0, USV_BC_COUNT);
  if (active) {
    load_state(b.state, i, e);
    load_consts<kDisturb>(b.consts, i, k);
    ls.prev_h = bs[USV_BS_PREV_H * kTile];
    ls.prev_pot = bs[USV_BS_PREV_POT * kTile];
    ls.outcome = __float_as_int(bs[USV_BS_OUTCOME * kTile]);
    do_reset = b.reset_buf[i] != 0;
    act = actions[i];
    const uint64_t gid = (uint64_t)(p.env_id_offset + i);
    if (do_reset && lp.com_rand) {  // MDD._randomize_com  [ref USV_disturbances.py:100-124]
      const Uniform4 rc = philox_uniform4(p.seed, gid, step, RS_RESET_COM);
      redraw_com(lp, rc, bc);
    }
    step_dynamics<kDisturb, true>(e, k, p, do_reset, act, gid, i, step, b.lut_left, b.lut_right, s);
  }
  // every lane of the warp (a ragged tail warp has inactive ones that issued copies too) waits for its own copies, then the warp
  // meets: a __syncwarp inside the `active` branch would pair with the one in write_obs_tile_b that the inactive lanes reach first
  if (kStage) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
  }
  if (active) {
    float* bcs = kStage ? s_bc + (threadIdx.x & 31) : bc;
    if (kStage && do_reset && lp.com_rand) {   // the staged copy predates this step's CoM re-draw of a resetting env
#pragma unroll
      for (int j = 0; j < 3; ++j) bcs[(USV_BC_COM_X + j) * kTile] = bc[(USV_BC_COM_X + j) * kTile];
    }
    post_live<kStats>(e, k, ls, bcs, lb.field + i * (int64_t)(kGridB * kGridB), p, lp, do_reset, any_reset, p.first_call != 0, s, o);
    store_state(b.state, i, e);
    if (do_reset) store_consts<kDisturb>(b.consts, i, k);
    bs[USV_BS_PREV_H * kTile] = ls.prev_h;
    bs[USV_BS_PREV_POT * kTile] = ls.prev_pot;
    bs[USV_BS_OUTCOME * kTile] = __int_as_float(ls.outcome);
    if (kStats) {
      float* __restrict__ st = lb.bstats + tile_base(i, USV_BST_COUNT);
#pragma unroll
      for (int f = 0; f < USV_BST_COUNT; ++f) st[f * kTile] = (do_reset ? 0.0f : st[f * kTile]) + o.st[f];
    }
    rew[i] = o.rew;
    b.reset_buf[i] = (int64_t)o.done;
    if (o.done) lb.reset_epoch[(step + 1) & 1] = step + 1;  // every writer stores the same value
    if (b.nonfinite_flag) {
      if (!o.finite) atomicOr(b.nonfinite_flag, 1u);
      if (!isfinite(act.x) || !isfinite(act.y)) atomicOr(b.nonfinite_flag, 2u);
    }
  }
  write_obs_tile_b(smem, obs, block_start, n, lp.priv_dim == 4 ? kObsB - 4 : kObsB);
}

// ---- Tier-3 tasks behind the same 33-dim observation (SURVEY row T) -------------------------------------------------
__device__ __forceinline__ float mode_reward(int mode, float err, float coeff) {
  // 1/(1+e) | 1/(1+e^2) | exp(-e/coeff)   [ref OIGE/tasks/USV/USV_task_rewards.py:206-325]
  if (mode == USV_REWARD_LINEAR) return __fdiv_rn(1.0f, 1.0f + err);
  if (mode == USV_REWARD_SQUARE) return __fdiv_rn(1.0f, 1.0f + err * err);
  return expf(-__fdiv_rn(err, coeff));
}

__device__ __forceinline__ void penalties_live(EnvState& e, const UsvStepParams& p, const DynOut& s, bool first_call, float speed,
                                               float& total) {
  const float pa0_ = s.pa0, pa1_ = s.pa1, wn = s.wn;
  const float asum = pa0_ + pa1_;
  const float dw = first_call ? 0.0f : (wn - e.prev_w);
  const float dasum = first_call ? 0.0f : (asum - e.prev_asum);
  float pen_lin = 0.0f, pen_ang = 0.0f, pen_angvar = 0.0f, pen_energy = 0.0f, pen_actvar = 0.0f;
  if (p.pen_linear_vel.form != USV_PEN_OFF) pen_lin = penalty_scalar(p.pen_linear_vel, speed);
  if (p.pen_angular_vel.form != USV_PEN_OFF) pen_ang = penalty_scalar(p.pen_angular_vel, wn);
  if (p.pen_angular_vel_variation.form != USV_PEN_OFF) pen_angvar = penalty_scalar(p.pen_angular_vel_variation, dw);
  if (p.pen_energy.form == USV_PEN_NEG_SUM) pen_energy = -(pa0_ + pa1_) * p.pen_energy.c1 + p.pen_energy.c2;
  else if (p.pen_energy.form == USV_PEN_EXP_NEG_SUMSQ) pen_energy = (__expf(-(pa0_ * pa0_ + pa1_ * pa1_)) - 1.0f) * p.pen_energy.c1;
  if (p.pen_action_variation.form != USV_PEN_OFF) pen_actvar = penalty_scalar(p.pen_action_variation, dasum);
  e.prev_w = wn;
  e.prev_asum = asum;
  total = pen_lin + pen_ang + pen_angvar + pen_energy + pen_actvar;
}

template <int kTask>
__device__ __forceinline__ void post_task(EnvState& e, const EnvConst& k, const float* __restrict__ bc, const UsvStepParams& p,
                                          const UsvLiveParams& lp, bool do_reset, bool first_call, const DynOut& s, LiveOut& o) {
  const float pxn = s.pxn, pyn = s.pyn, vxn = s.vxn, vyn = s.vyn;
  obs_head(o, s);
  float task_rew;
  int die;
  const float speed = sqrtf(__fmaf_rn(vyn, vyn, __fmul_rn(vxn, vxn)));  // torch.norm(linear_velocity, dim=-1)
  if (kTask == USV_TASK_TRACK_XY_VELOCITY) {
    // [ref USV_track_xy_velocity.py:64-128]
    const float evx = bc[USV_BC_TARGET_VX * kTile] - vxn, evy = bc[USV_BC_TARGET_VY * kTile] - vyn;
    o.put(3, evx);
    o.put(4, evy);
#pragma unroll
    for (int j = 5; j < 23; ++j) o.put(j, 0.0f);
    const float pd = sqrtf(__fadd_rn(__fmul_rn(pxn, pxn), __fmul_rn(pyn, pyn)));   // _position_error = position
    const float vd = sqrtf(__fadd_rn(__fmul_rn(evx, evx), __fmul_rn(evy, evy)));
    const int goal = (vd < lp.lin_vel_tolerance) ? 1 : 0;
    e.goal_cnt = e.goal_cnt * goal + goal;
    task_rew = mode_reward(p.reward_mode, vd, p.exponential_reward_coeff);
    die = (pd > p.kill_dist) ? 1 : 0;
    if (e.goal_cnt > p.kill_after_n_steps_in_tolerance) die = 1;      // strict '>' in this task (:123)
  } else {
    // GoToPose [ref USV_go_to_pose.py:81-209] / KeepXY [ref USV_keep_xy.py:80-179]
    const float ex = k.tx - pxn, ey = k.ty - pyn;
    const float theta = wrap_pi(s.yawn);
    const float beta = atan2f(ey, ex);
    const float xa = beta - theta + USV_PI_F;
    const float alpha = ((xa >= USV_2PI_F) ? xa - USV_2PI_F : xa) - USV_PI_F;
    float sa, ca;
    fsincos(alpha, &sa, &ca);
    const float d = sqrtf(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
    o.put(3, ca);
    o.put(4, sa);
    o.put(5, sqrtf(__fmaf_rn(ey, ey, __fmul_rn(ex, ex))));
    float herr = 0.0f;
    if (kTask == USV_TASK_GO_TO_POSE) {
      // heading error: fmod(target - theta + pi, 2pi) - pi, then atan2(sin, cos)
      const float xh = bc[USV_BC_TARGET_HEADING * kTile] - theta + USV_PI_F;   // in (-pi, 4pi): C fmod keeps the sign of the dividend
      const float hr = fmodf(xh, USV_2PI_F) - USV_PI_F;
      float sh, ch;
      fsincos(hr, &sh, &ch);
      herr = atan2f(sh, ch);
      float sh2, ch2;
      fsincos(herr, &sh2, &ch2);
      o.put(6, ch2);
      o.put(7, sh2);
    } else {
      o.put(6, 0.0f);
      o.put(7, 0.0f);
    }
#pragma unroll
    for (int j = 8; j < 23; ++j) o.put(j, 0.0f);
    if (kTask == USV_TASK_GO_TO_POSE) {
      if (do_reset) e.prev_d = 0.0f;                                    // reset(): prev_position_dist[env_ids] = 0  (:226)
      const float progress = 2.0f * fminf(fmaxf(e.prev_d - d, -2.0f), 2.0f);
      e.prev_d = d;
      const int goal = ((d < p.position_tolerance) && (speed < 0.1f)) ? 1 : 0;
      e.goal_cnt = e.goal_cnt * goal + goal;
      // GoToPoseReward.compute_reward  [ref USV_task_rewards.py:206-255]
      const float hw = 1.0f - __fdiv_rn(1.0f, 1.0f + expf(-lp.sig_gain * (d - 2.0f)));
      const float pos_rew = p.position_scale * mode_reward(p.reward_mode, d, p.exponential_reward_coeff);
      const float head_rew = hw * lp.heading_scale * mode_reward(lp.heading_reward_mode, fabsf(herr), lp.heading_exponential_reward_coeff);
      const float act_pen = -0.05f * (fabsf(s.raw0) + fabsf(s.raw1));
      task_rew = pos_rew + head_rew + progress + 2.0f * (float)goal + act_pen;
    } else {
      task_rew = mode_reward(p.reward_mode, d, p.exponential_reward_coeff);   // KeepXYReward; the goal counter is never fed (:118-141)
    }
    die = (d > p.kill_dist) ? 1 : 0;
    if (e.goal_cnt >= p.kill_after_n_steps_in_tolerance) die = 1;
  }
  obs_tail(o, s, k, bc, p, lp, do_reset);
  float pen;
  penalties_live(e, p, s, first_call, speed, pen);
  o.rew = task_rew + pen;
  if (lp.fixed_horizon_eval) die = 0;
  o.done = (e.progress >= p.max_episode_length - 1) ? 1 : die;
  o.finite = (fmaf(o.rew, 0.0f, o.chk) == 0.0f);
}

template <int kTask, int kDisturb>
__global__ void __launch_bounds__(kBlock, 3) step_task_kernel(UsvEnvBuffers b, UsvLiveBuffers lb, const float2* __restrict__ actions,
                                                              float* __restrict__ obs, float* __restrict__ rew, int64_t n,
                                                              const __grid_constant__ UsvStepParams p,
                                                              const __grid_constant__ UsvLiveParams lp) {
  extern __shared__ __align__(16) float smem[];
  const int64_t block_start = (int64_t)blockIdx.x * kBlock;
  const int64_t i = block_start + threadIdx.x;
  const bool active = i < n;
  const uint64_t step = p.step_counter + (b.step_offset ? *b.step_offset : 0ull);   // device-side addend: CUDA-graph replays
  LiveOut o;
  o.sw = smem + (threadIdx.x >> 5) * (32 * kObsB) + (threadIdx.x & 31) * kObsB;
  o.chk = 0.0f;
  o.clip = p.clip_obs;
  if (active) {
    EnvState e;
    EnvConst k;
    load_state(b.state, i, e);
    load_consts<kDisturb>(b.consts, i, k);
    float* __restrict__ bc = lb.bconsts + tile_base(i, USV_BC_COUNT);
    const bool do_reset = b.reset_buf[i] != 0;
    const float2 act = actions[i];
    const uint64_t gid = (uint64_t)(p.env_id_offset + i);
    if (do_reset) {
      const Uniform4 rc = philox_uniform4(p.seed, gid, step, RS_RESET_COM);
      if (lp.com_rand) redraw_com(lp, rc, bc);
      if (!p.reset_pose_external) {
        // task.get_goals at the end of reset_idx  [ref USV_go_to_pose.py:244-246 ; USV_track_xy_velocity.py:141-146]
        if (kTask == USV_TASK_GO_TO_POSE) bc[USV_BC_TARGET_HEADING * kTile] = rc.d * USV_PI_F * 2.0f;
        if (kTask == USV_TASK_TRACK_XY_VELOCITY) {
          const Uniform4 rt = philox_uniform4(p.seed, gid, step, RS_RESET_TASK);
          bc[USV_BC_TARGET_VX * kTile] = rt.a * lp.goal_random_velocity * 2.0f - lp.goal_random_velocity;
          bc[USV_BC_TARGET_VY * kTile] = rt.b * lp.goal_random_velocity * 2.0f - lp.goal_random_velocity;
        }
      }
    }
    DynOut s;
    step_dynamics<kDisturb, true>(e, k, p, do_reset, act, gid, i, step, b.lut_left, b.lut_right, s);
    post_task<kTask>(e, k, bc, p, lp, do_reset, p.first_call != 0, s, o);
    store_state(b.state, i, e);
    if (do_reset) store_consts<kDisturb>(b.consts, i, k);
    rew[i] = o.rew;
    b.reset_buf[i] = (int64_t)o.done;
    if (b.nonfinite_flag) {
      if (!o.finite) atomicOr(b.nonfinite_flag, 1u);
      if (!isfinite(act.x) || !isfinite(act.y)) atomicOr(b.nonfinite_flag, 2u);
    }
  }
  write_obs_tile_b(smem, obs, block_start, n, lp.priv_dim == 4 ? kObsB - 4 : kObsB);
}

}  // namespace usv

using namespace usv;

extern "C" int usv_step_live_f32(const UsvEnvBuffers* b, const UsvLiveBuffers* lb, const float* actions, float* obs, float* rew,
                                 int64_t n, const UsvStepParams* p, const UsvLiveParams* lp, void* stream) {
  if (!lb || !lp) return USV_E_NULL;
  int rc = check_common(b, n, p);
  if (rc) return rc;
  if (lp->task < USV_TASK_CAPTURE_OBSTACLES || lp->task > USV_TASK_TRACK_XY_VELOCITY) return USV_E_PARAM;
  const bool obst = lp->task == USV_TASK_CAPTURE_OBSTACLES;
  if (!lb->bconsts || (obst && (!lb->bstate || !lb->field || !lb->reset_epoch))) return USV_E_NULL;
  if (lb->bconsts_stride < n || (lb->bconsts_stride & 31)) return USV_E_SIZE;
  if (obst && (lb->bstate_stride < n || (lb->bstate_stride & 31))) return USV_E_SIZE;
  if (lb->bstats && (lb->bstats_stride < n || (lb->bstats_stride & 31))) return USV_E_SIZE;
  if (!(lp->map_size > 0.0f)) return USV_E_PARAM;
  if (lp->priv_mode < USV_PRIV_RAW || lp->priv_mode > USV_PRIV_MINMAX) return USV_E_PARAM;
  if (lp->priv_dim != 0 && lp->priv_dim != 4 && lp->priv_dim != 8) return USV_E_PARAM;
  if (n == 0) return USV_OK;
  if (!actions || !obs || !rew) return USV_E_NULL;
  if ((uintptr_t)actions & 7) return USV_E_ALIGN;
  const int grid = grid_for(n, kBlock);
  const bool dis = wants_disturb(p), st = lb->bstats != nullptr;
  // staged bconsts (cp.async into shared memory) vs direct loads, A/B on one B200 (r02, profiles/r02_live_kernels.md): 13.9 vs 14.9 us at
  // 16 384 envs, 16.8 vs 18.4 at 65 536, 41.5 vs 44.7 at 131 072 -- but 83.5 vs 76.1 us at 262 144, where the 24 GB of per-env fields make
  // every tap a DRAM access and the 36 KB of extra shared memory per CTA cost more L1 than the staging saves.
  const bool no_stage = n > 196608;
  // one wave at two CTAs per SM (and no statistics: the rarely used stats build stays on one register budget)
  const bool one_wave = !no_stage && grid <= 2 * num_sms();
  decltype(&step_live_kernel<false, false>) kernel;
#define USV_LIVE_KERNEL(D, S) \
  (no_stage ? step_live_kernel<D, S, false> : (one_wave && !S) ? step_live_kernel<D, false, true, 2> : step_live_kernel<D, S, true>)
#define USV_TASK_KERNEL(T) (dis ? step_task_kernel<T, true> : step_task_kernel<T, false>)
  if (lp->task == USV_TASK_GO_TO_POSE) kernel = USV_TASK_KERNEL(USV_TASK_GO_TO_POSE);
  else if (lp->task == USV_TASK_KEEP_XY) kernel = USV_TASK_KERNEL(USV_TASK_KEEP_XY);
  else if (lp->task == USV_TASK_TRACK_XY_VELOCITY) kernel = USV_TASK_KERNEL(USV_TASK_TRACK_XY_VELOCITY);
  else if (dis) kernel = st ? USV_LIVE_KERNEL(true, true) : USV_LIVE_KERNEL(true, false);
  else kernel = st ? USV_LIVE_KERNEL(false, true) : USV_LIVE_KERNEL(false, false);
#undef USV_LIVE_KERNEL
#undef USV_TASK_KERNEL
  size_t smem = (size_t)kBlock * kObsB * sizeof(float);
  if (obst && !no_stage) smem += (size_t)(kBlock / 32) * USV_BC_COUNT * kTile * sizeof(float);   // + the staged bconsts tiles
  ensure_dynamic_smem(kernel, smem);
  kernel<<<grid, kBlock, smem, (cudaStream_t)stream>>>(*b, *lb, (const float2*)actions, obs, rew, n, *p, *lp);
  return finish_launch();
}
