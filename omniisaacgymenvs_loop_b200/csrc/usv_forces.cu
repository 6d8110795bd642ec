// Stand-alone force-layer kernels (SURVEY rows A1-A6, A10) behind the reference's
// HydrostaticsObject / HydrodynamicsObject / DynamicsFirstOrder method surfaces.
// These are the 6-DOF, AoS-in / AoS-out drop-ins; the fused env step (usv_step.cu) carries the
// planar specialisation of the same maths.  All are pure streaming kernels (HBM-bound):
// one thread per env, row-major (n,k) tensors read/written with vector accesses where the
// row size allows (quat = float4; (n,6) rows as 3 x float2; (n,2) rows as float2).
#include <string.h>
#include "usv_common.cuh"
#include "philox.cuh"

namespace usv {

std::atomic<int64_t> g_launch_count{0};

// ------------------------------------------------------------------ A1 hydrostatics
__global__ void __launch_bounds__(256) hydrostatics_kernel(
    const float* __restrict__ vol, const float* __restrict__ rpy, const float4* __restrict__ quat,
    float2* __restrict__ out6, float* __restrict__ fg, float* __restrict__ tg, int64_t n, float rho_g,
    float neg_w, float neg_l, float avg_force, float amp) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float V = vol[i];
  const float roll = rpy[3 * i + 0], pitch = rpy[3 * i + 1];
  const float4 q = quat[i];
  // [ref Hydrostatics.py:67-69] Fz = -rho*g*V (world frame)
  const float Fz = rho_g * V;
  // [ref :83-92] the second assignment wins: torque uses the constant average force
  const float tx = neg_w * (sinf(roll) * avg_force);
  const float ty = neg_l * (sinf(pitch) * avg_force);
  // [ref :105-115] F_local = R^T F_global; F_global = (0,0,Fz)
  const Rot3 R = quat_to_matrix(q.x, q.y, q.z, q.w);
  float fx, fy, fz;
  rot_t_apply(R, 0.0f, 0.0f, Fz, fx, fy, fz);
  // [ref :123] torque is NOT rotated; [ref :127-132] hstack + amplify
  out6[3 * i + 0] = make_float2(fx, fy);
  out6[3 * i + 1] = make_float2(fz, tx * amp);
  out6[3 * i + 2] = make_float2(ty * amp, 0.0f * amp);
  if (fg) { fg[3 * i + 0] = 0.0f; fg[3 * i + 1] = 0.0f; fg[3 * i + 2] = Fz; }
  if (tg) { tg[3 * i + 0] = tx; tg[3 * i + 1] = ty; tg[3 * i + 2] = 0.0f; }
}

// ------------------------------------------------------------------ A2 hydrodynamics
struct HydroDevParams {
  float fwd[6];       // linear_damping_forward_speed + offset_lin_forward_damping_speed
  float off_lin, off_nl, scaling;
  int use_scale, use_current;
  float flow[3];
};

__global__ void __launch_bounds__(256) hydrodynamics_kernel(
    const float4* __restrict__ quat, const float2* __restrict__ vel6, const float2* __restrict__ lin6,
    const float2* __restrict__ quad6, const float* __restrict__ kdrag, float2* __restrict__ drag6,
    float2* __restrict__ local6, float2* __restrict__ damp6, int64_t n, HydroDevParams p) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = quat[i];
  const float2 va = vel6[3 * i], vb = vel6[3 * i + 1], vc = vel6[3 * i + 2];
  const float2 la = lin6[3 * i], lb = lin6[3 * i + 1], lc = lin6[3 * i + 2];
  const float2 qa = quad6[3 * i], qb = quad6[3 * i + 1], qc = quad6[3 * i + 2];
  const float k = p.use_scale ? kdrag[i] : 1.0f;
  const Rot3 R = quat_to_matrix(q.x, q.y, q.z, q.w);
  float v[6];
  // [ref Hydrodynamics.py:210-222] local = R^T world for linear and angular parts
  rot_t_apply(R, va.x, va.y, vb.x, v[0], v[1], v[2]);
  rot_t_apply(R, vb.y, vc.x, vc.y, v[3], v[4], v[5]);
  if (p.use_current) {  // [ref :224-237]
    float fx, fy, fz;
    rot_t_apply(R, p.flow[0], p.flow[1], p.flow[2], fx, fy, fz);
    v[0] -= fx; v[1] -= fy; v[2] -= fz;
  }
  const float L[6] = {la.x, la.y, lb.x, lb.y, lc.x, lc.y};
  const float Q[6] = {qa.x, qa.y, qb.x, qb.y, qc.x, qc.y};
  float d[6], Dm[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    // [ref :186-203] D = ((L + off - (fwd+off_fwd)) + (Q+off_nl)*|v|)*scaling [*k_drag]; [ref :243] drag = -D*v
    const float lin = (L[c] + p.off_lin) - p.fwd[c];
    const float qd = (Q[c] + p.off_nl) * fabsf(v[c]);
    float D = (lin + qd) * p.scaling;
    if (p.use_scale) D = D * k;
    Dm[c] = D;
    d[c] = -1.0f * D * v[c];
  }
  if (damp6) {
    damp6[3 * i + 0] = make_float2(Dm[0], Dm[1]);
    damp6[3 * i + 1] = make_float2(Dm[2], Dm[3]);
    damp6[3 * i + 2] = make_float2(Dm[4], Dm[5]);
  }
  drag6[3 * i + 0] = make_float2(d[0], d[1]);
  drag6[3 * i + 1] = make_float2(d[2], d[3]);
  drag6[3 * i + 2] = make_float2(d[4], d[5]);
  if (local6) {
    local6[3 * i + 0] = make_float2(v[0], v[1]);
    local6[3 * i + 1] = make_float2(v[2], v[3]);
    local6[3 * i + 2] = make_float2(v[4], v[5]);
  }
}

// ------------------------------------------------------------------ A4 thruster target
__global__ void __launch_bounds__(256) thruster_target_kernel(
    const float2* __restrict__ cmd, const float* __restrict__ lutL, const float* __restrict__ lutR, int n_lut,
    const float* __restrict__ mL, const float* __restrict__ mR, float2* __restrict__ before,
    float2* __restrict__ after, int64_t n) {
  extern __shared__ float s_lut[];  // [2][n_lut]: the LUT is gathered at random -> stage it once per CTA
  for (int t = threadIdx.x; t < n_lut; t += blockDim.x) {
    s_lut[t] = lutL[t];
    s_lut[n_lut + t] = lutR[t];
  }
  __syncthreads();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float2 c = cmd[i];
  const float fl = s_lut[lut_index(c.x, n_lut)];
  const float fr = s_lut[n_lut + lut_index(c.y, n_lut)];
  before[i] = make_float2(fl, fr);
  if (after) after[i] = make_float2(fl * (mL ? mL[i] : 1.0f), fr * (mR ? mR[i] : 1.0f));
}

// ------------------------------------------------------------------ A5 thruster lag
__global__ void __launch_bounds__(256) thruster_lag_kernel(float2* __restrict__ cur, const float2* __restrict__ tgt,
                                                           float alpha, float one_minus_alpha,
                                                           float* __restrict__ thr6, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float2 c = cur[i];
  const float2 t = tgt[i];
  // [ref ThrusterDynamics.py:133-136] cur*alpha + (1.0-alpha)*target, evaluated op by op as torch does
  c.x = __fadd_rn(__fmul_rn(c.x, alpha), __fmul_rn(one_minus_alpha, t.x));
  c.y = __fadd_rn(__fmul_rn(c.y, alpha), __fmul_rn(one_minus_alpha, t.y));
  cur[i] = c;
  // [ref :223-230] thrusters[:, [0,3]] = cur
  thr6[6 * i + 0] = c.x;
  thr6[6 * i + 3] = c.y;
}

// ------------------------------------------------------------------ LUT builder
__global__ void build_lut_kernel(const float* __restrict__ pts, int n_pts, float* __restrict__ lut, int n_out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  // ATen upsample_linear1d, align_corners=True: scale=(in-1)/(out-1); src=scale*i; i0=floor(src);
  // l1=src-i0; out=(1-l1)*in[i0]+l1*in[min(i0+1,in-1)]   [ref ThrusterDynamics.py:158-169]
  const float scale = n_out > 1 ? (float)(n_pts - 1) / (float)(n_out - 1) : 0.0f;
  const float src = __fmul_rn(scale, (float)i);
  int i0 = (int)floorf(src);
  if (i0 > n_pts - 1) i0 = n_pts - 1;
  float l1 = __fsub_rn(src, (float)i0);
  l1 = fminf(fmaxf(l1, 0.0f), 1.0f);
  const float l0 = __fsub_rn(1.0f, l1);
  const int i1 = i0 + (i0 < n_pts - 1 ? 1 : 0);
  // ATen's CPU kernel evaluates w0*x0 + w1*x1 as fma(w0, x0, w1*x1); pinned bit-exactly against the reference LUTs
  lut[i] = __fmaf_rn(l0, pts[i0], __fmul_rn(l1, pts[i1]));
}

// ------------------------------------------------------------------ A3/A6/A10 row re-draws
__global__ void __launch_bounds__(256) randomize_rows_kernel(float* __restrict__ dst, int64_t ld,
                                                             const int64_t* __restrict__ ids, int64_t n_ids, int ncols,
                                                             const float* __restrict__ base,
                                                             const float* __restrict__ lo,
                                                             const float* __restrict__ hi, int log_space,
                                                             uint64_t seed, uint64_t counter, uint32_t stream_id) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_ids) return;
  const int64_t env = ids[j];
  for (int c0 = 0; c0 < ncols; c0 += 4) {
    const Uniform4 u = philox_uniform4(seed, (uint64_t)env, counter, RS_ROWS + stream_id * 16u + (uint32_t)(c0 >> 2));
    const float uu[4] = {u.a, u.b, u.c, u.d};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = c0 + k;
      if (c < ncols) {
        float v;
        if (log_space) {  // [ref Hydrodynamics.py:130-133] exp(log(min) + u*(log(max)-log(min)))
          const float l0 = logf(lo[c]), l1 = logf(hi[c]);
          v = expf(l0 + uu[k] * (l1 - l0));
        } else {
          v = lo[c] + uu[k] * (hi[c] - lo[c]);
        }
        dst[env * ld + c] = base[c] + v;
      }
    }
  }
}

}  // namespace usv

using namespace usv;

namespace usv {

// ---- planar rigid body behind the simulator surface the task expects (row A7 as a stand-alone: HeronView / world.step()) ------------------
// wrench[i] = (Fx, Fy, Tz) in the BODY frame, accumulated over the apply_forces_and_torques_at_pos calls of one physics step
__global__ void planar_wrench_accumulate_kernel(float* __restrict__ wrench, const float* __restrict__ forces, const float* __restrict__ torques,
                                                const float* __restrict__ pose, float off_x, float off_y, int is_global, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float fx = forces ? forces[i * 3] : 0.f, fy = forces ? forces[i * 3 + 1] : 0.f;
  float tz = torques ? torques[i * 3 + 2] : 0.f;
  if (is_global) {   // world -> body: R(psi)^T
    float sn, cs;
    sincosf(pose[i * 3 + 2], &sn, &cs);
    const float bx = cs * fx + sn * fy, by = -sn * fx + cs * fy;
    fx = bx; fy = by;
  }
  // a force applied at the body-frame offset (off_x, off_y) adds the moment r x F
  tz += off_x * fy - off_y * fx;
  wrench[i * 3] += fx;
  wrench[i * 3 + 1] += fy;
  wrench[i * 3 + 2] += tz;
}

// semi-implicit Euler of the planar body (the fused step's integrator, usv_step_core.cuh): pose (x, y, psi), vel (vx, vy world, r);
// consumes and clears the accumulated wrench
__global__ void planar_rigid_step_kernel(float* __restrict__ pose, float* __restrict__ vel, float* __restrict__ wrench,
                                         const float* __restrict__ mass, const float* __restrict__ izz, float dt, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float sn, cs;
  sincosf(pose[i * 3 + 2], &sn, &cs);
  const float fx = wrench[i * 3], fy = wrench[i * 3 + 1], tz = wrench[i * 3 + 2];
  const float inv_m = 1.0f / mass[i];
  const float ax = (cs * fx - sn * fy) * inv_m, ay = (sn * fx + cs * fy) * inv_m;
  float vx = vel[i * 3] + dt * ax, vy = vel[i * 3 + 1] + dt * ay, r = vel[i * 3 + 2] + dt * (tz / izz[i]);
  vel[i * 3] = vx; vel[i * 3 + 1] = vy; vel[i * 3 + 2] = r;
  pose[i * 3] += dt * vx;
  pose[i * 3 + 1] += dt * vy;
  pose[i * 3 + 2] += dt * r;
  wrench[i * 3] = 0.f; wrench[i * 3 + 1] = 0.f; wrench[i * 3 + 2] = 0.f;
}

}  // namespace usv

extern "C" {

int usv_b200_abi_version(void) { return USV_B200_ABI_VERSION; }

int64_t usv_b200_launch_count(void) { return g_launch_count.load(); }

int64_t usv_b200_sizeof(const char* name) {
  if (!name) return -1;
#define USV_SZ(T) if (!strcmp(name, #T)) return (int64_t)sizeof(T)
  USV_SZ(UsvHydrostaticsParams);
  USV_SZ(UsvHydrodynamicsParams);
  USV_SZ(UsvPenaltyTerm);
  USV_SZ(UsvStepParams);
  USV_SZ(UsvEnvBuffers);
  USV_SZ(UsvCaptureXYIO);
  USV_SZ(UsvLiveParams);
  USV_SZ(UsvLiveBuffers);
  USV_SZ(PpoLossParams);
  USV_SZ(PpoAdamParams);
  USV_SZ(PpoPeerComm);
  USV_SZ(PpoLoopzNet);
  USV_SZ(PpoLoopzLossParams);
  USV_SZ(PpoLoopzAdamParams);
#undef USV_SZ
  return -1;
}

const char* usv_b200_error_string(int code) {
  switch (code) {
    case USV_OK: return "ok";
    case USV_E_NULL: return "usv_b200: required pointer is NULL";
    case USV_E_SIZE: return "usv_b200: negative or inconsistent size";
    case USV_E_PARAM: return "usv_b200: parameter outside supported range";
    case USV_E_ALIGN: return "usv_b200: pointer/stride not aligned as documented";
    case USV_E_UNSUPPORTED: return "usv_b200: unsupported configuration";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "usv_b200: unknown error";
}

int usv_hydrostatics_f32(const float* vol, const float* rpy, const float* quat, float* out6, float* fg, float* tg,
                         int64_t n, const UsvHydrostaticsParams* p, void* stream) {
  if (!p) return USV_E_NULL;
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!vol || !rpy || !quat || !out6) return USV_E_NULL;
  if (((uintptr_t)quat & 15) || ((uintptr_t)out6 & 7)) return USV_E_ALIGN;
  // python evaluates -rho*g, -1*width, -1*length in double before they meet the fp32 tensor
  const float rho_g = (float)(-(double)p->water_density * (double)p->gravity);
  hydrostatics_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      vol, rpy, (const float4*)quat, (float2*)out6, fg, tg, n, rho_g, -p->metacentric_width, -p->metacentric_length,
      p->average_hydrostatics_force_value, p->amplify_torque);
  return finish_launch();
}

int usv_hydrodynamics_f32(const float* quat, const float* vel6, const float* lin6, const float* quad6,
                          const float* drag_scale, float* drag6, float* local6, float* damp6, int64_t n,
                          const UsvHydrodynamicsParams* p, void* stream) {
  if (!p) return USV_E_NULL;
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!quat || !vel6 || !lin6 || !quad6 || !drag6) return USV_E_NULL;
  if (p->use_drag_scale && !drag_scale) return USV_E_NULL;
  if (((uintptr_t)quat & 15) || ((uintptr_t)vel6 & 7) || ((uintptr_t)lin6 & 7) || ((uintptr_t)quad6 & 7) ||
      ((uintptr_t)drag6 & 7) || ((uintptr_t)local6 & 7) || ((uintptr_t)damp6 & 7))
    return USV_E_ALIGN;
  HydroDevParams d;
  for (int c = 0; c < 6; ++c)
    d.fwd[c] = p->linear_damping_forward_speed[c] + p->offset_lin_forward_damping_speed;
  d.off_lin = p->offset_linear_damping;
  d.off_nl = p->offset_nonlin_damping;
  d.scaling = p->scaling_damping;
  d.use_scale = p->use_drag_scale;
  d.use_current = p->use_water_current;
  for (int c = 0; c < 3; ++c) d.flow[c] = p->flow_vel[c];
  hydrodynamics_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      (const float4*)quat, (const float2*)vel6, (const float2*)lin6, (const float2*)quad6, drag_scale,
      (float2*)drag6, (float2*)local6, (float2*)damp6, n, d);
  return finish_launch();
}

int usv_thruster_target_f32(const float* cmd2, const float* lutL, const float* lutR, int32_t n_lut, const float* mL,
                            const float* mR, float* before2, float* after2, int64_t n, void* stream) {
  if (n < 0 || n_lut < 2) return USV_E_SIZE;
  if (n_lut > 8192) return USV_E_PARAM;
  if (n == 0) return USV_OK;
  if (!cmd2 || !lutL || !lutR || !before2) return USV_E_NULL;
  if (((uintptr_t)cmd2 & 7) || ((uintptr_t)before2 & 7) || ((uintptr_t)after2 & 7)) return USV_E_ALIGN;
  const size_t smem = 2 * (size_t)n_lut * sizeof(float);
  ensure_dynamic_smem(thruster_target_kernel, smem);
  thruster_target_kernel<<<grid_for(n, 256), 256, smem, (cudaStream_t)stream>>>(
      (const float2*)cmd2, lutL, lutR, n_lut, mL, mR, (float2*)before2, (float2*)after2, n);
  return finish_launch();
}

int usv_thruster_lag_f32(float* cur2, const float* target2, float alpha, float* thr6, int64_t n, void* stream) {
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!cur2 || !target2 || !thr6) return USV_E_NULL;
  if (((uintptr_t)cur2 & 7) || ((uintptr_t)target2 & 7)) return USV_E_ALIGN;
  thruster_lag_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((float2*)cur2, (const float2*)target2, alpha,
                                                                          1.0f - alpha, thr6, n);
  return finish_launch();
}

int usv_thruster_build_lut_f32(const float* points, int32_t n_pts, float* lut, int32_t n_out, void* stream) {
  if (n_pts < 1 || n_out < 1) return USV_E_SIZE;
  if (!points || !lut) return USV_E_NULL;
  build_lut_kernel<<<grid_for(n_out, 256), 256, 0, (cudaStream_t)stream>>>(points, n_pts, lut, n_out);
  return finish_launch();
}

int usv_randomize_rows_f32(float* dst, int64_t ld, const int64_t* env_ids, int64_t n_ids, int32_t ncols,
                           const float* base, const float* lo, const float* hi, int32_t log_space, uint64_t seed,
                           uint64_t counter, uint32_t stream_id, void* stream) {
  if (n_ids < 0 || ncols < 1 || ncols > 64 || ld < ncols) return USV_E_SIZE;
  if (n_ids == 0) return USV_OK;
  if (!dst || !env_ids || !base || !lo || !hi) return USV_E_NULL;
  randomize_rows_kernel<<<grid_for(n_ids, 256), 256, 0, (cudaStream_t)stream>>>(dst, ld, env_ids, n_ids, ncols, base,
                                                                                lo, hi, log_space, seed, counter,
                                                                                stream_id);
  return finish_launch();
}


int usv_planar_wrench_accumulate_f32(float* wrench, const float* forces, const float* torques, const float* pose, float offset_x,
                                     float offset_y, int32_t is_global, int64_t n, void* stream) {
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!wrench || (!forces && !torques) || (is_global && !pose)) return USV_E_NULL;
  usv::planar_wrench_accumulate_kernel<<<usv::grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(wrench, forces, torques, pose, offset_x, offset_y,
                                                                                               is_global, n);
  return usv::finish_launch();
}

int usv_planar_rigid_step_f32(float* pose, float* vel, float* wrench, const float* mass, const float* izz, float dt, int64_t n, void* stream) {
  if (n < 0) return USV_E_SIZE;
  if (n == 0) return USV_OK;
  if (!pose || !vel || !wrench || !mass || !izz) return USV_E_NULL;
  if (!(dt > 0.0f)) return USV_E_PARAM;
  usv::planar_rigid_step_kernel<<<usv::grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(pose, vel, wrench, mass, izz, dt, n);
  return usv::finish_launch();
}

}  // extern "C"
