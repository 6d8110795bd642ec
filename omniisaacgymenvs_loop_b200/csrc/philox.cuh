// Philox4x32-10 counter-based RNG (Salmon et al., SC'11 -- the published Random123 algorithm).
// Keyed (seed_lo, seed_hi); counter = (env_id, step_lo, step_hi, stream).  Stateless: a reset or a
// noise draw needs no per-env RNG state in HBM.  oracle/philox.py is the bit-exact numpy mirror.
#pragma once
#include <stdint.h>

namespace usv {

struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#ifdef __CUDA_ARCH__
  hi = __umulhi(a, b);
  lo = a * b;
#else
  uint64_t p = (uint64_t)a * (uint64_t)b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(M0, c0, hi0, lo0);
    philox_mulhilo(M1, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

// The 10 round keys (k0 + r*W0, k1 + r*W1) of one Philox key.  A kernel whose draws all use one seed takes them as a parameter and
// reads them as constant-bank operands, instead of deriving them with 20 integer adds per draw.
struct PhiloxKeys { uint32_t k0[10], k1[10]; };
inline PhiloxKeys philox_round_keys(uint64_t seed) {
  PhiloxKeys K;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    K.k0[r] = k0; K.k1[r] = k1;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return K;
}
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys& K) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(M0, c0, hi0, lo0);
    philox_mulhilo(M1, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ K.k0[r];
    uint32_t n2 = hi0 ^ c3 ^ K.k1[r];
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  return Philox4{c0, c1, c2, c3};
}

// 24-bit uniform in [0,1), the same range contract as torch.rand (never returns 1.0)
__host__ __device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

struct Uniform4 { float a, b, c, d; };

__host__ __device__ __forceinline__ Uniform4 philox_uniform4(uint64_t seed, uint64_t env_id, uint64_t step,
                                                             uint32_t stream) {
  // env ids beyond 2^32 fold their high word into the stream word (never reached in practice)
  Philox4 r = philox4x32_10((uint32_t)env_id, (uint32_t)step, (uint32_t)(step >> 32),
                            stream ^ ((uint32_t)(env_id >> 32) << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
  return Uniform4{u01(r.x), u01(r.y), u01(r.z), u01(r.w)};
}

// 8 x 16-bit uniforms in [0,1) from ONE Philox call (per-step observation / action noise: amplitudes are
// <= 0.05, so 2^-16 resolution is ~1e-6 of the signal; halves the RNG cost of the step)
struct Uniform8 { float v[8]; };
__host__ __device__ __forceinline__ Uniform8 uniform8x16(const Philox4& r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  Uniform8 u;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    u.v[2 * i] = (float)(w[i] & 0xFFFFu) * (1.0f / 65536.0f);
    u.v[2 * i + 1] = (float)(w[i] >> 16) * (1.0f / 65536.0f);
  }
  return u;
}
__host__ __device__ __forceinline__ Uniform8 philox_uniform8x16(uint64_t seed, uint64_t env_id, uint64_t step,
                                                                uint32_t stream) {
  return uniform8x16(philox4x32_10((uint32_t)env_id, (uint32_t)step, (uint32_t)(step >> 32),
                                   stream ^ ((uint32_t)(env_id >> 32) << 8), (uint32_t)seed, (uint32_t)(seed >> 32)));
}
// the same draw from the round keys of `seed` (philox_round_keys)
__device__ __forceinline__ Uniform8 philox_uniform8x16(const PhiloxKeys& K, uint64_t env_id, uint64_t step, uint32_t stream) {
  return uniform8x16(philox4x32_10((uint32_t)env_id, (uint32_t)step, (uint32_t)(step >> 32),
                                   stream ^ ((uint32_t)(env_id >> 32) << 8), K));
}

// Philox stream ids used by the fused env step (DESIGN.md "RNG streams")
enum : uint32_t {
  RS_STEP_A = 0,   // 8x16-bit: act0, act1, vel_x, vel_y, vel_r, heading, pos_x, pos_y
  RS_STEP_B = 1,   // (reserved)
  RS_RESET_0 = 2,  // goal_x, goal_y, spawn_r, spawn_theta
  RS_RESET_1 = 3,  // spawn_yaw, vel_x, vel_y, mass
  RS_RESET_2 = 4,  // (com_x, com_y, com_z reserved), k_drag
  RS_RESET_3 = 5,  // lin_u, lin_v, lin_r, thr_shared
  RS_RESET_4 = 6,  // quad_u, quad_v, quad_r, thr_left
  RS_RESET_5 = 7,  // thr_right, k_Iz, force_x_freq, force_y_freq
  RS_RESET_6 = 8,  // force_x_shift, force_y_shift, force_amp, force_const_r
  RS_RESET_7 = 9,  // force_const_theta, torque_freq, torque_shift, torque_amp
  RS_RESET_8 = 10, // torque_const_r, torque_sign, -, -
  RS_RESET_COM = 11,  // live: com_x, com_y, com_z, target_heading (GoToPose)
  RS_RESET_TASK = 12, // TrackXYVelocity: target_vx, target_vy, -, -
  RS_OBST = 0x1000, // live scene builder: stream RS_OBST + round*8 + j/2 (round 0..20); obstacle j takes (a,b) if j even else (c,d)
  RS_ROWS = 64     // usv_randomize_rows_f32: stream = RS_ROWS + stream_id*16 + col/4
};

}  // namespace usv
