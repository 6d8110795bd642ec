// Shared host/device helpers for libusv_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include "../../include/usv_b200.h"

namespace usv {

extern std::atomic<int64_t> g_launch_count;

inline int finish_launch(int n_launches = 1) {
  g_launch_count.fetch_add(n_launches, std::memory_order_relaxed);
  cudaError_t e = cudaPeekAtLastError();
  return e == cudaSuccess ? USV_OK : (int)cudaGetLastError();
}

inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

// Attribute A of the current device, queried once per device; `fallback` when the query fails.  Concurrent first calls on one
// device store the same value.
template <cudaDeviceAttr A>
inline int device_attr(int fallback) {
  constexpr int kMaxDevices = 64;
  static std::atomic<int> cached[kMaxDevices];
  int dev = 0;
  cudaGetDevice(&dev);
  const bool keyed = dev >= 0 && dev < kMaxDevices;
  int n = keyed ? cached[dev].load(std::memory_order_relaxed) : 0;
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, A, dev) != cudaSuccess || n <= 0) n = fallback;
    if (keyed) cached[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

// SM count and L2 size in bytes of the current device (a B200's when the query fails)
inline int num_sms() { return device_attr<cudaDevAttrMultiProcessorCount>(148); }
inline int l2_bytes() { return device_attr<cudaDevAttrL2CacheSize>(126 << 20); }

// Lets `kernel` launch with `bytes` of dynamic shared memory on the current device.  The largest size set per (kernel, device) is
// remembered and the attribute is set again only when a request exceeds it: some kernels' sizes depend on their arguments.
inline void ensure_dynamic_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> set_bytes;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = set_bytes[{kernel, dev}];
  if (bytes > have && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess) have = bytes;
}
template <typename... Args>
inline void ensure_dynamic_smem(void (*kernel)(Args...), size_t bytes) {
  ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), bytes);
}

// rotation-matrix rows needed for R^T v with R = quaternion_to_matrix(q), q = (r,i,j,k) real-first,
// two_s = 2/|q|^2  (public PyTorch3D formula; see oracle/ref_shim.py for the restatement we pin)
struct Rot3 {
  float m00, m01, m02, m10, m11, m12, m20, m21, m22;
};

__device__ __forceinline__ Rot3 quat_to_matrix(float r, float i, float j, float k) {
  const float two_s = 2.0f / (r * r + i * i + j * j + k * k);
  Rot3 R;
  R.m00 = 1.0f - two_s * (j * j + k * k);
  R.m01 = two_s * (i * j - k * r);
  R.m02 = two_s * (i * k + j * r);
  R.m10 = two_s * (i * j + k * r);
  R.m11 = 1.0f - two_s * (i * i + k * k);
  R.m12 = two_s * (j * k - i * r);
  R.m20 = two_s * (i * k - j * r);
  R.m21 = two_s * (j * k + i * r);
  R.m22 = 1.0f - two_s * (i * i + j * j);
  return R;
}

// (R^T v)
__device__ __forceinline__ void rot_t_apply(const Rot3& R, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = R.m00 * x + R.m10 * y + R.m20 * z;
  oy = R.m01 * x + R.m11 * y + R.m21 * z;
  oz = R.m02 * x + R.m12 * y + R.m22 * z;
}

// thruster LUT index: clamp(round_half_even(((cmd+1)/2)*(n-1)), 0, n-1) with torch's op order
// (no FMA contraction: the index must be bit-exact)  [ref: OIGE/envs/USV/ThrusterDynamics.py:187-191]
__device__ __forceinline__ int lut_index(float cmd, int n_lut) {
  float t = __fmul_rn(__fmul_rn(__fadd_rn(cmd, 1.0f), 0.5f), (float)(n_lut - 1));
  float rr = rintf(t);  // round-half-to-even == torch.round
  int idx = (int)rr;
  // NaN -> (long)NaN is UB in the reference; we pin it to 0
  if (!(rr >= 0.0f)) idx = 0;
  if (idx > n_lut - 1) idx = n_lut - 1;
  return idx;
}

// Peer exchange packets: one 8-byte {fp32 payload, sequence number} store is both the value and its flag, so a receiver that sees this
// step's sequence number in a packet also sees its payload (the store is one 64-bit access).  Used by the fused rl_games minibatch
// tail (ppo_mlp_tc_impl.inc) and the loopz exchanges (ppo_loopz_peer.cu).  A peer that does not show up within kPeerSpinNs is an error.
constexpr unsigned long long kPeerSpinNs = 10ull * 1000 * 1000 * 1000;
__device__ __forceinline__ void st_packet(float* p, float v, uint32_t seq) {
  asm volatile("st.volatile.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(seq) : "memory");
}
__device__ __forceinline__ bool ld_packet(const float* p, uint32_t seq, float& v) {
  uint32_t a, b;
  asm volatile("ld.volatile.global.v2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "l"(p) : "memory");
  v = __uint_as_float(a);
  return b == seq;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

}  // namespace usv
