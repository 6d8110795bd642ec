// The USV SysID / DAgger student on the device (SURVEY 8(f) row 4, second half), sm_100a.
//
//   StateHistoryEncoder.forward            [ref: OIGE/algo/ppo/module.py:392-448]
//   USVSysIDTrainer._train_step            [ref: OIGE/algo/ppo/dagger.py:125-196]  MSE to the frozen teacher latent, Adam(5e-4)
//   teacher latent / frozen action head    [ref: OIGE/algo/ppo/dagger.py:50-66]    small LeakyReLU MLPs (mlp_forward_kernel)
//
// Network (tsteps = 50; 20 and 10 have two conv layers): per-step Linear(In, 32) + act over the T history frames, the (bs*T, 32)
// projection RESHAPED (not transposed -- reference quirk, kept) to (bs, 32 channels, T), Conv1d(32,32,k,s) + LeakyReLU stack down to
// length 3, flatten (96), Linear(96, Out) + act.  ~0.37 MFLOP forward per sample; 20 136 parameters at In = 25, Out = 8.
//
// Mapping.  Every layer has 32 output channels, so a WARP owns a sample and lane = output channel (forward) or = input channel (the
// transposed convolutions of the backward pass).  All weights live in shared memory once, in layouts that are bank-conflict-free for
// BOTH directions: conv weights as [ci][k][co] with the ci-stride padded by one word (lane = co: consecutive words; lane = ci: stride
// 32 k + 1, odd), the output layer as [i][j] with stride Out + 1.  Activations are broadcast reads.  A CTA (8 warps) walks chunks of
// 8 samples; between the per-warp stages of the backward pass the whole CTA accumulates the weight gradients of the chunk into
// REGISTERS (each thread owns ~83 fixed parameters for the CTA's lifetime: no atomics, fixed summation order, deterministic) and the
// gradient w.r.t. a layer's input then overwrites that layer's input in place.  One partial gradient per CTA goes to global memory;
// the Adam kernel sums the partials in a fixed order.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <type_traits>
#include "usv_common.cuh"

namespace dagger {

constexpr int C = 32;              // channels of every hidden layer
constexpr int kWarps = 8, kThreads = kWarps * 32;
constexpr float kLeaky = 0.01f;    // nn.LeakyReLU default slope (the USV script passes LeakyReLU as activation_fn as well)

__device__ __forceinline__ float lrelu(float x) { return x > 0.f ? x : kLeaky * x; }
__device__ __forceinline__ float dlrelu_from_out(float y) { return y > 0.f ? 1.0f : kLeaky; }   // sign(pre) == sign(post) for slope > 0

// conv stack per history length  [module.py:404-436]
template <int T> struct Spec;
#define DAGGER_SPEC(TT, NCV, K0, K1, K2, S0, S1, S2, L0, L1, L2, L3)                                                            \
  template <> struct Spec<TT> {                                                                                                   \
    static constexpr int NC = NCV;                                                                                                \
    __host__ __device__ static constexpr int K(int i) { return i == 0 ? K0 : (i == 1 ? K1 : K2); }                                \
    __host__ __device__ static constexpr int S(int i) { return i == 0 ? S0 : (i == 1 ? S1 : S2); }                                \
    __host__ __device__ static constexpr int L(int i) { return i == 0 ? L0 : (i == 1 ? L1 : (i == 2 ? L2 : L3)); }                \
  }
DAGGER_SPEC(50, 3, 8, 5, 5, 4, 1, 1, 50, 11, 7, 3);
DAGGER_SPEC(20, 2, 6, 4, 1, 2, 2, 1, 20, 8, 3, 3);
DAGGER_SPEC(10, 2, 4, 2, 1, 2, 1, 1, 10, 4, 3, 3);

struct Offsets {   // flat parameter vector, StateHistoryEncoder.parameters() order
  int w0, b0, wc[3], bc[3], wl, bl, P;
};
template <int T>
__host__ __device__ inline Offsets offsets(int In, int Out) {
  Offsets o;
  int p = 0;
  o.w0 = p; p += C * In; o.b0 = p; p += C;
  for (int i = 0; i < 3; ++i) {
    o.wc[i] = p; o.bc[i] = p;
    if (i < Spec<T>::NC) { p += C * C * Spec<T>::K(i); o.bc[i] = p; p += C; }
  }
  o.wl = p; p += Out * C * 3; o.bl = p; p += Out;
  o.P = p;
  return o;
}

// shared-memory weight block (floats): W0t[In][32] | b0[32] | per conv: Wc[ci][k][co] (ci-stride 32 k + 1) | bc[32] | Wl[i][j] (stride Out+1) | bl[Out]
template <int T>
struct SmemW {
  int w0, b0, wc[3], bc[3], wl, bl, total;
  __host__ __device__ SmemW(int In, int Out) {
    int p = 0;
    w0 = p; p += In * C; b0 = p; p += C;
    for (int i = 0; i < 3; ++i) {
      wc[i] = p; bc[i] = p;
      if (i < Spec<T>::NC) { p += C * (C * Spec<T>::K(i) + 1); bc[i] = p; p += C; }
    }
    wl = p; p += 3 * C * (Out + 1); bl = p; p += Out;
    total = (p + 3) & ~3;
  }
};
// per-sample activation block: hist[T*In] | y[32*T] | c_i[32*L_i] ... | dout[Out]   (the gradients overwrite y / c_i in place)
template <int T>
struct SmemA {
  int hist, y, c[3], dout, total;
  __host__ __device__ SmemA(int In, int Out) {
    int p = 0;
    hist = p; p += T * In; y = p; p += C * T;
    for (int i = 0; i < 3; ++i) { c[i] = p; if (i < Spec<T>::NC) p += C * Spec<T>::L(i + 1); }
    dout = p; p += Out;
    total = (p + 3) & ~3;
  }
};

template <int T>
__device__ void load_weights(float* sw, const float* __restrict__ prm, int In, int Out) {
  const Offsets o = offsets<T>(In, Out);
  const SmemW<T> s(In, Out);
  for (int q = threadIdx.x; q < C * In; q += blockDim.x) { const int f = q / In, d = q - f * In; sw[s.w0 + d * C + f] = prm[o.w0 + q]; }
  for (int q = threadIdx.x; q < C; q += blockDim.x) sw[s.b0 + q] = prm[o.b0 + q];
#pragma unroll
  for (int i = 0; i < Spec<T>::NC; ++i) {
    const int K = Spec<T>::K(i);
    for (int q = threadIdx.x; q < C * C * K; q += blockDim.x) {   // prm: [co][ci][k]
      const int co = q / (C * K), r = q - co * (C * K), ci = r / K, k = r - ci * K;
      sw[s.wc[i] + ci * (C * K + 1) + k * C + co] = prm[o.wc[i] + q];
    }
    for (int q = threadIdx.x; q < C; q += blockDim.x) sw[s.bc[i] + q] = prm[o.bc[i] + q];
  }
  for (int q = threadIdx.x; q < Out * 3 * C; q += blockDim.x) { const int j = q / (3 * C), i = q - j * (3 * C); sw[s.wl + i * (Out + 1) + j] = prm[o.wl + q]; }
  for (int q = threadIdx.x; q < Out; q += blockDim.x) sw[s.bl + q] = prm[o.bl + q];
}

// one conv layer forward for one sample: lane = co; in[ci*LIN + t], out[co*LOUT + l]
template <int K, int S, int LIN, int LOUT>
__device__ __forceinline__ void conv_fwd(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ in,
                                         float* __restrict__ out, int lane) {
  float acc[LOUT];
#pragma unroll
  for (int l = 0; l < LOUT; ++l) acc[l] = b[lane];
  for (int ci = 0; ci < C; ++ci) {
    const float* wr = w + ci * (C * K + 1) + lane;
    const float* xr = in + ci * LIN;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float wv = wr[k * C];
#pragma unroll
      for (int l = 0; l < LOUT; ++l) acc[l] = fmaf(wv, xr[l * S + k], acc[l]);
    }
  }
#pragma unroll
  for (int l = 0; l < LOUT; ++l) out[lane * LOUT + l] = lrelu(acc[l]);
}

// transposed conv for one sample: lane = ci; din[ci*LIN + t] = (sum_{co,k,l: l*S+k = t} W[co][ci][k] * dout[co*LOUT + l]) * act'(in[ci*LIN + t]),
// written IN PLACE over `in` (the forward input of the layer, post-activation of the layer below)
template <int K, int S, int LIN, int LOUT>
__device__ __forceinline__ void conv_bwd_input(const float* __restrict__ w, const float* __restrict__ dout, float* __restrict__ in, int lane) {
  float acc[LIN];
#pragma unroll
  for (int t = 0; t < LIN; ++t) acc[t] = 0.f;
  const float* wr = w + lane * (C * K + 1);
  for (int co = 0; co < C; ++co) {
    float d[LOUT];
#pragma unroll
    for (int l = 0; l < LOUT; ++l) d[l] = dout[co * LOUT + l];   // broadcast
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float wv = wr[k * C + co];
#pragma unroll
      for (int l = 0; l < LOUT; ++l) acc[l * S + k] = fmaf(wv, d[l], acc[l * S + k]);
    }
  }
#pragma unroll
  for (int t = 0; t < LIN; ++t) {
    float* p = in + lane * LIN + t;
    *p = acc[t] * dlrelu_from_out(*p);
  }
}

// forward of one sample by one warp; returns the Out outputs replicated in every lane's out[] (Out <= 8)
template <int T>
__device__ __forceinline__ void sample_forward(const float* sw, float* a, int In, int Out, int lane, float (&out)[8]) {
  using SP = Spec<T>;
  const SmemW<T> s(In, Out);
  const SmemA<T> m(In, Out);
  // per-step projection: y[step*32 + f] = act(b0[f] + sum_d W0[f][d] hist[step*In + d]),  lane = f
  for (int st = 0; st < T; ++st) {
    float acc = sw[s.b0 + lane];
    const float* h = a + m.hist + st * In;
    for (int d = 0; d < In; ++d) acc = fmaf(sw[s.w0 + d * C + lane], h[d], acc);
    a[m.y + st * C + lane] = lrelu(acc);
  }
  __syncwarp();
  // the reference's reshape: channel c of the conv input is flat[c*T .. c*T + T)
  conv_fwd<SP::K(0), SP::S(0), SP::L(0), SP::L(1)>(sw + s.wc[0], sw + s.bc[0], a + m.y, a + m.c[0], lane);
  __syncwarp();
  conv_fwd<SP::K(1), SP::S(1), SP::L(1), SP::L(2)>(sw + s.wc[1], sw + s.bc[1], a + m.c[0], a + m.c[1], lane);
  __syncwarp();
  if constexpr (SP::NC == 3) {
    conv_fwd<SP::K(2), SP::S(2), SP::L(2), SP::L(3)>(sw + s.wc[2], sw + s.bc[2], a + m.c[1], a + m.c[2], lane);
    __syncwarp();
  }
  const float* top = a + m.c[SP::NC - 1];       // 96 values, flatten order co*3 + l
  float part[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) part[j] = 0.f;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int i = r * C + lane;
    const float x = top[i];
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < Out) part[j] = fmaf(sw[s.wl + i * (Out + 1) + j], x, part[j]);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = part[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    out[j] = (j < Out) ? lrelu(v + sw[s.bl + (j < Out ? j : 0)]) : 0.f;
  }
}

template <int T>
__host__ __device__ inline size_t fwd_smem_bytes(int In, int Out) { return (size_t)(SmemW<T>(In, Out).total + kWarps * SmemA<T>(In, Out).total) * sizeof(float); }

__device__ __forceinline__ void stage_hist(float* dst, const float* __restrict__ src, int n, int lane) {
  for (int q = lane; q < n; q += 32) dst[q] = src[q];
}

// How a kernel finds sample r's window (T * In floats, oldest frame first).  RowWindows: row r of a [M][ld] matrix.
struct RowWindows {
  const float* __restrict__ hist;
  int64_t ld;
  __device__ __forceinline__ void operator()(float* dst, int64_t r, int n, int lane) const { stage_hist(dst, hist + r * ld, n, lane); }
};

// StoreWindows: the frame store of a rollout.  store[N][S][In] (S = T - 1 + H) holds each frame once: index t + T - 1 is the frame of
// rollout step t, indices 0 .. T - 1 the window of step 0.  refill[H][N] is the store index of the last "repeat" refill at or before
// step t (0: none).  Global row g = t * N + e (the time-major order of ObsStorage) is window(t) of env e, whose element k is
// store[e][max(t + k, refill[t][e])]: a contiguous span when nothing was refilled, else the refill frame repeated below it.
struct StoreWindows {
  const float* __restrict__ store;
  const int* __restrict__ refill;
  int64_t row0, N;
  int S, In;
  __device__ __forceinline__ void operator()(float* dst, int64_t r, int n, int lane) const {
    const int64_t g = row0 + r, t = g / N, e = g - t * N;
    const float* src = store + (e * S + t) * In;
    const int lo = (refill[g] - (int)t) * In;                          // elements below lo repeat the frame that starts at lo
    if (lo <= 0) stage_hist(dst, src, n, lane);                        // the common case keeps the row copy's pipelined loads
    else
      for (int q = lane; q < n; q += 32) dst[q] = src[q < lo ? lo + q % In : q];
  }
};

// ---- inference: out[M, Out] = StateHistoryEncoder(window of row r) ----------------------------------------------------------------------
template <int T, class Win>
__device__ __forceinline__ void encoder_forward(const float* __restrict__ prm, Win win, int In, int Out, float* __restrict__ out, int64_t M) {
  extern __shared__ __align__(16) float smem[];
  const SmemW<T> s(In, Out);
  const SmemA<T> m(In, Out);
  load_weights<T>(smem, prm, In, Out);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* a = smem + s.total + warp * m.total;
  for (int64_t r = (int64_t)blockIdx.x * kWarps + warp; r < M; r += (int64_t)gridDim.x * kWarps) {
    win(a + m.hist, r, T * In, lane);
    __syncwarp();
    float o[8];
    sample_forward<T>(smem, a, In, Out, lane, o);
    if (lane < Out) {
      float v = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) if (j == lane) v = o[j];
      out[r * Out + lane] = v;
    }
    __syncwarp();
  }
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) encoder_forward_kernel(const float* __restrict__ prm, const float* __restrict__ hist, int64_t ld,
                                                                      int In, int Out, float* __restrict__ out, int64_t M) {
  encoder_forward<T>(prm, RowWindows{hist, ld}, In, Out, out, M);
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) encoder_forward_store_kernel(const float* __restrict__ prm, StoreWindows win, int In, int Out,
                                                                            float* __restrict__ out, int64_t M) {
  encoder_forward<T>(prm, win, In, Out, out, M);
}

// ---- training: MSE(encoder(hist), zstar) forward + backward; one partial gradient per CTA -------------------------------------------------
// partial layout: [P gradient | sum of squared errors | unused x3], stride P + 4.  tid: threadIdx.x read in the kernel, whose
// __launch_bounds__ bound it there (the range does not reach reads inside an inlined body, and the owner maps below use it).
template <int T, class Win>
__device__ __forceinline__ void train(const float* __restrict__ prm, Win win, const float* __restrict__ zstar, int In, int Out,
                                      float* __restrict__ partial, int64_t M, unsigned tid) {
  using SP = Spec<T>;
  extern __shared__ __align__(16) float smem[];
  const SmemW<T> s(In, Out);
  const SmemA<T> m(In, Out);
  const Offsets o = offsets<T>(In, Out);
  load_weights<T>(smem, prm, In, Out);
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  float* abase = smem + s.total;
  float* a = abase + warp * m.total;
  constexpr int K0 = SP::K(0), K1 = SP::K(1), K2 = SP::K(2);
  constexpr int P0 = C * K0 / kWarps, P1 = C * K1 / kWarps, P2 = (SP::NC == 3) ? C * K2 / kWarps : 1;   // (ci,k) pairs per warp
  static_assert((C * K0) % kWarps == 0 && (C * K1) % kWarps == 0 && (C * K2) % kWarps == 0, "pairs divide over the warps");
  // register accumulators: lane = co (convs), f (W0), i mod 32 (Wl); the warp picks the (ci,k) pairs / input columns / output row
  float g0[4] = {0.f, 0.f, 0.f, 0.f}, gb0 = 0.f;          // dW0[f = lane][d = warp + 8 q], db0 (warp 0)
  float g1[P0], g2[P1], g3[P2], gbc[3] = {0.f, 0.f, 0.f}; // conv weights; biases owned by warp 0 / 1 / 2
  float gl[3] = {0.f, 0.f, 0.f}, gbl = 0.f;               // dWl[j = warp][i = lane + 32 r] (Out <= 8 rows per pass), dbl
  float sse = 0.f;
#pragma unroll
  for (int j = 0; j < P0; ++j) g1[j] = 0.f;
#pragma unroll
  for (int j = 0; j < P1; ++j) g2[j] = 0.f;
#pragma unroll
  for (int j = 0; j < P2; ++j) g3[j] = 0.f;
  const float inv = 2.0f / ((float)M * (float)Out);       // d mean((out - z)^2) / d out
  const int64_t nchunks = (M + kWarps - 1) / kWarps;
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t r = ch * kWarps + warp;
    const bool valid = r < M;
    // ---- per warp: forward, output gradient ----
    if (valid) {
      win(a + m.hist, r, T * In, lane);
      __syncwarp();
      float out[8];
      sample_forward<T>(smem, a, In, Out, lane, out);
      if (lane < Out) {
        float v = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j == lane) v = out[j];
        const float e = v - zstar[r * Out + lane];
        sse += e * e;
        a[m.dout + lane] = inv * e * dlrelu_from_out(v);
      }
    } else {
      // a padding sample contributes zeros everywhere: clear what the CTA-wide phases read
      for (int q = lane; q < m.total; q += 32) a[q] = 0.f;
    }
    __syncthreads();
    // ---- CTA: dWl[j][i] += dout[j] c_top[i];  warp = j (Out <= 8), lane + 32 r = i ----
    {
      const int top = m.c[SP::NC - 1];
      for (int sidx = 0; sidx < kWarps; ++sidx) {
        const float* as = abase + sidx * m.total;
        if (warp < Out) {
          const float d = as[m.dout + warp];
#pragma unroll
          for (int q = 0; q < 3; ++q) gl[q] = fmaf(d, as[top + q * C + lane], gl[q]);
          if (lane == 0) gbl += d;
        }
      }
    }
    __syncthreads();
    // ---- per warp: d c_top[i] = (sum_j Wl[j][i] dout[j]) * act'(c_top[i]), in place ----
    {
      float* top = a + m.c[SP::NC - 1];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int i = q * C + lane;
        float acc = 0.f;
        for (int j = 0; j < Out; ++j) acc = fmaf(smem[s.wl + i * (Out + 1) + j], a[m.dout + j], acc);
        top[i] = acc * dlrelu_from_out(top[i]);
      }
    }
    __syncthreads();
    // ---- conv layers from the top down: CTA-wide weight gradient, then the per-warp input gradient in place ----
    if constexpr (SP::NC == 3) {
      constexpr int LIN = SP::L(2), LOUT = SP::L(3);
      for (int sidx = 0; sidx < kWarps; ++sidx) {
        const float* as = abase + sidx * m.total;
        float d[LOUT];
#pragma unroll
        for (int l = 0; l < LOUT; ++l) d[l] = as[m.c[2] + lane * LOUT + l];
#pragma unroll
        for (int j = 0; j < P2; ++j) {
          const int pr = warp * P2 + j, ci = pr / K2, k = pr - ci * K2;
#pragma unroll
          for (int l = 0; l < LOUT; ++l) g3[j] = fmaf(d[l], as[m.c[1] + ci * LIN + l * SP::S(2) + k], g3[j]);
        }
        if (warp == 2) {
#pragma unroll
          for (int l = 0; l < LOUT; ++l) gbc[2] += d[l];
        }
      }
      __syncthreads();
      conv_bwd_input<K2, SP::S(2), LIN, LOUT>(smem + s.wc[2], a + m.c[2], a + m.c[1], lane);
      __syncthreads();
    }
    {
      constexpr int LIN = SP::L(1), LOUT = SP::L(2);
      for (int sidx = 0; sidx < kWarps; ++sidx) {
        const float* as = abase + sidx * m.total;
        float d[LOUT];
#pragma unroll
        for (int l = 0; l < LOUT; ++l) d[l] = as[m.c[1] + lane * LOUT + l];
#pragma unroll
        for (int j = 0; j < P1; ++j) {
          const int pr = warp * P1 + j, ci = pr / K1, k = pr - ci * K1;
#pragma unroll
          for (int l = 0; l < LOUT; ++l) g2[j] = fmaf(d[l], as[m.c[0] + ci * LIN + l * SP::S(1) + k], g2[j]);
        }
        if (warp == 1) {
#pragma unroll
          for (int l = 0; l < LOUT; ++l) gbc[1] += d[l];
        }
      }
      __syncthreads();
      conv_bwd_input<K1, SP::S(1), LIN, LOUT>(smem + s.wc[1], a + m.c[1], a + m.c[0], lane);
      __syncthreads();
    }
    {
      constexpr int LIN = SP::L(0), LOUT = SP::L(1);
      for (int sidx = 0; sidx < kWarps; ++sidx) {
        const float* as = abase + sidx * m.total;
        float d[LOUT];
#pragma unroll
        for (int l = 0; l < LOUT; ++l) d[l] = as[m.c[0] + lane * LOUT + l];
#pragma unroll
        for (int j = 0; j < P0; ++j) {
          const int pr = warp * P0 + j, ci = pr / K0, k = pr - ci * K0;
#pragma unroll
          for (int l = 0; l < LOUT; ++l) g1[j] = fmaf(d[l], as[m.y + ci * LIN + l * SP::S(0) + k], g1[j]);
        }
        if (warp == 0) {
#pragma unroll
          for (int l = 0; l < LOUT; ++l) gbc[0] += d[l];
        }
      }
      __syncthreads();
      conv_bwd_input<K0, SP::S(0), LIN, LOUT>(smem + s.wc[0], a + m.c[0], a + m.y, lane);
      __syncthreads();
    }
    // ---- CTA: dW0[f][d] += sum_step dy[step*32 + f] hist[step*In + d];  lane = f, d = warp + 8 q ----
    for (int sidx = 0; sidx < kWarps; ++sidx) {
      const float* as = abase + sidx * m.total;
      for (int st = 0; st < T; ++st) {
        const float dy = as[m.y + st * C + lane];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int d = warp + kWarps * q;
          if (d < In) g0[q] = fmaf(dy, as[m.hist + st * In + d], g0[q]);
        }
        if (warp == 0) gb0 += dy;
      }
    }
    __syncthreads();
  }
  // ---- this CTA's partial gradient (every parameter has exactly one owner thread) ----
  float* out = partial + (size_t)blockIdx.x * (o.P + 4);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int d = warp + kWarps * q;
    if (d < In) out[o.w0 + lane * In + d] = g0[q];
  }
  if (warp == 0) out[o.b0 + lane] = gb0;
#pragma unroll
  for (int j = 0; j < P0; ++j) { const int pr = warp * P0 + j, ci = pr / K0, k = pr - ci * K0; out[o.wc[0] + (lane * C + ci) * K0 + k] = g1[j]; }
#pragma unroll
  for (int j = 0; j < P1; ++j) { const int pr = warp * P1 + j, ci = pr / K1, k = pr - ci * K1; out[o.wc[1] + (lane * C + ci) * K1 + k] = g2[j]; }
  if constexpr (SP::NC == 3) {
#pragma unroll
    for (int j = 0; j < P2; ++j) { const int pr = warp * P2 + j, ci = pr / K2, k = pr - ci * K2; out[o.wc[2] + (lane * C + ci) * K2 + k] = g3[j]; }
  }
  if (warp < SP::NC) out[o.bc[warp] + lane] = warp == 0 ? gbc[0] : (warp == 1 ? gbc[1] : gbc[2]);
  if (warp < Out) {
#pragma unroll
    for (int q = 0; q < 3; ++q) out[o.wl + warp * (3 * C) + q * C + lane] = gl[q];
    if (lane == 0) out[o.bl + warp] = gbl;
  }
  // squared error: lanes < Out of every warp hold a share
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, of);
  __shared__ float s_sse[kWarps];
  if (lane == 0) s_sse[warp] = sse;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kWarps; ++w) t += s_sse[w];
    out[o.P] = t;
  }
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) train_kernel(const float* __restrict__ prm, const float* __restrict__ hist, int64_t ld,
                                                            const float* __restrict__ zstar, int In, int Out, float* __restrict__ partial, int64_t M) {
  train<T>(prm, RowWindows{hist, ld}, zstar, In, Out, partial, M, threadIdx.x);
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) train_store_kernel(const float* __restrict__ prm, StoreWindows win, const float* __restrict__ zstar,
                                                                  int In, int Out, float* __restrict__ partial, int64_t M) {
  train<T>(prm, win, zstar, In, Out, partial, M, threadIdx.x);
}

// second stage + Adam (torch.optim.Adam defaults, no clipping) in one launch: grads[P + 1] = [gradient | mse]
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ prm, const float* __restrict__ partial, int nparts, int P, float* __restrict__ grads,
                                                   float* __restrict__ m, float* __restrict__ v, const float* __restrict__ lr, int* __restrict__ step,
                                                   int parity, float inv_count, float* __restrict__ mse_accum) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int stp = step[parity] + 1;
  if (e < P) {
    float g = 0.f;
    for (int c = 0; c < nparts; ++c) g += partial[(size_t)c * (P + 4) + e];
    grads[e] = g;
    const double bc1 = 1.0 - pow(0.9, (double)stp), bc2 = 1.0 - pow(0.999, (double)stp);
    const float step_size = (float)((double)lr[0] / bc1), bc2_sqrt = (float)sqrt(bc2);
    const float mm = m[e] + (g - m[e]) * (1.0f - 0.9f);
    const float vv = v[e] * 0.999f + (1.0f - 0.999f) * g * g;
    m[e] = mm;
    v[e] = vv;
    prm[e] = prm[e] - step_size * (mm / (sqrtf(vv) / bc2_sqrt + 1e-8f));
  }
  if (e == P) {
    float t = 0.f;
    for (int c = 0; c < nparts; ++c) t += partial[(size_t)c * (P + 4) + P];
    grads[P] = t * inv_count;            // nn.MSELoss (mean over samples and latent dims) of this minibatch, before the update
    if (mse_accum) *mse_accum += t * inv_count;
    step[1 - parity] = stp;
  }
}

// ---- small LeakyReLU MLP forward (teacher mass encoder, frozen action head): up to 3 Linear layers, widths <= 128 ------------------------------
struct MlpDesc {
  int nl;            // layers (<= 3)
  int dim[4];        // in, h1, h2, out
  int w[3], b[3];    // offsets into the flat vector (nn.Linear: weight [out][in], bias [out])
  int tanh_out;      // 1: tanh on the last layer, 0: LeakyReLU on the last layer, 2: no activation on the last layer
};
__global__ void __launch_bounds__(256) mlp_forward_kernel(const float* __restrict__ prm, MlpDesc d, const float* __restrict__ x, int64_t ldx,
                                                          float* __restrict__ y, int64_t M) {
  extern __shared__ __align__(16) float smem[];
  // transposed weights [in][out] (lane = output unit: conflict-free), then per-warp activation ping-pong buffers of 128 floats
  int off[3], p = 0;
  for (int l = 0; l < d.nl; ++l) { off[l] = p; p += d.dim[l] * d.dim[l + 1] + d.dim[l + 1]; }
  for (int l = 0; l < d.nl; ++l) {
    const int I = d.dim[l], O = d.dim[l + 1];
    for (int q = threadIdx.x; q < I * O; q += blockDim.x) { const int o = q / I, i = q - o * I; smem[off[l] + i * O + o] = prm[d.w[l] + q]; }
    for (int q = threadIdx.x; q < O; q += blockDim.x) smem[off[l] + I * O + q] = prm[d.b[l] + q];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float* buf = smem + ((p + 3) & ~3) + warp * 256;
  for (int64_t r = (int64_t)blockIdx.x * nw + warp; r < M; r += (int64_t)gridDim.x * nw) {
    for (int q = lane; q < d.dim[0]; q += 32) buf[q] = x[r * ldx + q];
    __syncwarp();
    float* in = buf;
    float* out = buf + 128;
    for (int l = 0; l < d.nl; ++l) {
      const int I = d.dim[l], O = d.dim[l + 1];
      const float* w = smem + off[l];
      for (int o = lane; o < O; o += 32) {
        float acc = w[I * O + o];
        for (int i = 0; i < I; ++i) acc = fmaf(w[i * O + o], in[i], acc);
        const bool last = l == d.nl - 1;
        out[o] = (last && d.tanh_out == 1) ? tanhf(acc) : ((last && d.tanh_out == 2) ? acc : lrelu(acc));
      }
      __syncwarp();
      float* t = in; in = out; out = t;
    }
    for (int q = lane; q < d.dim[d.nl]; q += 32) y[r * d.dim[d.nl] + q] = in[q];
    __syncwarp();
  }
}

// ---- deployment: the student's control step = history ring update + encoder + frozen action head, one launch ----------------------------
// ring[M][T][D] holds each env's last T frames; slot[0] is the slot of the oldest frame, which the launch overwrites with the current frame,
// so the frames in chronological order are slots p+1, ..., p+T-1, p (mod T) afterwards.  slot[1] counts the CTAs that have read slot[0];
// the last one advances slot[0] and clears the count, so the index lives on the device and a captured graph can replay the launch.
// Head weights live in shared memory as [out][in + 1] (lane = output unit: row stride in + 1 is conflict-free, and the copy from the
// nn.Linear [out][in] layout is coalesced) followed by the bias.  Where they do not fit beside the encoder's weights and the 8 activation
// blocks (T = 50: 81 + 113 + 84 KB), the CTA works in two phases: the encoder, then the head weights copied over the dead activation
// blocks (from L2, coalesced), then the head.
__host__ __device__ inline int head_smem_floats(const MlpDesc& d, int* off) {
  int p = 0;
  for (int l = 0; l < d.nl; ++l) { off[l] = p; p += d.dim[l + 1] * (d.dim[l] + 1) + d.dim[l + 1]; }
  return (p + 3) & ~3;
}

__device__ void load_head(float* sh, const float* __restrict__ prm, const MlpDesc& d, const int* off) {
  for (int l = 0; l < d.nl; ++l) {
    const int I = d.dim[l], O = d.dim[l + 1];
    for (int q = threadIdx.x; q < I * O; q += blockDim.x) { const int o = q / I, i = q - o * I; sh[off[l] + o * (I + 1) + i] = prm[d.w[l] + q]; }
    for (int q = threadIdx.x; q < O; q += blockDim.x) sh[off[l] + O * (I + 1) + q] = prm[d.b[l] + q];
  }
}

// the frozen head on buf[0, dim[0]) for one sample by one warp, in mlp_forward_kernel's fmaf order (bit-identical); returns the output row
__device__ __forceinline__ const float* head_forward(const float* sh, const MlpDesc& d, const int* off, float* buf, int lane) {
  float* in = buf;
  float* out = buf + 128;
  for (int l = 0; l < d.nl; ++l) {
    const int I = d.dim[l], O = d.dim[l + 1];
    const float* w = sh + off[l];
    for (int o = lane; o < O; o += 32) {
      float acc = w[O * (I + 1) + o];
      const float* wr = w + o * (I + 1);
      for (int i = 0; i < I; ++i) acc = fmaf(wr[i], in[i], acc);
      const bool last = l == d.nl - 1;
      out[o] = (last && d.tanh_out == 1) ? tanhf(acc) : ((last && d.tanh_out == 2) ? acc : lrelu(acc));
    }
    __syncwarp();
    float* t = in; in = out; out = t;
  }
  return in;
}

template <int T>
__host__ __device__ inline size_t act_block_floats(int In, int Out) { return (size_t)kWarps * SmemA<T>(In, Out).total; }

// Shared memory: encoder weights | 8 activation blocks | head weights (resident only) | 8 head ping-pong buffers | per warp, the head
// inputs [frame | z^] of G samples.  Split CTAs run the encoder over G chunks of their grid-stride sequence, then copy the head over the
// activation blocks once and run it over the same G chunks: one head copy per G chunks (G = 16 covers 16 384 envs at T = 50 in one copy).
//
// The distillation's collect step (Collect = Distill) is the same step on rollout step t of H, plus: it writes window(t) into the frame
// store (StoreWindows: all T frames at t = 0, the new frame after that) and the refill index, and labels the sample with the frozen
// teacher's z* = mass_encoder(obs[:, D : D + priv]), in mlp_forward_kernel's fmaf order.  The teacher's weights sit behind the head's
// ([out][in + 1] as well), resident or over the dead activation blocks.  Deployment (Collect = NoDistill) compiles none of it.
struct NoDistill {
  static constexpr bool kOn = false;
};
struct Distill {
  static constexpr bool kOn = true;
  const float* __restrict__ teacher;   // flat parameters of the teacher's mass encoder
  MlpDesc td;                          // its layers: priv -> ... -> latent
  float* __restrict__ store;           // [M][S][D], S = T - 1 + H
  int* __restrict__ refill;            // [H][M]
  float* __restrict__ zstar;           // [H][M][latent]
  int t, S;
};

template <int T, class Collect>
__device__ __forceinline__ void student_step(const float* __restrict__ enc, const float* __restrict__ head, MlpDesc hd, float* __restrict__ ring,
                                             int* __restrict__ slot, const float* __restrict__ obs, int64_t obs_ld, int D, int Lat,
                                             const int64_t* __restrict__ dones, int repeat, int init, int resident, int G, float* __restrict__ mu,
                                             float* __restrict__ latent, int64_t M, Collect col) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int s_p;
  const SmemW<T> s(D, Lat);
  const SmemA<T> m(D, Lat);
  int hoff[3], toff[3];
  const int hfl = head_smem_floats(hd, hoff);
  int tfl = 0;
  if constexpr (Collect::kOn) tfl = head_smem_floats(col.td, toff);
  const int afl = (int)act_block_floats<T>(D, Lat);
  const int XS = D + Lat;
  float* act = smem + s.total;
  float* hw = resident ? act + afl : act;                                   // resident: beside the activations; else over them
  float* tw = hw + hfl;                                                     // the teacher's weights (collect only)
  float* bufs = resident ? hw + hfl + tfl : act + (afl > hfl + tfl ? afl : hfl + tfl);
  if (threadIdx.x == 0) s_p = slot[0];
  load_weights<T>(smem, enc, D, Lat);
  if (resident) {
    load_head(hw, head, hd, hoff);
    if constexpr (Collect::kOn) load_head(tw, col.teacher, col.td, toff);
  }
  __syncthreads();
  const int p = s_p;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* a = act + warp * m.total;
  float* buf = bufs + warp * 256;
  float* xs = bufs + kWarps * 256 + warp * G * XS;
  const int Oh = hd.dim[hd.nl];
  const int64_t nchunks = (M + kWarps - 1) / kWarps;
  const int64_t stride = (int64_t)gridDim.x * G;
  for (int64_t c0 = blockIdx.x; c0 < nchunks; c0 += stride) {
    // ---- phase 1, per warp: the ring update and the chronological staging in one pass, then the encoder; G chunks ----
    for (int g = 0; g < G; ++g) {
      const int64_t r = (c0 + (int64_t)g * gridDim.x) * kWarps + warp;
      if (r >= M) break;
      const bool fill = repeat && (init || (dones != nullptr && dones[r] != 0));
      if (lane < D) {
        const float f = obs[r * obs_ld + lane];
        float* rr = ring + r * (int64_t)T * D + lane;
        xs[g * XS + lane] = f;
        int sl = p + 1 == T ? 0 : p + 1;                                    // window element t lives in slot (p + 1 + t) mod T
#pragma unroll 10
        for (int t = 0; t < T; ++t) {
          const bool newest = t == T - 1;
          // "zeros" leaves a finished env's old frames in place (the reference zeroes an advanced-indexing copy); init zeroes the window
          const float v = (fill || newest) ? f : (init ? 0.f : rr[sl * D]);
          a[m.hist + t * D + lane] = v;
          if (fill || newest || init) rr[sl * D] = v;
          sl = sl + 1 == T ? 0 : sl + 1;
        }
        if constexpr (Collect::kOn)
          if (col.t > 0) col.store[(r * col.S + col.t + T - 1) * D + lane] = f;
      }
      __syncwarp();
      if constexpr (Collect::kOn) {
        if (col.t == 0)
          for (int q = lane; q < T * D; q += 32) col.store[r * col.S * D + q] = a[m.hist + q];
        if (lane == 0)
          col.refill[col.t * M + r] = fill ? col.t + T - 1 : (col.t == 0 ? 0 : col.refill[(col.t - 1) * M + r]);
      }
      float z[8];
      sample_forward<T>(smem, a, D, Lat, lane, z);
      if (lane < Lat) {
        float v = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j == lane) v = z[j];
        xs[g * XS + D + lane] = v;
        if (latent) latent[r * Lat + lane] = v;
      }
      __syncwarp();
    }
    if (!resident) {                       // every warp is past its encoder before the head overwrites the activation blocks
      __syncthreads();
      load_head(hw, head, hd, hoff);
      if constexpr (Collect::kOn) load_head(tw, col.teacher, col.td, toff);
      __syncthreads();
    }
    // ---- phase 2, per warp: the frozen head over the same G chunks ----
    for (int g = 0; g < G; ++g) {
      const int64_t r = (c0 + (int64_t)g * gridDim.x) * kWarps + warp;
      if (r >= M) break;
      if constexpr (Collect::kOn) {        // the label z* = teacher(priv tail)
        for (int q = lane; q < col.td.dim[0]; q += 32) buf[q] = obs[r * obs_ld + D + q];
        __syncwarp();
        const float* y = head_forward(tw, col.td, toff, buf, lane);
        for (int q = lane; q < Lat; q += 32) col.zstar[(col.t * M + r) * Lat + q] = y[q];
        __syncwarp();
      }
      for (int q = lane; q < XS; q += 32) buf[q] = xs[g * XS + q];
      __syncwarp();
      const float* y = head_forward(hw, hd, hoff, buf, lane);
      for (int q = lane; q < Oh; q += 32) mu[r * Oh + q] = y[q];
      __syncwarp();
    }
    if (!resident) __syncthreads();        // the next chunks' staging overwrites the head weights
  }
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(slot + 1, 1) == (int)gridDim.x - 1) {
      slot[0] = p + 1 == T ? 0 : p + 1;
      slot[1] = 0;
    }
  }
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) student_act_kernel(const float* __restrict__ enc, const float* __restrict__ head, MlpDesc hd,
                                                                  float* __restrict__ ring, int* __restrict__ slot, const float* __restrict__ obs,
                                                                  int64_t obs_ld, int D, int Lat, const int64_t* __restrict__ dones, int repeat,
                                                                  int init, int resident, int G, float* __restrict__ mu, float* __restrict__ latent,
                                                                  int64_t M) {
  student_step<T>(enc, head, hd, ring, slot, obs, obs_ld, D, Lat, dones, repeat, init, resident, G, mu, latent, M, NoDistill{});
}

template <int T>
__global__ void __launch_bounds__(kThreads, 1) sysid_collect_kernel(const float* __restrict__ enc, const float* __restrict__ head, MlpDesc hd,
                                                                    float* __restrict__ ring, int* __restrict__ slot, const float* __restrict__ obs,
                                                                    int64_t obs_ld, int D, int Lat, const int64_t* __restrict__ dones, int repeat,
                                                                    int init, int resident, int G, float* __restrict__ mu, int64_t M, Distill col) {
  student_step<T>(enc, head, hd, ring, slot, obs, obs_ld, D, Lat, dones, repeat, init, resident, G, mu, nullptr, M, col);
}

// col: the collect step's extra outputs, or nullptr for the deployment step
template <int T>
static int launch_student_act(const float* enc, const float* head, const MlpDesc& hd, float* ring, int* slot, const float* obs, int64_t obs_ld,
                              int D, int Lat, const int64_t* dones, int repeat, int init, float* mu, float* latent, int64_t M, const Distill* col,
                              cudaStream_t st) {
  constexpr size_t kMax = 227 * 1024 / sizeof(float);
  int hoff[3];
  const size_t hfl = (size_t)head_smem_floats(hd, hoff) + (col ? (size_t)head_smem_floats(col->td, hoff) : 0);   // + the teacher's
  const size_t afl = act_block_floats<T>(D, Lat), wfl = (size_t)SmemW<T>(D, Lat).total;
  const size_t bufs = (size_t)kWarps * 256, xs = (size_t)kWarps * (D + Lat);                       // xs: per sample of G
  const int resident = wfl + afl + hfl + bufs + xs <= kMax;
  const size_t fixed = resident ? wfl + afl + hfl + bufs : wfl + (afl > hfl ? afl : hfl) + bufs;
  if (fixed + xs > kMax) return USV_E_SIZE;
  const int G = resident ? 1 : (int)((kMax - fixed) / xs < 16 ? (kMax - fixed) / xs : 16);
  const size_t smem = (fixed + G * xs) * sizeof(float);
  const int64_t want = (M + kWarps - 1) / kWarps;
  const int sms = usv::num_sms();
  const int grid = (int)(want < sms ? want : sms);
  if (col) {
    usv::ensure_dynamic_smem(sysid_collect_kernel<T>, smem);
    sysid_collect_kernel<T><<<grid, kThreads, smem, st>>>(enc, head, hd, ring, slot, obs, obs_ld, D, Lat, dones, repeat, init, resident, G, mu, M,
                                                          *col);
  } else {
    usv::ensure_dynamic_smem(student_act_kernel<T>, smem);
    student_act_kernel<T><<<grid, kThreads, smem, st>>>(enc, head, hd, ring, slot, obs, obs_ld, D, Lat, dones, repeat, init, resident, G, mu,
                                                        latent, M);
  }
  return usv::finish_launch();
}

template <int T, class Win>
static int launch_forward(const float* prm, const Win& win, int In, int Out, float* out, int64_t M, cudaStream_t st) {
  const size_t smem = fwd_smem_bytes<T>(In, Out);
  if (smem > 227 * 1024) return USV_E_SIZE;
  const int64_t want = (M + kWarps - 1) / kWarps;
  const int sms = usv::num_sms();
  const int grid = (int)(want < sms ? want : sms);
  if constexpr (std::is_same<Win, RowWindows>::value) {
    usv::ensure_dynamic_smem(encoder_forward_kernel<T>, smem);
    encoder_forward_kernel<T><<<grid, kThreads, smem, st>>>(prm, win.hist, win.ld, In, Out, out, M);
  } else {
    usv::ensure_dynamic_smem(encoder_forward_store_kernel<T>, smem);
    encoder_forward_store_kernel<T><<<grid, kThreads, smem, st>>>(prm, win, In, Out, out, M);
  }
  return usv::finish_launch();
}

template <int T, class Win>
static int launch_train(const float* prm, const Win& win, const float* zstar, int In, int Out, float* partial, int64_t M, int* nparts,
                        cudaStream_t st) {
  const size_t smem = fwd_smem_bytes<T>(In, Out);
  if (smem > 227 * 1024) return USV_E_SIZE;
  const int64_t want = (M + kWarps - 1) / kWarps;
  const int sms = usv::num_sms();
  const int grid = (int)(want < sms ? want : sms);
  *nparts = grid;
  if constexpr (std::is_same<Win, RowWindows>::value) {
    usv::ensure_dynamic_smem(train_kernel<T>, smem);
    train_kernel<T><<<grid, kThreads, smem, st>>>(prm, win.hist, win.ld, zstar, In, Out, partial, M);
  } else {
    usv::ensure_dynamic_smem(train_store_kernel<T>, smem);
    train_store_kernel<T><<<grid, kThreads, smem, st>>>(prm, win, zstar, In, Out, partial, M);
  }
  return usv::finish_launch();
}

// one minibatch: the training kernel over the windows `win` names, then Adam
template <class Win>
static int minibatch_step(float* params, const Win& win, const float* zstar, int32_t input_size, int32_t tsteps, int32_t output_size, float* grads,
                          float* scratch, float* exp_avg, float* exp_avg_sq, const float* lr, int32_t* step, int32_t parity, float* mse_accum,
                          int64_t M, cudaStream_t st) {
  const int64_t P = dagger_history_encoder_param_count(input_size, tsteps, output_size);
  if (P < 0) return USV_E_UNSUPPORTED;
  int nparts = 0, rc;
  if (tsteps == 50) rc = launch_train<50>(params, win, zstar, input_size, output_size, scratch, M, &nparts, st);
  else if (tsteps == 20) rc = launch_train<20>(params, win, zstar, input_size, output_size, scratch, M, &nparts, st);
  else rc = launch_train<10>(params, win, zstar, input_size, output_size, scratch, M, &nparts, st);
  if (rc) return rc;
  adam_kernel<<<(int)((P + 1 + 255) / 256), 256, 0, st>>>(params, scratch, nparts, (int)P, grads, exp_avg, exp_avg_sq, lr, step, parity,
                                                         1.0f / ((float)M * (float)output_size), mse_accum);
  return usv::finish_launch();
}

}  // namespace dagger

using namespace dagger;

#define DAGGER_DISPATCH(T, expr50, expr20, expr10) \
  do {                                             \
    if ((T) == 50) return expr50;                  \
    if ((T) == 20) return expr20;                  \
    if ((T) == 10) return expr10;                  \
    return USV_E_UNSUPPORTED;                      \
  } while (0)

extern "C" {

int64_t dagger_history_encoder_param_count(int32_t input_size, int32_t tsteps, int32_t output_size) {
  if (input_size < 1 || input_size > 32 || output_size < 1 || output_size > 8) return -1;
  if (tsteps == 50) return offsets<50>(input_size, output_size).P;
  if (tsteps == 20) return offsets<20>(input_size, output_size).P;
  if (tsteps == 10) return offsets<10>(input_size, output_size).P;
  return -1;
}

int64_t dagger_train_scratch_floats(int32_t input_size, int32_t tsteps, int32_t output_size) {
  const int64_t P = dagger_history_encoder_param_count(input_size, tsteps, output_size);
  return P < 0 ? -1 : (int64_t)160 * (P + 4);
}

int dagger_history_encoder_forward_f32(const float* params, const float* hist, int64_t hist_ld, int32_t input_size, int32_t tsteps,
                                       int32_t output_size, float* latent, int64_t M, void* stream) {
  if (M < 0 || input_size < 1 || input_size > 32 || output_size < 1 || output_size > 8 || hist_ld < (int64_t)input_size * tsteps) return USV_E_SIZE;
  if (M == 0) return USV_OK;
  if (!params || !hist || !latent) return USV_E_NULL;
  cudaStream_t st = (cudaStream_t)stream;
  const RowWindows win{hist, hist_ld};
  DAGGER_DISPATCH(tsteps, launch_forward<50>(params, win, input_size, output_size, latent, M, st),
                  launch_forward<20>(params, win, input_size, output_size, latent, M, st),
                  launch_forward<10>(params, win, input_size, output_size, latent, M, st));
}

int dagger_sysid_minibatch_step_f32(float* params, const float* hist, int64_t hist_ld, const float* zstar, int32_t input_size, int32_t tsteps,
                                    int32_t output_size, float* grads, float* scratch, float* exp_avg, float* exp_avg_sq, const float* lr,
                                    int32_t* step, int32_t parity, float* mse_accum, int64_t M, void* stream) {
  if (M <= 0 || input_size < 1 || input_size > 32 || output_size < 1 || output_size > 8 || hist_ld < (int64_t)input_size * tsteps) return USV_E_SIZE;
  if (!params || !hist || !zstar || !grads || !scratch || !exp_avg || !exp_avg_sq || !lr || !step) return USV_E_NULL;
  if (parity != 0 && parity != 1) return USV_E_PARAM;
  return minibatch_step(params, RowWindows{hist, hist_ld}, zstar, input_size, tsteps, output_size, grads, scratch, exp_avg, exp_avg_sq, lr, step,
                        parity, mse_accum, M, (cudaStream_t)stream);
}

// the frame store's shape and the rows [row0, row0 + M) of its H * N windows
static int check_store(int32_t input_size, int32_t output_size, int64_t num_envs, int32_t horizon, int64_t row0, int64_t M) {
  if (M < 0 || input_size < 1 || input_size > 32 || output_size < 1 || output_size > 8 || num_envs < 1 || horizon < 1 || row0 < 0) return USV_E_SIZE;
  if (num_envs > INT32_MAX || row0 + M > (int64_t)horizon * num_envs) return USV_E_SIZE;
  return USV_OK;
}

int dagger_history_encoder_forward_store_f32(const float* params, const float* store, const int32_t* refill, int64_t num_envs, int32_t horizon,
                                             int64_t row0, int32_t input_size, int32_t tsteps, int32_t output_size, float* latent, int64_t M,
                                             void* stream) {
  if (!params || !store || !refill || !latent) return USV_E_NULL;
  if (tsteps != 50 && tsteps != 20 && tsteps != 10) return USV_E_UNSUPPORTED;
  if (const int rc = check_store(input_size, output_size, num_envs, horizon, row0, M)) return rc;
  if (M == 0) return USV_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const StoreWindows win{store, refill, row0, num_envs, tsteps - 1 + horizon, input_size};
  DAGGER_DISPATCH(tsteps, launch_forward<50>(params, win, input_size, output_size, latent, M, st),
                  launch_forward<20>(params, win, input_size, output_size, latent, M, st),
                  launch_forward<10>(params, win, input_size, output_size, latent, M, st));
}

int dagger_sysid_minibatch_step_store_f32(float* params, const float* store, const int32_t* refill, int64_t num_envs, int32_t horizon, int64_t row0,
                                          const float* zstar, int32_t input_size, int32_t tsteps, int32_t output_size, float* grads, float* scratch,
                                          float* exp_avg, float* exp_avg_sq, const float* lr, int32_t* step, int32_t parity, float* mse_accum,
                                          int64_t M, void* stream) {
  if (!params || !store || !refill || !zstar || !grads || !scratch || !exp_avg || !exp_avg_sq || !lr || !step) return USV_E_NULL;
  if (tsteps != 50 && tsteps != 20 && tsteps != 10) return USV_E_UNSUPPORTED;
  if (M <= 0) return USV_E_SIZE;
  if (const int rc = check_store(input_size, output_size, num_envs, horizon, row0, M)) return rc;
  if (parity != 0 && parity != 1) return USV_E_PARAM;
  const StoreWindows win{store, refill, row0, num_envs, tsteps - 1 + horizon, input_size};
  return minibatch_step(params, win, zstar + row0 * output_size, input_size, tsteps, output_size, grads, scratch, exp_avg, exp_avg_sq, lr, step,
                        parity, mse_accum, M, (cudaStream_t)stream);
}

int dagger_mlp_forward_f32(const float* params, int32_t n_layers, const int32_t* dims, const int32_t* w_offsets, const int32_t* b_offsets,
                           int32_t last_activation, const float* x, int64_t x_ld, float* y, int64_t M, void* stream) {
  if (M < 0 || n_layers < 1 || n_layers > 3 || !dims || !w_offsets || !b_offsets) return USV_E_SIZE;
  if (M == 0) return USV_OK;
  if (!params || !x || !y) return USV_E_NULL;
  if (last_activation < 0 || last_activation > 2) return USV_E_PARAM;
  MlpDesc d{};
  d.nl = n_layers;
  d.tanh_out = last_activation;
  size_t fl = 0;
  for (int l = 0; l <= n_layers; ++l) {
    if (dims[l] < 1 || dims[l] > 128) return USV_E_SIZE;
    d.dim[l] = dims[l];
  }
  if (x_ld < dims[0]) return USV_E_SIZE;
  for (int l = 0; l < n_layers; ++l) { d.w[l] = w_offsets[l]; d.b[l] = b_offsets[l]; fl += (size_t)dims[l] * dims[l + 1] + dims[l + 1]; }
  const size_t smem = (((fl + 3) & ~(size_t)3) + 8 * 256) * sizeof(float);
  if (smem > 227 * 1024) return USV_E_SIZE;
  usv::ensure_dynamic_smem(mlp_forward_kernel, smem);
  const int64_t want = (M + 7) / 8;
  const int sms = usv::num_sms();
  const int grid = (int)(want < sms ? want : sms);
  mlp_forward_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(params, d, x, x_ld, y, M);
  return usv::finish_launch();
}

// a small MLP's layers from host arrays: USV_E_SIZE for a bad shape, USV_E_PARAM for a bad last activation
static int mlp_desc(int32_t n_layers, const int32_t* dims, const int32_t* w_offsets, const int32_t* b_offsets, int32_t last_activation, MlpDesc* d) {
  if (n_layers < 1 || n_layers > 3) return USV_E_SIZE;
  for (int l = 0; l <= n_layers; ++l)
    if (dims[l] < 1 || dims[l] > 128) return USV_E_SIZE;
  if (last_activation < 0 || last_activation > 2) return USV_E_PARAM;
  *d = MlpDesc{};
  d->nl = n_layers;
  d->tanh_out = last_activation;
  for (int l = 0; l <= n_layers; ++l) d->dim[l] = dims[l];
  for (int l = 0; l < n_layers; ++l) { d->w[l] = w_offsets[l]; d->b[l] = b_offsets[l]; }
  return USV_OK;
}

// dagger_student_act_f32 and, with col, dagger_sysid_collect_f32 past the collect step's own checks
static int student_act(const float* encoder_params, const float* head_params, int32_t head_layers, const int32_t* head_dims,
                       const int32_t* head_w_offsets, const int32_t* head_b_offsets, int32_t head_last_activation, float* ring, int32_t* slot,
                       const float* obs, int64_t obs_ld, int32_t obs_nonpriv_dim, int32_t tsteps, int32_t latent_dim, const int64_t* dones,
                       int32_t fill_mode, int32_t init, float* mu_out, float* latent_out, int64_t M, const Distill* col, void* stream) {
  if (!encoder_params || !head_params || !head_dims || !head_w_offsets || !head_b_offsets || !ring || !slot || !obs || !mu_out) return USV_E_NULL;
  if (tsteps != 50 && tsteps != 20 && tsteps != 10) return USV_E_UNSUPPORTED;
  if (M < 0 || obs_nonpriv_dim < 1 || obs_nonpriv_dim > 32 || latent_dim < 1 || latent_dim > 8 || obs_ld < obs_nonpriv_dim) return USV_E_SIZE;
  if (head_layers < 1 || head_layers > 3) return USV_E_SIZE;
  for (int l = 0; l <= head_layers; ++l)
    if (head_dims[l] < 1 || head_dims[l] > 128) return USV_E_SIZE;
  if (head_dims[0] != obs_nonpriv_dim + latent_dim) return USV_E_SIZE;
  if (head_last_activation < 0 || head_last_activation > 2 || (fill_mode != 0 && fill_mode != 1) || (init != 0 && init != 1)) return USV_E_PARAM;
  MlpDesc d{};
  d.nl = head_layers;
  d.tanh_out = head_last_activation;
  for (int l = 0; l <= head_layers; ++l) d.dim[l] = head_dims[l];
  for (int l = 0; l < head_layers; ++l) { d.w[l] = head_w_offsets[l]; d.b[l] = head_b_offsets[l]; }
  if (M == 0) return USV_OK;
  cudaStream_t st = (cudaStream_t)stream;
  DAGGER_DISPATCH(tsteps,
                  launch_student_act<50>(encoder_params, head_params, d, ring, slot, obs, obs_ld, obs_nonpriv_dim, latent_dim, dones, fill_mode, init,
                                         mu_out, latent_out, M, col, st),
                  launch_student_act<20>(encoder_params, head_params, d, ring, slot, obs, obs_ld, obs_nonpriv_dim, latent_dim, dones, fill_mode, init,
                                         mu_out, latent_out, M, col, st),
                  launch_student_act<10>(encoder_params, head_params, d, ring, slot, obs, obs_ld, obs_nonpriv_dim, latent_dim, dones, fill_mode, init,
                                         mu_out, latent_out, M, col, st));
}

int dagger_student_act_f32(const float* encoder_params, const float* head_params, int32_t head_layers, const int32_t* head_dims,
                           const int32_t* head_w_offsets, const int32_t* head_b_offsets, int32_t head_last_activation, float* ring,
                           int32_t* slot, const float* obs, int64_t obs_ld, int32_t obs_nonpriv_dim, int32_t tsteps, int32_t latent_dim,
                           const int64_t* dones, int32_t fill_mode, int32_t init, float* mu_out, float* latent_out, int64_t M, void* stream) {
  return student_act(encoder_params, head_params, head_layers, head_dims, head_w_offsets, head_b_offsets, head_last_activation, ring, slot, obs,
                     obs_ld, obs_nonpriv_dim, tsteps, latent_dim, dones, fill_mode, init, mu_out, latent_out, M, nullptr, stream);
}

int dagger_sysid_collect_f32(const float* encoder_params, const float* head_params, int32_t head_layers, const int32_t* head_dims,
                             const int32_t* head_w_offsets, const int32_t* head_b_offsets, int32_t head_last_activation, const float* teacher_params,
                             int32_t teacher_layers, const int32_t* teacher_dims, const int32_t* teacher_w_offsets, const int32_t* teacher_b_offsets,
                             int32_t teacher_last_activation, float* ring, int32_t* slot, const float* obs, int64_t obs_ld, int32_t obs_nonpriv_dim,
                             int32_t tsteps, int32_t latent_dim, const int64_t* dones, int32_t fill_mode, int32_t init, float* store, int32_t* refill,
                             float* zstar, int32_t t, int32_t horizon, float* mu_out, int64_t M, void* stream) {
  if (!teacher_params || !teacher_dims || !teacher_w_offsets || !teacher_b_offsets || !store || !refill || !zstar) return USV_E_NULL;
  Distill col{};
  if (const int rc = mlp_desc(teacher_layers, teacher_dims, teacher_w_offsets, teacher_b_offsets, teacher_last_activation, &col.td)) return rc;
  if (teacher_dims[teacher_layers] != latent_dim || obs_ld < (int64_t)obs_nonpriv_dim + teacher_dims[0]) return USV_E_SIZE;
  if (horizon < 1 || t < 0 || t >= horizon) return USV_E_SIZE;
  if (init && t != 0) return USV_E_PARAM;                 // the store keeps one window per rollout: it starts at step 0
  col.teacher = teacher_params;
  col.store = store;
  col.refill = refill;
  col.zstar = zstar;
  col.t = t;
  col.S = tsteps - 1 + horizon;
  return student_act(encoder_params, head_params, head_layers, head_dims, head_w_offsets, head_b_offsets, head_last_activation, ring, slot, obs,
                     obs_ld, obs_nonpriv_dim, tsteps, latent_dim, dones, fill_mode, init, mu_out, nullptr, M, &col, stream);
}

}  // extern "C"
