// USV_PPOcontinuous_MLP on the GPU: fused normalise -> Linear+tanh -> Linear+tanh -> {mu, value} forward,
// fused PPO loss + full backward, deterministic two-stage gradient reduction, and a fused
// grad-norm-clip + Adam + adaptive-KL learning-rate step (rows P4, P5 of SURVEY 8).
// [ref: RLG/algos_torch/models.py:366-401 ; network_builder.py:1577-1629 ; a2c_continuous.py:78-217 ;
//       RLG/common/common_losses.py:10-48 ; a2c_common.py:308-330 ; schedulers.py:19-32 ; torch_ext.py:27-36]
//
// This file is the fp32 SIMT implementation: one CTA owns a tile of 64 samples, the whole network (18.7 k
// parameters) sits in shared memory, activations never leave the SM, and each thread keeps an 8x8 block of the
// 128x128 weight gradient in registers across tiles.  It is the numerics reference for the tensor-core path.
#include <math_constants.h>
#include "philox.cuh"
#include "usv_common.cuh"

namespace ppo {

constexpr int H = PPO_HIDDEN;       // 128
constexpr int A = PPO_ACTIONS;      // 2
constexpr int TM = 64;              // samples per tile
constexpr int NT = 256;             // threads per CTA
constexpr int HS = H + 4;           // padded activation / W2T row stride (floats); keeps float4 alignment
constexpr float kHalfLog2Pi2 = 1.8378770664093453f;  // 0.5*log(2*pi)*2

struct Layout {  // offsets into the flat parameter vector (rl_games model.parameters() order)
  int D, sigma, w1, b1, w2, b2, wv, bv, wmu, bmu, P;
  __host__ __device__ explicit Layout(int d) {
    D = d; sigma = 0; w1 = 2; b1 = w1 + H * d; w2 = b1 + H; b2 = w2 + H * H; wv = b2 + H; bv = wv + H; wmu = bv + 1;
    bmu = wmu + A * H; P = bmu + A;
  }
};

// ---------------------------------------------------------------------------------------------
// shared-memory carve-up (floats)
struct Smem {
  float *w1t, *b1, *w2t, *b2, *w3, *b3, *xs, *h1, *h2, *dz3, *gw1, *gw3, *gb;
  int xstride;
};
__host__ __device__ inline int xs_stride(int D) { return D | 1; }
__host__ __device__ inline size_t smem_floats(int D, bool train) {
  size_t n = (size_t)D * H + H + (size_t)H * HS + H + 3 * H + 4 + (size_t)TM * xs_stride(D) + 2 * (size_t)TM * HS;
  if (train) n += TM * 4 + (size_t)H * D + 3 * H + (2 * H + 4);
  return n;
}
__device__ inline Smem carve(float* base, int D, bool train) {
  Smem s;
  s.xstride = xs_stride(D);
  float* p = base;
  s.w2t = p; p += H * HS;       // first: 16 B aligned rows
  s.h1 = p; p += TM * HS;
  s.h2 = p; p += TM * HS;
  s.w1t = p; p += D * H;
  s.b1 = p; p += H;
  s.b2 = p; p += H;
  s.w3 = p; p += 3 * H;         // rows: mu0, mu1, value
  s.b3 = p; p += 4;
  s.xs = p; p += TM * s.xstride;
  if (train) {
    s.dz3 = p; p += TM * 4;
    s.gw1 = p; p += H * D;
    s.gw3 = p; p += 3 * H;
    s.gb = p; p += 2 * H + 4;   // db1[128], db2[128], db3[3]
  }
  return s;
}

__device__ inline void load_weights(const Smem& s, const float* __restrict__ prm, const Layout& L) {
  const int t = threadIdx.x;
  for (int e = t; e < H * L.D; e += NT) {            // W1[o][d] -> w1t[d][o]
    const int o = e / L.D, d = e - o * L.D;
    s.w1t[d * H + o] = prm[L.w1 + e];
  }
  for (int e = t; e < H * H; e += NT) {              // W2[o][i] -> w2t[i][o] (stride HS)
    const int o = e >> 7, i = e & (H - 1);
    s.w2t[i * HS + o] = prm[L.w2 + e];
  }
  for (int e = t; e < H; e += NT) {
    s.b1[e] = prm[L.b1 + e];
    s.b2[e] = prm[L.b2 + e];
    s.w3[2 * H + e] = prm[L.wv + e];
    s.w3[e] = prm[L.wmu + e];
    s.w3[H + e] = prm[L.wmu + H + e];
  }
  if (t == 0) { s.b3[0] = prm[L.bmu]; s.b3[1] = prm[L.bmu + 1]; s.b3[2] = prm[L.bv]; s.b3[3] = 0.f; }
}

// normalised, clamped observations of a tile -> xs  [ref running_mean_std.py:113-116]
__device__ inline void load_obs_tile(const Smem& s, const float* __restrict__ obs, int D, const float* __restrict__ mean,
                                     const float* __restrict__ var, int64_t row0, int64_t M) {
  for (int e = threadIdx.x; e < TM * D; e += NT) {
    const int r = e / D, d = e - r * D;
    float y = 0.f;
    if (row0 + r < M) {
      const float x = obs[(row0 + r) * D + d];
      y = (x - mean[d]) / sqrtf(var[d] + 1e-5f);
      y = fminf(fmaxf(y, -5.0f), 5.0f);
    }
    s.xs[r * s.xstride + d] = y;
  }
}

// C[4 rows][8 cols] += A[rows ty*4..][0..K) * B[0..K)[cols tx*8..]   (A row stride lda, B row stride ldb)
template <int KU>
__device__ inline void gemm_4x8(const float* __restrict__ Asm, int lda, const float* __restrict__ Bsm, int ldb, int K,
                                int ty, int tx, float (&acc)[4][8]) {
  const float* a0 = Asm + (ty * 4) * lda;
  const float* b0 = Bsm + tx * 8;
#pragma unroll KU
  for (int k = 0; k < K; ++k) {
    const float4 bl = *reinterpret_cast<const float4*>(b0 + k * ldb);
    const float4 bh = *reinterpret_cast<const float4*>(b0 + k * ldb + 4);
    const float b[8] = {bl.x, bl.y, bl.z, bl.w, bh.x, bh.y, bh.z, bh.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = a0[j * lda + k];
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[j][c] = fmaf(a, b[c], acc[j][c]);
    }
  }
}

// trunk: xs -> h1 -> h2 (tanh after each Linear)   [ref network_builder.py:1577-1600]
__device__ inline void trunk_forward(const Smem& s, int D) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  float acc[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[j][c] = s.b1[tx * 8 + c];
  gemm_4x8<1>(s.xs, s.xstride, s.w1t, H, D, ty, tx, acc);
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) s.h1[(ty * 4 + j) * HS + tx * 8 + c] = tanhf(acc[j][c]);
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[j][c] = s.b2[tx * 8 + c];
  gemm_4x8<4>(s.h1, HS, s.w2t, HS, H, ty, tx, acc);
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) s.h2[(ty * 4 + j) * HS + tx * 8 + c] = tanhf(acc[j][c]);
  __syncthreads();
}

// heads: out[r][j] = h2[r] . w3[j] + b3[j], j = mu0, mu1, value.  4 threads per row (j = 0..2 active).
__device__ inline float head_out(const Smem& s, int r, int j) {
  float acc = 0.f;
  const float* h = s.h2 + r * HS;
  const float* w = s.w3 + j * H;
#pragma unroll 8
  for (int k = 0; k < H; k += 4) {
    const float4 hv = *reinterpret_cast<const float4*>(h + k);
    const float4 wv = *reinterpret_cast<const float4*>(w + k);
    acc = fmaf(hv.x, wv.x, acc); acc = fmaf(hv.y, wv.y, acc); acc = fmaf(hv.z, wv.z, acc); acc = fmaf(hv.w, wv.w, acc);
  }
  return acc + s.b3[j];
}

// ---------------------------------------------------------------------------------------------
// inference: rollout action sampling / value read-out
__global__ void __launch_bounds__(NT, 1) forward_kernel(
    const float* __restrict__ prm, const float* __restrict__ obs, int D, const float* __restrict__ omean,
    const float* __restrict__ ovar, const float* __restrict__ vmean, const float* __restrict__ vvar, uint64_t seed,
    uint64_t counter_in, const uint64_t* __restrict__ counter_offset, int64_t row_offset, float* __restrict__ actions, float* __restrict__ neglogp,
    float* __restrict__ values, float* __restrict__ mus, float* __restrict__ sigmas, int64_t M) {
  extern __shared__ __align__(16) float smem[];
  const Layout L(D);
  const Smem s = carve(smem, D, false);
  load_weights(s, prm, L);
  const uint64_t counter = counter_in + (counter_offset ? *counter_offset : 0ull);
  const float ls0 = prm[L.sigma], ls1 = prm[L.sigma + 1];
  const float sg0 = expf(ls0), sg1 = expf(ls1);
  const int64_t ntiles = (M + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * TM;
    __syncthreads();
    load_obs_tile(s, obs, D, omean, ovar, row0, M);
    __syncthreads();
    trunk_forward(s, D);
    const int r = threadIdx.x >> 2, j = threadIdx.x & 3;
    const int64_t row = row0 + r;
    float o = (j < 3) ? head_out(s, r, j) : 0.f;
    // gather the row's three outputs on its j==0 lane
    const float mu0 = __shfl_sync(0xffffffffu, o, (threadIdx.x & 31 & ~3) + 0);
    const float mu1 = __shfl_sync(0xffffffffu, o, (threadIdx.x & 31 & ~3) + 1);
    const float v = __shfl_sync(0xffffffffu, o, (threadIdx.x & 31 & ~3) + 2);
    if (j == 0 && row < M) {
      if (mus) { mus[row * 2] = mu0; mus[row * 2 + 1] = mu1; }
      if (sigmas) { sigmas[row * 2] = sg0; sigmas[row * 2 + 1] = sg1; }
      if (values) {  // denorm_value: clamp(v,+-5)*sqrt(var+eps)+mean  [ref running_mean_std.py:108-110]
        const float y = fminf(fmaxf(v, -5.0f), 5.0f);
        values[row] = vmean ? sqrtf(vvar[0] + 1e-5f) * y + vmean[0] : v;
      }
      if (actions) {
        // a ~ Normal(mu, sigma): Box-Muller on Philox uniforms keyed (seed; global row, counter)
        const usv::Philox4 rr = usv::philox4x32_10((uint32_t)(row + row_offset), (uint32_t)counter, (uint32_t)(counter >> 32),
                                                   100u ^ ((uint32_t)((uint64_t)(row + row_offset) >> 32) << 8), (uint32_t)seed,
                                                   (uint32_t)(seed >> 32));
        const float u1 = (float)((rr.x >> 8) + 1u) * (1.0f / 16777216.0f);   // (0,1]
        const float u2 = (float)(rr.y >> 8) * (1.0f / 16777216.0f);          // [0,1)
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincosf(6.28318530717958647692f * u2, &sn, &cs);
        const float a0 = mu0 + sg0 * (rad * cs), a1 = mu1 + sg1 * (rad * sn);
        actions[row * 2] = a0;
        actions[row * 2 + 1] = a1;
        if (neglogp) {
          const float d0 = (a0 - mu0) / sg0, d1 = (a1 - mu1) / sg1;
          neglogp[row] = 0.5f * (d0 * d0 + d1 * d1) + kHalfLog2Pi2 + (ls0 + ls1);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// training: forward + PPO losses + backward for the tiles of one CTA; partial gradients per CTA
struct LossIn {
  const float *actions, *old_nlp, *adv, *old_v, *ret;
  float *old_mu, *old_sigma;
};

__global__ void __launch_bounds__(NT, 1) train_kernel(const float* __restrict__ prm, const float* __restrict__ obs, int D,
                                                     const float* __restrict__ omean, const float* __restrict__ ovar,
                                                     LossIn in, PpoLossParams lp, float* __restrict__ partial, int64_t M) {
  extern __shared__ __align__(16) float smem[];
  const Layout L(D);
  const Smem s = carve(smem, D, true);
  const int t = threadIdx.x;
  load_weights(s, prm, L);
  for (int e = t; e < H * D; e += NT) s.gw1[e] = 0.f;
  for (int e = t; e < 3 * H; e += NT) s.gw3[e] = 0.f;
  for (int e = t; e < 2 * H + 4; e += NT) s.gb[e] = 0.f;
  const float ls0 = prm[L.sigma], ls1 = prm[L.sigma + 1];
  const float sg0 = expf(ls0), sg1 = expf(ls1);
  const float invM = 1.0f / (float)M;
  float gW2[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) gW2[a][b] = 0.f;
  float st_a = 0.f, st_c = 0.f, st_e = 0.f, st_b = 0.f, st_kl = 0.f, g_ls0 = 0.f, g_ls1 = 0.f;  // per-thread partial sums
  const int ty = t >> 4, tx = t & 15;
  const int64_t ntiles = (M + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * TM;
    __syncthreads();
    load_obs_tile(s, obs, D, omean, ovar, row0, M);
    __syncthreads();
    trunk_forward(s, D);
    // ---- heads + per-sample losses: 4 lanes per row ------------------------------------------------
    {
      const int r = t >> 2, j = t & 3;
      const int64_t row = row0 + r;
      const float o = (j < 3) ? head_out(s, r, j) : 0.f;
      const int base = (t & 31) & ~3;
      const float mu0 = __shfl_sync(0xffffffffu, o, base), mu1 = __shfl_sync(0xffffffffu, o, base + 1);
      const float v = __shfl_sync(0xffffffffu, o, base + 2);
      float d_mu0 = 0.f, d_mu1 = 0.f, d_v = 0.f;
      if (j == 0 && row < M) {
        const float a0 = in.actions[row * 2], a1 = in.actions[row * 2 + 1];
        const float e0 = (a0 - mu0) / sg0, e1 = (a1 - mu1) / sg1;
        const float nlp = 0.5f * (e0 * e0 + e1 * e1) + kHalfLog2Pi2 + (ls0 + ls1);      // [ref models.py:398-401]
        const float adv = in.adv[row];
        // actor_loss  [ref common_losses.py:39-48]
        const float ratio = expf(in.old_nlp[row] - nlp);
        const float s1 = adv * ratio;
        const float s2 = adv * fminf(fmaxf(ratio, 1.0f - lp.e_clip), 1.0f + lp.e_clip);
        const float a_loss = fmaxf(-s1, -s2);
        const float g_nlp = (-s1 >= -s2) ? s1 : 0.f;          // d a_loss / d nlp  (= adv*ratio on the unclipped branch)
        // critic loss  [ref common_losses.py:10-20]
        const float ov = in.old_v[row], ret = in.ret[row];
        float c_loss, g_v;
        if (lp.clip_value) {
          const float dvc = fminf(fmaxf(v - ov, -lp.e_clip), lp.e_clip);
          const float vpc = ov + dvc;
          const float l1 = (v - ret) * (v - ret), l2 = (vpc - ret) * (vpc - ret);
          c_loss = fmaxf(l1, l2);
          const bool inside = fabsf(v - ov) <= lp.e_clip;
          g_v = (l1 >= l2) ? 2.0f * (v - ret) : (inside ? 2.0f * (vpc - ret) : 0.f);
        } else {
          c_loss = (ret - v) * (ret - v);
          g_v = 2.0f * (v - ret);
        }
        // bound loss  [ref a2c_continuous.py:209-217]
        const float h0 = fmaxf(mu0 - lp.bound_soft, 0.f), l0 = fminf(mu0 + lp.bound_soft, 0.f);
        const float h1v = fmaxf(mu1 - lp.bound_soft, 0.f), l1v = fminf(mu1 + lp.bound_soft, 0.f);
        const float b_loss = (l0 * l0 + h0 * h0) + (l1v * l1v + h1v * h1v);
        const float ent = (0.5f + 0.5f * 1.8378770664093453f + ls0) + (0.5f + 0.5f * 1.8378770664093453f + ls1);
        // policy_kl(new, old)  [ref torch_ext.py:27-36]
        const float om0 = in.old_mu[row * 2], om1 = in.old_mu[row * 2 + 1];
        const float os0 = in.old_sigma[row * 2], os1 = in.old_sigma[row * 2 + 1];
        const float kl0 = logf(os0 / sg0 + 1e-5f) + (sg0 * sg0 + (om0 - mu0) * (om0 - mu0)) / (2.0f * (os0 * os0 + 1e-5f)) - 0.5f;
        const float kl1 = logf(os1 / sg1 + 1e-5f) + (sg1 * sg1 + (om1 - mu1) * (om1 - mu1)) / (2.0f * (os1 * os1 + 1e-5f)) - 0.5f;
        st_a += a_loss; st_c += c_loss; st_e += ent; st_b += b_loss; st_kl += kl0 + kl1;
        // loss = mean(a) + 0.5*critic_coef*mean(c) - entropy_coef*mean(ent) + bounds_coef*mean(b)  [ref a2c_continuous.py:159]
        const float wa = invM, wc = 0.5f * lp.critic_coef * invM, wb = lp.bounds_loss_coef * invM, we = lp.entropy_coef * invM;
        d_mu0 = wa * g_nlp * (-(a0 - mu0) / (sg0 * sg0)) + wb * 2.0f * (h0 + l0);
        d_mu1 = wa * g_nlp * (-(a1 - mu1) / (sg1 * sg1)) + wb * 2.0f * (h1v + l1v);
        d_v = wc * g_v;
        g_ls0 += wa * g_nlp * (1.0f - e0 * e0) - we;
        g_ls1 += wa * g_nlp * (1.0f - e1 * e1) - we;
        in.old_mu[row * 2] = mu0; in.old_mu[row * 2 + 1] = mu1;           // dataset.update_mu_sigma  [ref datasets.py:25-29]
        in.old_sigma[row * 2] = sg0; in.old_sigma[row * 2 + 1] = sg1;
      }
      if (j == 0) { s.dz3[r * 4 + 0] = d_mu0; s.dz3[r * 4 + 1] = d_mu1; s.dz3[r * 4 + 2] = d_v; s.dz3[r * 4 + 3] = 0.f; }
    }
    __syncthreads();
    // ---- head gradients: gw3[j][k] += sum_r dz3[r][j]*h2[r][k] ; db3 ------------------------------------
    for (int e = t; e < 3 * H; e += NT) {
      const int j = e >> 7, k = e & (H - 1);
      float acc = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) acc = fmaf(s.dz3[r * 4 + j], s.h2[r * HS + k], acc);
      s.gw3[e] += acc;
    }
    if (t < 3) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.dz3[r * 4 + t];
      s.gb[2 * H + t] += acc;
    }
    __syncthreads();
    // ---- dz2 = (dz3 . W3) * (1 - h2^2), in place over h2 ------------------------------------------------
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = ty * 4 + j;
      const float g0 = s.dz3[r * 4], g1 = s.dz3[r * 4 + 1], g2 = s.dz3[r * 4 + 2];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int k = tx * 8 + c;
        const float h = s.h2[r * HS + k];
        const float dh = g0 * s.w3[k] + g1 * s.w3[H + k] + g2 * s.w3[2 * H + k];
        s.h2[r * HS + k] = dh * (1.0f - h * h);
      }
    }
    __syncthreads();
    // ---- gW2[o][i] += sum_r dz2[r][o]*h1[r][i]  (8x8 block per thread, registers) ; db2 ------------------
    {
      const float* za = s.h2 + ty * 8;   // o block
      const float* hb = s.h1 + tx * 8;   // i block
#pragma unroll 4
      for (int r = 0; r < TM; ++r) {
        const float4 al = *reinterpret_cast<const float4*>(za + r * HS), ah = *reinterpret_cast<const float4*>(za + r * HS + 4);
        const float4 bl = *reinterpret_cast<const float4*>(hb + r * HS), bh = *reinterpret_cast<const float4*>(hb + r * HS + 4);
        const float av[8] = {al.x, al.y, al.z, al.w, ah.x, ah.y, ah.z, ah.w};
        const float bv[8] = {bl.x, bl.y, bl.z, bl.w, bh.x, bh.y, bh.z, bh.w};
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) gW2[a][b] = fmaf(av[a], bv[b], gW2[a][b]);
      }
      if (t < H) {
        float acc = 0.f;
        for (int r = 0; r < TM; ++r) acc += s.h2[r * HS + t];
        s.gb[H + t] += acc;
      }
    }
    // ---- dz1 = (dz2 . W2) * (1 - h1^2), in place over h1.  B[k=o][n=i] = w2t[i][o]: columns interleaved (i = tx+16c)
    {
      float acc[4][8];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;
      const float* a0 = s.h2 + (ty * 4) * HS;
#pragma unroll 2
      for (int k = 0; k < H; k += 4) {
        float4 av[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) av[j] = *reinterpret_cast<const float4*>(a0 + j * HS + k);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 bv = *reinterpret_cast<const float4*>(s.w2t + (tx + 16 * c) * HS + k);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc[j][c] = fmaf(av[j].x, bv.x, acc[j][c]);
            acc[j][c] = fmaf(av[j].y, bv.y, acc[j][c]);
            acc[j][c] = fmaf(av[j].z, bv.z, acc[j][c]);
            acc[j][c] = fmaf(av[j].w, bv.w, acc[j][c]);
          }
        }
      }
      __syncthreads();   // every thread is done reading h1 (gW2) before it is overwritten
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int r = ty * 4 + j, i = tx + 16 * c;
          const float h = s.h1[r * HS + i];
          s.h1[r * HS + i] = acc[j][c] * (1.0f - h * h);
        }
    }
    __syncthreads();
    // ---- gw1[o][d] += sum_r dz1[r][o]*x[r][d] ; db1 ------------------------------------------------------
    for (int e = t; e < H * D; e += NT) {
      const int d = e >> 7, o = e & (H - 1);       // consecutive threads -> consecutive o (conflict-free dz1 reads)
      float acc = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) acc = fmaf(s.h1[r * HS + o], s.xs[r * s.xstride + d], acc);
      s.gw1[o * D + d] += acc;
    }
    if (t < H) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.h1[r * HS + t];
      s.gb[t] += acc;
    }
  }
  __syncthreads();
  // ---- write this CTA's partial gradient + statistics ------------------------------------------------------
  float* out = partial + (size_t)blockIdx.x * (L.P + PPO_STAT_COUNT);
  for (int e = t; e < H * D; e += NT) out[L.w1 + e] = s.gw1[e];
  for (int e = t; e < H; e += NT) {
    out[L.b1 + e] = s.gb[e];
    out[L.b2 + e] = s.gb[H + e];
    out[L.wv + e] = s.gw3[2 * H + e];
    out[L.wmu + e] = s.gw3[e];
    out[L.wmu + H + e] = s.gw3[H + e];
  }
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) out[L.w2 + (ty * 8 + a) * H + tx * 8 + b] = gW2[a][b];
  // block-reduce the per-thread scalars (a, c, ent, b, kl, dlogstd0, dlogstd1)
  __shared__ float red[7][NT / 32];
  float vals[7] = {st_a, st_c, st_e, st_b, st_kl, g_ls0, g_ls1};
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    float v = vals[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((t & 31) == 0) red[q][t >> 5] = v;
  }
  __syncthreads();
  if (t == 0) {
    float tot[7];
    for (int q = 0; q < 7; ++q) {
      float v = 0.f;
      for (int w = 0; w < NT / 32; ++w) v += red[q][w];
      tot[q] = v;
    }
    out[L.sigma] = tot[5];
    out[L.sigma + 1] = tot[6];
    out[L.bmu] = s.gb[2 * H];
    out[L.bmu + 1] = s.gb[2 * H + 1];
    out[L.bv] = s.gb[2 * H + 2];
    out[L.P + PPO_STAT_A_LOSS] = tot[0] * invM;
    out[L.P + PPO_STAT_C_LOSS] = tot[1] * invM;
    out[L.P + PPO_STAT_ENTROPY] = tot[2] * invM;
    out[L.P + PPO_STAT_B_LOSS] = tot[3] * invM;
    out[L.P + PPO_STAT_KL] = tot[4] * invM;
    out[L.P + PPO_STAT_LOSS] = 0.f;
    out[L.P + PPO_STAT_GRAD_NORM] = 0.f;
    out[L.P + PPO_STAT_LR] = 0.f;
  }
}

// second stage: grads[e] = sum over CTAs of partial[c][e]  (fixed order -> deterministic).
// 64 columns x 4 row-groups per block: four 32-long dependent load chains instead of one 128-long one.
__global__ void __launch_bounds__(256) reduce_kernel(const float* __restrict__ partial, int nparts, int n,
                                                     float* __restrict__ grads, PpoLossParams lp, int P) {
  __shared__ float sm[4][64];
  const int col = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int e = blockIdx.x * 64 + col;
  float acc = 0.f;
  if (e < n)
    for (int c = grp; c < nparts; c += 4) acc += partial[(size_t)c * n + e];
  sm[grp][col] = acc;
  __syncthreads();
  // the total-loss slot belongs to block 0 (below): the column sum of that slot is 0 and, written from another block, raced with it
  if (grp == 0 && e < n && e != P + PPO_STAT_LOSS) {
    float v = (sm[0][col] + sm[1][col]) + (sm[2][col] + sm[3][col]);
    grads[e] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // total loss from the component means
    float a = 0.f, cl = 0.f, en = 0.f, b = 0.f;
    for (int c = 0; c < nparts; ++c) {
      const float* q = partial + (size_t)c * n + P;
      a += q[PPO_STAT_A_LOSS]; cl += q[PPO_STAT_C_LOSS]; en += q[PPO_STAT_ENTROPY]; b += q[PPO_STAT_B_LOSS];
    }
    grads[P + PPO_STAT_LOSS] = a + 0.5f * cl * lp.critic_coef - en * lp.entropy_coef + b * lp.bounds_loss_coef;
  }
}

// clip_grad_norm_ + Adam + adaptive-KL lr.  Multi-CTA: every CTA recomputes the global gradient norm from the (L2-resident)
// 75 KB gradient in the same fixed order (deterministic, no atomics, no second launch), then updates its own slice.
// lr/step live in device memory: read by every CTA at entry; the LAST launch-ordered writer is CTA 0, and the next
// kernel that reads them is a later launch, so there is no intra-kernel hazard (they are written from *_in copies).
constexpr int kAdamThreads = 256;
__global__ void __launch_bounds__(kAdamThreads) adam_kernel(float* __restrict__ prm, float* __restrict__ g, float* __restrict__ m,
                                                            float* __restrict__ v, const float* __restrict__ lr_in,
                                                            const int* __restrict__ step_in, float* __restrict__ lr_out,
                                                            int* __restrict__ step_out, int P, PpoAdamParams ap) {
  __shared__ float red[kAdamThreads / 32];
  __shared__ float s_coef;
  const int t = threadIdx.x;
  // all-reduce delivered the SUM over ranks: average  [ref a2c_common.py:311-323]
  float ss = 0.f;
  for (int e = t; e < P; e += kAdamThreads) {
    const float x = g[e] * ap.inv_world;
    ss = fmaf(x, x, ss);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((t & 31) == 0) red[t >> 5] = ss;
  __syncthreads();
  if (t == 0) {
    float x = 0.f;
    for (int w = 0; w < kAdamThreads / 32; ++w) x += red[w];
    const float norm = sqrtf(x);
    // torch.nn.utils.clip_grad_norm_: coef = max_norm/(norm+1e-6), clamped to 1
    s_coef = (ap.grad_norm > 0.f) ? fminf(ap.grad_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    red[0] = norm;
  }
  __syncthreads();
  const float coef = s_coef * ap.inv_world;
  const float lr = *lr_in;
  const int step = *step_in + 1;
  // torch.optim.Adam (amsgrad=False, weight_decay=0); bias corrections evaluated in double like torch's scalar path
  const double bc1 = 1.0 - pow((double)ap.beta1, (double)step), bc2 = 1.0 - pow((double)ap.beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  const int e = blockIdx.x * kAdamThreads + t;
  if (e < P) {
    const float gr = g[e] * coef;
    const float mm = m[e] + (gr - m[e]) * (1.0f - ap.beta1);           // exp_avg.lerp_(grad, 1-beta1)
    const float vv = v[e] * ap.beta2 + (1.0f - ap.beta2) * gr * gr;    // exp_avg_sq.mul_(beta2).addcmul_(g,g,1-beta2)
    m[e] = mm;
    v[e] = vv;
    const float denom = sqrtf(vv) / bc2_sqrt + ap.eps;
    prm[e] = prm[e] - step_size * (mm / denom);
  }
  if (blockIdx.x == gridDim.x - 1) {   // the last CTA owns the statistics tail (no other CTA touches g[P..])
    if (t < PPO_STAT_COUNT) {
      float x = g[P + t] * ap.inv_world;
      if (t == PPO_STAT_GRAD_NORM) x = red[0];
      if (t == PPO_STAT_LR) x = lr;
      g[P + t] = x;
      if (t == PPO_STAT_KL) {
        float nl = lr;
        if (ap.adaptive_lr) {  // AdaptiveScheduler.update, 'legacy' per-minibatch schedule  [ref schedulers.py:26-32]
          if (x > 2.0f * ap.kl_threshold) nl = fmaxf(lr / 1.5f, ap.min_lr);
          if (x < 0.5f * ap.kl_threshold) nl = fminf(lr * 1.5f, ap.max_lr);
        }
        *lr_out = nl;
        *step_out = step;
      }
    }
  }
}

// RunningMeanStd.forward in training mode, fused: batch mean / unbiased variance per feature (fp32 inputs, fp64 accumulation)
// + the Chan parallel-variance merge into the fp64 running moments + the fp32 copies the network kernels read.
// One CTA per feature.  [ref: RLG/algos_torch/running_mean_std.py:69-89]
__global__ void __launch_bounds__(256) rms_update_kernel(const float* __restrict__ x, int64_t M, int D, double* __restrict__ mean,
                                                         double* __restrict__ var, double* __restrict__ count,
                                                         float* __restrict__ mean32, float* __restrict__ var32) {
  __shared__ double sh[2][8];
  const int d = blockIdx.x, t = threadIdx.x;
  // pass 1: mean
  double s = 0.0;
  for (int64_t r = t; r < M; r += 256) s += (double)x[r * D + d];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((t & 31) == 0) sh[0][t >> 5] = s;
  __syncthreads();
  double bm = 0.0;
  for (int w = 0; w < 8; ++w) bm += sh[0][w];
  bm /= (double)M;
  // pass 2: centred sum of squares (the batch is L2-resident)
  double q = 0.0;
  for (int64_t r = t; r < M; r += 256) {
    const double c = (double)x[r * D + d] - bm;
    q += c * c;
  }
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if ((t & 31) == 0) sh[1][t >> 5] = q;
  __syncthreads();
  if (t == 0) {
    double ss = 0.0;
    for (int w = 0; w < 8; ++w) ss += sh[1][w];
    // torch computes the batch moments in fp32 (input.mean / input.var) before they are promoted: round-trip through float
    const double bmean = (double)(float)bm, bvar = (double)(float)(M > 1 ? ss / (double)(M - 1) : 0.0);
    const double cnt = *count, bc = (double)M, tot = cnt + bc;
    const double delta = bmean - mean[d];
    const double new_mean = mean[d] + delta * bc / tot;
    const double M2 = var[d] * cnt + bvar * bc + delta * delta * cnt * bc / tot;
    mean[d] = new_mean;
    var[d] = M2 / tot;
    mean32[d] = (float)new_mean;
    var32[d] = (float)(M2 / tot);
  }
}
__global__ void rms_count_kernel(double* count, double add) { *count += add; }
__global__ void adam_roll_kernel(float* lr, int* step) { lr[0] = lr[1]; step[0] = step[1]; }

constexpr int kMaxParts = 160;

void launch_reduce(const float* scratch, int nparts, int n, float* grads, const PpoLossParams& lp, int P, cudaStream_t s) {
  reduce_kernel<<<(n + 63) / 64, 256, 0, s>>>(scratch, nparts, n, grads, lp, P);
}

}  // namespace ppo

using namespace ppo;

extern "C" {

int64_t ppo_param_count(int32_t obs_dim) { return Layout(obs_dim).P; }

int64_t ppo_train_scratch_floats(int32_t obs_dim) { return (int64_t)kMaxParts * (Layout(obs_dim).P + PPO_STAT_COUNT); }

int ppo_policy_forward_f32(const float* params, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                           const float* value_mean, const float* value_var, uint64_t seed, uint64_t counter, const uint64_t* counter_offset,
                           int64_t row_offset, float* actions, float* neglogp, float* values, float* mus, float* sigmas, int64_t M,
                           void* stream) {
  if (M < 0 || obs_dim < 1 || obs_dim > PPO_MAX_OBS) return USV_E_SIZE;
  if (M == 0) return USV_OK;
  if (!params || !obs || !obs_mean || !obs_var) return USV_E_NULL;
  if ((value_mean == nullptr) != (value_var == nullptr)) return USV_E_NULL;
  const size_t smem = smem_floats(obs_dim, false) * sizeof(float);
  usv::ensure_dynamic_smem(forward_kernel, smem);
  const int64_t ntiles = (M + TM - 1) / TM;
  const int sms = usv::num_sms();
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  forward_kernel<<<grid, NT, smem, (cudaStream_t)stream>>>(params, obs, obs_dim, obs_mean, obs_var, value_mean, value_var, seed,
                                                           counter, counter_offset, row_offset, actions, neglogp, values, mus, sigmas, M);
  return usv::finish_launch();
}

int ppo_minibatch_grad_f32(const float* params, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                           const float* actions, const float* old_neglogp, const float* advantages, const float* old_values,
                           const float* returns, float* old_mu, float* old_sigma, const PpoLossParams* lp, float* grads,
                           float* scratch, int64_t M, void* stream) {
  if (M <= 0 || obs_dim < 1 || obs_dim > PPO_MAX_OBS) return USV_E_SIZE;
  if (!params || !obs || !obs_mean || !obs_var || !actions || !old_neglogp || !advantages || !old_values || !returns || !old_mu ||
      !old_sigma || !lp || !grads || !scratch)
    return USV_E_NULL;
  const Layout L(obs_dim);
  const size_t smem = smem_floats(obs_dim, true) * sizeof(float);
  if (smem > 227 * 1024) return USV_E_UNSUPPORTED;
  usv::ensure_dynamic_smem(train_kernel, smem);
  const int64_t ntiles = (M + TM - 1) / TM;
  const int sms = usv::num_sms();
  int grid = (int)(ntiles < sms ? ntiles : sms);
  if (grid > kMaxParts) grid = kMaxParts;
  LossIn in{actions, old_neglogp, advantages, old_values, returns, old_mu, old_sigma};
  train_kernel<<<grid, NT, smem, (cudaStream_t)stream>>>(params, obs, obs_dim, obs_mean, obs_var, in, *lp, scratch, M);
  const int n = L.P + PPO_STAT_COUNT;
  reduce_kernel<<<(n + 63) / 64, 256, 0, (cudaStream_t)stream>>>(scratch, grid, n, grads, *lp, L.P);
  return usv::finish_launch(2);
}

int ppo_adam_step_f32(float* params, float* grads, float* exp_avg, float* exp_avg_sq, float* lr, int32_t* step, int64_t P,
                      const PpoAdamParams* ap, void* stream) {
  if (P <= 0) return USV_E_SIZE;
  if (!params || !grads || !exp_avg || !exp_avg_sq || !lr || !step || !ap) return USV_E_NULL;
  // lr/step are double-buffered ([0] = current, [1] = next) so that no CTA can observe the update of another CTA
  adam_kernel<<<(int)((P + kAdamThreads - 1) / kAdamThreads), kAdamThreads, 0, (cudaStream_t)stream>>>(
      params, grads, exp_avg, exp_avg_sq, lr, step, lr + 1, step + 1, (int)P, *ap);
  adam_roll_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(lr, step);
  return usv::finish_launch(2);
}

int ppo_rms_update_f64(const float* x, int64_t M, int32_t D, double* mean, double* var, double* count, float* mean32, float* var32,
                       void* stream) {
  if (M <= 0 || D < 1) return USV_E_SIZE;
  if (!x || !mean || !var || !count || !mean32 || !var32) return USV_E_NULL;
  rms_update_kernel<<<D, 256, 0, (cudaStream_t)stream>>>(x, M, D, mean, var, count, mean32, var32);
  rms_count_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(count, (double)M);   // after every feature has read the old count
  return usv::finish_launch(2);
}

}  // extern "C"
