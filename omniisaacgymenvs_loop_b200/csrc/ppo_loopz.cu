// The loopz PPO learner on the GPU (SURVEY 8(f) row 4): separate actor / critic MLPEncode networks
//   obs = [speed | task | mass] -> mass encoder Linear(Md,64)+LeakyReLU -> Linear(64,16)+LeakyReLU -> Linear(16,8)+LeakyReLU
//       -> cat(speed, task, latent) -> Linear(IN,128)+LeakyReLU -> Linear(128,128)+LeakyReLU -> Linear(128,OUT) [+ tanh]
// a tanh-squashed diagonal Gaussian with a free std parameter, the storage's GAE variant with advantage standardisation,
// clipped-surrogate / clipped-value minibatch gradients, and clip_grad_norm_ + Adam.
// [ref: OIGE/algo/ppo/module.py:184-361 (MLPEncode), :517-659 (SquashedGaussianDiagonalCovariance), :54-115 (Actor, Critic);
//       OIGE/algo/ppo/storage.py:92-124 (compute_returns), :126-148 (minibatch generators);
//       OIGE/algo/ppo/ppo.py:232-321 (_train_step); OIGE/scripts/rlgames_train_loopz.py:784-842 (network / PPO configuration)]
//
// fp32 SIMT design (same skeleton as ppo_mlp.cu): one CTA owns tiles of 64 samples, one whole network (22.9 k parameters)
// sits in shared memory, activations never leave the SM, each thread keeps an 8x8 block of the 128x128 weight gradient in
// registers across its tiles.  blockIdx.y selects the network: the actor's loss depends only on the actor, the critic's only
// on the critic, so the two backward passes are independent CTAs of ONE launch.
#include <math_constants.h>
#include "philox.cuh"
#include "usv_common.cuh"

namespace loopz {

constexpr int H = PPO_HIDDEN;          // 128
constexpr int TM = 64;                 // samples per tile
constexpr int NT = 256;                // threads per CTA
constexpr int HS = H + 4;              // padded activation / W2T row stride
constexpr int E1 = PPO_LOOPZ_ENC1;     // 64
constexpr int E2 = PPO_LOOPZ_ENC2;     // 16
constexpr int E3 = PPO_LOOPZ_LATENT;   // 8
constexpr int E1S = E1 + 1, E2S = E2 + 1;
constexpr int MS = PPO_LOOPZ_MAX_MASS + 1;   // mass-tile row stride
constexpr float kSlope = 0.01f;        // nn.LeakyReLU default negative_slope
constexpr float kHalfLog2Pi = 0.91893853320467274178f;   // log(sqrt(2*pi))
constexpr int kMaxParts = 148;

__device__ __forceinline__ float lrelu(float x) { return x > 0.f ? x : kSlope * x; }
__device__ __forceinline__ float lrelu_grad(float y) { return y > 0.f ? 1.0f : kSlope; }   // sign(y) == sign(x)
__device__ __forceinline__ float sanitize0(float x) { return isfinite(x) ? x : 0.f; }     // torch.nan_to_num(x, 0, 0, 0)

struct NetLayout {   // offsets of one network inside its span of the flat parameter vector (nn.Module registration order)
  int D, Md, IN, OUT, e1w, e1b, e2w, e2b, e3w, e3b, w1, b1, w2, b2, w3, b3, P;
  __host__ __device__ NetLayout(int d, int md, int out) {
    D = d; Md = md; IN = d - md + E3; OUT = out;
    e1w = 0; e1b = e1w + E1 * md; e2w = e1b + E1; e2b = e2w + E2 * E1; e3w = e2b + E2; e3b = e3w + E3 * E2;
    w1 = e3b + E3; b1 = w1 + H * IN; w2 = b1 + H; b2 = w2 + H * H; w3 = b2 + H; b3 = w3 + out * H; P = b3 + out;
  }
};
struct Spans {       // flat vector: actor architecture | std[2] | critic architecture
  int actor, std, critic, P, PA, PC;
  __host__ __device__ explicit Spans(const PpoLoopzNet& n) {
    PA = NetLayout(n.obs_dim, n.mass_dim, 2).P; PC = NetLayout(n.obs_dim, n.mass_dim, 1).P;
    actor = 0; std = PA; critic = PA + 2; P = PA + 2 + PC;
  }
};
__host__ __device__ inline int part_stride(const Spans& sp) { return sp.PA + 2 + 2; }   // grads | std grads | 2 statistics

struct Smem {
  float *w2t, *h1, *h2, *w1t, *b1, *b2, *w3, *b3, *we1t, *be1, *we2t, *be2, *we3t, *be3, *xs, *ms, *e1, *e2;
  float *dz3, *gw1, *gw3, *gb, *gwe1, *gbe1, *gwe2, *gbe2, *gwe3, *gbe3, *dlat;
  int xstride;
};
__host__ __device__ inline int xs_stride(int D, int IN) { return (D > IN ? D : IN) | 1; }
__host__ __device__ inline size_t smem_floats(int D, int Md, bool train) {
  const int IN = D - Md + E3;
  size_t n = (size_t)H * HS + 2 * (size_t)TM * HS + (size_t)IN * H + 2 * H + 2 * H + 4 + (size_t)Md * E1 + E1 + E1 * E2 + E2 + E2 * E3 + E3 +
             (size_t)TM * xs_stride(D, IN) + TM * MS + TM * E1S + TM * E2S;
  if (train) n += TM * 4 + (size_t)H * IN + 2 * H + (2 * H + 4) + (size_t)Md * E1 + E1 + E1 * E2 + E2 + E2 * E3 + E3 + TM * MS;
  return n;
}
__device__ inline Smem carve(float* base, int D, int Md, bool train) {
  const int IN = D - Md + E3;
  Smem s;
  s.xstride = xs_stride(D, IN);
  float* p = base;
  s.w2t = p; p += H * HS;       // 16 B aligned rows first
  s.h1 = p; p += TM * HS;
  s.h2 = p; p += TM * HS;
  s.w1t = p; p += IN * H;
  s.b1 = p; p += H;
  s.b2 = p; p += H;
  s.w3 = p; p += 2 * H;
  s.b3 = p; p += 4;
  s.we1t = p; p += Md * E1;
  s.be1 = p; p += E1;
  s.we2t = p; p += E1 * E2;
  s.be2 = p; p += E2;
  s.we3t = p; p += E2 * E3;
  s.be3 = p; p += E3;
  s.xs = p; p += TM * s.xstride;
  s.ms = p; p += TM * MS;
  s.e1 = p; p += TM * E1S;
  s.e2 = p; p += TM * E2S;
  if (train) {
    s.dz3 = p; p += TM * 4;
    s.gw1 = p; p += H * IN;
    s.gw3 = p; p += 2 * H;
    s.gb = p; p += 2 * H + 4;
    s.gwe1 = p; p += Md * E1;
    s.gbe1 = p; p += E1;
    s.gwe2 = p; p += E1 * E2;
    s.gbe2 = p; p += E2;
    s.gwe3 = p; p += E2 * E3;
    s.gbe3 = p; p += E3;
    s.dlat = p; p += TM * MS;
  }
  return s;
}

__device__ inline void load_weights(const Smem& s, const float* __restrict__ prm, const NetLayout& L) {
  const int t = threadIdx.x;
  for (int e = t; e < E1 * L.Md; e += NT) { const int o = e / L.Md, k = e - o * L.Md; s.we1t[k * E1 + o] = prm[L.e1w + e]; }
  for (int e = t; e < E2 * E1; e += NT) { const int o = e / E1, k = e - o * E1; s.we2t[k * E2 + o] = prm[L.e2w + e]; }
  for (int e = t; e < E3 * E2; e += NT) { const int o = e / E2, k = e - o * E2; s.we3t[k * E3 + o] = prm[L.e3w + e]; }
  for (int e = t; e < E1; e += NT) s.be1[e] = prm[L.e1b + e];
  if (t < E2) s.be2[t] = prm[L.e2b + t];
  if (t < E3) s.be3[t] = prm[L.e3b + t];
  for (int e = t; e < H * L.IN; e += NT) { const int o = e / L.IN, d = e - o * L.IN; s.w1t[d * H + o] = prm[L.w1 + e]; }
  for (int e = t; e < H * H; e += NT) { const int o = e >> 7, i = e & (H - 1); s.w2t[i * HS + o] = prm[L.w2 + e]; }
  for (int e = t; e < H; e += NT) {
    s.b1[e] = prm[L.b1 + e];
    s.b2[e] = prm[L.b2 + e];
    s.w3[e] = prm[L.w3 + e];
    s.w3[H + e] = (L.OUT > 1) ? prm[L.w3 + H + e] : 0.f;
  }
  if (t == 0) { s.b3[0] = prm[L.b3]; s.b3[1] = (L.OUT > 1) ? prm[L.b3 + 1] : 0.f; s.b3[2] = 0.f; s.b3[3] = 0.f; }
}

// rows of a tile (optionally gathered through `index`: shuffled minibatches), non-finite observations zeroed like the storage does
__device__ inline void load_obs_tile(const Smem& s, const float* __restrict__ obs, const int64_t* __restrict__ index, int D,
                                     int64_t row0, int64_t M) {
  for (int e = threadIdx.x; e < TM * D; e += NT) {
    const int r = e / D, d = e - r * D;
    float y = 0.f;
    if (row0 + r < M) {
      const int64_t row = index ? index[row0 + r] : row0 + r;
      y = sanitize0(obs[row * D + d]);
    }
    s.xs[r * s.xstride + d] = y;
  }
}

// C[4 rows][8 cols] += A[rows ty*4..][0..K) * B[0..K)[cols].  A thread's 8 columns are tx*4..+3 and 64+tx*4..+3, so the 16 threads
// of a half-warp read two contiguous 256 B runs of a B row: conflict-free LDS.128 (8 consecutive columns per thread cost 2 wavefronts
// more per load; the first capture of this kernel ran the shared-memory pipe at 76 % with 35 % of the wavefronts bank conflicts).
__device__ __forceinline__ int tile_col(int tx, int c) { return (c < 4) ? tx * 4 + c : 64 + tx * 4 + (c - 4); }
template <int KU, bool A4>
__device__ inline void gemm_4x8(const float* __restrict__ Asm, int lda, const float* __restrict__ Bsm, int ldb, int K, int ty, int tx,
                                float (&acc)[4][8]) {
  const float* a0 = Asm + (ty * 4) * lda;
  const float* b0 = Bsm + tx * 4;
  if constexpr (A4) {   // lda and K multiples of 4, A rows 16 B aligned
#pragma unroll KU
    for (int k = 0; k < K; k += 4) {
      float4 av[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) av[j] = *reinterpret_cast<const float4*>(a0 + j * lda + k);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 bl = *reinterpret_cast<const float4*>(b0 + (k + kk) * ldb);
        const float4 bh = *reinterpret_cast<const float4*>(b0 + (k + kk) * ldb + 64);
        const float b[8] = {bl.x, bl.y, bl.z, bl.w, bh.x, bh.y, bh.z, bh.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float a = kk == 0 ? av[j].x : (kk == 1 ? av[j].y : (kk == 2 ? av[j].z : av[j].w));
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[j][c] = fmaf(a, b[c], acc[j][c]);
        }
      }
    }
  } else {
#pragma unroll KU
    for (int k = 0; k < K; ++k) {
      const float4 bl = *reinterpret_cast<const float4*>(b0 + k * ldb);
      const float4 bh = *reinterpret_cast<const float4*>(b0 + k * ldb + 64);
      const float b[8] = {bl.x, bl.y, bl.z, bl.w, bh.x, bh.y, bh.z, bh.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float a = a0[j * lda + k];
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[j][c] = fmaf(a, b[c], acc[j][c]);
      }
    }
  }
}
// bias -> accumulators, accumulators -> LeakyReLU -> activation tile (two float4 per row)
__device__ __forceinline__ void acc_init(float (&acc)[4][8], const float* __restrict__ bias, int tx) {
  const float4 bl = *reinterpret_cast<const float4*>(bias + tx * 4), bh = *reinterpret_cast<const float4*>(bias + 64 + tx * 4);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    acc[j][0] = bl.x; acc[j][1] = bl.y; acc[j][2] = bl.z; acc[j][3] = bl.w;
    acc[j][4] = bh.x; acc[j][5] = bh.y; acc[j][6] = bh.z; acc[j][7] = bh.w;
  }
}
__device__ __forceinline__ void acc_store_lrelu(const float (&acc)[4][8], float* __restrict__ h, int ty, int tx) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float* row = h + (ty * 4 + j) * HS;
    *reinterpret_cast<float4*>(row + tx * 4) = make_float4(lrelu(acc[j][0]), lrelu(acc[j][1]), lrelu(acc[j][2]), lrelu(acc[j][3]));
    *reinterpret_cast<float4*>(row + 64 + tx * 4) = make_float4(lrelu(acc[j][4]), lrelu(acc[j][5]), lrelu(acc[j][6]), lrelu(acc[j][7]));
  }
}

// xs (raw obs tile) -> mass encoder -> latent written over the mass columns of xs -> h1 -> h2   [ref module.py:340-361]
__device__ inline void net_forward(const Smem& s, const NetLayout& L) {
  const int t = threadIdx.x;
  const int m0 = L.D - L.Md;   // first mass column == first latent column of the main input
  for (int e = t; e < TM * L.Md; e += NT) { const int r = e / L.Md, k = e - r * L.Md; s.ms[r * MS + k] = s.xs[r * s.xstride + m0 + k]; }
  __syncthreads();
  for (int e = t; e < TM * E1; e += NT) {
    const int r = e / E1, o = e - r * E1;
    float acc = s.be1[o];
    for (int k = 0; k < L.Md; ++k) acc = fmaf(s.ms[r * MS + k], s.we1t[k * E1 + o], acc);
    s.e1[r * E1S + o] = lrelu(acc);
  }
  __syncthreads();
  {   // thread = (row, 4 outputs): one broadcast word of e1 + one LDS.128 of W_e2^T feed 4 FMAs
    static_assert(TM * E2 == NT * 4, "e2 tiling");
    const int r = t >> 2, o4 = (t & 3) * 4;
    float4 acc = *reinterpret_cast<const float4*>(s.be2 + o4);
    const float* er = s.e1 + r * E1S;
#pragma unroll 8
    for (int k = 0; k < E1; ++k) {
      const float a = er[k];
      const float4 w = *reinterpret_cast<const float4*>(s.we2t + k * E2 + o4);
      acc.x = fmaf(a, w.x, acc.x); acc.y = fmaf(a, w.y, acc.y); acc.z = fmaf(a, w.z, acc.z); acc.w = fmaf(a, w.w, acc.w);
    }
    float* out = s.e2 + r * E2S + o4;
    out[0] = lrelu(acc.x); out[1] = lrelu(acc.y); out[2] = lrelu(acc.z); out[3] = lrelu(acc.w);
  }
  __syncthreads();
  for (int e = t; e < TM * E3; e += NT) {
    const int r = e / E3, o = e - r * E3;
    float acc = s.be3[o];
#pragma unroll
    for (int k = 0; k < E2; ++k) acc = fmaf(s.e2[r * E2S + k], s.we3t[k * E3 + o], acc);
    s.xs[r * s.xstride + m0 + o] = lrelu(acc);
  }
  __syncthreads();
  const int ty = t >> 4, tx = t & 15;
  float acc[4][8];
  acc_init(acc, s.b1, tx);
  gemm_4x8<1, false>(s.xs, s.xstride, s.w1t, H, L.IN, ty, tx, acc);
  acc_store_lrelu(acc, s.h1, ty, tx);
  __syncthreads();
  acc_init(acc, s.b2, tx);
  gemm_4x8<2, true>(s.h1, HS, s.w2t, HS, H, ty, tx, acc);
  acc_store_lrelu(acc, s.h2, ty, tx);
  __syncthreads();
}

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

// log pi(a) of the tanh-squashed, scaled Gaussian for the pre-squash sample u   [ref module.py:555-566]
__device__ inline float squashed_log_prob(float u0, float u1, float m0, float m1, float s0, float s1, float scale, float eps) {
  const float t0 = tanhf(u0), t1 = tanhf(u1);
  const float d0 = u0 - m0, d1 = u1 - m1;
  const float lpu = (-(d0 * d0) / (2.0f * (s0 * s0)) - logf(s0) - kHalfLog2Pi) + (-(d1 * d1) / (2.0f * (s1 * s1)) - logf(s1) - kHalfLog2Pi);
  const float log_det = 2.0f * logf(scale + eps) + (logf(1.0f - t0 * t0 + eps) + logf(1.0f - t1 * t1 + eps));
  return lpu - log_det;
}

// ---------------------------------------------------------------------------------------------
// rollout: actor.sample(obs) and critic.predict(obs)   [ref module.py:67-70,104-105,568-583 ; ppo.py:97-148]
__global__ void __launch_bounds__(NT, 1) act_kernel(const float* __restrict__ prm, PpoLoopzNet cfg, int first_net,
                                                   const float* __restrict__ obs_actor, const float* __restrict__ obs_critic, uint64_t seed,
                                                   uint64_t counter_in, const uint64_t* __restrict__ counter_offset, int64_t row_offset,
                                                   const float* __restrict__ eval_actions, float* __restrict__ actions,
                                                   float* __restrict__ log_prob, float* __restrict__ means, float* __restrict__ values,
                                                   int64_t M) {
  extern __shared__ __align__(16) float smem[];
  const int net = first_net + blockIdx.y;   // 0 = actor, 1 = critic
  const Spans sp(cfg);
  const NetLayout L(cfg.obs_dim, cfg.mass_dim, net == 0 ? 2 : 1);
  const Smem s = carve(smem, L.D, L.Md, false);
  const float* np = prm + (net == 0 ? sp.actor : sp.critic);
  const float* obs = net == 0 ? obs_actor : obs_critic;
  load_weights(s, np, L);
  const uint64_t counter = counter_in + (counter_offset ? *counter_offset : 0ull);
  const float sd0 = prm[sp.std], sd1 = prm[sp.std + 1];
  const int64_t ntiles = (M + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * TM;
    __syncthreads();
    load_obs_tile(s, obs, nullptr, L.D, row0, M);
    __syncthreads();
    net_forward(s, L);
    const int r = threadIdx.x >> 2, j = threadIdx.x & 3;
    const int64_t row = row0 + r;
    const float o = (j < L.OUT) ? head_out(s, r, j) : 0.f;
    const int base = (threadIdx.x & 31) & ~3;
    const float o0 = __shfl_sync(0xffffffffu, o, base), o1 = __shfl_sync(0xffffffffu, o, base + 1);
    if (j != 0 || row >= M) continue;
    if (net == 1) {
      values[row] = o0;
      continue;
    }
    const float m0 = cfg.tanh_out ? tanhf(o0) : o0, m1 = cfg.tanh_out ? tanhf(o1) : o1;
    if (means) { means[row * 2] = m0; means[row * 2 + 1] = m1; }
    if (eval_actions) {   // actor.evaluate(obs, actions): log-prob of given actions   [ref module.py:586-637]
      const float lim = 1.0f - cfg.eps;
      const float as0 = fminf(fmaxf(eval_actions[row * 2] / (cfg.action_scale + cfg.eps), -lim), lim);
      const float as1 = fminf(fmaxf(eval_actions[row * 2 + 1] / (cfg.action_scale + cfg.eps), -lim), lim);
      const float u0 = 0.5f * (log1pf(as0) - log1pf(-as0)), u1 = 0.5f * (log1pf(as1) - log1pf(-as1));
      log_prob[row] = squashed_log_prob(u0, u1, isfinite(m0) ? m0 : 0.f, isfinite(m1) ? m1 : 0.f, isfinite(sd0) ? sd0 : 1.0f,
                                        isfinite(sd1) ? sd1 : 1.0f, cfg.action_scale, cfg.eps);
    } else if (actions) {
      // u ~ Normal(mean, std): Box-Muller on Philox uniforms keyed (seed; global row, counter)
      const usv::Philox4 rr = usv::philox4x32_10((uint32_t)(row + row_offset), (uint32_t)counter, (uint32_t)(counter >> 32),
                                                 101u ^ ((uint32_t)((uint64_t)(row + row_offset) >> 32) << 8), (uint32_t)seed,
                                                 (uint32_t)(seed >> 32));
      const float u1 = (float)((rr.x >> 8) + 1u) * (1.0f / 16777216.0f);   // (0,1]
      const float u2 = (float)(rr.y >> 8) * (1.0f / 16777216.0f);          // [0,1)
      const float rad = sqrtf(-2.0f * logf(u1));
      float sn, cs;
      sincosf(6.28318530717958647692f * u2, &sn, &cs);
      const float x0 = m0 + sd0 * (rad * cs), x1 = m1 + sd1 * (rad * sn);
      actions[row * 2] = tanhf(x0) * cfg.action_scale;
      actions[row * 2 + 1] = tanhf(x1) * cfg.action_scale;
      if (log_prob) log_prob[row] = squashed_log_prob(x0, x1, m0, m1, sd0, sd1, cfg.action_scale, cfg.eps);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// training: forward + loss + backward of one network for the tiles of one CTA; partial gradients per CTA
struct LossIn {
  const float *actions, *old_log_prob, *adv, *target_values, *returns;
  const int64_t* index;
};

__global__ void __launch_bounds__(NT, 1) train_kernel(const float* __restrict__ prm, PpoLoopzNet cfg, const float* __restrict__ obs_actor,
                                                     const float* __restrict__ obs_critic, LossIn in, PpoLoopzLossParams lp,
                                                     float* __restrict__ partial, int64_t M) {
  extern __shared__ __align__(16) float smem[];
  const int net = blockIdx.y;
  const Spans sp(cfg);
  const NetLayout L(cfg.obs_dim, cfg.mass_dim, net == 0 ? 2 : 1);
  const Smem s = carve(smem, L.D, L.Md, true);
  const float* np = prm + (net == 0 ? sp.actor : sp.critic);
  const float* obs = net == 0 ? obs_actor : obs_critic;
  const int t = threadIdx.x;
  load_weights(s, np, L);
  for (int e = t; e < H * L.IN; e += NT) s.gw1[e] = 0.f;
  for (int e = t; e < 2 * H; e += NT) s.gw3[e] = 0.f;
  for (int e = t; e < 2 * H + 4; e += NT) s.gb[e] = 0.f;
  for (int e = t; e < E1 * L.Md; e += NT) s.gwe1[e] = 0.f;
  for (int e = t; e < E1 * E2; e += NT) s.gwe2[e] = 0.f;
  for (int e = t; e < E2 * E3; e += NT) s.gwe3[e] = 0.f;
  if (t < E1) s.gbe1[t] = 0.f;
  if (t < E2) s.gbe2[t] = 0.f;
  if (t < E3) s.gbe3[t] = 0.f;
  float sd0 = prm[sp.std], sd1 = prm[sp.std + 1];
  if (!isfinite(sd0)) sd0 = 1.0f;     // evaluate(): nan_to_num(std, 1, 1, 1)  [ref module.py:607-615]
  if (!isfinite(sd1)) sd1 = 1.0f;
  const float invM = 1.0f / (float)M;
  const int m0c = L.D - L.Md;
  float gW2[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) gW2[a][b] = 0.f;
  float st_loss = 0.f, st_lp = 0.f, g_sd0 = 0.f, g_sd1 = 0.f;
  const int ty = t >> 4, tx = t & 15;
  const int64_t ntiles = (M + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * TM;
    __syncthreads();
    load_obs_tile(s, obs, in.index, L.D, row0, M);
    __syncthreads();
    net_forward(s, L);
    // ---- output layer + per-sample loss gradient: 4 lanes per row ----------------------------------------
    {
      const int r = t >> 2, j = t & 3;
      const float o = (j < L.OUT) ? head_out(s, r, j) : 0.f;
      const int base = (t & 31) & ~3;
      const float o0 = __shfl_sync(0xffffffffu, o, base), o1 = __shfl_sync(0xffffffffu, o, base + 1);
      float dz0 = 0.f, dz1 = 0.f;
      if (j == 0 && row0 + r < M) {
        const int64_t row = in.index ? in.index[row0 + r] : row0 + r;
        if (net == 0) {
          float m0 = cfg.tanh_out ? tanhf(o0) : o0, m1 = cfg.tanh_out ? tanhf(o1) : o1;
          const bool f0 = isfinite(m0), f1 = isfinite(m1);        // evaluate(): nan_to_num(logits)  [ref module.py:591-604]
          if (!f0) m0 = 0.f;
          if (!f1) m1 = 0.f;
          // stored action -> pre-squash u = atanh(clamp(a / (scale + eps)))   [ref module.py:620-626]
          const float lim = 1.0f - cfg.eps;
          const float as0 = fminf(fmaxf(in.actions[row * 2] / (cfg.action_scale + cfg.eps), -lim), lim);
          const float as1 = fminf(fmaxf(in.actions[row * 2 + 1] / (cfg.action_scale + cfg.eps), -lim), lim);
          const float u0 = 0.5f * (log1pf(as0) - log1pf(-as0)), u1 = 0.5f * (log1pf(as1) - log1pf(-as1));
          const float logp = squashed_log_prob(u0, u1, m0, m1, sd0, sd1, cfg.action_scale, cfg.eps);
          // clipped surrogate   [ref ppo.py:252-258]
          const float adv = in.adv[row];
          const float ratio = expf(logp - in.old_log_prob[row]);
          const float lo = 1.0f - lp.clip_param, hi = 1.0f + lp.clip_param;
          const float su = -adv * ratio, sc = -adv * fminf(fmaxf(ratio, lo), hi);
          const float loss = fmaxf(su, sc);
          const bool inside = ratio >= lo && ratio <= hi;
          const float w = su > sc ? 1.0f : (su == sc ? (inside ? 1.0f : 0.5f) : 0.f);    // torch.max splits ties evenly
          // rl_loss = mean(surrogate + value_coef*value_loss - entropy_coef*entropy), entropy := -log_prob  [ref ppo.py:276-277, module.py:632-637]
          const float g_lp = (-adv * ratio * w + lp.entropy_coef) * invM;
          const float d0 = u0 - m0, d1 = u1 - m1;
          const float gm0 = g_lp * d0 / (sd0 * sd0), gm1 = g_lp * d1 / (sd1 * sd1);
          g_sd0 += g_lp * (d0 * d0 / (sd0 * sd0 * sd0) - 1.0f / sd0);
          g_sd1 += g_lp * (d1 * d1 / (sd1 * sd1 * sd1) - 1.0f / sd1);
          dz0 = f0 ? (cfg.tanh_out ? gm0 * (1.0f - m0 * m0) : gm0) : 0.f;
          dz1 = f1 ? (cfg.tanh_out ? gm1 * (1.0f - m1 * m1) : gm1) : 0.f;
          st_loss += loss;
          st_lp += logp;
        } else {
          // (clipped) value loss   [ref ppo.py:261-268]
          const float v = o0, tv = in.target_values[row], ret = in.returns[row];
          float vl, g;
          if (lp.use_clipped_value_loss) {
            const float dv = v - tv;
            const float vc = tv + fminf(fmaxf(dv, -lp.clip_param), lp.clip_param);
            const float l1 = (v - ret) * (v - ret), l2 = (vc - ret) * (vc - ret);
            vl = fmaxf(l1, l2);
            const float g1 = 2.0f * (v - ret);
            const float g2 = (dv >= -lp.clip_param && dv <= lp.clip_param) ? 2.0f * (vc - ret) : 0.f;
            g = l1 > l2 ? g1 : (l1 == l2 ? 0.5f * (g1 + g2) : g2);
          } else {
            vl = (ret - v) * (ret - v);
            g = 2.0f * (v - ret);
          }
          dz0 = lp.value_loss_coef * g * invM;
          st_loss += vl;
        }
      }
      if (j == 0) { s.dz3[r * 4 + 0] = dz0; s.dz3[r * 4 + 1] = dz1; s.dz3[r * 4 + 2] = 0.f; s.dz3[r * 4 + 3] = 0.f; }
    }
    __syncthreads();
    // ---- output-layer gradients ---------------------------------------------------------------------------
    for (int e = t; e < L.OUT * H; e += NT) {
      const int j = e >> 7, k = e & (H - 1);
      float acc = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) acc = fmaf(s.dz3[r * 4 + j], s.h2[r * HS + k], acc);
      s.gw3[e] += acc;
    }
    if (t < L.OUT) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.dz3[r * 4 + t];
      s.gb[2 * H + t] += acc;
    }
    __syncthreads();
    // ---- dz2 = (dz3 . W3) * lrelu'(h2), in place over h2 --------------------------------------------------
    {
      float4 wa[2], wb[2];
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        wa[hh] = *reinterpret_cast<const float4*>(s.w3 + hh * 64 + tx * 4);
        wb[hh] = *reinterpret_cast<const float4*>(s.w3 + H + hh * 64 + tx * 4);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = ty * 4 + j;
        const float g0 = s.dz3[r * 4], g1 = s.dz3[r * 4 + 1];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          float4* hp = reinterpret_cast<float4*>(s.h2 + r * HS + hh * 64 + tx * 4);
          const float4 h = *hp;
          *hp = make_float4((g0 * wa[hh].x + g1 * wb[hh].x) * lrelu_grad(h.x), (g0 * wa[hh].y + g1 * wb[hh].y) * lrelu_grad(h.y),
                            (g0 * wa[hh].z + g1 * wb[hh].z) * lrelu_grad(h.z), (g0 * wa[hh].w + g1 * wb[hh].w) * lrelu_grad(h.w));
        }
      }
    }
    __syncthreads();
    // ---- gW2[o][i] += sum_r dz2[r][o]*h1[r][i]  (8x8 block per thread, registers) ; db2 --------------------
    {
      const float* za = s.h2 + ty * 8;
      const float* hb = s.h1 + tx * 4;   // i columns tx*4..+3 and 64+tx*4..+3 (conflict-free float4)
#pragma unroll 4
      for (int r = 0; r < TM; ++r) {
        const float4 al = *reinterpret_cast<const float4*>(za + r * HS), ah = *reinterpret_cast<const float4*>(za + r * HS + 4);
        const float4 bl = *reinterpret_cast<const float4*>(hb + r * HS), bh = *reinterpret_cast<const float4*>(hb + r * HS + 64);
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
    // ---- dz1 = (dz2 . W2) * lrelu'(h1), in place over h1 (columns interleaved: i = tx + 16c) ---------------
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
          s.h1[r * HS + i] = acc[j][c] * lrelu_grad(s.h1[r * HS + i]);
        }
    }
    __syncthreads();
    // ---- gw1[o][d] += sum_r dz1[r][o]*zin[r][d] ; db1 ; d(latent) -----------------------------------------
    {   // 4 outputs x <= 8 input columns per thread: one LDS.128 of dz1 + one broadcast word of zin feed 4 FMAs each
      const int o4 = (t & 31) * 4, dg = t >> 5;
      float g1a[8][4];
#pragma unroll
      for (int q = 0; q < 8; ++q) { g1a[q][0] = 0.f; g1a[q][1] = 0.f; g1a[q][2] = 0.f; g1a[q][3] = 0.f; }
#pragma unroll 2
      for (int r = 0; r < TM; ++r) {
        const float4 dz = *reinterpret_cast<const float4*>(s.h1 + r * HS + o4);
        const float* xr = s.xs + r * s.xstride + dg;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (dg + 8 * q < L.IN) {
            const float x = xr[8 * q];
            g1a[q][0] = fmaf(dz.x, x, g1a[q][0]); g1a[q][1] = fmaf(dz.y, x, g1a[q][1]);
            g1a[q][2] = fmaf(dz.z, x, g1a[q][2]); g1a[q][3] = fmaf(dz.w, x, g1a[q][3]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int d = dg + 8 * q;
        if (d < L.IN) {
#pragma unroll
          for (int i = 0; i < 4; ++i) s.gw1[(o4 + i) * L.IN + d] += g1a[q][i];
        }
      }
    }
    if (t < H) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.h1[r * HS + t];
      s.gb[t] += acc;
    }
    for (int e = t; e < TM * E3; e += NT) {       // dlat_pre[r][j] = (dz1[r] . W1[:, m0c+j]) * lrelu'(lat[r][j]); a warp = 32 rows, one j
      const int j = e / TM, r = e - j * TM;
      const float* dz = s.h1 + r * HS;
      const float* w = s.w1t + (m0c + j) * H;
      float acc = 0.f;
#pragma unroll 8
      for (int o = 0; o < H; o += 4) {
        const float4 a = *reinterpret_cast<const float4*>(dz + o);
        const float4 b = *reinterpret_cast<const float4*>(w + o);
        acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
      }
      s.dlat[r * MS + j] = acc * lrelu_grad(s.xs[r * s.xstride + m0c + j]);
    }
    __syncthreads();
    // ---- encoder layer 3: gwe3[o][k] += sum_r dlat[r][o]*e2[r][k] ; de2 in place -----------------------------
    if (t < E3 * E2) {
      const int o = t / E2, k = t - o * E2;
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc = fmaf(s.dlat[r * MS + o], s.e2[r * E2S + k], acc);
      s.gwe3[t] += acc;
    } else if (t < E3 * E2 + E3) {
      const int o = t - E3 * E2;
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.dlat[r * MS + o];
      s.gbe3[o] += acc;
    }
    __syncthreads();
    for (int e = t; e < TM * E2; e += NT) {
      const int r = e / E2, k = e - r * E2;
      float acc = 0.f;
#pragma unroll
      for (int o = 0; o < E3; ++o) acc = fmaf(s.dlat[r * MS + o], s.we3t[k * E3 + o], acc);
      s.e2[r * E2S + k] = acc * lrelu_grad(s.e2[r * E2S + k]);
    }
    __syncthreads();
    // ---- encoder layer 2: gwe2[o][k] += sum_r de2[r][o]*e1[r][k] ; de1 in place ------------------------------
    {   // thread = (k, 4 outputs o): one word of e1 + 4 broadcast words of de2 feed 4 FMAs
      static_assert(E2 * E1 == NT * 4, "gwe2 tiling");
      const int k = t & (E1 - 1), og = (t >> 6) * 4;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) {
        const float x = s.e1[r * E1S + k];
        const float* d = s.e2 + r * E2S + og;
        a0 = fmaf(d[0], x, a0); a1 = fmaf(d[1], x, a1); a2 = fmaf(d[2], x, a2); a3 = fmaf(d[3], x, a3);
      }
      s.gwe2[(og + 0) * E1 + k] += a0; s.gwe2[(og + 1) * E1 + k] += a1; s.gwe2[(og + 2) * E1 + k] += a2; s.gwe2[(og + 3) * E1 + k] += a3;
    }
    if (t < E2) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.e2[r * E2S + t];
      s.gbe2[t] += acc;
    }
    __syncthreads();
    {   // thread = (row, 16 columns k): the row's de2 in registers, W_e2^T rows by LDS.128 (a per-output loop reads W_e2^T with a
        // 16-way bank conflict: stride 16 words)
      static_assert(TM * 4 == NT, "de1 tiling");
      const int r = t >> 2, kb = (t & 3) * 16;
      float d[E2];
#pragma unroll
      for (int o = 0; o < E2; ++o) d[o] = s.e2[r * E2S + o];
#pragma unroll 4
      for (int kk = 0; kk < 16; ++kk) {
        const float* w = s.we2t + (kb + kk) * E2;
        float acc = 0.f;
#pragma unroll
        for (int o = 0; o < E2; o += 4) {
          const float4 wv = *reinterpret_cast<const float4*>(w + o);
          acc = fmaf(d[o], wv.x, acc); acc = fmaf(d[o + 1], wv.y, acc); acc = fmaf(d[o + 2], wv.z, acc); acc = fmaf(d[o + 3], wv.w, acc);
        }
        float* ep = s.e1 + r * E1S + kb + kk;
        *ep = acc * lrelu_grad(*ep);
      }
    }
    __syncthreads();
    // ---- encoder layer 1: gwe1[o][k] += sum_r de1[r][o]*mass[r][k] -------------------------------------------
    for (int e = t; e < E1 * L.Md; e += NT) {
      const int k = e / E1, o = e - k * E1;      // consecutive threads -> consecutive o
      float acc = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) acc = fmaf(s.e1[r * E1S + o], s.ms[r * MS + k], acc);
      s.gwe1[o * L.Md + k] += acc;
    }
    if (t < E1) {
      float acc = 0.f;
      for (int r = 0; r < TM; ++r) acc += s.e1[r * E1S + t];
      s.gbe1[t] += acc;
    }
  }
  __syncthreads();
  // ---- this CTA's partial gradient + statistics --------------------------------------------------------------
  const int S = part_stride(sp);
  float* out = partial + ((size_t)net * gridDim.x + blockIdx.x) * S;
  for (int e = t; e < E1 * L.Md; e += NT) out[L.e1w + e] = s.gwe1[e];
  for (int e = t; e < E2 * E1; e += NT) out[L.e2w + e] = s.gwe2[e];
  for (int e = t; e < E3 * E2; e += NT) out[L.e3w + e] = s.gwe3[e];
  if (t < E1) out[L.e1b + t] = s.gbe1[t];
  if (t < E2) out[L.e2b + t] = s.gbe2[t];
  if (t < E3) out[L.e3b + t] = s.gbe3[t];
  for (int e = t; e < H * L.IN; e += NT) out[L.w1 + e] = s.gw1[e];
  for (int e = t; e < H; e += NT) { out[L.b1 + e] = s.gb[e]; out[L.b2 + e] = s.gb[H + e]; }
  for (int e = t; e < L.OUT * H; e += NT) out[L.w3 + e] = s.gw3[e];
  if (t < L.OUT) out[L.b3 + t] = s.gb[2 * H + t];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) out[L.w2 + (ty * 8 + a) * H + tile_col(tx, b)] = gW2[a][b];
  __shared__ float red[4][NT / 32];
  float vals[4] = {st_loss, st_lp, g_sd0, g_sd1};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float v = vals[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((t & 31) == 0) red[q][t >> 5] = v;
  }
  __syncthreads();
  if (t < 4) {
    float v = 0.f;
    for (int w = 0; w < NT / 32; ++w) v += red[t][w];
    // [S-4, S-3] = std gradient (actor CTAs), [S-2] = sum of the per-sample loss, [S-1] = sum of log-probs
    out[S - 4 + (t < 2 ? t + 2 : t - 2)] = v;
  }
}

// second stage: grads = sum over CTAs (fixed order -> deterministic); statistics tail
__global__ void __launch_bounds__(256) reduce_kernel(const float* __restrict__ partial, int nparts, PpoLoopzNet cfg, PpoLoopzLossParams lp,
                                                     float* __restrict__ grads) {
  __shared__ float sm[4][64];
  const Spans sp(cfg);
  const int S = part_stride(sp);
  const int col = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int e = blockIdx.x * 64 + col;
  const int n = sp.P + PPO_LOOPZ_STAT_COUNT;
  // where element e lives in the per-CTA records
  int net = 0, c0 = 0;
  bool live = e < n;
  if (e < sp.PA) { net = 0; c0 = e; }
  else if (e < sp.PA + 2) { net = 0; c0 = S - 4 + (e - sp.PA); }
  else if (e < sp.P) { net = 1; c0 = e - sp.critic; }
  else if (e == sp.P + PPO_LOOPZ_STAT_SURROGATE) { net = 0; c0 = S - 2; }
  else if (e == sp.P + PPO_LOOPZ_STAT_VALUE_LOSS) { net = 1; c0 = S - 2; }
  else if (e == sp.P + PPO_LOOPZ_STAT_LOG_PROB) { net = 0; c0 = S - 1; }
  else live = false;
  float acc = 0.f;
  if (live)
    for (int c = grp; c < nparts; c += 4) acc += partial[((size_t)net * nparts + c) * S + c0];
  sm[grp][col] = acc;
  __syncthreads();
  if (grp == 0 && live) grads[e] = (sm[0][col] + sm[1][col]) + (sm[2][col] + sm[3][col]);
}

// clip_grad_norm_ + Adam over the whole flat vector; the step is skipped when the loss is not finite   [ref ppo.py:286-299]
constexpr int kAdamThreads = 256;
__global__ void __launch_bounds__(kAdamThreads) adam_kernel(float* __restrict__ prm, float* __restrict__ g, float* __restrict__ m,
                                                            float* __restrict__ v, const float* __restrict__ lr_dev,
                                                            const int* __restrict__ step_in, int* __restrict__ step_out,
                                                            float* __restrict__ accum, int P, float inv_M, PpoLoopzLossParams lp,
                                                            PpoLoopzAdamParams ap) {
  __shared__ float red[kAdamThreads / 32];
  __shared__ float s_coef;
  const int t = threadIdx.x;
  float ss = 0.f;
  for (int e = t; e < P; e += kAdamThreads) ss = fmaf(g[e], g[e], ss);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((t & 31) == 0) red[t >> 5] = ss;
  __syncthreads();
  if (t == 0) {
    float x = 0.f;
    for (int w = 0; w < kAdamThreads / 32; ++w) x += red[w];
    const float norm = sqrtf(x);
    s_coef = (ap.max_grad_norm > 0.f) ? fminf(ap.max_grad_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    red[0] = norm;
  }
  __syncthreads();
  const float surr = g[P + PPO_LOOPZ_STAT_SURROGATE] * inv_M, vloss = g[P + PPO_LOOPZ_STAT_VALUE_LOSS] * inv_M;
  const float mlp = g[P + PPO_LOOPZ_STAT_LOG_PROB] * inv_M;
  const float loss = surr + lp.value_loss_coef * vloss + lp.entropy_coef * mlp;
  const bool ok = isfinite(loss);
  const int step = *step_in + (ok ? 1 : 0);
  const int e = blockIdx.x * kAdamThreads + t;
  if (ok && e < P) {
    const float lr = *lr_dev;
    const double bc1 = 1.0 - pow((double)ap.beta1, (double)step), bc2 = 1.0 - pow((double)ap.beta2, (double)step);
    const float step_size = (float)((double)lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float gr = g[e] * s_coef;
    const float mm = m[e] + (gr - m[e]) * (1.0f - ap.beta1);
    const float vv = v[e] * ap.beta2 + (1.0f - ap.beta2) * gr * gr;
    m[e] = mm;
    v[e] = vv;
    prm[e] = prm[e] - step_size * (mm / (sqrtf(vv) / bc2_sqrt + ap.eps));
  }
  if (blockIdx.x == gridDim.x - 1 && t == 0) {   // the statistics tail has one owner
    *step_out = step;
    g[P + PPO_LOOPZ_STAT_LOSS] = loss;
    g[P + PPO_LOOPZ_STAT_GRAD_NORM] = red[0];
    g[P + PPO_LOOPZ_STAT_SKIPPED] = ok ? 0.f : 1.f;
    if (accum) {   // mean_value_loss / mean_surrogate_loss over the valid updates   [ref ppo.py:301-318]
      if (isfinite(vloss)) accum[0] += vloss;
      if (isfinite(surr)) accum[1] += surr;
      if (ok) accum[2] += 1.0f;
    }
  }
}

// the statistics the adam kernel reads are SUMS; turn the tail into means afterwards (separate tiny launch: every CTA of the adam
// kernel reads the sums)
__global__ void stat_mean_kernel(float* g, int P, float inv_M) {
  const int t = threadIdx.x;
  if (t == PPO_LOOPZ_STAT_SURROGATE || t == PPO_LOOPZ_STAT_VALUE_LOSS || t == PPO_LOOPZ_STAT_LOG_PROB) g[P + t] *= inv_M;
}

__global__ void min_std_kernel(float* std, const float* min_std, int dim) {   // [ref module.py:649-659]
  const int j = threadIdx.x;
  if (j < dim) {
    const float lo = min_std[j];
    const float cur = isfinite(std[j]) ? std[j] : lo;
    std[j] = fmaxf(cur, lo);
  }
}

// ---------------------------------------------------------------------------------------------
// RolloutStorage.compute_returns: reverse scan per env (coalesced over envs), then advantage standardisation over the batch
constexpr int kRetBlocks = 1184;   // 8 x 148
__global__ void __launch_bounds__(256) returns_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                                      const uint8_t* __restrict__ dones, const float* __restrict__ last_values, float gamma,
                                                      float lam, float* __restrict__ returns, float* __restrict__ adv, double* __restrict__ part,
                                                      int T, int64_t n) {
  double s1 = 0.0, s2 = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    float nextv = sanitize0(last_values[j]);
    float a = 0.f;
#pragma unroll 4
    for (int t = T - 1; t >= 0; --t) {
      const int64_t q = (int64_t)t * n + j;
      const float r = sanitize0(rewards[q]), v = sanitize0(values[q]);
      const float nnt = 1.0f - (float)dones[q];                  // the done flag of THIS step   [ref storage.py:109]
      const float ng = __fmul_rn(nnt, gamma);
      const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(ng, nextv)), v);
      a = __fadd_rn(delta, __fmul_rn(__fmul_rn(ng, lam), a));
      const float ret = __fadd_rn(a, v);
      const float ad = __fsub_rn(ret, v);                        // advantages = returns - values   [ref storage.py:114]
      returns[q] = sanitize0(ret);
      adv[q] = ad;
      s1 += (double)ad;
      s2 += (double)ad * (double)ad;
      nextv = v;
    }
  }
  __shared__ double sh[2][8];
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s1; sh[1][threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
    part[2 * blockIdx.x] = a;
    part[2 * blockIdx.x + 1] = b;
  }
}
// moments over `total` entries (all ranks' batches when the moments were exchanged), normalising the `count` local entries
__global__ void __launch_bounds__(256) adv_norm_kernel(float* __restrict__ adv, const double* __restrict__ part, int nparts, int64_t total,
                                                       int64_t count) {
  __shared__ double sh[2][8];
  __shared__ float s_mean, s_inv;
  double s1 = 0.0, s2 = 0.0;
  for (int c = threadIdx.x; c < nparts; c += 256) { s1 += part[2 * c]; s2 += part[2 * c + 1]; }
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s1; sh[1][threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
    const double mean = a / (double)total;
    double var = total > 1 ? (b - a * mean) / (double)(total - 1) : CUDART_NAN;   // torch.std: unbiased
    if (var < 0.0) var = 0.0;
    float sd = (float)sqrt(var);
    if (!isfinite(sd)) sd = 0.f;                                                   // nan_to_num(adv_std)   [ref storage.py:117]
    s_mean = (float)mean;
    s_inv = sd + 1e-8f;
  }
  __syncthreads();
  const float mean = s_mean, den = s_inv;
  for (int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x; q < count; q += (int64_t)gridDim.x * 256)
    adv[q] = sanitize0((adv[q] - mean) / den);
}

// ---------------------------------------------------------------------------------------------
// data-parallel training over `world` ranks (one process per GPU, CUDA-IPC windows of ppo_peer_window_alloc / _open).  Two exchanges
// share one window set and one sequence counter, in the order every rank issues them: the advantage moments once per update, the
// minibatch gradient once per minibatch.  Window of rank q: [2 parities][world][ecap] packets {fp32 payload, sequence} (usv::st_packet),
// ecap = cap / (2 world).  A rank stores its packet for entry e straight into slot [seq & 1][its rank][e] of every peer's window and
// polls its own window until every peer's packet of entry e carries this sequence number, then adds the values in rank order: every
// rank gets the same bits.  Double buffering by parity: a peer can be at most one exchange ahead (it needs this rank's packets of
// exchange s+1 to finish s+1), and its packets of s+1 land in the other parity.
// seq_dev = device uint32[2] {sequence number of the last exchange, arrival counter}, zero at start and the same on every rank; the last
// CTA to finish advances the sequence, i.e. after every CTA has read it.  A peer that does not arrive within usv::kPeerSpinNs sets the
// sticky err_flag; from then on the exchanges stop waiting and the gradient exchange marks its statistics non-finite, so Adam skips the
// step on un-reduced gradients (the host reads the flag: PPO.check_peers).
constexpr int kXThreads = 256;

__device__ inline bool wait_packet(const float* src, uint32_t seq, float& x, const uint32_t* err_flag) {
  if (usv::ld_packet(src, seq, x)) return true;
  const unsigned long long t0 = usv::global_ns();
  uint32_t spins = 0;
  while (!usv::ld_packet(src, seq, x))
    if ((++spins & 255u) == 0 && (usv::global_ns() - t0 > usv::kPeerSpinNs || *reinterpret_cast<const volatile uint32_t*>(err_flag))) return false;
  return true;
}

// grads[0, n) summed over ranks; the gradient entries [0, P) are means over each rank's minibatch, so their sum is scaled by 1/world
// (the mean over all ranks' samples); the statistics behind them are sums and stay sums (Adam divides them by world x M).
// CTA b handles entries b, b + grid, ... on every rank and only waits for CTA b of its peers, so each CTA needs its peers' CTAs to be
// resident at some point, never its own rank's other CTAs.  The grid is at most one CTA per SM (one wave of a kernel without shared
// memory), so all CTAs of a launch are resident together; there is no grid-wide barrier, hence no cooperative launch.
__global__ void __launch_bounds__(kXThreads) grad_exchange_kernel(PpoPeerComm c, float* __restrict__ g, int n, int P, float inv_world,
                                                                  uint32_t* __restrict__ seq_dev, uint32_t* __restrict__ err_flag) {
  __shared__ uint32_t s_seq;
  __shared__ int s_bad;
  if (threadIdx.x == 0) { s_seq = seq_dev[0] + 1u; s_bad = *reinterpret_cast<volatile uint32_t*>(err_flag) != 0; }
  __syncthreads();
  const uint32_t seq = s_seq;
  const int64_t ecap = c.cap / (2 * c.world);
  const int64_t par = (int64_t)(seq & 1u) * c.world;
  if (!s_bad) {
    for (int e = blockIdx.x * kXThreads + threadIdx.x; e < n; e += gridDim.x * kXThreads) {
      const float v = g[e];
      for (int p = 0; p < c.world; ++p)
        if (p != c.rank) usv::st_packet(c.windows[p] + ((par + c.rank) * ecap + e) * 2, v, seq);
    }
    bool bad = false;
    const float* mine = c.windows[c.rank];
    for (int e = blockIdx.x * kXThreads + threadIdx.x; e < n && !bad; e += gridDim.x * kXThreads) {
      const float own = g[e];
      float acc = 0.f;
      for (int p = 0; p < c.world && !bad; ++p) {
        float x = own;
        if (p != c.rank) bad = !wait_packet(mine + ((par + p) * ecap + e) * 2, seq, x, err_flag);
        acc = p == 0 ? x : acc + x;
      }
      if (!bad) g[e] = e < P ? acc * inv_world : acc;
    }
    if (bad) { atomicOr(err_flag, 1u); s_bad = 1; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(seq_dev + 1, 1u) == gridDim.x - 1) {   // the last CTA: every CTA has read the sequence number and written its entries
      seq_dev[1] = 0u;
      seq_dev[0] = seq;
      if (*reinterpret_cast<volatile uint32_t*>(err_flag)) g[P + PPO_LOOPZ_STAT_SURROGATE] = CUDART_NAN_F;   // Adam skips the step
    }
  }
}

// the advantage moments: this rank's fp64 (sum a, sum a^2) reduced from the per-block partials of returns_kernel, exchanged as four
// packets (low and high words of each), added in rank order into part[0], part[1].  One CTA.
__global__ void __launch_bounds__(256) moment_exchange_kernel(PpoPeerComm c, double* __restrict__ part, int nparts,
                                                              uint32_t* __restrict__ seq_dev, uint32_t* __restrict__ err_flag) {
  __shared__ double sh[2][8];
  __shared__ double s_mom[16][2];
  __shared__ int s_bad;
  double s1 = 0.0, s2 = 0.0;
  for (int k = threadIdx.x; k < nparts; k += 256) { s1 += part[2 * k]; s2 += part[2 * k + 1]; }
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s1; sh[1][threadIdx.x >> 5] = s2; }
  if (threadIdx.x == 0) s_bad = *reinterpret_cast<volatile uint32_t*>(err_flag) != 0;
  __syncthreads();
  const uint32_t seq = seq_dev[0] + 1u;
  const int64_t ecap = c.cap / (2 * c.world);
  const int64_t par = (int64_t)(seq & 1u) * c.world;
  double a = 0.0, b = 0.0;
  for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
  const int p = threadIdx.x;                  // thread p trades packets with rank p
  if (p < c.world) {
    const uint64_t ua = (uint64_t)__double_as_longlong(a), ub = (uint64_t)__double_as_longlong(b);
    const float words[4] = {__uint_as_float((uint32_t)ua), __uint_as_float((uint32_t)(ua >> 32)), __uint_as_float((uint32_t)ub),
                            __uint_as_float((uint32_t)(ub >> 32))};
    float got[4] = {words[0], words[1], words[2], words[3]};
    if (p != c.rank && !s_bad) {
      for (int k = 0; k < 4; ++k) usv::st_packet(c.windows[p] + ((par + c.rank) * ecap + k) * 2, words[k], seq);
      bool ok = true;
      for (int k = 0; k < 4 && ok; ++k) ok = wait_packet(c.windows[c.rank] + ((par + p) * ecap + k) * 2, seq, got[k], err_flag);
      if (!ok) { atomicOr(err_flag, 1u); s_bad = 1; }
    }
    s_mom[p][0] = __longlong_as_double((long long)(((uint64_t)__float_as_uint(got[1]) << 32) | __float_as_uint(got[0])));
    s_mom[p][1] = __longlong_as_double((long long)(((uint64_t)__float_as_uint(got[3]) << 32) | __float_as_uint(got[2])));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = s_mom[0][0], tb = s_mom[0][1];
    for (int q = 1; q < c.world; ++q) { ta += s_mom[q][0]; tb += s_mom[q][1]; }
    part[0] = s_bad ? CUDART_NAN : ta;          // a failed exchange leaves no moments: the advantages come out zero
    part[1] = s_bad ? CUDART_NAN : tb;
    seq_dev[0] = seq;
  }
}

static int check_comm(const PpoPeerComm* c, int64_t entries, const uint32_t* seq_dev, const uint32_t* err_flag) {
  if (!c || !seq_dev || !err_flag) return USV_E_NULL;
  if (c->world < 1 || c->world > 16 || c->rank < 0 || c->rank >= c->world) return USV_E_PARAM;
  if (c->cap < (int64_t)c->world * entries * 2) return USV_E_SIZE;
  for (int r = 0; r < c->world; ++r)
    if (!c->windows[r]) return USV_E_NULL;
    else if ((uintptr_t)c->windows[r] & 7) return USV_E_ALIGN;
  return USV_OK;
}

static int check_net(const PpoLoopzNet* net) {
  if (!net) return USV_E_NULL;
  if (net->mass_dim < 1 || net->mass_dim > PPO_LOOPZ_MAX_MASS || net->obs_dim <= net->mass_dim || net->obs_dim > PPO_MAX_OBS) return USV_E_SIZE;
  if (smem_floats(net->obs_dim, net->mass_dim, true) * sizeof(float) > 227 * 1024) return USV_E_UNSUPPORTED;
  return USV_OK;
}

}  // namespace loopz

using namespace loopz;

extern "C" {

int64_t ppo_loopz_param_count(const PpoLoopzNet* net) { return check_net(net) == USV_OK ? Spans(*net).P : -1; }
int64_t ppo_loopz_actor_param_count(const PpoLoopzNet* net) { return check_net(net) == USV_OK ? Spans(*net).PA : -1; }
int64_t ppo_loopz_train_scratch_floats(const PpoLoopzNet* net) {
  return check_net(net) == USV_OK ? (int64_t)2 * kMaxParts * part_stride(Spans(*net)) : -1;
}
int64_t ppo_loopz_returns_scratch_bytes(void) { return (int64_t)2 * kRetBlocks * sizeof(double); }

int ppo_loopz_act_f32(const float* params, const PpoLoopzNet* net, const float* actor_obs, const float* critic_obs, uint64_t seed,
                      uint64_t counter, const uint64_t* counter_offset, int64_t row_offset, const float* eval_actions, float* actions,
                      float* log_prob, float* means, float* values, int64_t M, void* stream) {
  int rc = check_net(net);
  if (rc != USV_OK) return rc;
  if (M < 0) return USV_E_SIZE;
  if (M == 0) return USV_OK;
  if (!params) return USV_E_NULL;
  const bool do_actor = actions || means || eval_actions, do_critic = values != nullptr;
  if (!do_actor && !do_critic) return USV_E_NULL;
  if ((do_actor && !actor_obs) || (do_critic && !critic_obs) || (log_prob && !actions && !eval_actions) || (eval_actions && (actions || !log_prob)))
    return USV_E_NULL;
  const size_t smem = smem_floats(net->obs_dim, net->mass_dim, false) * sizeof(float);
  usv::ensure_dynamic_smem(act_kernel, smem);
  const int64_t ntiles = (M + TM - 1) / TM;
  const int nn = (do_actor ? 1 : 0) + (do_critic ? 1 : 0);
  const int sms = usv::num_sms();
  const int cap = sms / nn > 0 ? sms / nn : 1;
  const int gx = (int)(ntiles < cap ? ntiles : cap);
  act_kernel<<<dim3(gx, nn), NT, smem, (cudaStream_t)stream>>>(params, *net, do_actor ? 0 : 1, actor_obs, critic_obs, seed, counter,
                                                               counter_offset, row_offset, eval_actions, actions, log_prob, means, values, M);
  return usv::finish_launch();
}

int ppo_loopz_returns_f32(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, float gamma, float lam,
                          float* returns, float* advantages, void* scratch, int32_t T, int64_t n, void* stream) {
  if (T < 0 || n < 0) return USV_E_SIZE;
  if (T == 0 || n == 0) return USV_OK;
  if (!rewards || !values || !dones || !last_values || !returns || !advantages || !scratch) return USV_E_NULL;
  int64_t blocks = (n + 255) / 256;
  if (blocks > kRetBlocks) blocks = kRetBlocks;
  returns_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, gamma, lam, returns, advantages,
                                                                (double*)scratch, T, n);
  const int64_t total = (int64_t)T * n;
  int64_t nb = (total + 255) / 256;
  if (nb > kRetBlocks) nb = kRetBlocks;
  adv_norm_kernel<<<(int)nb, 256, 0, (cudaStream_t)stream>>>(advantages, (const double*)scratch, (int)blocks, total, total);
  return usv::finish_launch(2);
}

int64_t ppo_loopz_peer_entries(const PpoLoopzNet* net) {
  return check_net(net) == USV_OK ? (int64_t)(Spans(*net).P + PPO_LOOPZ_STAT_COUNT + 63) / 64 * 64 : -1;
}

int ppo_loopz_returns_peer_f32(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, float gamma,
                               float lam, float* returns, float* advantages, void* scratch, int32_t T, int64_t n,
                               const PpoPeerComm* comm, uint32_t* seq_dev, uint32_t* err_flag, void* stream) {
  if (T <= 0 || n <= 0) return USV_E_SIZE;     // every rank takes part in every exchange: no empty shard
  if (!rewards || !values || !dones || !last_values || !returns || !advantages || !scratch) return USV_E_NULL;
  const int rc = check_comm(comm, 4, seq_dev, err_flag);
  if (rc != USV_OK) return rc;
  int64_t blocks = (n + 255) / 256;
  if (blocks > kRetBlocks) blocks = kRetBlocks;
  cudaStream_t st = (cudaStream_t)stream;
  returns_kernel<<<(int)blocks, 256, 0, st>>>(rewards, values, dones, last_values, gamma, lam, returns, advantages, (double*)scratch, T, n);
  moment_exchange_kernel<<<1, 256, 0, st>>>(*comm, (double*)scratch, (int)blocks, seq_dev, err_flag);
  const int64_t count = (int64_t)T * n;
  int64_t nb = (count + 255) / 256;
  if (nb > kRetBlocks) nb = kRetBlocks;
  adv_norm_kernel<<<(int)nb, 256, 0, st>>>(advantages, (const double*)scratch, 1, count * comm->world, count);
  return usv::finish_launch(3);
}

int ppo_loopz_minibatch_grad_f32(const float* params, const PpoLoopzNet* net, const float* actor_obs, const float* critic_obs,
                                 const float* actions, const float* old_log_prob, const float* advantages, const float* target_values,
                                 const float* returns, const int64_t* index, const PpoLoopzLossParams* lp, float* grads, float* scratch,
                                 int64_t M, void* stream) {
  int rc = check_net(net);
  if (rc != USV_OK) return rc;
  if (M <= 0) return USV_E_SIZE;
  if (!params || !actor_obs || !critic_obs || !actions || !old_log_prob || !advantages || !target_values || !returns || !lp || !grads || !scratch)
    return USV_E_NULL;
  const size_t smem = smem_floats(net->obs_dim, net->mass_dim, true) * sizeof(float);
  usv::ensure_dynamic_smem(train_kernel, smem);
  const int64_t ntiles = (M + TM - 1) / TM;
  int gx = usv::num_sms() / 2;
  if (gx > kMaxParts) gx = kMaxParts;
  if (gx < 1) gx = 1;
  if (ntiles < gx) gx = (int)ntiles;
  LossIn in{actions, old_log_prob, advantages, target_values, returns, index};
  train_kernel<<<dim3(gx, 2), NT, smem, (cudaStream_t)stream>>>(params, *net, actor_obs, critic_obs, in, *lp, scratch, M);
  const int n = Spans(*net).P + PPO_LOOPZ_STAT_COUNT;
  reduce_kernel<<<(n + 63) / 64, 256, 0, (cudaStream_t)stream>>>(scratch, gx, *net, *lp, grads);
  return usv::finish_launch(2);
}

int ppo_loopz_grad_exchange_f32(const PpoPeerComm* comm, const PpoLoopzNet* net, float* grads, uint32_t* seq_dev, uint32_t* err_flag,
                                void* stream) {
  int rc = check_net(net);
  if (rc != USV_OK) return rc;
  if (!grads) return USV_E_NULL;
  const int P = Spans(*net).P, n = P + PPO_LOOPZ_STAT_LOG_PROB + 1;   // the gradient and the three statistic sums
  rc = check_comm(comm, ppo_loopz_peer_entries(net), seq_dev, err_flag);
  if (rc != USV_OK) return rc;
  int grid = (n + kXThreads - 1) / kXThreads;
  if (grid > usv::num_sms()) grid = usv::num_sms();
  grad_exchange_kernel<<<grid, kXThreads, 0, (cudaStream_t)stream>>>(*comm, grads, n, P, 1.0f / (float)comm->world, seq_dev, err_flag);
  return usv::finish_launch();
}

int ppo_loopz_adam_step_f32(float* params, float* grads, float* exp_avg, float* exp_avg_sq, const float* lr, int32_t* step, int32_t parity,
                            float* accum, int64_t P, int64_t M, const PpoLoopzLossParams* lp, const PpoLoopzAdamParams* ap, void* stream) {
  if (P <= 0 || M <= 0 || parity < 0 || parity > 1) return USV_E_SIZE;
  if (!params || !grads || !exp_avg || !exp_avg_sq || !lr || !step || !lp || !ap) return USV_E_NULL;
  const float inv_M = 1.0f / (float)M;
  adam_kernel<<<(int)((P + kAdamThreads - 1) / kAdamThreads), kAdamThreads, 0, (cudaStream_t)stream>>>(
      params, grads, exp_avg, exp_avg_sq, lr, step + parity, step + (1 - parity), accum, (int)P, inv_M, *lp, *ap);
  stat_mean_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(grads, (int)P, inv_M);
  return usv::finish_launch(2);
}

int ppo_loopz_enforce_min_std_f32(float* std, const float* min_std, int32_t dim, void* stream) {
  if (dim < 1 || dim > 32) return USV_E_SIZE;
  if (!std || !min_std) return USV_E_NULL;
  min_std_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(std, min_std, dim);
  return usv::finish_launch();
}

}  // extern "C"
