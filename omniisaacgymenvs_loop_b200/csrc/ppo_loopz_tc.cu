// The loopz PPO minibatch gradient with the two 128-wide layers of each MLPEncode network on the 5th-generation tensor cores.
//
// The trunk of a loopz network -- Linear(IN,128)+LeakyReLU -> Linear(128,128)+LeakyReLU -> Linear(128,OUT) -- has exactly the GEMM
// shapes of the rl_games policy, so it runs on the same two kernels (ppo_mlp_tc_impl.inc compiled with PPOTC_LOOPZ: LeakyReLU
// epilogues, raw inputs, the loopz losses): T1 = forward + per-sample loss + backprop to dz1 (tcgen05.mma kind::tf32, accumulators
// in TMEM), T2 = weight gradients with K = samples.  What the trunk does not cover stays fp32 SIMT and is small:
//   enc_fwd_kernel : mass tail -> Linear(Md,64) -> Linear(64,16) -> Linear(16,8) (LeakyReLU) -> main-input rows [speed | task | latent]
//   enc_bwd_kernel : d latent = dz1 . W1[:, latent columns] (from T1's feature-major dz1 slab) -> encoder backward + weight gradients
//   reduce_kernel  : trunk gradients (T2 slots) + head biases / std / statistics (T1 slots) + encoder gradients -> the flat gradient
// Per network the launches are sequential (one slab workspace serves both).  TF32 operands put this path at ~1e-3 relative of
// ppo_loopz.cu, which stays the numerics reference.   [ref: OIGE/algo/ppo/module.py:184-361 ; ppo.py:232-284]
#include <math_constants.h>
#include "philox.cuh"
#include "usv_common.cuh"

#define PPOTC_NS loopztc
#define PPOTC_DP 48
#define PPOTC_LOOPZ 1
#include "ppo_mlp_tc_impl.inc"
#undef PPOTC_NS
#undef PPOTC_DP

namespace loopztc {

constexpr int E1 = PPO_LOOPZ_ENC1, E2 = PPO_LOOPZ_ENC2, E3 = PPO_LOOPZ_LATENT;
constexpr int ETM = 64, ENT = 256, E1S = E1 + 1, E2S = E2 + 1, MS = PPO_LOOPZ_MAX_MASS + 1;
constexpr float kSlope = 0.01f;
constexpr int kEncSlots = 320;          // partial-gradient slots of the encoder backward kernel (>= its grid)
__device__ __forceinline__ float lrelu(float x) { return x > 0.f ? x : kSlope * x; }
__device__ __forceinline__ float lrelu_grad(float y) { return y > 0.f ? 1.0f : kSlope; }

__host__ __device__ inline int enc_floats(int md) { return E1 * md + E1 + E2 * E1 + E2 + E3 * E2 + E3; }
__host__ __device__ inline int packed_dims(int in, int md, int out) { return in | (md << 8) | (out << 16); }
struct Spans {   // flat vector: actor | std[2] | critic  (ppo_loopz.cu)
  int IN, PA, PC, std, critic, P;
  __host__ __device__ explicit Spans(const PpoLoopzNet& n) {
    IN = n.obs_dim - n.mass_dim + E3;
    PA = Layout(packed_dims(IN, n.mass_dim, 2)).P; PC = Layout(packed_dims(IN, n.mass_dim, 1)).P;
    std = PA; critic = PA + 2; P = PA + 2 + PC;
  }
};

struct EncSmem {
  float *we1t, *be1, *we2t, *be2, *we3t, *be3, *ms, *e1, *e2, *lat;
};
__device__ inline float* carve_enc(float* p, int md, EncSmem& s) {
  s.we2t = p; p += E1 * E2;    // 16 B aligned first
  s.be2 = p; p += E2;
  s.we1t = p; p += md * E1;
  s.be1 = p; p += E1;
  s.we3t = p; p += E2 * E3;
  s.be3 = p; p += E3;
  s.ms = p; p += ETM * MS;
  s.e1 = p; p += ETM * E1S;
  s.e2 = p; p += ETM * E2S;
  s.lat = p; p += ETM * MS;
  return p;
}
__host__ __device__ inline int enc_smem_floats(int md) { return E1 * E2 + E2 + md * E1 + E1 + E2 * E3 + E3 + 2 * ETM * MS + ETM * E1S + ETM * E2S; }

__device__ inline void load_enc_weights(const EncSmem& s, const float* __restrict__ prm, int md) {
  const int t = threadIdx.x;
  const int e1w = 0, e1b = E1 * md, e2w = e1b + E1, e2b = e2w + E2 * E1, e3w = e2b + E2, e3b = e3w + E3 * E2;
  for (int e = t; e < E1 * md; e += ENT) { const int o = e / md, k = e - o * md; s.we1t[k * E1 + o] = prm[e1w + e]; }
  for (int e = t; e < E2 * E1; e += ENT) { const int o = e / E1, k = e - o * E1; s.we2t[k * E2 + o] = prm[e2w + e]; }
  for (int e = t; e < E3 * E2; e += ENT) { const int o = e / E2, k = e - o * E2; s.we3t[k * E3 + o] = prm[e3w + e]; }
  for (int e = t; e < E1; e += ENT) s.be1[e] = prm[e1b + e];
  if (t < E2) s.be2[t] = prm[e2b + t];
  if (t < E3) s.be3[t] = prm[e3b + t];
}

// mass tail of a 64-row tile -> ms, e1, e2, lat (post-activation)   [ref module.py:340-355]
__device__ inline void encoder_forward(const EncSmem& s, const float* __restrict__ obs, int D, int md, int64_t row0, int64_t M) {
  const int t = threadIdx.x, m0 = D - md;
  for (int e = t; e < ETM * md; e += ENT) {
    const int r = e / md, k = e - r * md;
    float x = 0.f;
    if (row0 + r < M) { x = obs[(row0 + r) * D + m0 + k]; if (!isfinite(x)) x = 0.f; }
    s.ms[r * MS + k] = x;
  }
  __syncthreads();
  for (int e = t; e < ETM * E1; e += ENT) {
    const int r = e / E1, o = e - r * E1;
    float acc = s.be1[o];
    for (int k = 0; k < md; ++k) acc = fmaf(s.ms[r * MS + k], s.we1t[k * E1 + o], acc);
    s.e1[r * E1S + o] = lrelu(acc);
  }
  __syncthreads();
  {
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
  for (int e = t; e < ETM * E3; e += ENT) {
    const int r = e / E3, o = e - r * E3;
    float acc = s.be3[o];
#pragma unroll
    for (int k = 0; k < E2; ++k) acc = fmaf(s.e2[r * E2S + k], s.we3t[k * E3 + o], acc);
    s.lat[r * MS + o] = lrelu(acc);
  }
  __syncthreads();
}

// zin[net][row][IN] = [obs[:, :D-Md] | latent]
__global__ void __launch_bounds__(ENT) enc_fwd_kernel(const float* __restrict__ prm, PpoLoopzNet cfg, const float* __restrict__ obs_actor,
                                                     const float* __restrict__ obs_critic, float* __restrict__ zin, int64_t M) {
  extern __shared__ __align__(1024) float smem[];
  const int net = blockIdx.y, D = cfg.obs_dim, md = cfg.mass_dim, m0 = D - md, IN = m0 + E3;
  const Spans sp(cfg);
  EncSmem s;
  carve_enc(smem, md, s);
  const float* obs = net == 0 ? obs_actor : obs_critic;
  load_enc_weights(s, prm + (net == 0 ? 0 : sp.critic), md);
  float* z = zin + (size_t)net * M * IN;
  const int64_t ntiles = (M + ETM - 1) / ETM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * ETM;
    __syncthreads();
    encoder_forward(s, obs, D, md, row0, M);
    for (int e = threadIdx.x; e < ETM * IN; e += ENT) {
      const int r = e / IN, d = e - r * IN;
      if (row0 + r < M) {
        float x;
        if (d < m0) { x = obs[(row0 + r) * D + d]; if (!isfinite(x)) x = 0.f; }
        else x = s.lat[r * MS + d - m0];
        z[(row0 + r) * IN + d] = x;
      }
    }
  }
}

// encoder backward of one network: per-CTA partial gradients [enc_floats]
__global__ void __launch_bounds__(ENT) enc_bwd_kernel(const float* __restrict__ prm_net, PpoLoopzNet cfg, const float* __restrict__ obs,
                                                     const float* __restrict__ dz1t, int64_t ld, float* __restrict__ partial, int64_t M) {
  extern __shared__ __align__(1024) float smem[];
  const int D = cfg.obs_dim, md = cfg.mass_dim, m0 = D - md, IN = m0 + E3, t = threadIdx.x;
  EncSmem s;
  float* p = carve_enc(smem, md, s);
  float* dz = p; p += 4 * ETM * MS;       // partial sums of d latent over the four feature quarters
  float* w1l = p; p += E3 * H;            // W1[:, latent columns], [8][128]
  float* dlat = p; p += ETM * MS;
  float* gwe1 = p; p += md * E1;
  float* gbe1 = p; p += E1;
  float* gwe2 = p; p += E1 * E2;
  float* gbe2 = p; p += E2;
  float* gwe3 = p; p += E2 * E3;
  float* gbe3 = p; p += E3;
  load_enc_weights(s, prm_net, md);
  const int w1 = enc_floats(md);
  for (int e = t; e < E3 * H; e += ENT) { const int j = e / H, o = e - j * H; w1l[e] = prm_net[w1 + o * IN + m0 + j]; }
  for (int e = t; e < enc_floats(md); e += ENT) gwe1[e] = 0.f;     // gwe1 .. gbe3 are contiguous
  const int64_t ntiles = (M + ETM - 1) / ETM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * ETM;
    __syncthreads();
    encoder_forward(s, obs, D, md, row0, M);     // ends with __syncthreads()
    // d latent straight from the feature-major dz1 slab (ld is padded to 128, rows beyond M are zero): thread = (sample r, quarter q
    // of the 128 features); a warp reads 32 consecutive samples of one feature = one 128 B line (L2 hits: T1 has just written it)
    {
      const int r = t & (ETM - 1), q = t >> 6;
      float acc[E3];
#pragma unroll
      for (int j = 0; j < E3; ++j) acc[j] = 0.f;
      const float* g = dz1t + (int64_t)(q * 32) * ld + row0 + r;
#pragma unroll 4
      for (int o = 0; o < 32; ++o) {
        const float d = g[(int64_t)o * ld];
#pragma unroll
        for (int j = 0; j < E3; ++j) acc[j] = fmaf(d, w1l[j * H + q * 32 + o], acc[j]);
      }
#pragma unroll
      for (int j = 0; j < E3; ++j) dz[(q * ETM + r) * MS + j] = acc[j];     // partial sums [4][64][8] in the (otherwise unused) dz area
    }
    __syncthreads();
    for (int e = t; e < ETM * E3; e += ENT) {
      const int r = e / E3, j = e - r * E3;
      const float v = (dz[(0 * ETM + r) * MS + j] + dz[(1 * ETM + r) * MS + j]) + (dz[(2 * ETM + r) * MS + j] + dz[(3 * ETM + r) * MS + j]);
      dlat[r * MS + j] = (row0 + r < M) ? v * lrelu_grad(s.lat[r * MS + j]) : 0.f;
    }
    __syncthreads();
    if (t < E3 * E2) {
      const int o = t / E2, k = t - o * E2;
      float acc = 0.f;
      for (int r = 0; r < ETM; ++r) acc = fmaf(dlat[r * MS + o], s.e2[r * E2S + k], acc);
      gwe3[t] += acc;
    } else if (t < E3 * E2 + E3) {
      const int o = t - E3 * E2;
      float acc = 0.f;
      for (int r = 0; r < ETM; ++r) acc += dlat[r * MS + o];
      gbe3[o] += acc;
    }
    __syncthreads();
    for (int e = t; e < ETM * E2; e += ENT) {
      const int r = e / E2, k = e - r * E2;
      float acc = 0.f;
#pragma unroll
      for (int o = 0; o < E3; ++o) acc = fmaf(dlat[r * MS + o], s.we3t[k * E3 + o], acc);
      s.e2[r * E2S + k] = acc * lrelu_grad(s.e2[r * E2S + k]);
    }
    __syncthreads();
    {
      const int k = t & (E1 - 1), og = (t >> 6) * 4;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int r = 0; r < ETM; ++r) {
        const float x = s.e1[r * E1S + k];
        const float* d = s.e2 + r * E2S + og;
        a0 = fmaf(d[0], x, a0); a1 = fmaf(d[1], x, a1); a2 = fmaf(d[2], x, a2); a3 = fmaf(d[3], x, a3);
      }
      gwe2[(og + 0) * E1 + k] += a0; gwe2[(og + 1) * E1 + k] += a1; gwe2[(og + 2) * E1 + k] += a2; gwe2[(og + 3) * E1 + k] += a3;
    }
    if (t < E2) {
      float acc = 0.f;
      for (int r = 0; r < ETM; ++r) acc += s.e2[r * E2S + t];
      gbe2[t] += acc;
    }
    __syncthreads();
    {
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
    for (int e = t; e < E1 * md; e += ENT) {
      const int k = e / E1, o = e - k * E1;
      float acc = 0.f;
#pragma unroll 8
      for (int r = 0; r < ETM; ++r) acc = fmaf(s.e1[r * E1S + o], s.ms[r * MS + k], acc);
      gwe1[o * md + k] += acc;
    }
    if (t < E1) {
      float acc = 0.f;
      for (int r = 0; r < ETM; ++r) acc += s.e1[r * E1S + t];
      gbe1[t] += acc;
    }
  }
  __syncthreads();
  // partial record in the parameter order of the encoder: e1w | e1b | e2w | e2b | e3w | e3b
  float* out = partial + (size_t)blockIdx.x * enc_floats(md);
  const int e1b = E1 * md, e2w = e1b + E1, e2b = e2w + E2 * E1, e3w = e2b + E2, e3b = e3w + E3 * E2;
  for (int e = t; e < E1 * md; e += ENT) out[e] = gwe1[e];
  if (t < E1) out[e1b + t] = gbe1[t];
  for (int e = t; e < E2 * E1; e += ENT) out[e2w + e] = gwe2[e];
  if (t < E2) out[e2b + t] = gbe2[t];
  if (t < E3 * E2) out[e3w + t] = gwe3[t];
  if (t < E3) out[e3b + t] = gbe3[t];
}

struct RedIn {
  const float* t1[2];    // [g1][16]
  const float* t2[2];    // [g2][P_net]
  const float* enc[2];   // [g3][enc_floats]
  int g1[2], g2[2], g3[2];
};
// flat gradient + statistics (sums) in the layout ppo_loopz_adam_step_f32 expects.  64 entries x 4 slot groups per block (four short
// dependent load chains instead of one long one), fixed order: deterministic
__global__ void __launch_bounds__(256) reduce_kernel(RedIn in, PpoLoopzNet cfg, float* __restrict__ grads) {
  __shared__ float sm[4][64];
  const Spans sp(cfg);
  const int col = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int e = blockIdx.x * 64 + col;
  const int n = sp.P + PPO_LOOPZ_STAT_COUNT;
  const int encn = enc_floats(cfg.mass_dim);
  // source of entry e: base pointer, slot count, slot stride, column
  const float* src = nullptr;
  int cnt = 0, stride = 0, c0 = 0;
  if (e < n) {
    if (e >= sp.P) {
      const int k = e - sp.P;
      if (k == PPO_LOOPZ_STAT_SURROGATE) { src = in.t1[0]; cnt = in.g1[0]; stride = 16; c0 = 0; }
      else if (k == PPO_LOOPZ_STAT_LOG_PROB) { src = in.t1[0]; cnt = in.g1[0]; stride = 16; c0 = 1; }
      else if (k == PPO_LOOPZ_STAT_VALUE_LOSS) { src = in.t1[1]; cnt = in.g1[1]; stride = 16; c0 = 0; }
    } else if (e >= sp.std && e < sp.std + 2) {
      src = in.t1[0]; cnt = in.g1[0]; stride = 16; c0 = 5 + (e - sp.std);
    } else {
      const int net = e < sp.std ? 0 : 1;
      const int loc = e - (net == 0 ? 0 : sp.critic);
      const Layout L(packed_dims(sp.IN, cfg.mass_dim, net == 0 ? 2 : 1));
      if (loc < encn) { src = in.enc[net]; cnt = in.g3[net]; stride = encn; c0 = loc; }
      else if (loc >= L.b3) { src = in.t1[net]; cnt = in.g1[net]; stride = 16; c0 = 7 + (loc - L.b3); }
      else { src = in.t2[net]; cnt = in.g2[net]; stride = slot_stride(L); c0 = slot_pad(L) + loc; }
    }
  }
  float acc = 0.f;
  for (int c = grp; c < cnt; c += 4) acc += src[(size_t)c * stride + c0];
  sm[grp][col] = acc;
  __syncthreads();
  if (grp == 0 && e < n) grads[e] = (sm[0][col] + sm[1][col]) + (sm[2][col] + sm[3][col]);
}

}  // namespace loopztc

using namespace loopztc;

extern "C" {

int64_t ppo_loopz_tc_workspace_floats(const PpoLoopzNet* net, int64_t M) {
  if (!net || M <= 0 || net->mass_dim < 1 || net->mass_dim > PPO_LOOPZ_MAX_MASS || net->obs_dim <= net->mass_dim) return -1;
  const Spans sp(*net);
  if (sp.IN >= DP) return -1;
  const int64_t ld = (M + 127) / 128 * 128;
  const int64_t slabs = (4 * (int64_t)H + DP + 16) * ld;
  const int64_t zin = 2 * M * sp.IN + 8;
  const int64_t packed = 2 * (int64_t)PK_TOTAL;
  const int64_t slots = 2 * (160 * 16 + (int64_t)kWgradCtas * slot_stride(Layout(packed_dims(sp.IN, net->mass_dim, 2))) +
                             kEncSlots * (int64_t)enc_floats(net->mass_dim));
  return slabs + zin + packed + slots + 64;
}

int ppo_loopz_minibatch_grad_tc(const float* params, const PpoLoopzNet* net, const float* actor_obs, const float* critic_obs,
                                const float* actions, const float* old_log_prob, const float* advantages, const float* target_values,
                                const float* returns, const PpoLoopzLossParams* lp, float* grads, float* workspace, int64_t M, void* stream) {
  if (!net) return USV_E_NULL;
  if (M <= 0 || net->mass_dim < 1 || net->mass_dim > PPO_LOOPZ_MAX_MASS || net->obs_dim <= net->mass_dim) return USV_E_SIZE;
  if (!params || !actor_obs || !critic_obs || !actions || !old_log_prob || !advantages || !target_values || !returns || !lp || !grads || !workspace)
    return USV_E_NULL;
  if ((uintptr_t)workspace & 15) return USV_E_ALIGN;
  const Spans sp(*net);
  if (sp.IN >= DP) return USV_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int md = net->mass_dim, encn = enc_floats(md);
  // workspace carve-up (every piece a multiple of 4 floats): the T1 / T2 slabs first, whole 128-sample T1 tiles
  const TrainSetup t = train_setup(workspace, M, TM);
  const TrainWs& ws = t.ws;
  const int64_t ld = ws.ld;
  float* p = ws.dz3t + 16 * ld;
  float* zin = p; p += (2 * M * sp.IN + 7) / 8 * 8;
  float* pk[2]; pk[0] = p; p += PK_TOTAL; pk[1] = p; p += PK_TOTAL;
  float* t1s[2]; float* t2s[2]; float* encs[2];
  for (int k = 0; k < 2; ++k) { t1s[k] = p; p += 160 * 16; }
  for (int k = 0; k < 2; ++k) { t2s[k] = p; p += (size_t)kWgradCtas * slot_stride(Layout(packed_dims(sp.IN, md, 2))); }
  for (int k = 0; k < 2; ++k) { encs[k] = p; p += (size_t)kEncSlots * encn; }
  const int sms = usv::num_sms();
  const int64_t etiles = (M + ETM - 1) / ETM;
  int g3 = (int)(etiles < 2 * sms ? etiles : 2 * sms);       // 55 KB of shared memory: two or more CTAs per SM
  if (g3 > kEncSlots) g3 = kEncSlots;
  const size_t smem_ef = (size_t)enc_smem_floats(md) * sizeof(float);
  const size_t smem_eb = (size_t)(enc_smem_floats(md) + 4 * ETM * MS + E3 * H + ETM * MS + encn) * sizeof(float);
  usv::ensure_dynamic_smem(enc_fwd_kernel, smem_ef);
  usv::ensure_dynamic_smem(enc_bwd_kernel, smem_eb);
  cudaMemsetAsync(ws.dz3t, 0, sizeof(float) * 16 * ld, st);               // rows >= 2 of dz3^T are structurally zero
  const int gef = (int)(etiles < 2 * sms ? etiles : 2 * sms);   // x 2 networks: four CTAs per SM (33 KB of shared memory each)
  enc_fwd_kernel<<<dim3(gef, 2), ENT, smem_ef, st>>>(params, *net, actor_obs, critic_obs, zin, M);
  LossInTc in{actions, old_log_prob, advantages, target_values, returns, nullptr, nullptr};
  for (int k = 0; k < 2; ++k) {
    const float* prm_net = params + (k == 0 ? 0 : sp.critic);
    const int dims = packed_dims(sp.IN, md, k == 0 ? 2 : 1);
    pack_weights_kernel<<<(PK_TOTAL + 255) / 256, 256, 0, st>>>(prm_net, dims, pk[k]);
    train_fwd_bwd_tc_kernel<<<t.g1, NT, train_smem_bytes(), st>>>(prm_net, pk[k], zin + (size_t)k * M * sp.IN, dims, params + sp.std, k, *net, in,
                                                                *lp, ws, t1s[k], M);
    wgrad_tc_kernel<<<t.g2, NT, wgrad_smem_bytes(), st>>>(ws, dims, t2s[k], 0, t.nchunks);
    enc_bwd_kernel<<<g3, ENT, smem_eb, st>>>(prm_net, *net, k == 0 ? actor_obs : critic_obs, ws.dz1t, ld, encs[k], M);
  }
  RedIn ri;
  for (int k = 0; k < 2; ++k) { ri.t1[k] = t1s[k]; ri.t2[k] = t2s[k]; ri.enc[k] = encs[k]; ri.g1[k] = t.g1; ri.g2[k] = t.g2; ri.g3[k] = g3; }
  const int n = sp.P + PPO_LOOPZ_STAT_COUNT;
  reduce_kernel<<<(n + 63) / 64, 256, 0, st>>>(ri, *net, grads);
  return usv::finish_launch(10);
}

}  // extern "C"
