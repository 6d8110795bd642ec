// USV_PPOcontinuous_MLP on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a only.
//
// One CTA owns a tile of 128 samples.  The three Linear layers are tcgen05.mma.kind::tf32 instructions issued by one
// thread, with fp32 accumulators in tensor memory; the activations never leave the SM:
//
//   X[128x16] (obs, normalised, col 13 = 1 so b1 rides along as a weight column)
//     --UMMA 128x128x16-->  TMEM acc  --tcgen05.ld, tanh.approx--> H1[128x128] in smem (UMMA K-major operand layout)
//     --UMMA 128x128x128--> TMEM acc  --tcgen05.ld, +b2, tanh-->   H2[128x128] in smem
//     --UMMA 128x16x128-->  TMEM      --tcgen05.ld, +b3-->          (mu0, mu1, value)
//
// Operand tiles use the un-swizzled ("interleave") canonical layout: 8 x 16 B core matrices,
//     off(outer, inner) = (outer/8)*KC*32 + (inner/4)*32 + (outer%8)*4 + (inner%4)      [floats], KC = inner extent / 4.
// The same bytes are a K-major operand (outer = M/N index, inner = K) for the forward GEMMs and an MN-major operand
// (outer = K, inner = M/N) for the weight-gradient GEMMs of the training kernel, so the PyTorch-layout weights
// W[out][in] and the row-per-thread activations are staged exactly once.
//
// TF32 inputs (10-bit mantissa) + tanh.approx (2^-11) put this path at ~1e-3 relative of the fp32 kernels in ppo_mlp.cu,
// which remain the numerics reference (DESIGN.md section 6).
#include <cooperative_groups.h>
#include <math_constants.h>
#include <string.h>
#include "philox.cuh"
#include "usv_common.cuh"

#define PPOTC_NS ppotc16
#define PPOTC_DP 16
#include "ppo_mlp_tc_impl.inc"
#undef PPOTC_NS
#undef PPOTC_DP
#define PPOTC_NS ppotc48
#define PPOTC_DP 48
#include "ppo_mlp_tc_impl.inc"
#undef PPOTC_NS
#undef PPOTC_DP

// ---- C ABI: dispatch on the padded observation width (one column is reserved for the bias): obs_dim <= 15 -> 16, <= 47 -> 48
#define PPOTC_DISPATCH(obs_dim, call)                      \
  do {                                                     \
    if ((obs_dim) >= 1 && (obs_dim) < 16) return ppotc16::call; \
    if ((obs_dim) >= 16 && (obs_dim) < 48) return ppotc48::call; \
    return USV_E_SIZE;                                     \
  } while (0)

extern "C" int64_t ppo_packed_weight_floats(void) { return ppotc48::packed_weight_floats(); }   // the larger of the two layouts

extern "C" int ppo_pack_weights_tc(const float* params, int32_t obs_dim, float* packed, void* stream) {
  PPOTC_DISPATCH(obs_dim, host_pack_weights(params, obs_dim, packed, stream));
}

extern "C" int ppo_policy_forward_tc(const float* params, const float* packed, const float* obs, int32_t obs_dim, const float* obs_mean,
                                     const float* obs_var, const float* value_mean, const float* value_var, uint64_t seed,
                                     uint64_t counter, const uint64_t* counter_offset, int64_t row_offset, float* actions, float* neglogp,
                                     float* values, float* mus, float* sigmas, int64_t M, void* stream) {
  PPOTC_DISPATCH(obs_dim, host_policy_forward(params, packed, obs, obs_dim, obs_mean, obs_var, value_mean, value_var, seed, counter,
                                              counter_offset, row_offset, actions, neglogp, values, mus, sigmas, M, stream));
}

extern "C" int64_t ppo_train_tc_workspace_floats(int64_t M) { return ppotc48::train_workspace_floats(M); }

extern "C" int ppo_minibatch_grad_tc(const float* params, const float* packed, const float* obs, int32_t obs_dim, const float* obs_mean,
                                     const float* obs_var, const float* actions, const float* old_neglogp, const float* advantages,
                                     const float* old_values, const float* returns, float* old_mu, float* old_sigma,
                                     const PpoLossParams* lp, float* grads, float* scratch, float* workspace, int64_t M, void* stream) {
  PPOTC_DISPATCH(obs_dim, host_minibatch_grad(params, packed, obs, obs_dim, obs_mean, obs_var, actions, old_neglogp, advantages, old_values,
                                              returns, old_mu, old_sigma, lp, grads, scratch, workspace, M, stream));
}

extern "C" int ppo_minibatch_step_tc(float* params, float* packed, const float* obs, int32_t obs_dim, const float* obs_mean,
                                     const float* obs_var, const float* actions, const float* old_neglogp, const float* advantages,
                                     const float* old_values, const float* returns, float* old_mu, float* old_sigma,
                                     const PpoLossParams* lp, float* grads, float* scratch, float* workspace, float* exp_avg,
                                     float* exp_avg_sq, float* lr, int32_t* step, const PpoAdamParams* ap, int64_t M, void* stream) {
  PPOTC_DISPATCH(obs_dim, host_minibatch_step(params, packed, obs, obs_dim, obs_mean, obs_var, actions, old_neglogp, advantages, old_values,
                                              returns, old_mu, old_sigma, lp, grads, scratch, workspace, exp_avg, exp_avg_sq, lr, step, ap,
                                              nullptr, nullptr, nullptr, M, stream));
}

extern "C" int64_t ppo_minibatch_step_peer_entries(int32_t obs_dim) {
  if (obs_dim >= 1 && obs_dim < 16) return ppotc16::tail_entries(obs_dim);
  if (obs_dim >= 16 && obs_dim < 48) return ppotc48::tail_entries(obs_dim);
  return -1;
}

extern "C" int ppo_minibatch_step_peer_tc(float* params, float* packed, const float* obs, int32_t obs_dim, const float* obs_mean,
                                          const float* obs_var, const float* actions, const float* old_neglogp, const float* advantages,
                                          const float* old_values, const float* returns, float* old_mu, float* old_sigma,
                                          const PpoLossParams* lp, float* grads, float* scratch, float* workspace, float* exp_avg,
                                          float* exp_avg_sq, float* lr, int32_t* step, const PpoAdamParams* ap, const PpoPeerComm* comm,
                                          uint32_t* seq_dev, uint32_t* err_flag, int64_t M, void* stream) {
  if (!comm) return USV_E_NULL;
  PPOTC_DISPATCH(obs_dim, host_minibatch_step(params, packed, obs, obs_dim, obs_mean, obs_var, actions, old_neglogp, advantages, old_values,
                                              returns, old_mu, old_sigma, lp, grads, scratch, workspace, exp_avg, exp_avg_sq, lr, step, ap,
                                              comm, seq_dev, err_flag, M, stream));
}
