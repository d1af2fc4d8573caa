// K4c: the PPO loss starting from a diagonal-Gaussian actor head (continuous actions; see include/srl_b200.h).
//
// The head's log-prob and entropy are those of torch.distributions.Normal(mean, exp(log_std)), summed over the D action
// dimensions -- what a PyTorch Gaussian policy computes.  No line of the reference pins a Gaussian head: its policies are
// categorical (K4b), so the definition here is torch's:
//   logp = sum_d [ -(a_d - mu_d)^2 / (2 sigma_d^2) - log sigma_d - log sqrt(2 pi) ]
//   H    = sum_d [ 0.5 + 0.5 log(2 pi) + log sigma_d ]
// and the per-transition loss is K4's element<RuntimeCfg>, unchanged.  The backward of the head follows from the loss's
// d loss / d logp (g_lp) and d loss / d H (g_en):
//   d loss / d mu_d      = g_lp (a_d - mu_d) / sigma_d^2
//   d loss / d log_std_d = g_lp ((a_d - mu_d)^2 / sigma_d^2 - 1) + g_en
// `log_std` is either per transition ([T*n, D], the output of a network head) or one [D] parameter shared by every
// transition (the usual PPO Gaussian policy); its gradient is then the sum of the second line over the minibatch.
//
// The kernel, its launch and host setup are ppo_loss_head.cuh's, with mean as P0 and log_std as P1; this file has the
// Gaussian's math (GaussianHead) and the entries.  One difference between the element types: the float row pass leaves
// 1 / sigma^2 in the staged log_std slot for the column pass; a bfloat16 slot would round it, so there the column pass
// recomputes expf(-2 s) from the staged s -- the same expression on the same float.
#include "ppo_loss_head.cuh"

namespace srl {
namespace loss {
namespace {

constexpr double kLogSqrt2Pi = 0.918938533204672742;  // log(sqrt(2 pi))

struct GaussianHead {
  static constexpr bool kShared = true;
  static constexpr const char* kNames[4] = {"mean", "log_std", "g_mean", "g_log_std"};

  // the two sums in float64, rounded once: the loss sees logp through exp(logp - old_logp), and a float32 sum of
  // D = 64 terms of a |logp| ~ 100 is off by ~1e-5 -- the ratio's whole error budget
  struct Row {
    double sq, ssum;
  };
  static __device__ __forceinline__ Row row_begin(double ls_sum) { return Row{0.0, ls_sum}; }

  // s_iv: a shared log_std's 1 / sigma_d^2
  template <bool SHARED, typename T>
  static __device__ __forceinline__ void row_term(Row& r, const float* sac, const T* smu, T* sls, int i,
                                                  const double* s_iv, int d) {
    const double diff = static_cast<double>(sac[i]) - static_cast<double>(to_float(smu[i]));  // exact
    double iv;
    if (SHARED) {
      iv = s_iv[d];
    } else {
      const float s = to_float(sls[i]);
      const float ivf = expf(-2.f * s);
      r.ssum += static_cast<double>(s);
      if constexpr (std::is_same<T, float>::value) sls[i] = ivf;  // the column pass needs 1 / sigma^2, not log sigma
      iv = static_cast<double>(ivf);
    }
    r.sq = fma(diff * diff, iv, r.sq);
  }

  static __device__ __forceinline__ void row_end(const Row& r, int D, float& logp, float& ent) {
    logp = static_cast<float>(-0.5 * r.sq - r.ssum - D * kLogSqrt2Pi);
    ent = static_cast<float>(D * (0.5 + kLogSqrt2Pi) + r.ssum);
  }

  // d loss / d mean in place of the mean, d loss / d log_std in place of 1 / sigma^2 (per row; a bfloat16 slot still
  // holds log sigma, whose 1 / sigma^2 is the row pass's expression again); a shared log_std's terms go to g_acc
  template <bool SHARED, typename T>
  static __device__ __forceinline__ void column(const float* sac, T* smu, T* sls, int idx, float gl, float ge, float iv_c,
                                                double iv_cd, double& g_acc) {
    const float a = sac[idx], mu = to_float(smu[idx]);
    const float diff = a - mu;
    float iv = iv_c;
    if constexpr (std::is_same<T, float>::value) {
      if (!SHARED) iv = sls[idx];
    } else {
      if (!SHARED) iv = expf(-2.f * to_float(sls[idx]));
    }
    const float z = diff * iv;
    smu[idx] = from_float<T>(gl * z);
    if (SHARED) {
      // formed in float64 too: (a - mu)^2 / sigma^2 - 1 cancels near sigma, and T * n of these terms are summed
      const double dd = static_cast<double>(a) - static_cast<double>(mu);
      g_acc += fma(static_cast<double>(gl), fma(dd * dd, iv_cd, -1.0), static_cast<double>(ge));
    } else {
      sls[idx] = from_float<T>(fmaf(gl, fmaf(diff, z, -1.f), ge));
    }
  }
};

}  // namespace
}  // namespace loss
}  // namespace srl

extern "C" size_t srl_ppo_loss_gaussian_workspace_bytes(int T, int n, int D, int log_std_shared) {
  return srl::loss::head_workspace_bytes(T, n, D, log_std_shared != 0);
}

extern "C" int srl_ppo_loss_from_gaussian(const float* mean, const float* log_std, int log_std_shared, const float* action,
                                          int D, const float* v_pred, const float* old_logp, const float* old_value,
                                          const float* ret, const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                          const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                          const double* local_stats, const double* popart_mean_std,
                                          const srl_ppo_hyper* hyper, float* g_mean, float* g_log_std, float* g_value,
                                          float* logp_out, float* entropy_out, double* out, float* out_f32, void* workspace,
                                          size_t workspace_bytes, srl_stream_t stream) {
  return srl::loss::ppo_loss_from_head<srl::loss::GaussianHead>(
      "srl_ppo_loss_from_gaussian", sizeof(float), mean, log_std, log_std_shared != 0, action, D, v_pred, old_logp,
      old_value, ret, adv, on_reset_next, ld_smp, nullptr, 0, lane_idx, T, n, norm_stats, local_stats, popart_mean_std,
      hyper, g_mean, g_log_std, g_value, logp_out, entropy_out, out, out_f32, workspace, workspace_bytes,
      static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_gaussian_bf16(const uint16_t* mean, const void* log_std, int log_std_shared,
                                               const float* action, int D, const uint16_t* v_pred, const float* old_logp,
                                               const float* old_value, const float* ret, const float* adv,
                                               const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx,
                                               int T, int n, const double* norm_stats, const double* local_stats,
                                               const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                               uint16_t* g_mean, void* g_log_std, uint16_t* g_value, float* logp_out,
                                               float* entropy_out, double* out, float* out_f32, void* workspace,
                                               size_t workspace_bytes, srl_stream_t stream) {
  return srl::loss::ppo_loss_from_head<srl::loss::GaussianHead>(
      "srl_ppo_loss_from_gaussian_bf16", sizeof(__nv_bfloat16), mean, log_std, log_std_shared != 0, action, D, v_pred,
      old_logp, old_value, ret, adv, on_reset_next, ld_smp, nullptr, 0, lane_idx, T, n, norm_stats, local_stats,
      popart_mean_std, hyper, g_mean, g_log_std, g_value, logp_out, entropy_out, out, out_f32, workspace,
      workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_gaussian_pack(const void* mean, const void* log_std, int log_std_shared, const float* action,
                                               int D, int elem_bytes, const void* v_pred, const float* pack,
                                               int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
                                               const double* norm_stats, const double* local_stats,
                                               const double* popart_mean_std, const srl_ppo_hyper* hyper, void* g_mean,
                                               void* g_log_std, void* g_value, float* logp_out, float* entropy_out,
                                               double* out, float* out_f32, void* workspace, size_t workspace_bytes,
                                               srl_stream_t stream) {
  constexpr const char* fn = "srl_ppo_loss_from_gaussian_pack";
  const int rc = srl::loss::check_head_pack(fn, elem_bytes, pack, pack_row_lo, lane_idx, pack_lanes, n);
  if (rc != SRL_OK) return rc;
  return srl::loss::ppo_loss_from_head<srl::loss::GaussianHead>(
      fn, static_cast<size_t>(elem_bytes), mean, log_std, log_std_shared != 0, action, D, v_pred, nullptr, nullptr,
      nullptr, nullptr, nullptr, pack_lanes, pack, pack_row_lo, lane_idx, T, n, norm_stats, local_stats,
      popart_mean_std, hyper, g_mean, g_log_std, g_value, logp_out, entropy_out, out, out_f32, workspace,
      workspace_bytes, static_cast<cudaStream_t>(stream));
}
