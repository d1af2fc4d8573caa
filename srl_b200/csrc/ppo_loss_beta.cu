// K4d: the PPO loss starting from a Beta actor head (actions bounded to an interval; see include/srl_b200.h).
//
// The head's log-prob and entropy are those of torch.distributions.Beta(c1, c0) (c1 = concentration1 = alpha,
// c0 = concentration0 = beta), summed over the D action dimensions, with the action x in (0, 1) -- what a PyTorch Beta
// policy computes (Chou et al., 2017).  No line of the reference pins a Beta head, so the definition is torch's:
//   logp = sum_d [ (c1 - 1) log x + (c0 - 1) log(1 - x) + lgamma(c1 + c0) - lgamma(c1) - lgamma(c0) ]
//   H    = sum_d [ lgamma(c1) + lgamma(c0) - lgamma(c1 + c0) - (c1 - 1) psi(c1) - (c0 - 1) psi(c0)
//                  + (c1 + c0 - 2) psi(c1 + c0) ]
// and the per-transition loss is K4's element<RuntimeCfg>, unchanged.  With (g_lp, g_en) = d loss / d (logp, H):
//   d loss / d c1 = g_lp (log x - psi(c1) + psi(c1 + c0)) + g_en ((c1 + c0 - 2) psi'(c1 + c0) - (c1 - 1) psi'(c1))
//   d loss / d c0 = the same with c0 and log(1 - x)
// The kernel, its launch and host setup are ppo_loss_head.cuh's, with concentration1 as P0 and concentration0 as P1;
// this file has the Beta's math (BetaHead) and the entries.
//
// Precision: for concentrations of 10 and more, lgamma(c1 + c0) - lgamma(c1) - lgamma(c0) cancels (at c1 + c0 = 200 one
// float32 ulp of lgamma(200) ~ 857 is 6e-5), so every per-dimension term and the sums over d are float64, and logp and
// H are rounded to float once, before element().  The column pass forms the gradients in float64 from the staged
// (float) c1, c0 and x again -- psi and psi' of c1, c0 and c1 + c0 -- and rounds each once: nothing is left in the
// staged slots, which a bfloat16 launch could not hold in any case.  CUDA has lgamma but no psi / psi': digamma_trigamma
// below takes the recurrence up to x >= 6, then the asymptotic series (truncation error below 2e-11 there).
#include "ppo_loss_head.cuh"

namespace srl {
namespace loss {
namespace {

// psi(x) and psi'(x) for x > 0, in float64: psi(x) = psi(x + 1) - 1 / x, psi'(x) = psi'(x + 1) + 1 / x^2 up to x >= 6,
// then psi(x) ~ log x - 1/(2x) - sum_k B_2k / (2k x^2k), psi'(x) ~ 1/x + 1/(2x^2) + sum_k B_2k / x^(2k+1) to k = 6.
// A caller that does not use psi' gets its arithmetic removed by the compiler.  x <= 0 and NaN give NaN for both: the
// recurrence would not end for x = -inf or x <= -2^53 (x + 1 == x), and a concentration there is outside the contract;
// the recurrence then runs at most 6 steps.
__device__ __forceinline__ void digamma_trigamma(double x, double& psi, double& tri) {
  if (!(x > 0.0)) {
    psi = tri = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  double ps = 0.0, tr = 0.0;
  while (x < 6.0) {
    const double r = 1.0 / x;
    ps -= r;
    tr = fma(r, r, tr);
    x += 1.0;
  }
  const double r = 1.0 / x, r2 = r * r;
  // -(1/12 - r2 (1/120 - r2 (1/252 - r2 (1/240 - r2 (1/132 - r2 691/32760))))) r2
  double s = fma(r2, -691.0 / 32760.0, 1.0 / 132.0);
  s = fma(r2, -s, 1.0 / 240.0);
  s = fma(r2, -s, 1.0 / 252.0);
  s = fma(r2, -s, 1.0 / 120.0);
  s = fma(r2, -s, 1.0 / 12.0);
  psi = ps + (log(x) - 0.5 * r - s * r2);
  // 1/6 - r2 (1/30 - r2 (1/42 - r2 (1/30 - r2 (5/66 - r2 691/2730))))
  double t = fma(r2, -691.0 / 2730.0, 5.0 / 66.0);
  t = fma(r2, -t, 1.0 / 30.0);
  t = fma(r2, -t, 1.0 / 42.0);
  t = fma(r2, -t, 1.0 / 30.0);
  t = fma(r2, -t, 1.0 / 6.0);
  tri = tr + r * (1.0 + r * (0.5 + r * t));
}

struct BetaHead {
  static constexpr bool kShared = false;
  static constexpr const char* kNames[4] = {"concentration1", "concentration0", "g_concentration1", "g_concentration0"};

  struct Row {
    double lp, h;
  };
  static __device__ __forceinline__ Row row_begin(double) { return Row{0.0, 0.0}; }

  template <bool SHARED, typename T>
  static __device__ __forceinline__ void row_term(Row& r, const float* sac, const T* sc1, const T* sc0, int i,
                                                  const double*, int) {
    const double x = static_cast<double>(sac[i]);
    const double c1 = static_cast<double>(to_float(sc1[i])), c0 = static_cast<double>(to_float(sc0[i]));
    const double s = c1 + c0;
    const double lnorm = lgamma(s) - lgamma(c1) - lgamma(c0);  // -log B(c1, c0)
    double p1, p0, ps, unused;
    digamma_trigamma(c1, p1, unused);
    digamma_trigamma(c0, p0, unused);
    digamma_trigamma(s, ps, unused);
    r.lp += fma(c1 - 1.0, log(x), fma(c0 - 1.0, log1p(-x), lnorm));
    r.h += fma(s - 2.0, ps, -fma(c1 - 1.0, p1, fma(c0 - 1.0, p0, lnorm)));
  }

  static __device__ __forceinline__ void row_end(const Row& r, int, float& logp, float& ent) {
    logp = static_cast<float>(r.lp);
    ent = static_cast<float>(r.h);
  }

  template <bool SHARED, typename T>
  static __device__ __forceinline__ void column(const float* sac, T* sc1, T* sc0, int idx, float gl, float ge, float,
                                                double, double&) {
    const double x = static_cast<double>(sac[idx]);
    const double c1 = static_cast<double>(to_float(sc1[idx])), c0 = static_cast<double>(to_float(sc0[idx]));
    const double s = c1 + c0;
    double p1, t1, p0, t0, ps, ts;
    digamma_trigamma(c1, p1, t1);
    digamma_trigamma(c0, p0, t0);
    digamma_trigamma(s, ps, ts);
    const double gld = static_cast<double>(gl), ged = static_cast<double>(ge);
    const double hs = (s - 2.0) * ts;
    const double g1 = fma(gld, log(x) - p1 + ps, ged * (hs - (c1 - 1.0) * t1));
    const double g0 = fma(gld, log1p(-x) - p0 + ps, ged * (hs - (c0 - 1.0) * t0));
    sc1[idx] = from_float<T>(static_cast<float>(g1));
    sc0[idx] = from_float<T>(static_cast<float>(g0));
  }
};

}  // namespace
}  // namespace loss
}  // namespace srl

extern "C" int srl_ppo_loss_from_beta(const float* concentration1, const float* concentration0, const float* action, int D,
                                      const float* v_pred, const float* old_logp, const float* old_value, const float* ret,
                                      const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                      const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                      const double* local_stats, const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                      float* g_concentration1, float* g_concentration0, float* g_value, float* logp_out,
                                      float* entropy_out, double* out, float* out_f32, void* workspace,
                                      size_t workspace_bytes, srl_stream_t stream) {
  return srl::loss::ppo_loss_from_head<srl::loss::BetaHead>(
      "srl_ppo_loss_from_beta", sizeof(float), concentration1, concentration0, false, action, D, v_pred, old_logp,
      old_value, ret, adv, on_reset_next, ld_smp, nullptr, 0, lane_idx, T, n, norm_stats, local_stats, popart_mean_std,
      hyper, g_concentration1, g_concentration0, g_value, logp_out, entropy_out, out, out_f32, workspace,
      workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_beta_bf16(const uint16_t* concentration1, const uint16_t* concentration0,
                                           const float* action, int D, const uint16_t* v_pred, const float* old_logp,
                                           const float* old_value, const float* ret, const float* adv,
                                           const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T,
                                           int n, const double* norm_stats, const double* local_stats,
                                           const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                           uint16_t* g_concentration1, uint16_t* g_concentration0, uint16_t* g_value,
                                           float* logp_out, float* entropy_out, double* out, float* out_f32,
                                           void* workspace, size_t workspace_bytes, srl_stream_t stream) {
  return srl::loss::ppo_loss_from_head<srl::loss::BetaHead>(
      "srl_ppo_loss_from_beta_bf16", sizeof(__nv_bfloat16), concentration1, concentration0, false, action, D, v_pred,
      old_logp, old_value, ret, adv, on_reset_next, ld_smp, nullptr, 0, lane_idx, T, n, norm_stats, local_stats,
      popart_mean_std, hyper, g_concentration1, g_concentration0, g_value, logp_out, entropy_out, out, out_f32,
      workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_beta_pack(const void* concentration1, const void* concentration0, const float* action,
                                           int D, int elem_bytes, const void* v_pred, const float* pack,
                                           int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
                                           const double* norm_stats, const double* local_stats,
                                           const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                           void* g_concentration1, void* g_concentration0, void* g_value,
                                           float* logp_out, float* entropy_out, double* out, float* out_f32,
                                           void* workspace, size_t workspace_bytes, srl_stream_t stream) {
  constexpr const char* fn = "srl_ppo_loss_from_beta_pack";
  const int rc = srl::loss::check_head_pack(fn, elem_bytes, pack, pack_row_lo, lane_idx, pack_lanes, n);
  if (rc != SRL_OK) return rc;
  return srl::loss::ppo_loss_from_head<srl::loss::BetaHead>(
      fn, static_cast<size_t>(elem_bytes), concentration1, concentration0, false, action, D, v_pred, nullptr, nullptr,
      nullptr, nullptr, nullptr, pack_lanes, pack, pack_row_lo, lane_idx, T, n, norm_stats, local_stats,
      popart_mean_std, hyper, g_concentration1, g_concentration0, g_value, logp_out, entropy_out, out, out_f32,
      workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}
