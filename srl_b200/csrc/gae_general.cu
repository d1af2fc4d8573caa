// The rest of the GAE family's API surface (include/srl_b200.h: srl_gae_trace, srl_traj_gae):
//
// 1. srl_gae_trace -- everything modules.gae_trace accepts that the specialised K2 kernels do not
//    (legacy/algorithm/modules/gae.py:8-97): vector critics (reward / value [.., N, Nc] with the flags broadcast over
//    Nc, gae.py:26-30), per-element discount and lambda tensors (gae.py:31-34,51-60) and a ready-made importance ratio
//    (gae.py:36,64-65,88-89).  One thread owns one (lane, critic) column for the whole trajectory; adjacent threads own
//    adjacent columns, so every row access of a warp is one coalesced segment.  Rows are taken newest first in chunks of
//    CH: all loads of a chunk are issued before the first dependent float64 operation, so a thread exposes one DRAM
//    round trip per CH rows.  The per-cell arithmetic is K2's (gae_common.cuh) -> bit-identical to the reference.
//
// 2. srl_traj_gae -- TrajGAE.process (gae.py:100-139): GAE along whole episodes, one after another in memory
//    ([total_steps, W] with an offset table), in the arrays' own dtype (numpy semantics: float32 arrays stay float32,
//    the python scalars gamma and gamma * lmbda are rounded to that dtype first).  One thread per (trajectory, element).
#include "common.cuh"
#include "gae_common.cuh"

namespace srl {
namespace {

struct TraceParams {
  const float* reward;      // [L-1(+), NC]
  const float* value;       // [L, NC]
  const uint8_t* done;      // [L, N] or null
  const uint8_t* truncated; // [L, N]
  const uint8_t* on_reset;  // [L, N]
  const float* gamma_t;     // [L-1, N] or null
  const float* lmbda_t;     // [L-1, N] or null
  const float* imp_ratio;   // [L-1, N] or null
  float* adv;               // [L-1 or L, NC]
  float* ret;               // same or null
  int L, N, Nc, pad_last_row;
  double gamma, lmbda, rho, c;
};

constexpr int kTraceThreads = 128;
constexpr int kTraceChunk = 4;

template <bool HAS_G, bool HAS_L, bool HAS_R, bool ONE_CRITIC>
__global__ void __launch_bounds__(kTraceThreads) gae_trace_kernel(const TraceParams p) {
  constexpr int CH = kTraceChunk;
  const long long NC = static_cast<long long>(p.N) * p.Nc;
  const long long col = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (col >= NC) return;
  const long long lane = ONE_CRITIC ? col : col / p.Nc;
  const int L = p.L;
  const long long N = p.N;

  // v'[L-1]: the bootstrap value of the newest row
  float vnext = __ldg(p.value + static_cast<long long>(L - 1) * NC + col);
  if (p.done != nullptr)
    vnext = gae_vprime(vnext, __ldg(p.done + static_cast<long long>(L - 1) * N + lane) != 0, false, 0.0, 1.0);
  if (p.pad_last_row) {  // mappo.py:254-256
    p.adv[static_cast<long long>(L - 1) * NC + col] = 0.f;
    if (p.ret != nullptr) p.ret[static_cast<long long>(L - 1) * NC + col] = 0.f;
  }
  const double gl_const = __dmul_rn(p.gamma, p.lmbda);  // python evaluates gamma * lmbda first (gae.py:87)
  double g = 0.0;
  for (int t = L - 2; t >= 0; t -= CH) {
    float rw[CH], vv[CH], gm[CH], lm[CH], ir[CH];
    uint32_t dn[CH], tr[CH], rs[CH];
#pragma unroll
    for (int u = 0; u < CH; ++u) {
      const int row = t - u;
      rw[u] = vv[u] = gm[u] = lm[u] = ir[u] = 0.f;
      dn[u] = tr[u] = rs[u] = 0u;
      if (row >= 0) {
        const long long e = static_cast<long long>(row) * NC + col;
        const long long f = static_cast<long long>(row) * N + lane;
        rw[u] = ldg_stream(p.reward + e);
        vv[u] = ldg_stream(p.value + e);
        if (p.done != nullptr) dn[u] = __ldg(p.done + f);
        tr[u] = __ldg(p.truncated + f + N);  // flags of row + 1
        rs[u] = __ldg(p.on_reset + f + N);
        if (HAS_G) gm[u] = __ldg(p.gamma_t + f);
        if (HAS_L) lm[u] = __ldg(p.lmbda_t + f);
        if (HAS_R) ir[u] = __ldg(p.imp_ratio + f);
      }
    }
#pragma unroll
    for (int u = 0; u < CH; ++u) {
      const int row = t - u;
      if (row >= 0) {
        const float v0 = p.done != nullptr ? gae_vprime(vv[u], dn[u] != 0, false, 0.0, 1.0) : vv[u];
        const bool reset1 = rs[u] != 0, trunc1 = tr[u] != 0;
        const double gam = HAS_G ? static_cast<double>(gm[u]) : p.gamma;
        double d = gae_delta(&rw[u], v0, vnext, reset1, gam);
        const double gl = (HAS_G || HAS_L) ? __dmul_rn(gam, HAS_L ? static_cast<double>(lm[u]) : p.lmbda) : gl_const;
        double m = gae_carry_product(gl, reset1, trunc1);  // any per-element gamma / lmbda: the product, not a select
        if (HAS_R) gae_vtrace_scale(d, m, static_cast<double>(ir[u]), p.rho, p.c);
        g = gae_step(d, m, g);
        const float a = static_cast<float>(g);  // gae.py:97
        const long long e = static_cast<long long>(row) * NC + col;
        stg_stream(p.adv + e, a);
        if (p.ret != nullptr) stg_stream(p.ret + e, gae_value_target(a, v0));
        vnext = v0;
      }
    }
  }
}

template <bool G, bool Lm, bool R>
int launch_trace(const TraceParams& p, cudaStream_t st) {
  const long long NC = static_cast<long long>(p.N) * p.Nc;
  const long long grid = (NC + kTraceThreads - 1) / kTraceThreads;
  if (p.Nc == 1)
    gae_trace_kernel<G, Lm, R, true><<<static_cast<unsigned>(grid), kTraceThreads, 0, st>>>(p);
  else
    gae_trace_kernel<G, Lm, R, false><<<static_cast<unsigned>(grid), kTraceThreads, 0, st>>>(p);
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}

// ---- TrajGAE ----------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T mul_rn(T a, T b);
template <>
__device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }
template <>
__device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }
template <typename T>
__device__ __forceinline__ T add_rn(T a, T b);
template <>
__device__ __forceinline__ float add_rn<float>(float a, float b) { return __fadd_rn(a, b); }
template <>
__device__ __forceinline__ double add_rn<double>(double a, double b) { return __dadd_rn(a, b); }

template <typename T>
__global__ void __launch_bounds__(128) traj_gae_kernel(const T* __restrict__ reward, const T* __restrict__ value,
                                                       const int64_t* __restrict__ offsets,
                                                       const uint8_t* __restrict__ final_truncated,
                                                       const uint8_t* __restrict__ final_has_value, int n_traj, int W,
                                                       double gamma, double lmbda, T* __restrict__ adv,
                                                       T* __restrict__ ret) {
  const long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (e >= static_cast<long long>(n_traj) * W) return;
  const int traj = static_cast<int>(e / W);
  const int w = static_cast<int>(e % W);
  const long long lo = offsets[traj], hi = offsets[traj + 1];
  const long long len = hi - lo;
  if (len < 2) return;  // gae.py:113: `step = ep_len - 2` < 0 -> nothing is written
  // numpy: a python float meeting a float32 array is rounded to float32 first; gamma * lmbda is a python product
  const T gam = static_cast<T>(gamma);
  const T gl = static_cast<T>(__dmul_rn(gamma, lmbda));
  // gae.py:117-123: bootstrap of the last computed step = value[last] * truncated[last], or 0 when the final step
  // carries no analyzed_result
  T boot = static_cast<T>(0);
  if (final_has_value[traj])
    boot = mul_rn<T>(value[(hi - 1) * W + w], static_cast<T>(final_truncated[static_cast<long long>(traj) * W + w] != 0));
  T g = static_cast<T>(0);
  for (long long s = hi - 2; s >= lo; --s) {
    const T r = reward[s * W + w];
    const T v = value[s * W + w];
    const T delta = add_rn<T>(add_rn<T>(r, mul_rn<T>(gam, boot)), -v);  // gae.py:127
    g = add_rn<T>(mul_rn<T>(gl, g), delta);                              // gae.py:128
    adv[s * W + w] = g;                                                  // gae.py:130
    ret[s * W + w] = add_rn<T>(g, v);                                    // gae.py:131
    boot = v;                                                            // gae.py:125
  }
}

}  // namespace
}  // namespace srl

extern "C" int srl_gae_trace(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                             const uint8_t* on_reset, const float* gamma_t, const float* lmbda_t,
                             const float* imp_ratio, int L, int N, int critic_dim, double gamma, double lmbda, double rho,
                             double c, int pad_last_row, float* adv, float* ret, srl_stream_t stream) {
  using namespace srl;
  SRL_REQUIRE(L >= 2 && N >= 1 && critic_dim >= 1, SRL_ERR_INVALID_ARG,
              "srl_gae_trace: need L >= 2, N >= 1, critic_dim >= 1 (got L=%d N=%d critic_dim=%d)", L, N, critic_dim);
  SRL_REQUIRE(reward && value && truncated && on_reset && adv, SRL_ERR_INVALID_ARG, "srl_gae_trace: null tensor pointer");
  SRL_REQUIRE(static_cast<long long>(N) * critic_dim <= 0x7fffffffLL * kTraceThreads, SRL_ERR_UNSUPPORTED,
              "srl_gae_trace: N * critic_dim too large for one grid");
  TraceParams p;
  p.reward = reward;
  p.value = value;
  p.done = done;
  p.truncated = truncated;
  p.on_reset = on_reset;
  p.gamma_t = gamma_t;
  p.lmbda_t = lmbda_t;
  p.imp_ratio = imp_ratio;
  p.adv = adv;
  p.ret = ret;
  p.L = L;
  p.N = N;
  p.Nc = critic_dim;
  p.pad_last_row = pad_last_row;
  p.gamma = gamma;
  p.lmbda = lmbda;
  p.rho = rho;
  p.c = c;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int key = (gamma_t ? 4 : 0) | (lmbda_t ? 2 : 0) | (imp_ratio ? 1 : 0);
  switch (key) {
    case 0: return launch_trace<false, false, false>(p, st);
    case 1: return launch_trace<false, false, true>(p, st);
    case 2: return launch_trace<false, true, false>(p, st);
    case 3: return launch_trace<false, true, true>(p, st);
    case 4: return launch_trace<true, false, false>(p, st);
    case 5: return launch_trace<true, false, true>(p, st);
    case 6: return launch_trace<true, true, false>(p, st);
    default: return launch_trace<true, true, true>(p, st);
  }
}

extern "C" int srl_traj_gae(const void* reward, const void* value, const int64_t* offsets, const uint8_t* final_truncated,
                            const uint8_t* final_has_value, int n_traj, int width, int is_float64, double gamma,
                            double lmbda, void* adv, void* ret, srl_stream_t stream) {
  using namespace srl;
  SRL_REQUIRE(n_traj >= 0 && width >= 1, SRL_ERR_INVALID_ARG, "srl_traj_gae: need n_traj >= 0 and width >= 1 (got %d, %d)",
              n_traj, width);
  if (n_traj == 0) return SRL_OK;
  SRL_REQUIRE(reward && value && offsets && final_truncated && final_has_value && adv && ret, SRL_ERR_INVALID_ARG,
              "srl_traj_gae: null pointer");
  const long long threads = static_cast<long long>(n_traj) * width;
  const long long grid = (threads + 127) / 128;
  SRL_REQUIRE(grid <= 0x7fffffffLL, SRL_ERR_UNSUPPORTED, "srl_traj_gae: too many trajectories for one grid");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (is_float64)
    traj_gae_kernel<double><<<static_cast<unsigned>(grid), 128, 0, st>>>(
        static_cast<const double*>(reward), static_cast<const double*>(value), offsets, final_truncated, final_has_value,
        n_traj, width, gamma, lmbda, static_cast<double*>(adv), static_cast<double*>(ret));
  else
    traj_gae_kernel<float><<<static_cast<unsigned>(grid), 128, 0, st>>>(
        static_cast<const float*>(reward), static_cast<const float*>(value), offsets, final_truncated, final_has_value,
        n_traj, width, gamma, lmbda, static_cast<float*>(adv), static_cast<float*>(ret));
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}
