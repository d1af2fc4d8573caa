// Shared by the GAE scan kernels (gae_scan.cu: shared-memory tile kernel; gae_scan_tma.cu: one-warp TMA kernel;
// gae_scan_ws.cu: warp-specialised kernel) and srl_gae_trace (gae_general.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "perm.cuh"

namespace srl {

struct GaeParams {
  const float* reward;
  const float* value;
  const uint8_t* done;
  const uint8_t* truncated;
  const uint8_t* on_reset;
  const float* vt_new_logp;
  const float* vt_old_logp;
  const double* popart;  // {mean, std} or null
  const float* old_logp;  // [L, N] or null (only for the pack)
  float* adv;
  float* ret;
  double* lane_part;
  double* lane_aos;  // [N][4] f64 {sum mask, sum adv*mask, sum (adv*mask)^2, 0} or null: the loss kernel's gather form
  float* pack;  // pair-interleaved [ceil(L/2)][N][2] float4 or null (include/srl_b200.h)
  int L, N, row_lo, row_hi;
  double gamma, gamma_lmbda, rho, c;
  PermJob perm;  // srl_gae_scan_perm: a permutation computed on the side (gae_scan_ws.cu only); out == nullptr: none
};

// Position (in float4 items) of transition (t, lane) in the loss pack: the two rows of a row pair sit next to each other,
// so a permuted minibatch fetches 32 contiguous, 32-byte aligned bytes per lane and row pair.
__host__ __device__ inline size_t pack_index(int t, int N, int lane) {
  return (static_cast<size_t>(t >> 1) * N + lane) * 2 + (t & 1);
}
// The advantage slot of a pack item the loss masks out (on_reset[t+1] set, or the padding row L-1): a quiet NaN.
constexpr int kPackMaskedAdv = 0x7fc00000;

bool gae_tma_eligible(const GaeParams& p);
int launch_gae_tma(const GaeParams& p, cudaStream_t st);
bool gae_ws_eligible(const GaeParams& p);
int launch_gae_ws(const GaeParams& p, cudaStream_t st);

#ifdef __CUDACC__
// ---- the reference's per-cell arithmetic ----------------------------------------------------------------------------
// Bit-identical to the reference's float64 scan only if every kernel rounds exactly as it does: each operation below is an
// explicit _rn intrinsic, a conversion or a plain add, so no -fmad setting can contract them.

// v' = value * (1 - done) in fp32 (mappo.py:120-124); with PopArt the value is denormalised first,
// (x.double() * std + mean).float() (utils.py:146-151)
__device__ __forceinline__ float gae_vprime(float value, bool done, bool popart, double pa_mean, double pa_std) {
  if (popart) value = static_cast<float>(__dadd_rn(__dmul_rn(static_cast<double>(value), pa_std), pa_mean));
  return __fmul_rn(value, done ? 0.f : 1.f);
}

// delta_t = reward + gamma * value[1:] * (1 - on_reset[1:]) - value[:-1] in float64   gae.py:63
// The operands come as stored (float or double) and the reward is read where it is added, so each kernel keeps the
// instruction schedule it had with this statement written out in place.
template <class V, class R>
__device__ __forceinline__ double gae_delta(const R* reward, V v0, V v1, bool reset1, double gamma) {
  double d = __dmul_rn(__dmul_rn(gamma, static_cast<double>(v1)), reset1 ? 0.0 : 1.0);
  d = __dadd_rn(static_cast<double>(*reward), d);
  return __dsub_rn(d, static_cast<double>(v0));
}

// m_t = gamma * lmbda * (1 - on_reset[1:]) * (1 - truncated[1:])   gae.py:87
__device__ __forceinline__ double gae_carry_product(double gl, bool reset1, bool trunc1) {
  return __dmul_rn(__dmul_rn(gl, reset1 ? 0.0 : 1.0), trunc1 ? 0.0 : 1.0);
}
// ... with gamma * lmbda a finite non-negative constant it is exactly 0 or gamma * lmbda: a select
__device__ __forceinline__ double gae_carry(bool carries, double gl) { return carries ? gl : 0.0; }

// V-trace: delta_t and m_t scaled by the clipped importance ratio   gae.py:64-65,88-89
__device__ __forceinline__ void gae_vtrace_scale(double& d, double& m, double ratio, double rho, double c) {
  d = __dmul_rn(d, fmin(ratio, rho));
  m = __dmul_rn(m, fmin(ratio, c));
}

// A_t = delta_t + m_t * A_{t+1}: separate multiply and add, as the reference's two torch ops   gae.py:92
__device__ __forceinline__ double gae_step(double d, double m, double a_next) { return __dadd_rn(d, __dmul_rn(m, a_next)); }

// value target = adv + v'[:-1] in fp32   mappo.py:143
__device__ __forceinline__ float gae_value_target(float adv, float vprime) { return __fadd_rn(adv, vprime); }

// one transition of the loss pack (include/srl_b200.h); `keep` = the loss mask of the transition
__device__ __forceinline__ float4 pack_item(float old_logp, float value, float ret, float adv, bool keep) {
  return make_float4(old_logp, value, ret, keep ? adv : __int_as_float(kPackMaskedAdv));
}

// A lane's running statistics over its loss rows (lane_part rows 0..6, include/srl_b200.h).
struct LaneStats {
  double s1 = 0, s2 = 0, s3 = 0, s4 = 0;
  int cnt = 0, dn = 0, tr = 0;
  // one row: `in_rows` = the row lies in [row_lo, row_hi); `mask` = in_rows and 1 - on_reset[t+1]   mappo.py:259-261
  __device__ __forceinline__ void add(bool in_rows, bool mask, float adv, float ret, bool done, bool trunc) {
    const double x = static_cast<double>(mask ? adv : 0.f);
    const double y = static_cast<double>(mask ? ret : 0.f);
    cnt += mask ? 1 : 0;
    s1 += x;
    s2 = __fma_rn(x, x, s2);
    s3 += y;
    s4 = __fma_rn(y, y, s4);
    dn += (in_rows && done) ? 1 : 0;
    tr += (in_rows && trunc) ? 1 : 0;
  }
};

// lane_part (SRL_LANE_PART rows, row 7 zero) and lane_aos ({cnt, s1, s2, 0}) of the block's LW lanes from a
// [GROUPS][7][LW] table of partial sums, added in group order (a fixed order).  All THREADS threads of the block take part;
// on_sum(k, ln, sum) sees every sum of rows k < 7 as well.
template <int LW, int GROUPS, int THREADS, class OnSum>
__device__ __forceinline__ void fold_lane_sums(const GaeParams& p, const double* red, OnSum on_sum) {
  for (int o = threadIdx.x; o < SRL_LANE_PART * LW; o += THREADS) {
    const int k = o / LW, ln = o % LW;
    const int col = blockIdx.x * LW + ln;
    if (col < p.N) {
      double s = 0.0;
      if (k < 7)
        for (int g = 0; g < GROUPS; ++g) s += red[(g * 7 + k) * LW + ln];
      p.lane_part[static_cast<size_t>(k) * p.N + col] = s;
      if (p.lane_aos != nullptr && k < 4) p.lane_aos[static_cast<size_t>(col) * 4 + k] = k < 3 ? s : 0.0;
      on_sum(k, ln, s);
    }
  }
}
#endif  // __CUDACC__

}  // namespace srl
