// K4b-wide: the fused categorical PPO loss of ppo_loss.cu's K4b for rows of up to SRL_K4B_WIDE_MAX_SUM_K logits (Go's 362
// actions, chess's 4672, a language model's vocabulary), where K4b's staged [256, sum K] tile no longer fits shared memory.
//
// A warp owns one transition's row at a time (rows dealt round-robin over the grid's warps) and walks it head by head:
//  * first pass: lane l reads logits k = k0 + 32 u + l (u < kWideUnroll: that many independent coalesced loads in flight per
//    lane) and keeps running values of the head -- max m, s = sum e^{z-m}, w = sum e^{z-m} (z - m) -- merged across the warp
//    by a fixed butterfly of shuffles whose merge is rounded explicitly, so every lane ends with the same bits.  Then
//    l = fl(m + log s) and H = (l - m) - w / s: the head's log-sum-exp and entropy with one exponential per logit;
//  * element<RuntimeCfg> once per row (every lane, on the same values; lane 0 adds the row to the sums and stores);
//  * second pass: the row is read again (from L2 when it is still there) and d loss / d logits written, coalesced.
// The element-to-lane assignment and every operation are the same for float32 and bfloat16 (a bfloat16 logit is widened
// where it is read), so the bfloat16 instantiation returns the float32 one's logp and entropy on the widened values and its
// gradients rounded once.  Offsets into the logits are 64-bit: T * n * sum K exceeds 2^31 at these widths.
#include "ppo_loss.cuh"

namespace srl {
namespace loss {
namespace {

constexpr int kWideWarps = 8;   // warps of a CTA (256 threads), one row each at a time
constexpr int kWideUnroll = 8;  // logits per lane and step of a pass

// running log-sum-exp state of a head: max m, s = sum e^{z-m}, w = sum e^{z-m} (z - m).  The empty state is
// {-FLT_MAX, 0, 0}: a -inf logit (an unmasked policy's dead agent) then gives e = 0 and a clamped z - m, never 0 * inf.
struct Lse {
  float m, s, w;
};

// a and b rescaled to the larger max and added.  Rounded explicitly (no contraction), so merge(a, b) and merge(b, a) are the
// same bits: both lanes of a shuffle pair go on with one state.
__device__ __forceinline__ Lse merge(const Lse& a, const Lse& b) {
  const float m = fmaxf(a.m, b.m);
  const float da = fmaxf(a.m - m, -FLT_MAX), db = fmaxf(b.m - m, -FLT_MAX);
  const float ea = expf(da), eb = expf(db);
  Lse r;
  r.m = m;
  r.s = __fadd_rn(__fmul_rn(ea, a.s), __fmul_rn(eb, b.s));
  r.w = __fadd_rn(__fmul_rn(ea, __fadd_rn(a.w, __fmul_rn(da, a.s))), __fmul_rn(eb, __fadd_rn(b.w, __fmul_rn(db, b.s))));
  return r;
}

// first pass over one head of K logits at z (its mask bytes at mk): the warp's merged state, the same in every lane
template <bool MASKED, typename T>
__device__ __forceinline__ Lse head_lse(const T* z, const uint8_t* mk, int K, int lane) {
  Lse st{-FLT_MAX, 0.f, 0.f};
  for (int k0 = 0; k0 < K; k0 += 32 * kWideUnroll) {
    float v[kWideUnroll];
#pragma unroll
    for (int u = 0; u < kWideUnroll; ++u) {
      const int k = k0 + 32 * u + lane;
      v[u] = k < K ? logit_at<MASKED>(z, mk, k) : -INFINITY;
    }
    float mc = v[0];
#pragma unroll
    for (int u = 1; u < kWideUnroll; ++u) mc = fmaxf(mc, v[u]);
    const float m = fmaxf(st.m, mc);
    // this step's terms summed first, then added to the running sums: a chain of K / (32 kWideUnroll) additions per lane
    float cs = 0.f, cw = 0.f;
#pragma unroll
    for (int u = 0; u < kWideUnroll; ++u) {
      const float x = fmaxf(v[u] - m, -FLT_MAX);
      const float e = expf(x);
      cs += e;
      cw += e * x;
    }
    const float d = fmaxf(st.m - m, -FLT_MAX);
    const float a = expf(d);
    st.w = a * (st.w + d * st.s) + cw;
    st.s = a * st.s + cs;
    st.m = m;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Lse p;
    p.m = __shfl_xor_sync(0xffffffffu, st.m, o);
    p.s = __shfl_xor_sync(0xffffffffu, st.s, o);
    p.w = __shfl_xor_sync(0xffffffffu, st.w, o);
    st = merge(st, p);
  }
  return st;
}

// MASKED: an unavailable logit reads as kUnavailableLogit and gets exactly 0 gradient.  T: float or __nv_bfloat16.
// PACK: the sample side is K2's loss pack (load_pack_item), else the five leaves.
template <bool MASKED, typename T, bool PACK>
__global__ void __launch_bounds__(256, 3) ppo_loss_logits_wide_kernel(const __grid_constant__ LogitsParams q) {
  __shared__ float2 s_head[kWideWarps][SRL_MAX_HEADS];  // per warp and head: {log-sum-exp, entropy} for the second pass
  const LossShared& p = q.s;
  const Problem& pr = q.pr;
  const LossHyperDev& h = p.h;
  double mask_sum;
  const Uniforms u = load_uniforms(pr.norm_stats, pr.local_stats, p.popart, h.adv_eps, mask_sum);
  Acc acc;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long SK = q.SK;
  const long long W = static_cast<long long>(p.T) * p.n;
  for (long long i = static_cast<long long>(blockIdx.x) * kWideWarps + warp; i < W;
       i += static_cast<long long>(gridDim.x) * kWideWarps) {
    // the sample side of the row (every lane loads the same words: one transaction each), in flight under the first pass
    float ol, ov = 0.f, rt, ad;
    bool valid;
    const int t = static_cast<int>(i / p.n);
    const int j = static_cast<int>(i - static_cast<long long>(t) * p.n);
    const int c = pr.lane_idx ? pr.lane_idx[j] : j;
    const float vp = to_float(reinterpret_cast<const T*>(pr.v_pred)[i]);
    if constexpr (PACK) {
      load_pack_item(p, t, c, ol, ov, rt, ad, valid);
    } else {
      const long long os = t * p.ld_smp + c;
      ol = __ldg(p.old_logp + os), rt = __ldg(p.ret + os), ad = __ldg(p.adv + os);
      ov = h.clip_value ? __ldg(p.old_value + os) : 0.f;
      valid = __ldg(p.reset_next + os) == 0;
    }
    const T* z = static_cast<const T*>(q.logits) + i * SK;
    const uint8_t* mk = MASKED ? q.available + i * SK : nullptr;
    const int32_t* act = q.action + i * q.heads;
    float logp = 0.f, ent = 0.f;
    int off = 0;
#pragma unroll 1
    for (int hd = 0; hd < q.heads; ++hd) {
      const int K = q.head_size[hd];
      const Lse st = head_lse<MASKED>(z + off, MASKED ? mk + off : nullptr, K, lane);
      const float l = st.m + logf(st.s);
      // -sum_k p_k (z_k - l) with p_k = e^{z_k - m} / s and l already rounded: torch's lp_k = z_k - l, so a head whose logits
      // are all unavailable (l rounds to -1e10 = m, w = 0) has entropy exactly 0, not log K
      const float hh = (l - st.m) - st.w / st.s;
      const int a = __ldg(act + hd);
      logp += logit_at<MASKED>(z + off, MASKED ? mk + off : nullptr, a) - l;
      ent += hh;
      if (lane == 0) s_head[warp][hd] = make_float2(l, hh);
      off += K;
    }
    __syncwarp();
    float g_lp, g_v, g_en;
    RowSums rs;
    element<RuntimeCfg>(h, u, logp, vp, ent, ol, ov, rt, ad, valid, g_lp, g_v, g_en, rs);
    if (lane == 0) {
      acc.add(rs);
      stg_stream(reinterpret_cast<T*>(pr.g_value) + i, from_float<T>(g_v));
      if (q.logp_out) q.logp_out[i] = logp;
      if (q.entropy_out) q.entropy_out[i] = ent;
    }
    T* g = static_cast<T*>(q.g_logits) + i * SK;
    off = 0;
#pragma unroll 1
    for (int hd = 0; hd < q.heads; ++hd) {
      const int K = q.head_size[hd];
      const float2 lh = s_head[warp][hd];
      const int a = __ldg(act + hd);
      for (int k0 = 0; k0 < K; k0 += 32 * kWideUnroll) {
        float v[kWideUnroll];
#pragma unroll
        for (int uu = 0; uu < kWideUnroll; ++uu) {
          const int k = k0 + 32 * uu + lane;
          v[uu] = k < K ? to_float(ldg_stream(z + off + k)) : 0.f;
        }
#pragma unroll
        for (int uu = 0; uu < kWideUnroll; ++uu) {
          const int k = k0 + 32 * uu + lane;
          if (k < K) {
            const float lp = v[uu] - lh.x;
            const float pk = expf(lp);
            // d logp / d z_k = [k == a] - p_k ;  d H / d z_k = -p_k (lp_k + H)
            const float gk = g_lp * ((k == a ? 1.f : 0.f) - pk) - g_en * pk * (fmaxf(lp, -FLT_MAX) + lh.y);
            stg_stream(g + off + k, from_float<T>((MASKED && __ldg(mk + off + k) == 0) ? 0.f : gk));
          }
        }
      }
      off += K;
    }
    __syncwarp();  // s_head is rewritten by the next row
  }
  reduce_and_finalize(pr, h, acc, mask_sum, blockIdx.x, gridDim.x);
}

// at most kMaxGrid CTAs (one partial row each in the workspace slot), no more than are resident at once.  The grid follows the
// float32 instantiation's residency for both element types, so that they fold their partial rows alike.
template <bool MASKED, typename T, bool PACK>
int launch_wide(const LogitsParams& q, cudaStream_t stream) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_loss_logits_wide_kernel<MASKED, float, PACK>, 256, 0) !=
          cudaSuccess ||
      per_sm < 1)
    per_sm = 1;
  const long long rows = static_cast<long long>(q.s.T) * q.s.n;
  long long grid = static_cast<long long>(sm_count()) * per_sm;
  if (grid > kMaxGrid) grid = kMaxGrid;
  if (grid > (rows + kWideWarps - 1) / kWideWarps) grid = (rows + kWideWarps - 1) / kWideWarps;
  ppo_loss_logits_wide_kernel<MASKED, T, PACK><<<static_cast<int>(grid), 256, 0, stream>>>(q);
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}

int launch_logits_wide(const LogitsParams& q, size_t elem_bytes, bool masked, bool pack, cudaStream_t stream) {
  const bool bf16 = elem_bytes == sizeof(__nv_bfloat16);
  if (pack) {
    if (bf16)
      return masked ? launch_wide<true, __nv_bfloat16, true>(q, stream) : launch_wide<false, __nv_bfloat16, true>(q, stream);
    return masked ? launch_wide<true, float, true>(q, stream) : launch_wide<false, float, true>(q, stream);
  }
  if (bf16)
    return masked ? launch_wide<true, __nv_bfloat16, false>(q, stream) : launch_wide<false, __nv_bfloat16, false>(q, stream);
  return masked ? launch_wide<true, float, false>(q, stream) : launch_wide<false, float, false>(q, stream);
}

}  // namespace
}  // namespace loss
}  // namespace srl

extern "C" int srl_ppo_loss_from_logits_wide(const void* logits, int elem_bytes, const uint8_t* available,
                                             const int32_t* action, const int32_t* head_sizes_host, int heads,
                                             const void* v_pred, const float* old_logp, const float* old_value,
                                             const float* ret, const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                             const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                             const double* local_stats, const double* popart_mean_std,
                                             const srl_ppo_hyper* hyper, void* g_logits, void* g_value, float* logp_out,
                                             float* entropy_out, double* out, float* out_f32, void* workspace,
                                             size_t workspace_bytes, srl_stream_t stream) {
  constexpr const char* fn = "srl_ppo_loss_from_logits_wide";
  SRL_REQUIRE(elem_bytes == 4 || elem_bytes == 2, SRL_ERR_INVALID_ARG, "%s: elem_bytes=%d, need 4 (float32) or 2 (bfloat16)",
              fn, elem_bytes);
  return srl::loss::ppo_loss_from_logits(fn, SRL_K4B_WIDE_MAX_SUM_K, SRL_K4B_WIDE_MAX_SUM_K, srl::loss::launch_logits_wide,
                                         static_cast<size_t>(elem_bytes), logits, available, action, head_sizes_host, heads,
                                         v_pred, old_logp, old_value, ret, adv, on_reset_next, ld_smp, nullptr, 0, lane_idx,
                                         T, n, norm_stats, local_stats, popart_mean_std, hyper, g_logits, g_value, logp_out,
                                         entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_logits_wide_pack(const void* logits, int elem_bytes, const uint8_t* available,
                                                  const int32_t* action, const int32_t* head_sizes_host, int heads,
                                                  const void* v_pred, const float* pack, int64_t pack_lanes, int pack_row_lo,
                                                  const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                                  const double* local_stats, const double* popart_mean_std,
                                                  const srl_ppo_hyper* hyper, void* g_logits, void* g_value,
                                                  float* logp_out, float* entropy_out, double* out, float* out_f32,
                                                  void* workspace, size_t workspace_bytes, srl_stream_t stream) {
  constexpr const char* fn = "srl_ppo_loss_from_logits_wide_pack";
  const int rc = srl::loss::check_logits_pack(fn, elem_bytes, pack, pack_lanes, pack_row_lo, lane_idx, n);
  if (rc != SRL_OK) return rc;
  return srl::loss::ppo_loss_from_logits(fn, SRL_K4B_WIDE_MAX_SUM_K, SRL_K4B_WIDE_MAX_SUM_K, srl::loss::launch_logits_wide,
                                         static_cast<size_t>(elem_bytes), logits, available, action, head_sizes_host, heads,
                                         v_pred, nullptr, nullptr, nullptr, nullptr, nullptr, pack_lanes, pack, pack_row_lo,
                                         lane_idx, T, n, norm_stats, local_stats, popart_mean_std, hyper, g_logits, g_value,
                                         logp_out, entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}
