// K4: fused PPO / MAPPO loss forward + backward (see include/srl_b200.h; replaces mappo.py:146-217,
// utils.py:10-67,228-265 and the autograd backward to new_logp / state_values / entropy).
//
// One pass over the [T, n] minibatch: each element reads 29 B (25 B without value clipping) and
// writes 12 B of gradients.  The advantage-normalisation statistics arrive pre-reduced (and, on
// several GPUs, pre-all-reduced) from K2 + srl_group_stats, so there is no second pass and no grid
// barrier.
//
// Work decomposition (r1c; profiles/r1c_notes.md has the ncu evidence behind each choice):
//  * a launch covers up to SRL_MAX_LOSS_BATCH minibatches ("problems") of one shape -- blockIdx.y picks the
//    problem -- so the 32 tiny per-minibatch launches of a 4 x 8 PPO schedule become one grid that fills the
//    machine;
//  * inside a problem a CTA walks tiles of `rows_per_tile` rows x (blockDim * 4) lanes; a thread owns four
//    adjacent lanes (128-bit accesses on the dense policy side) and keeps its four gather indices in
//    registers for all rows of the tile, so index loads and the run-of-4 test are paid once per tile;
//  * the sample side comes in one of three forms: dense leaves (whole batch, no permutation), leaves
//    gathered through lane_idx (any alignment), or K2's `pack` (float4 = old_logp, old_value, ret, adv-or-NaN per
//    transition, the two rows of a row pair next to each other): one gather per lane and row pair instead of five
//    1..4-byte ones per transition -- permuted minibatches of even width run ppo_loss_pair.cu, this file's row-tile
//    kernel keeps the odd shapes of that form;
//  * per-element arithmetic is fp32 except the advantage / PopArt normalisation, which stays in float64
//    (reference: utils.py:38-67,139-144) as subtract + multiply by a correctly rounded reciprocal + one
//    Newton residual step (3 fp64 instructions instead of a ~25-instruction IEEE division; the quotient is
//    the correctly rounded one, then cast to float as the reference does);
//  * eight masked sums: four lanes are summed in fp32, then accumulated in float64 per thread, reduced
//    warp-shuffle -> shared memory -> one float64 partial row per CTA in the problem's workspace slot.
// Finalisation: immediate (out != NULL): the last CTA of the problem (atomic ticket) folds the rows in a fixed
// order; deferred (out == NULL): srl_ppo_loss_finalize folds any number of slots later in ONE launch.
// Either way the result is deterministic for a given launch shape and nothing syncs with the host.
#include <stdlib.h>
#include <string.h>

#include "ppo_loss.cuh"
#include "tma_util.cuh"

namespace srl {
namespace loss {
namespace {

__global__ void __launch_bounds__(256) loss_finalize_kernel(unsigned char* __restrict__ ws, size_t slot_bytes,
                                                            double* __restrict__ out, float* __restrict__ out_f32) {
  __shared__ double sred[kNumSums][8];
  unsigned char* base = ws + static_cast<size_t>(blockIdx.x) * slot_bytes;
  const SlotHeader* hd = reinterpret_cast<const SlotHeader*>(base);
  fold_rows_and_write(reinterpret_cast<double*>(base + kPartialsOffset), static_cast<int>(hd->n_rows),
                      hd->mask_sum, hd->wv, hd->we, sred, out + static_cast<size_t>(blockIdx.x) * SRL_LOSS_OUT_LEN,
                      out_f32 ? out_f32 + static_cast<size_t>(blockIdx.x) * 4 : nullptr);
}

// ---- K4b: the same loss starting from the actor head's logits -----------------------------------
// (actor_critic_policy.py:303-324: Categorical(logits=slice).log_prob / .entropy per head, summed.)
// A CTA takes 256 consecutive transitions; their [256, sumK] logits block is contiguous in memory, so
// it is staged through shared memory with coalesced loads (row stride sumK+1 words: conflict-free
// per-thread row walks), turned into d loss / d logits in place, and streamed back out coalesced.
// The policy side (logits, v_pred, g_logits, g_value) is float or bfloat16, the kernel's element type T; pr.v_pred and
// pr.g_value point at T as well (Problem is K4's struct, typed float).  Everything else, the arithmetic included, is float.
struct LogitsParams {
  LossShared s;
  Problem pr;             // new_logp / entropy / g_logp / g_entropy are unused here
  const void* logits;     // [T*n, SK] of T
  const int32_t* action;  // [T*n, heads]
  void* g_logits;         // [T*n, SK] of T
  float* logp_out;        // [T*n] or null
  float* entropy_out;     // [T*n] or null
  int heads, SK;
  int head_size[SRL_MAX_HEADS];
  const uint8_t* available;  // [T*n, SK], 0 = unavailable (MASKED instantiations only)
};

// How the kernel got here (ncu, T=128 N=4096 K=18: profiles/r2_notes.md).  First version: 2180 instructions per transition --
// the staged [256, SK + 1] block was walked once per pass (max, exp / sum, entropy, gradient) with a run-time trip count,
// staged in and out element by element with an integer division each, every shared-memory store behind its own global
// load -- 98 us for 91 MB, neither bandwidth- nor issue-bound.  Now:
//  * staging is ONE bulk asynchronous copy per tile and direction (tma::bulk_load / bulk_store, completion on an mbarrier /
//    a bulk group): the block is contiguous in global memory and dense in shared memory;
//  * a head of <= 32 actions lives in registers for the forward passes and again for the gradient pass, in instantiations
//    of 4, 8, ... 32 registers (loops unrolled, addresses immediate); e_k = exp(z_k - max) is kept in a second dense block
//    when both fit (CACHE_E), so the gradient pass needs no exponential; wider heads keep the row walk;
//  * the sample side is loaded before the passes, so its DRAM round trip hides under them.
#ifndef SRL_K4B_MIN_BLOCKS
#define SRL_K4B_MIN_BLOCKS 2
#endif
constexpr int kStage = 9;  // manual staging batch per thread (last, partial tile only)

// actor_critic_policy.py:135-136: logits.masked_fill(available_action == 0, -1e10) before the Categorical
constexpr float kUnavailableLogit = -1e10f;

// logit k of a row as the Categorical sees it
template <bool MASKED, typename T>
__device__ __forceinline__ float logit_at(const T* z, const uint8_t* m, int k) {
  return (MASKED && m[k] == 0) ? kUnavailableLogit : to_float(z[k]);
}

// forward passes of one head held in registers: log-sum-exp, 1 / sum, entropy; e_k to `ez` when CACHE_E.  With MASKED,
// `m` is the head's availability bytes and an unavailable logit reads as kUnavailableLogit (its e_k is 0 unless the whole
// head is unavailable: then every lp_k is 0, as in torch, and the head adds nothing to logp or the entropy)
template <int KM, bool CACHE_E, bool MASKED, typename T>
__device__ __forceinline__ void head_forward(const T* z, float* ez, const uint8_t* m, int K, float& l, float& inv,
                                             float& hh) {
  float v[KM];
#pragma unroll
  for (int k = 0; k < KM; ++k) v[k] = k < K ? logit_at<MASKED>(z, m, k) : -INFINITY;
  float mx = v[0];
#pragma unroll
  for (int k = 1; k < KM; ++k) mx = fmaxf(mx, v[k]);
  float e[KM];
  float se = 0.f;
#pragma unroll
  for (int k = 0; k < KM; ++k) {
    e[k] = expf(v[k] - mx);  // exp(-inf) = 0 for the padding registers
    se += e[k];
  }
  l = mx + logf(se);
  inv = 1.f / se;
  hh = 0.f;
#pragma unroll
  for (int k = 0; k < KM; ++k) {
    if (k < K) {
      const float lp = fmaxf(v[k] - l, -FLT_MAX);  // Categorical.entropy clamps at finfo.min
      const float pk = CACHE_E ? e[k] * inv : expf(lp);
      hh -= pk * lp;
      if (CACHE_E) ez[k] = e[k];
    }
  }
}

// gradient pass of one head: z_k <- d loss / d z_k; with MASKED an unavailable logit gets exactly 0 (masked_fill passes
// no gradient), also when it is the chosen action, where the expression below is not 0
template <int KM, bool CACHE_E, bool MASKED, typename T>
__device__ __forceinline__ void head_backward(T* z, const float* ez, const uint8_t* m, int K, int a, float l, float inv,
                                              float hh, float g_lp, float g_en) {
  float v[KM], e[KM];
#pragma unroll
  for (int k = 0; k < KM; ++k) {
    v[k] = k < K ? to_float(z[k]) : 0.f;
    e[k] = (CACHE_E && k < K) ? ez[k] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < KM; ++k) {
    if (k < K) {
      const float lp = v[k] - l;
      const float pk = CACHE_E ? e[k] * inv : expf(lp);
      // d logp / d z_k = [k == a] - p_k ;  d H / d z_k = -p_k (lp_k + H)
      const float g = g_lp * ((k == a ? 1.f : 0.f) - pk) - g_en * pk * (fmaxf(lp, -FLT_MAX) + hh);
      z[k] = from_float<T>((MASKED && m[k] == 0) ? 0.f : g);
    }
  }
}

#define SRL_HEAD_DISPATCH(FN, K, ...)                         \
  do {                                                        \
    if ((K) <= 4) FN<4, CACHE_E, MASKED>(__VA_ARGS__);        \
    else if ((K) <= 8) FN<8, CACHE_E, MASKED>(__VA_ARGS__);   \
    else if ((K) <= 12) FN<12, CACHE_E, MASKED>(__VA_ARGS__); \
    else if ((K) <= 16) FN<16, CACHE_E, MASKED>(__VA_ARGS__); \
    else if ((K) <= 20) FN<20, CACHE_E, MASKED>(__VA_ARGS__); \
    else if ((K) <= 24) FN<24, CACHE_E, MASKED>(__VA_ARGS__); \
    else if ((K) <= 28) FN<28, CACHE_E, MASKED>(__VA_ARGS__); \
    else FN<32, CACHE_E, MASKED>(__VA_ARGS__);                \
  } while (0)

// MASKED: the [256, SK] availability bytes of the tile follow the float blocks in shared memory, brought in with the logits
// (same mbarrier and expect_tx, or the same element-wise staging); every pass over a head reads them.
// T: the policy side's element type (float or __nv_bfloat16); the staged block holds T, the cached exponentials float.
template <bool CACHE_E, bool MASKED, typename T>
__global__ void __launch_bounds__(256, SRL_K4B_MIN_BLOCKS) ppo_loss_logits_kernel(const __grid_constant__ LogitsParams q) {
  // [256 * SK] of T, dense (+ [256 * SK] floats with CACHE_E), (+ [256 * SK] bytes with MASKED), then the mbarrier
  extern __shared__ __align__(128) float smem[];
  constexpr int kElem = sizeof(T);
  const LossShared& p = q.s;
  const Problem& pr = q.pr;
  const LossHyperDev& h = p.h;
  double mask_sum;
  const Uniforms u = load_uniforms(pr.norm_stats, pr.local_stats, p.popart, h.adv_eps, mask_sum);
  Acc acc;
  const int SK = q.SK;
  // offsets in floats: the staged block is 256 * SK * kElem bytes = 64 * kElem * SK floats (a multiple of 16 bytes), the
  // exponentials 256 * SK floats
  T* srow = reinterpret_cast<T*>(smem);
  float* erow = smem + 64 * kElem * SK;
  uint8_t* mrow = reinterpret_cast<uint8_t*>(smem + (CACHE_E ? 64 * kElem + 256 : 64 * kElem) * SK);
  uint64_t* bar = reinterpret_cast<uint64_t*>(mrow + (MASKED ? 256 * SK : 0));  // 256 * SK bytes keep it 8-byte aligned
  if (threadIdx.x == 0) {
    tma::mbar_init(bar, 1);
    tma::mbar_fence_init();
  }
  __syncthreads();
  uint32_t parity = 0;
  const bool bulk_ok = ((reinterpret_cast<uintptr_t>(q.logits) | reinterpret_cast<uintptr_t>(q.g_logits) |
                         (MASKED ? reinterpret_cast<uintptr_t>(q.available) : 0)) & 15) == 0;
  const long long W = static_cast<long long>(p.T) * p.n;
  const long long tiles = (W + 255) / 256;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long i0 = tile * 256;
    const int cnt = static_cast<int>(min(256ll, W - i0));
    const int total = cnt * SK;
    const T* src = static_cast<const T*>(q.logits) + i0 * SK;
    T* dst = static_cast<T*>(q.g_logits) + i0 * SK;
    // 256 * SK * kElem bytes of logits and 256 * SK bytes of mask: multiples of 16 at 16-byte aligned addresses
    const bool bulk = bulk_ok && cnt == 256;
    const uint8_t* msrc = MASKED ? q.available + i0 * SK : nullptr;
    if (bulk) {
      if (threadIdx.x == 0) {
        const uint32_t bytes = static_cast<uint32_t>(total) * kElem;
        tma::mbar_expect_tx(bar, MASKED ? bytes + static_cast<uint32_t>(total) : bytes);
        tma::bulk_load(srow, src, bytes, bar);
        if (MASKED) tma::bulk_load(mrow, msrc, static_cast<uint32_t>(total), bar);
      }
    } else {
      for (int e0 = threadIdx.x; e0 < total; e0 += 256 * kStage) {
        T v[kStage];
#pragma unroll
        for (int b = 0; b < kStage; ++b)
          v[b] = (e0 + b * 256 < total) ? ldg_stream(src + e0 + b * 256) : from_float<T>(0.f);
#pragma unroll
        for (int b = 0; b < kStage; ++b)
          if (e0 + b * 256 < total) srow[e0 + b * 256] = v[b];
      }
      if (MASKED) {
        for (int e0 = threadIdx.x; e0 < total; e0 += 256 * kStage) {
          uint8_t v[kStage];
#pragma unroll
          for (int b = 0; b < kStage; ++b) v[b] = (e0 + b * 256 < total) ? __ldg(msrc + e0 + b * 256) : 0;
#pragma unroll
          for (int b = 0; b < kStage; ++b)
            if (e0 + b * 256 < total) mrow[e0 + b * 256] = v[b];
        }
      }
    }
    // the sample side of this thread's transition, in flight while the block lands
    const bool mine = static_cast<int>(threadIdx.x) < cnt;
    const long long i = i0 + threadIdx.x;
    float vp = 0.f, ol = 0.f, rt = 0.f, ad = 0.f, ov = 0.f;
    bool valid = false;
    int act[SRL_MAX_HEADS];
    if (mine) {
      const int t = static_cast<int>(i / p.n);
      const int j = static_cast<int>(i - static_cast<long long>(t) * p.n);
      const int c = pr.lane_idx ? pr.lane_idx[j] : j;
      const long long os = t * p.ld_smp + c;
      vp = to_float(ldg_stream(reinterpret_cast<const T*>(pr.v_pred) + i));
      ol = __ldg(p.old_logp + os), rt = __ldg(p.ret + os), ad = __ldg(p.adv + os);
      ov = h.clip_value ? __ldg(p.old_value + os) : 0.f;
      valid = __ldg(p.reset_next + os) == 0;
#pragma unroll
      for (int hd = 0; hd < SRL_MAX_HEADS; ++hd) act[hd] = hd < q.heads ? q.action[i * q.heads + hd] : 0;
    }
    if (bulk) {
      tma::mbar_wait(bar, parity);
      parity ^= 1u;
    } else {
      __syncthreads();
    }
    if (mine) {
      T* z = srow + threadIdx.x * SK;
      float* ez = erow + threadIdx.x * SK;
      const uint8_t* m = mrow + threadIdx.x * SK;
      // (the head loops are NOT unrolled: with the dispatch over eight widths inlined in each of SRL_MAX_HEADS slots the kernel
      // was 128 copies of the passes and spent 27 % of its warp samples waiting for instructions; the per-head scalars
      // below are indexed at run time and live in local memory -- four words per head)
      float lse[SRL_MAX_HEADS], hent[SRL_MAX_HEADS], rse[SRL_MAX_HEADS];
      float logp = 0.f, ent = 0.f;
      int off = 0;
#pragma unroll 1
      for (int hd = 0; hd < q.heads; ++hd) {
        {
          const int K = q.head_size[hd];
          float l, inv, hh;
          if (K <= 32) {
            SRL_HEAD_DISPATCH(head_forward, K, z + off, ez + off, m + off, K, l, inv, hh);
          } else {
            float mx = -INFINITY;
            for (int k = 0; k < K; ++k) mx = fmaxf(mx, logit_at<MASKED>(z, m, off + k));
            float se = 0.f;
            for (int k = 0; k < K; ++k) {
              const float ek = expf(logit_at<MASKED>(z, m, off + k) - mx);
              if (CACHE_E) ez[off + k] = ek;
              se += ek;
            }
            l = mx + logf(se);
            inv = 1.f / se;
            hh = 0.f;
            for (int k = 0; k < K; ++k) {
              const float lp = fmaxf(logit_at<MASKED>(z, m, off + k) - l, -FLT_MAX);
              const float pk = CACHE_E ? ez[off + k] * inv : expf(lp);
              hh -= pk * lp;
            }
          }
          lse[hd] = l;
          rse[hd] = inv;
          hent[hd] = hh;
          logp += logit_at<MASKED>(z, m, off + act[hd]) - l;
          ent += hh;
          off += K;
        }
      }
      float g_lp, g_v, g_en;
      RowSums rs;
      element<RuntimeCfg>(h, u, logp, vp, ent, ol, ov, rt, ad, valid, g_lp, g_v, g_en, rs);
      acc.add(rs);
      stg_stream(reinterpret_cast<T*>(pr.g_value) + i, from_float<T>(g_v));
      if (q.logp_out) q.logp_out[i] = logp;
      if (q.entropy_out) q.entropy_out[i] = ent;
      off = 0;
#pragma unroll 1
      for (int hd = 0; hd < q.heads; ++hd) {
        {
          const int K = q.head_size[hd];
          if (K <= 32) {
            SRL_HEAD_DISPATCH(head_backward, K, z + off, ez + off, m + off, K, act[hd], lse[hd], rse[hd], hent[hd], g_lp,
                              g_en);
          } else {
            for (int k = 0; k < K; ++k) {
              const float lp = to_float(z[off + k]) - lse[hd];
              const float pk = CACHE_E ? ez[off + k] * rse[hd] : expf(lp);
              const float g = g_lp * ((k == act[hd] ? 1.f : 0.f) - pk) - g_en * pk * (fmaxf(lp, -FLT_MAX) + hent[hd]);
              z[off + k] = from_float<T>((MASKED && m[off + k] == 0) ? 0.f : g);
            }
          }
          off += K;
        }
      }
    }
    if (bulk) {
      tma::fence_proxy_async_smem();  // the gradients above, before the bulk copy reads them
      __syncthreads();
      if (threadIdx.x == 0) tma::bulk_store(dst, srow, static_cast<uint32_t>(total) * kElem);  // read before the next tile
      __syncthreads();
    } else {
      __syncthreads();
      for (int e0 = threadIdx.x; e0 < total; e0 += 256 * kStage) {
        T v[kStage];
#pragma unroll
        for (int b = 0; b < kStage; ++b) v[b] = (e0 + b * 256 < total) ? srow[e0 + b * 256] : from_float<T>(0.f);
#pragma unroll
        for (int b = 0; b < kStage; ++b)
          if (e0 + b * 256 < total) stg_stream(dst + e0 + b * 256, v[b]);
      }
      __syncthreads();
    }
  }
  reduce_and_finalize(pr, h, acc, mask_sum, blockIdx.x, gridDim.x);
}
#undef SRL_HEAD_DISPATCH

// The widest rows, the same for both element types: the largest sum K whose float32 block (and mask bytes) fit the 200 KiB
// opt-in below (include/srl_b200.h states both limits).  A bfloat16 block is half as wide, so it fits there as well.
static_assert(256 * SRL_K4B_MAX_SUM_K * 4 + 16 <= 200 * 1024 && 256 * (SRL_K4B_MAX_SUM_K + 1) * 4 + 16 > 200 * 1024, "");
static_assert(256 * SRL_K4B_MAX_SUM_K_MASKED * 5 + 16 <= 200 * 1024 && 256 * (SRL_K4B_MAX_SUM_K_MASKED + 1) * 5 + 16 > 200 * 1024,
              "");
static_assert(256 * SRL_K4B_MAX_SUM_K * 2 + 16 <= 200 * 1024 && 256 * SRL_K4B_MAX_SUM_K_MASKED * 3 + 16 <= 200 * 1024, "");

// one resident wave of ppo_loss_logits_kernel<CACHE_E, MASKED, T> over the T * n transitions of q
template <bool MASKED, typename T>
int launch_logits(const LogitsParams& q, bool cache_e, size_t smem, cudaStream_t stream) {
  int rc;
  if ((rc = opt_in_smem<ppo_loss_logits_kernel<true, MASKED, T>>(200 * 1024)) != SRL_OK) return rc;
  if ((rc = opt_in_smem<ppo_loss_logits_kernel<false, MASKED, T>>(200 * 1024)) != SRL_OK) return rc;
  const long long tiles = (static_cast<long long>(q.s.T) * q.s.n + 255) / 256;
  // one wave: as many CTAs as are resident with this much shared memory (2048 tiles on 1184 assumed slots were 1024 CTAs on
  // the 740 real ones -- a second, partial wave)
  int per_sm = 0;
  if ((cache_e ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_loss_logits_kernel<true, MASKED, T>, 256, smem)
               : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_loss_logits_kernel<false, MASKED, T>, 256, smem)) !=
          cudaSuccess ||
      per_sm < 1)
    per_sm = 1;
  const long long slots = static_cast<long long>(sm_count()) * per_sm;
  const long long cap = slots < kMaxGrid ? slots : kMaxGrid;
  // every CTA the same number of tiles (2048 tiles on 1184 slots would leave most CTAs one tile and the rest two)
  const long long per_cta = (tiles + cap - 1) / cap;
  const int grid = static_cast<int>((tiles + per_cta - 1) / per_cta);
  if (cache_e)
    ppo_loss_logits_kernel<true, MASKED, T><<<grid, 256, smem, stream>>>(q);
  else
    ppo_loss_logits_kernel<false, MASKED, T><<<grid, 256, smem, stream>>>(q);
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}

// srl_ppo_loss_from_logits (available == NULL) and srl_ppo_loss_from_logits_masked (elem_bytes = 4), and their _bf16 twins
// (elem_bytes = 2: logits, v_pred, g_logits and g_value are bfloat16)
int ppo_loss_from_logits(const char* fn, size_t elem_bytes, const void* logits, const uint8_t* available,
                         const int32_t* action, const int32_t* head_sizes_host, int heads, const void* v_pred,
                         const float* old_logp, const float* old_value, const float* ret, const float* adv,
                         const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
                         const double* norm_stats, const double* local_stats, const double* popart_mean_std,
                         const srl_ppo_hyper* hyper, void* g_logits, void* g_value, float* logp_out, float* entropy_out,
                         double* out, float* out_f32, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  SRL_REQUIRE(T >= 1 && n >= 1, SRL_ERR_INVALID_ARG, "%s: need T >= 1 and n >= 1", fn);
  SRL_REQUIRE(heads >= 1 && heads <= SRL_MAX_HEADS && head_sizes_host, SRL_ERR_INVALID_ARG,
              "%s: heads=%d outside [1, %d]", fn, heads, SRL_MAX_HEADS);
  SRL_REQUIRE(logits && action && v_pred && old_logp && ret && adv && on_reset_next && g_logits && g_value &&
                  norm_stats && local_stats && workspace,
              SRL_ERR_INVALID_ARG, "%s: null pointer", fn);
  SRL_REQUIRE(ld_smp >= (lane_idx ? 1 : n), SRL_ERR_INVALID_ARG, "%s: ld_smp smaller than the row", fn);
  SRL_REQUIRE(workspace_bytes >= srl_ppo_loss_workspace_bytes(T, n), SRL_ERR_INVALID_ARG,
              "%s: workspace too small (%zu bytes)", fn, workspace_bytes);
  LogitsParams q;
  int rc = fill_loss_hyper(hyper, popart_mean_std, q.s.h);
  if (rc != SRL_OK) return rc;
  SRL_REQUIRE(!(q.s.h.clip_value && old_value == nullptr), SRL_ERR_INVALID_ARG, "%s: clip_value needs old_value", fn);
  long long sk = 0;
  for (int i = 0; i < SRL_MAX_HEADS; ++i) {
    q.head_size[i] = i < heads ? head_sizes_host[i] : 0;
    SRL_REQUIRE(i >= heads || head_sizes_host[i] >= 1, SRL_ERR_INVALID_ARG, "%s: head %d has no actions", fn, i);
    sk += q.head_size[i];
  }
  const bool masked = available != nullptr;
  const int max_sk = masked ? SRL_K4B_MAX_SUM_K_MASKED : SRL_K4B_MAX_SUM_K;
  SRL_REQUIRE(sk <= max_sk, SRL_ERR_UNSUPPORTED, "%s: sum K = %lld too wide (max %d)", fn, sk, max_sk);
  const size_t row_bytes = static_cast<size_t>(256) * sk * elem_bytes;     // dense [256, sum K] block of the element type
  const size_t e_bytes = static_cast<size_t>(256) * sk * sizeof(float);    // the cached exponentials, float either way
  const size_t mask_bytes = masked ? static_cast<size_t>(256) * sk : 0;    // + its [256, sum K] availability bytes
  const bool cache_e = row_bytes + e_bytes + mask_bytes + 16 <= 200 * 1024;  // all fit: one exponential per logit
  const size_t smem = row_bytes + (cache_e ? e_bytes : 0) + mask_bytes + 16;  // + the mbarrier of the bulk copies
  q.heads = heads;
  q.SK = static_cast<int>(sk);
  q.logits = logits;
  q.available = available;
  q.action = action;
  q.g_logits = g_logits;
  q.logp_out = logp_out;
  q.entropy_out = entropy_out;
  LossShared& p = q.s;
  p.old_logp = old_logp;
  p.old_value = old_value;
  p.ret = ret;
  p.adv = adv;
  p.reset_next = on_reset_next;
  p.pack = nullptr;
  p.lane_aos = nullptr;
  p.part = nullptr;
  p.part_ctas = p.part_first = 0;
  p.row_lo = 0;
  p.popart = popart_mean_std;
  p.ld_pol = n;
  p.ld_grad = n;
  p.ld_smp = ld_smp;
  p.T = T;
  p.n = n;
  p.rows_per_tile = p.col_tiles = p.n_tiles = 0;
  p.smp_vec_ok = 0;
  Problem& pr = q.pr;
  pr.new_logp = pr.entropy = nullptr;
  pr.v_pred = static_cast<const float*>(v_pred);  // of the element type, as g_value
  pr.lane_idx = lane_idx;
  pr.norm_stats = norm_stats;
  pr.local_stats = local_stats;
  pr.g_logp = pr.g_entropy = nullptr;
  pr.g_value = static_cast<float*>(g_value);
  pr.out = out;
  pr.out_f32 = out_f32;
  pr.slot = reinterpret_cast<SlotHeader*>(workspace);
  if (elem_bytes == sizeof(__nv_bfloat16))
    return masked ? launch_logits<true, __nv_bfloat16>(q, cache_e, smem, stream)
                  : launch_logits<false, __nv_bfloat16>(q, cache_e, smem, stream);
  return masked ? launch_logits<true, float>(q, cache_e, smem, stream) : launch_logits<false, float>(q, cache_e, smem, stream);
}

}  // namespace

int fill_loss_hyper(const srl_ppo_hyper* hyper, const double* popart_mean_std, LossHyperDev& h) {
  SRL_REQUIRE(hyper != nullptr, SRL_ERR_INVALID_ARG, "ppo loss: null hyper pointer");
  SRL_REQUIRE(hyper->value_loss >= SRL_VL_MSE && hyper->value_loss <= SRL_VL_SMOOTHL1, SRL_ERR_INVALID_ARG,
              "ppo loss: unknown value_loss %d (0 mse, 1 huber, 2 smoothl1)", hyper->value_loss);
  SRL_REQUIRE(!(hyper->normalize_old_value && popart_mean_std == nullptr), SRL_ERR_INVALID_ARG,
              "ppo loss: normalize_old_value needs popart statistics");
  h.clip_lo = static_cast<float>(1.0 - hyper->eps_clip);  // python: 1 - self.eps_clip, then cast by torch.clamp
  h.clip_hi = static_cast<float>(1.0 + hyper->eps_clip);
  h.veps = static_cast<float>(hyper->value_eps_clip);
  h.c_clip = static_cast<float>(hyper->c_clip);
  h.wv = static_cast<float>(hyper->value_loss_weight);
  h.we = static_cast<float>(hyper->entropy_bonus_weight);
  h.vl_param = static_cast<float>(hyper->vl_param);
  h.adv_eps = hyper->adv_eps;
  h.value_loss = hyper->value_loss;
  h.clip_value = hyper->clip_value;
  h.dual_clip = hyper->dual_clip;
  h.normalize_old_value = hyper->normalize_old_value;
  return SRL_OK;
}

}  // namespace loss
}  // namespace srl

extern "C" size_t srl_ppo_loss_workspace_bytes(int, int) {
  return srl::loss::kPartialsOffset + static_cast<size_t>(srl::loss::kMaxGrid) * srl::loss::kNumSums * sizeof(double);
}

extern "C" int srl_ppo_loss_finalize(void* workspace, size_t slot_bytes, int n_slots, double* out, float* out_f32,
                                     srl_stream_t stream) {
  using namespace srl;
  using namespace srl::loss;
  SRL_REQUIRE(n_slots >= 0, SRL_ERR_INVALID_ARG, "srl_ppo_loss_finalize: negative slot count");
  if (n_slots == 0) return SRL_OK;
  SRL_REQUIRE(workspace && out, SRL_ERR_INVALID_ARG, "srl_ppo_loss_finalize: null pointer");
  SRL_REQUIRE(slot_bytes >= srl_ppo_loss_workspace_bytes(1, 1) && slot_bytes % 8 == 0, SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_finalize: slot_bytes=%zu smaller than one workspace or not 8-byte aligned", slot_bytes);
  loss_finalize_kernel<<<n_slots, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<unsigned char*>(workspace), slot_bytes, out, out_f32);
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}

extern "C" int srl_ppo_loss_fwd_bwd_batched(const srl_loss_problem* problems, int n_problems, int64_t ld_pol,
                                            int64_t ld_grad, const float* old_logp, const float* old_value,
                                            const float* ret, const float* adv, const uint8_t* on_reset_next,
                                            int64_t ld_smp, const float* pack, int pack_row_lo, const double* lane_aos,
                                            const double* minibatch_part, int part_ctas, int part_first, int T, int n,
                                            const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                            size_t workspace_bytes, srl_xchg* xchg, srl_stream_t stream) {
  using namespace srl;
  using namespace srl::loss;
  SRL_REQUIRE(n_problems >= 0, SRL_ERR_INVALID_ARG, "srl_ppo_loss_fwd_bwd_batched: negative problem count");
  if (n_problems == 0) return SRL_OK;
  SRL_REQUIRE(problems != nullptr, SRL_ERR_INVALID_ARG, "srl_ppo_loss_fwd_bwd_batched: null problem table");
  SRL_REQUIRE(T >= 1 && n >= 1, SRL_ERR_INVALID_ARG, "srl_ppo_loss_fwd_bwd: need T >= 1 and n >= 1 (got %d, %d)", T, n);
  SRL_REQUIRE(workspace_bytes >= srl_ppo_loss_workspace_bytes(T, n), SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd: workspace too small (%zu bytes)", workspace_bytes);
  LossShared s;
  int rc = fill_loss_hyper(hyper, popart_mean_std, s.h);
  if (rc != SRL_OK) return rc;
  if (pack == nullptr) {
    SRL_REQUIRE(old_logp && ret && adv && on_reset_next, SRL_ERR_INVALID_ARG, "srl_ppo_loss_fwd_bwd: null pointer");
    SRL_REQUIRE(!(s.h.clip_value && old_value == nullptr), SRL_ERR_INVALID_ARG,
                "srl_ppo_loss_fwd_bwd: clip_value needs old_value");
  } else {
    SRL_REQUIRE(aligned(pack, 32) && pack_row_lo >= 0, SRL_ERR_INVALID_ARG,
                "srl_ppo_loss_fwd_bwd: pack must be 32-byte aligned and pack_row_lo >= 0");
  }
  bool any_idx = false, all_idx = true;
  bool dense_ok = (n % 4 == 0) && (ld_pol % 4 == 0) && (ld_grad % 4 == 0);
  for (int k = 0; k < n_problems; ++k) {
    const srl_loss_problem& q = problems[k];
    SRL_REQUIRE(q.new_logp && q.v_pred && q.entropy && q.g_logp && q.g_value && q.g_entropy && q.workspace &&
                    (lane_aos != nullptr || (q.norm_stats && q.local_stats)),
                SRL_ERR_INVALID_ARG, "srl_ppo_loss_fwd_bwd: null pointer");
    any_idx = any_idx || q.lane_idx != nullptr;
    all_idx = all_idx && q.lane_idx != nullptr;
    dense_ok = dense_ok && aligned(q.new_logp, 16) && aligned(q.v_pred, 16) && aligned(q.entropy, 16) &&
               aligned(q.g_logp, 16) && aligned(q.g_value, 16) && aligned(q.g_entropy, 16) &&
               (q.lane_idx == nullptr || aligned(q.lane_idx, 16));
  }
  SRL_REQUIRE(any_idx == all_idx, SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd_batched: either every problem has a lane_idx or none has");
  SRL_REQUIRE(ld_pol >= n && ld_grad >= n && ld_smp >= (any_idx ? 1 : n), SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd: row strides smaller than the row");
  s.old_logp = old_logp;
  s.old_value = old_value;
  s.ret = ret;
  s.adv = adv;
  s.reset_next = on_reset_next;
  s.pack = reinterpret_cast<const float4*>(pack);
  s.popart = popart_mean_std;
  SRL_REQUIRE(lane_aos == nullptr || (popart_mean_std == nullptr && pack != nullptr && all_idx && aligned(lane_aos, 32)),
              SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd_batched: self-computed statistics (lane_aos) need the pack form with lane indices, no "
              "PopArt and a 32-byte aligned table");
  s.lane_aos = lane_aos;
  SRL_REQUIRE(minibatch_part == nullptr ||
                  (lane_aos != nullptr && aligned(minibatch_part, 32) && part_ctas >= 1 && part_first >= 0 &&
                   part_first + n_problems <= kMaxBatch),
              SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd_batched: minibatch_part needs lane_aos, a 32-byte aligned table, part_ctas >= 1 and table "
              "slots part_first .. part_first + n_problems - 1 within %d", kMaxBatch);
  s.part = minibatch_part;
  s.part_ctas = part_ctas;
  s.part_first = part_first;
  s.row_lo = pack ? pack_row_lo : 0;
  s.ld_pol = ld_pol;
  s.ld_grad = ld_grad;
  s.ld_smp = ld_smp;
  s.T = T;
  s.n = n;
  const bool smp_vec = pack == nullptr && (ld_smp % 4 == 0) && aligned(old_logp, 16) && aligned(ret, 16) &&
                       aligned(adv, 16) && (!s.h.clip_value || aligned(old_value, 16)) && aligned(on_reset_next, 4);
  s.smp_vec_ok = smp_vec ? 1 : 0;
  bool aligned8 = true;  // the pair kernel's 64-bit policy-side accesses
  for (int k = 0; k < n_problems; ++k) {
    const srl_loss_problem& q = problems[k];
    aligned8 = aligned8 && aligned(q.new_logp, 8) && aligned(q.v_pred, 8) && aligned(q.entropy, 8) && aligned(q.g_logp, 8) &&
               aligned(q.g_value, 8) && aligned(q.g_entropy, 8) && (q.lane_idx == nullptr || aligned(q.lane_idx, 8));
  }
  const bool pair = loss_pair_eligible(s, aligned8);
  SRL_REQUIRE(lane_aos == nullptr || pair, SRL_ERR_UNSUPPORTED,
              "srl_ppo_loss_fwd_bwd_batched: self-computed statistics need an even minibatch width <= 1024 lanes, even row "
              "strides and 8-byte aligned policy-side tensors (n = %d)", n);
  const int mode = pack ? kPack : ((!any_idx && dense_ok && smp_vec) ? kDense : kGather);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto fill = [](Problem& p, const srl_loss_problem& q) {
    p.new_logp = q.new_logp;
    p.v_pred = q.v_pred;
    p.entropy = q.entropy;
    p.lane_idx = q.lane_idx;
    p.norm_stats = q.norm_stats;
    p.local_stats = q.local_stats;
    p.g_logp = q.g_logp;
    p.g_value = q.g_value;
    p.g_entropy = q.g_entropy;
    p.out = q.out;
    p.out_f32 = q.out_f32;
    p.slot = reinterpret_cast<SlotHeader*>(q.workspace);
  };
  const XchgView* xv = xchg_view(xchg);
  SRL_REQUIRE(xchg == nullptr || (xv != nullptr && lane_aos != nullptr && xv->cap >= 3 * kMaxBatch), SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_fwd_bwd_batched: the in-kernel exchange needs a connected srl_xchg of >= %d doubles and the "
              "self-computed statistics (lane_aos)", 3 * kMaxBatch);
  for (int k = 0; k < n_problems && xv != nullptr; ++k)
    SRL_REQUIRE(problems[k].out != nullptr, SRL_ERR_INVALID_ARG,
                "srl_ppo_loss_fwd_bwd_batched: the in-kernel exchange needs immediate finalisation (out != NULL): the last CTA "
                "of each problem ends the exchange round");
  for (int k0 = 0; k0 < n_problems; k0 += kMaxBatch) {
    const int nb = n_problems - k0 < kMaxBatch ? n_problems - k0 : kMaxBatch;
    LossBatch b;
    b.s = s;
    b.s.part_first = part_first + k0;
    if (xv != nullptr && xv->world > 1) {
      b.xv = *xv;
    } else {
      memset(&b.xv, 0, sizeof(b.xv));
    }
    for (int k = 0; k < kMaxBatch; ++k) fill(b.prob[k], problems[k0 + (k < nb ? k : 0)]);
    if (mode == kPack && pair)
      rc = launch_loss_pair(b, nb, st);
    else if (mode == kPack)
      rc = launch_loss_pack(b, nb, dense_ok, st);
    else if (mode == kDense)
      rc = launch_loss_dense(b, nb, dense_ok, st);
    else
      rc = launch_loss_gather(b, nb, dense_ok, st);
    if (rc != SRL_OK) return rc;
  }
  return SRL_OK;
}

extern "C" int srl_ppo_loss_fwd_bwd(const float* new_logp, const float* v_pred, const float* entropy, int64_t ld_pol,
                                    const float* old_logp, const float* old_value, const float* ret,
                                    const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                    const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                    const double* local_stats, const double* popart_mean_std,
                                    const srl_ppo_hyper* hyper, float* g_logp, float* g_value, float* g_entropy,
                                    int64_t ld_grad, double* out, float* out_f32, void* workspace,
                                    size_t workspace_bytes, srl_stream_t stream) {
  srl_loss_problem q;
  q.new_logp = new_logp;
  q.v_pred = v_pred;
  q.entropy = entropy;
  q.lane_idx = lane_idx;
  q.norm_stats = norm_stats;
  q.local_stats = local_stats;
  q.g_logp = g_logp;
  q.g_value = g_value;
  q.g_entropy = g_entropy;
  q.out = out;
  q.out_f32 = out_f32;
  q.workspace = workspace;
  return srl_ppo_loss_fwd_bwd_batched(&q, 1, ld_pol, ld_grad, old_logp, old_value, ret, adv, on_reset_next, ld_smp,
                                      nullptr, 0, nullptr, nullptr, 0, 0, T, n, popart_mean_std, hyper, workspace_bytes, nullptr,
                                      stream);
}

extern "C" int srl_ppo_loss_from_logits(const float* logits, const int32_t* action, const int32_t* head_sizes_host,
                                        int heads, const float* v_pred, const float* old_logp,
                                        const float* old_value, const float* ret, const float* adv,
                                        const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T,
                                        int n, const double* norm_stats, const double* local_stats,
                                        const double* popart_mean_std, const srl_ppo_hyper* hyper, float* g_logits,
                                        float* g_value, float* logp_out, float* entropy_out, double* out,
                                        float* out_f32, void* workspace, size_t workspace_bytes,
                                        srl_stream_t stream) {
  return srl::loss::ppo_loss_from_logits("srl_ppo_loss_from_logits", sizeof(float), logits, nullptr, action, head_sizes_host,
                                         heads, v_pred, old_logp, old_value, ret, adv, on_reset_next, ld_smp, lane_idx, T, n,
                                         norm_stats, local_stats, popart_mean_std, hyper, g_logits, g_value, logp_out,
                                         entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_logits_masked(const float* logits, const uint8_t* available, const int32_t* action,
                                               const int32_t* head_sizes_host, int heads, const float* v_pred,
                                               const float* old_logp, const float* old_value, const float* ret,
                                               const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                               const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                               const double* local_stats, const double* popart_mean_std,
                                               const srl_ppo_hyper* hyper, float* g_logits, float* g_value,
                                               float* logp_out, float* entropy_out, double* out, float* out_f32,
                                               void* workspace, size_t workspace_bytes, srl_stream_t stream) {
  SRL_REQUIRE(available != nullptr, SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_from_logits_masked: null pointer available (use srl_ppo_loss_from_logits without a mask)");
  return srl::loss::ppo_loss_from_logits("srl_ppo_loss_from_logits_masked", sizeof(float), logits, available, action,
                                         head_sizes_host, heads, v_pred, old_logp, old_value, ret, adv, on_reset_next, ld_smp,
                                         lane_idx, T, n, norm_stats, local_stats, popart_mean_std, hyper, g_logits, g_value,
                                         logp_out, entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_logits_bf16(const uint16_t* logits, const int32_t* action, const int32_t* head_sizes_host,
                                             int heads, const uint16_t* v_pred, const float* old_logp,
                                             const float* old_value, const float* ret, const float* adv,
                                             const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T,
                                             int n, const double* norm_stats, const double* local_stats,
                                             const double* popart_mean_std, const srl_ppo_hyper* hyper, uint16_t* g_logits,
                                             uint16_t* g_value, float* logp_out, float* entropy_out, double* out,
                                             float* out_f32, void* workspace, size_t workspace_bytes,
                                             srl_stream_t stream) {
  return srl::loss::ppo_loss_from_logits("srl_ppo_loss_from_logits_bf16", sizeof(__nv_bfloat16), logits, nullptr, action,
                                         head_sizes_host, heads, v_pred, old_logp, old_value, ret, adv, on_reset_next, ld_smp,
                                         lane_idx, T, n, norm_stats, local_stats, popart_mean_std, hyper, g_logits, g_value,
                                         logp_out, entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}

extern "C" int srl_ppo_loss_from_logits_masked_bf16(const uint16_t* logits, const uint8_t* available, const int32_t* action,
                                                    const int32_t* head_sizes_host, int heads, const uint16_t* v_pred,
                                                    const float* old_logp, const float* old_value, const float* ret,
                                                    const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                                    const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                                    const double* local_stats, const double* popart_mean_std,
                                                    const srl_ppo_hyper* hyper, uint16_t* g_logits, uint16_t* g_value,
                                                    float* logp_out, float* entropy_out, double* out, float* out_f32,
                                                    void* workspace, size_t workspace_bytes, srl_stream_t stream) {
  SRL_REQUIRE(available != nullptr, SRL_ERR_INVALID_ARG,
              "srl_ppo_loss_from_logits_masked_bf16: null pointer available (use srl_ppo_loss_from_logits_bf16 without a "
              "mask)");
  return srl::loss::ppo_loss_from_logits("srl_ppo_loss_from_logits_masked_bf16", sizeof(__nv_bfloat16), logits, available,
                                         action, head_sizes_host, heads, v_pred, old_logp, old_value, ret, adv, on_reset_next,
                                         ld_smp, lane_idx, T, n, norm_stats, local_stats, popart_mean_std, hyper, g_logits,
                                         g_value, logp_out, entropy_out, out, out_f32, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}
