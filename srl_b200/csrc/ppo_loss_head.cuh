// The per-transition head losses K4c (Gaussian, ppo_loss_gaussian.cu) and K4d (Beta, ppo_loss_beta.cu): one kernel, one
// launch rule and one host setup, generic over the head's per-dimension math.
//
// A head has two [T*n, D] parameter blocks P0 and P1 of the element type T (mean / log_std, concentration1 /
// concentration0) and a float32 [T*n, D] action block; the loss is K4's element<RuntimeCfg>, unchanged.  The head struct
// supplies the math only:
//   Row                          the running sums of one transition over its D dimensions
//   row_begin(ls_sum)            an empty Row (ls_sum: the Gaussian's sum_d s_d when log_std is shared)
//   row_term<SHARED, T>(...)     add dimension d of the row's staged elements; may leave a value for the column pass in
//                                the staged P1 slot (the Gaussian's 1 / sigma^2)
//   row_end(row, D, logp, H)     the transition's log-prob and entropy, rounded to float once
//   column<SHARED, T>(...)       d loss / d P0 and d loss / d P1 of one (row, d) element, in place of the staged P0 / P1
// and kShared: whether P1 may be ONE [D] float vector for every transition (the Gaussian's state-independent log_std;
// its gradient is then folded across the CTAs of the grid, see below).  SHARED is a template parameter, so a head
// without it has no such branch in its code.
//
// Structure (K4b's, ppo_loss.cu): a CTA takes 256 consecutive transitions; the [256, D] blocks of P0, action and a
// per-row P1 are contiguous in global memory and arrive by one bulk copy each on one mbarrier while the sample side
// is loaded; the gradients are written back in place and leave by bulk copy.  The last, partial tile and pointers that
// are not 16-byte aligned are staged element by element.  Two passes over the staged tile:
//  * per row (thread t owns transition t): the two sums over d, then element() -- the row walk starts at column t % D,
//    so that the 32 rows a warp reads at once spread over the banks (about 2 words per bank and step for 4- and 2-byte
//    elements alike; more where D + 1 is a multiple of 8, up to 32 at D = 63: DESIGN.md section 4);
//  * per column (thread (k, d) owns column d of the rows k, k + K, ..., K = 256 / D): the two gradients -- consecutive
//    threads touch consecutive words, and with a shared P1 each thread adds its column's terms in float64 across all
//    its tiles (one register, no per-thread [D] array).
// The shared P1 gradient: the (k, d) accumulators are added in k order through shared memory into one float64 [D]
// row per CTA, stored as self-validating words (ppo_loss.cuh: box / unbox; 0 = "not there yet") after the K4 slot of the
// workspace; CTA 0 waits for every row, adds them in CTA order and clears them -- in both finalisation modes, so the [D]
// gradient is complete when the launch is.  The wait ends because the grid is one resident wave (launch_head_wave:
// never more CTAs than the SMs hold at once).  Deterministic for a given launch shape; no floating-point atomics.
//
// The policy side (P0, a per-row P1, v_pred and their gradients) is float or bfloat16, the kernel's element type T.  The
// staged P0 and P1 blocks hold T, the action block stays float (the sampled actions, never rounded); each element is
// widened where it is read and all arithmetic is the float32 entry's, so a bfloat16 launch computes what the float32 one
// computes on the widened values, with each gradient rounded to bfloat16 once.  A shared [D] P1 and its gradient are
// float for both types.
#pragma once

#include <type_traits>

#include "ppo_loss.cuh"
#include "tma_util.cuh"

namespace srl {
namespace loss {
namespace {

constexpr int kHeadMaxD = 64;
constexpr int kGStage = 8;      // manual staging batch per thread (last, partial tile only)
constexpr int kGFoldBatch = 8;  // rows CTA 0 reads at once per thread while it folds

// pr.v_pred and pr.g_value point at T (Problem is K4's struct, typed float)
struct HeadParams {
  LossShared s;
  Problem pr;                      // new_logp / entropy / g_logp / g_entropy are unused here
  const void* p0;                  // [T*n, D] of T
  const void* p1;                  // [T*n, D] of T, or [D] float (shared)
  const float* action;             // [T*n, D]
  void* g0;                        // [T*n, D] of T
  void* g1;                        // [T*n, D] of T, or [D] float (shared)
  float* logp_out;                 // [T*n] or null
  float* entropy_out;              // [T*n] or null
  unsigned long long* ls_rows;     // shared P1: [gridDim.x][D] boxed float64 partial rows (workspace after the slot)
  int D;
};

template <typename E>
__device__ __forceinline__ void stage_in(E* __restrict__ dst, const E* __restrict__ src, int total) {
  for (int e0 = threadIdx.x; e0 < total; e0 += 256 * kGStage) {
    E v[kGStage];
#pragma unroll
    for (int b = 0; b < kGStage; ++b) v[b] = (e0 + b * 256 < total) ? ldg_stream(src + e0 + b * 256) : from_float<E>(0.f);
#pragma unroll
    for (int b = 0; b < kGStage; ++b)
      if (e0 + b * 256 < total) dst[e0 + b * 256] = v[b];
  }
}

template <typename E>
__device__ __forceinline__ void stage_out(E* __restrict__ dst, const E* __restrict__ src, int total) {
  for (int e0 = threadIdx.x; e0 < total; e0 += 256 * kGStage) {
    E v[kGStage];
#pragma unroll
    for (int b = 0; b < kGStage; ++b) v[b] = (e0 + b * 256 < total) ? src[e0 + b * 256] : from_float<E>(0.f);
#pragma unroll
    for (int b = 0; b < kGStage; ++b)
      if (e0 + b * 256 < total) stg_stream(dst + e0 + b * 256, v[b]);
  }
}

// PACK: the sample side is K2's loss pack (load_pack_item, ppo_loss.cuh), else the five leaves.
template <typename Head, bool SHARED, typename T, bool PACK>
__global__ void __launch_bounds__(256, 2) ppo_loss_head_kernel(const __grid_constant__ HeadParams q) {
  static_assert(Head::kShared || !SHARED, "this head has no shared [D] parameter");
  // [256 * D] P0 of T, [256 * D] action floats (, [256 * D] P1 of T per row), then the mbarrier; every block is a
  // multiple of 16 bytes
  extern __shared__ __align__(128) float sblk[];
  constexpr int kElem = sizeof(T);
  __shared__ float s_glp[256], s_gen[256];  // the rows' d loss / d logp and d loss / d H, for the column pass
  __shared__ float s_ls[kHeadMaxD];   // shared P1: s_d
  __shared__ double s_iv[kHeadMaxD];  // shared P1: 1 / sigma_d^2 = exp(-2 s_d), in float64 (D exponentials per CTA)
  __shared__ double s_red[256];
  const LossShared& p = q.s;
  const Problem& pr = q.pr;
  const LossHyperDev& h = p.h;
  double mask_sum;
  const Uniforms u = load_uniforms(pr.norm_stats, pr.local_stats, p.popart, h.adv_eps, mask_sum);
  Acc acc;
  const int D = q.D;
  // offsets in floats: a [256 * D] block of T is 64 * kElem * D of them, the action block 256 * D
  T* smu = reinterpret_cast<T*>(sblk);
  float* sac = sblk + 64 * kElem * D;
  T* sls = reinterpret_cast<T*>(sblk + (64 * kElem + 256) * D);  // per-row P1 only
  uint64_t* bar = reinterpret_cast<uint64_t*>(sblk + (SHARED ? 64 * kElem + 256 : 128 * kElem + 256) * D);
  if (threadIdx.x == 0) {
    tma::mbar_init(bar, 1);
    tma::mbar_fence_init();
  }
  if (SHARED && static_cast<int>(threadIdx.x) < D) {
    const float s = __ldg(static_cast<const float*>(q.p1) + threadIdx.x);
    s_ls[threadIdx.x] = s;
    s_iv[threadIdx.x] = exp(-2.0 * static_cast<double>(s));
  }
  __syncthreads();
  // row pass: this thread's first column; column pass: this thread's column and first row, K rows apart
  const int d0 = static_cast<int>(threadIdx.x) % D;
  const int K = 256 / D;
  const int kc = static_cast<int>(threadIdx.x) / D;
  const bool col_thread = kc < K;
  double ls_sum = 0.0;  // shared P1: sum_d s_d
  double iv_cd = 0.0;   // shared P1: this thread's column's 1 / sigma^2
  if (SHARED) {
    for (int d = 0; d < D; ++d) ls_sum += static_cast<double>(s_ls[d]);
    iv_cd = s_iv[d0];
  }
  const float iv_c = static_cast<float>(iv_cd);
  double g_acc = 0.0;  // shared P1: this thread's column's gradient terms
  uint32_t parity = 0;
  uintptr_t align_bits = reinterpret_cast<uintptr_t>(q.p0) | reinterpret_cast<uintptr_t>(q.action) |
                         reinterpret_cast<uintptr_t>(q.g0);
  if (!SHARED) align_bits |= reinterpret_cast<uintptr_t>(q.p1) | reinterpret_cast<uintptr_t>(q.g1);
  const bool bulk_ok = (align_bits & 15) == 0;
  const long long W = static_cast<long long>(p.T) * p.n;
  const long long tiles = (W + 255) / 256;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long i0 = tile * 256;
    const int cnt = static_cast<int>(min(256ll, W - i0));
    const int total = cnt * D;
    const long long e0 = i0 * D;
    // 256 * D * kElem (and * 4) bytes: multiples of 16 at 16-byte aligned addresses
    const bool bulk = bulk_ok && cnt == 256;
    if (bulk) {
      if (threadIdx.x == 0) {
        const uint32_t bytes = static_cast<uint32_t>(total) * kElem;  // a block of T
        const uint32_t abytes = static_cast<uint32_t>(total) * 4u;    // the action block
        tma::mbar_expect_tx(bar, static_cast<uint32_t>(total) * ((SHARED ? 1u : 2u) * kElem + 4u));
        tma::bulk_load(smu, static_cast<const T*>(q.p0) + e0, bytes, bar);
        tma::bulk_load(sac, q.action + e0, abytes, bar);
        if (!SHARED) tma::bulk_load(sls, static_cast<const T*>(q.p1) + e0, bytes, bar);
      }
    } else {
      stage_in(smu, static_cast<const T*>(q.p0) + e0, total);
      stage_in(sac, q.action + e0, total);
      if (!SHARED) stage_in(sls, static_cast<const T*>(q.p1) + e0, total);
    }
    // the sample side of this thread's transition, in flight while the blocks land
    const bool mine = static_cast<int>(threadIdx.x) < cnt;
    const long long i = i0 + threadIdx.x;
    float vp = 0.f, ol = 0.f, rt = 0.f, ad = 0.f, ov = 0.f;
    bool valid = false;
    if (mine) {
      const int t = static_cast<int>(i / p.n);
      const int j = static_cast<int>(i - static_cast<long long>(t) * p.n);
      const int c = pr.lane_idx ? pr.lane_idx[j] : j;
      if constexpr (PACK) {
        vp = to_float(ldg_stream(reinterpret_cast<const T*>(pr.v_pred) + i));
        load_pack_item(p, t, c, ol, ov, rt, ad, valid);
      } else {
        const long long os = t * p.ld_smp + c;
        vp = to_float(ldg_stream(reinterpret_cast<const T*>(pr.v_pred) + i));
        ol = __ldg(p.old_logp + os), rt = __ldg(p.ret + os), ad = __ldg(p.adv + os);
        ov = h.clip_value ? __ldg(p.old_value + os) : 0.f;
        valid = __ldg(p.reset_next + os) == 0;
      }
    }
    if (bulk) {
      tma::mbar_wait(bar, parity);
      parity ^= 1u;
    } else {
      __syncthreads();
    }
    // ---- row pass: log-prob and entropy of this thread's transition, then the loss element ----
    if (mine) {
      const int rb = static_cast<int>(threadIdx.x) * D;
      typename Head::Row row = Head::row_begin(SHARED ? ls_sum : 0.0);
      int d = d0;
      for (int k = 0; k < D; ++k) {
        Head::template row_term<SHARED>(row, sac, smu, sls, rb + d, s_iv, d);
        d = (d + 1 == D) ? 0 : d + 1;
      }
      float logp, ent;
      Head::row_end(row, D, logp, ent);
      float g_lp, g_v, g_en;
      RowSums rs;
      element<RuntimeCfg>(h, u, logp, vp, ent, ol, ov, rt, ad, valid, g_lp, g_v, g_en, rs);
      acc.add(rs);
      stg_stream(reinterpret_cast<T*>(pr.g_value) + i, from_float<T>(g_v));
      if (q.logp_out) q.logp_out[i] = logp;
      if (q.entropy_out) q.entropy_out[i] = ent;
      s_glp[threadIdx.x] = g_lp;
      s_gen[threadIdx.x] = g_en;
    }
    __syncthreads();
    // ---- column pass: d loss / d P0 in place of P0, d loss / d P1 in place of P1 (per row) ----
    if (col_thread) {
      int idx = static_cast<int>(threadIdx.x);
      for (int r = kc; r < cnt; r += K, idx += K * D)
        Head::template column<SHARED>(sac, smu, sls, idx, s_glp[r], s_gen[r], iv_c, iv_cd, g_acc);
    }
    if (bulk) {
      tma::fence_proxy_async_smem();  // the gradients above, before the bulk copies read them
      __syncthreads();
      if (threadIdx.x == 0) {
        const uint32_t bytes = static_cast<uint32_t>(total) * kElem;
        tma::bulk_store(static_cast<T*>(q.g0) + e0, smu, bytes);  // read before the next tile
        if (!SHARED) tma::bulk_store(static_cast<T*>(q.g1) + e0, sls, bytes);
      }
      __syncthreads();
    } else {
      __syncthreads();
      stage_out(static_cast<T*>(q.g0) + e0, smu, total);
      if (!SHARED) stage_out(static_cast<T*>(q.g1) + e0, sls, total);
      __syncthreads();
    }
  }
  if (SHARED) {
    // this CTA's [D] row: the K accumulators of each column added in k order
    s_red[threadIdx.x] = g_acc;
    __syncthreads();
    if (static_cast<int>(threadIdx.x) < D) {
      double s = 0.0;
      for (int k = 0; k < K; ++k) s += s_red[k * D + threadIdx.x];
      reinterpret_cast<volatile unsigned long long*>(q.ls_rows)[static_cast<size_t>(blockIdx.x) * D + threadIdx.x] = box(s);
    }
  }
  reduce_and_finalize(pr, h, acc, mask_sum, blockIdx.x, gridDim.x);
  if (!SHARED || blockIdx.x != 0) return;
  // CTA 0 folds the rows: thread (k, d) adds the rows k, k + K, ... of column d in order, waiting for each word to appear
  // and clearing it behind itself; then the K sums of a column are added in k order.  Every CTA of the grid is resident
  // (one wave), so the wait ends; its bound is the pair kernel's (ppo_loss_pair.cu), after which the result is NaN.
  double s = 0.0;
  if (col_thread) {
    volatile unsigned long long* rows = q.ls_rows;
    const long long limit = 2 * kDefaultSpinLimit;
    const long long t0 = clock64();
    const int n_rows = static_cast<int>(gridDim.x);
    for (int r0 = kc; r0 < n_rows; r0 += K * kGFoldBatch) {
      unsigned long long w[kGFoldBatch];
      bool all = false, ok = true;
      while (!all) {
        all = true;
#pragma unroll
        for (int b = 0; b < kGFoldBatch; ++b) {
          const int r = r0 + K * b;
          w[b] = r < n_rows ? rows[static_cast<size_t>(r) * D + d0] : 1ull;
          all = all && w[b] != 0ull;
        }
        if (!all && clock64() - t0 > limit) {
          ok = false;
          break;
        }
      }
#pragma unroll
      for (int b = 0; b < kGFoldBatch; ++b) {
        const int r = r0 + K * b;
        if (r < n_rows) {
          s += ok ? unbox(w[b]) : __longlong_as_double(0x7ff8000000000000ll);  // a CTA never arrived: NaN
          rows[static_cast<size_t>(r) * D + d0] = 0ull;
        }
      }
    }
  }
  __syncthreads();  // s_red's last readers (the row above) are done
  s_red[threadIdx.x] = s;
  __syncthreads();
  if (static_cast<int>(threadIdx.x) < D) {
    double g = 0.0;
    for (int k = 0; k < K; ++k) g += s_red[k * D + threadIdx.x];
    static_cast<float*>(q.g1)[threadIdx.x] = static_cast<float>(g);
  }
}

// one resident wave of ppo_loss_head_kernel<Head, SHARED, T, PACK> over the T * n transitions of q
template <typename Head, bool SHARED, typename T, bool PACK>
int launch_head_wave(const HeadParams& q, size_t smem, cudaStream_t stream) {
  int rc;
  auto kern = ppo_loss_head_kernel<Head, SHARED, T, PACK>;
  if ((rc = opt_in_smem<ppo_loss_head_kernel<Head, SHARED, T, PACK>>(200 * 1024)) != SRL_OK) return rc;
  const long long tiles = (static_cast<long long>(q.s.T) * q.s.n + 255) / 256;
  // ONE resident wave, as srl_ppo_loss_from_logits sizes its grid: as many CTAs as the SMs hold at once with this much
  // shared memory, at most kMaxGrid.  With a shared P1 this is also what makes CTA 0's wait for the other CTAs' rows
  // finite -- keep the grid within the resident capacity.
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  const long long slots = static_cast<long long>(sm_count()) * per_sm;
  const long long cap = slots < kMaxGrid ? slots : kMaxGrid;
  // every CTA the same number of tiles
  const long long per_cta = (tiles + cap - 1) / cap;
  const int grid = static_cast<int>((tiles + per_cta - 1) / per_cta);
  kern<<<grid, 256, smem, stream>>>(q);
  SRL_CUDA(cudaGetLastError());
  return SRL_OK;
}

template <typename Head, typename T, bool PACK>
int launch_head(const HeadParams& q, bool shared, size_t smem, cudaStream_t stream) {
  if constexpr (Head::kShared) {
    if (shared) return launch_head_wave<Head, true, T, PACK>(q, smem, stream);
  }
  return launch_head_wave<Head, false, T, PACK>(q, smem, stream);
}

// The workspace of a head loss: a K4 slot, then (shared P1) the float64 partial rows of its gradient.
inline size_t head_workspace_bytes(int T, int n, int D, bool shared) {
  const size_t slot = srl_ppo_loss_workspace_bytes(T, n);
  if (!shared || D < 1) return slot;
  return slot + static_cast<size_t>(kMaxGrid) * static_cast<size_t>(D) * sizeof(double);
}

// The leaf entries (elem_bytes = 4: float32, 2: bfloat16 policy side) and the pack entries (pack != NULL: the sample side
// is K2's pack, ld_smp its lanes, pack_row_lo the absolute row of loss row 0; the five leaves are not read) of a head.
// Head::kNames are the argument names of P0, P1, g0 and g1 in the messages.
template <typename Head>
int ppo_loss_from_head(const char* fn, size_t elem_bytes, const void* p0, const void* p1, bool shared,
                       const float* action, int D, const void* v_pred, const float* old_logp, const float* old_value,
                       const float* ret, const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                       const float* pack, int pack_row_lo, const int32_t* lane_idx, int T, int n,
                       const double* norm_stats, const double* local_stats, const double* popart_mean_std,
                       const srl_ppo_hyper* hyper, void* g0, void* g1, void* g_value, float* logp_out,
                       float* entropy_out, double* out, float* out_f32, void* workspace, size_t workspace_bytes,
                       cudaStream_t stream) {
  SRL_REQUIRE(T >= 1 && n >= 1, SRL_ERR_INVALID_ARG, "%s: need T >= 1 and n >= 1 (got %d, %d)", fn, T, n);
  SRL_REQUIRE(D >= 1 && D <= kHeadMaxD, SRL_ERR_INVALID_ARG, "%s: D=%d action dimensions outside [1, %d]", fn, D,
              kHeadMaxD);
  const void* pk = pack;  // the pack form reads no leaf: the pack stands in for the four in the null test
  const struct {
    const void* p;
    const char* name;
  } required[] = {{p0, Head::kNames[0]},   {p1, Head::kNames[1]},    {action, "action"},     {v_pred, "v_pred"},
                  {pk ? pk : old_logp, "old_logp"}, {pk ? pk : ret, "ret"}, {pk ? pk : adv, "adv"},
                  {pk ? pk : on_reset_next, "on_reset_next"},
                  {norm_stats, "norm_stats"}, {local_stats, "local_stats"}, {g0, Head::kNames[2]}, {g1, Head::kNames[3]},
                  {g_value, "g_value"},   {workspace, "workspace"}};
  for (const auto& r : required) SRL_REQUIRE(r.p != nullptr, SRL_ERR_INVALID_ARG, "%s: null pointer %s", fn, r.name);
  SRL_REQUIRE(ld_smp >= (lane_idx ? 1 : n), SRL_ERR_INVALID_ARG, "%s: %s=%lld smaller than the row", fn,
              pack ? "pack_lanes" : "ld_smp", static_cast<long long>(ld_smp));
  const size_t need = head_workspace_bytes(T, n, D, shared);
  SRL_REQUIRE(workspace_bytes >= need, SRL_ERR_INVALID_ARG, "%s: workspace too small (%zu bytes, need %zu)", fn,
              workspace_bytes, need);
  HeadParams q;
  int rc = fill_loss_hyper(hyper, popart_mean_std, q.s.h);
  if (rc != SRL_OK) return rc;
  SRL_REQUIRE(pack || !(q.s.h.clip_value && old_value == nullptr), SRL_ERR_INVALID_ARG, "%s: clip_value needs old_value",
              fn);
  const size_t blk_bytes = static_cast<size_t>(256) * D * elem_bytes;  // one dense [256, D] block of the element type
  const size_t act_bytes = static_cast<size_t>(256) * D * sizeof(float);  // the [256, D] action block
  const size_t smem = (shared ? 1 : 2) * blk_bytes + act_bytes + 16;     // + the mbarrier of the bulk copies
  SRL_REQUIRE(smem <= 200 * 1024, SRL_ERR_UNSUPPORTED, "%s: D = %d too wide for shared memory", fn, D);
  q.p0 = p0;
  q.p1 = p1;
  q.action = action;
  q.g0 = g0;
  q.g1 = g1;
  q.logp_out = logp_out;
  q.entropy_out = entropy_out;
  q.ls_rows = shared ? reinterpret_cast<unsigned long long*>(static_cast<unsigned char*>(workspace) +
                                                              srl_ppo_loss_workspace_bytes(T, n))
                     : nullptr;
  q.D = D;
  LossShared& p = q.s;
  p.old_logp = old_logp;
  p.old_value = old_value;
  p.ret = ret;
  p.adv = adv;
  p.reset_next = on_reset_next;
  p.pack = reinterpret_cast<const float4*>(pack);
  p.lane_aos = nullptr;
  p.part = nullptr;
  p.part_ctas = p.part_first = 0;
  p.row_lo = pack ? pack_row_lo : 0;
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
  const bool bf16 = elem_bytes == sizeof(__nv_bfloat16);
  if (pack) return bf16 ? launch_head<Head, __nv_bfloat16, true>(q, shared, smem, stream)
                        : launch_head<Head, float, true>(q, shared, smem, stream);
  return bf16 ? launch_head<Head, __nv_bfloat16, false>(q, shared, smem, stream)
              : launch_head<Head, float, false>(q, shared, smem, stream);
}

// The pack entries' own checks, before ppo_loss_from_head's.
inline int check_head_pack(const char* fn, int elem_bytes, const float* pack, int pack_row_lo,
                           const int32_t* lane_idx, int64_t pack_lanes, int n) {
  SRL_REQUIRE(elem_bytes == 4 || elem_bytes == 2, SRL_ERR_INVALID_ARG, "%s: elem_bytes=%d, need 4 (float32) or 2 (bfloat16)",
              fn, elem_bytes);
  SRL_REQUIRE(pack != nullptr && aligned(pack, 16), SRL_ERR_INVALID_ARG, "%s: pack is null or not 16-byte aligned", fn);
  SRL_REQUIRE(pack_row_lo >= 0, SRL_ERR_INVALID_ARG, "%s: pack_row_lo=%d < 0", fn, pack_row_lo);
  SRL_REQUIRE(lane_idx != nullptr || pack_lanes >= n, SRL_ERR_INVALID_ARG,
              "%s: pack_lanes=%lld < n=%d without lane_idx", fn, static_cast<long long>(pack_lanes), n);
  return SRL_OK;
}

}  // namespace
}  // namespace loss
}  // namespace srl
