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
// Structure (K4b's, ppo_loss.cu): a CTA takes 256 consecutive transitions; the [256, D] blocks of mean, action and a
// per-row log_std are contiguous in global memory and arrive by one bulk copy each on one mbarrier while the sample side
// is loaded; the gradients are written back in place and leave by bulk copy.  The last, partial tile and pointers that
// are not 16-byte aligned are staged element by element.  Two passes over the staged tile:
//  * per row (thread t owns transition t): the two sums over d, then element() -- the row walk starts at column t % D,
//    so that the 32 rows a warp reads at once spread over the banks (about 2 words per bank and step for 4- and 2-byte
//    elements alike; more where D + 1 is a multiple of 8, up to 32 at D = 63: DESIGN.md section 4);
//  * per column (thread (k, d) owns column d of the rows k, k + K, ..., K = 256 / D): the two gradients -- consecutive
//    threads touch consecutive words, and with a shared log_std each thread adds its column's terms in float64 across all
//    its tiles (one register, no per-thread [D] array).
// The shared log_std gradient: the (k, d) accumulators are added in k order through shared memory into one float64 [D]
// row per CTA, stored as self-validating words (ppo_loss.cuh: box / unbox; 0 = "not there yet") after the K4 slot of the
// workspace; CTA 0 waits for every row, adds them in CTA order and clears them -- in both finalisation modes, so the [D]
// gradient is complete when the launch is.  The wait ends because the grid is one resident wave (the sizing rule in
// srl_ppo_loss_from_gaussian: never more CTAs than the SMs hold at once).  Deterministic for a given launch shape; no
// floating-point atomics.
//
// The policy side (mean, a per-row log_std, v_pred and their gradients) is float or bfloat16, the kernel's element type T
// (srl_ppo_loss_from_gaussian_bf16: a policy under torch.autocast).  The staged mean and log_std blocks hold T, the action
// block stays float (the sampled actions, never rounded); each element is widened where it is read and all arithmetic is
// the float32 entry's, so a bfloat16 launch computes what the float32 one computes on the widened values, with each
// gradient rounded to bfloat16 once.  A shared [D] log_std and its gradient are float for both types.  One difference in
// the passes: the float row pass leaves 1 / sigma^2 in the staged log_std slot for the column pass; a bfloat16 slot would
// round it, so there the column pass recomputes expf(-2 s) from the staged s -- the same expression on the same float.
#include <type_traits>

#include "ppo_loss.cuh"
#include "tma_util.cuh"

namespace srl {
namespace loss {
namespace {

constexpr int kMaxD = 64;
constexpr double kLogSqrt2Pi = 0.918938533204672742;  // log(sqrt(2 pi))
constexpr int kGStage = 8;                            // manual staging batch per thread (last, partial tile only)
constexpr int kGFoldBatch = 8;                        // rows CTA 0 reads at once per thread while it folds

// pr.v_pred and pr.g_value point at T (Problem is K4's struct, typed float)
struct GaussianParams {
  LossShared s;
  Problem pr;                      // new_logp / entropy / g_logp / g_entropy are unused here
  const void* mean;                // [T*n, D] of T
  const void* log_std;             // [T*n, D] of T, or [D] float
  const float* action;             // [T*n, D]
  void* g_mean;                    // [T*n, D] of T
  void* g_log_std;                 // [T*n, D] of T, or [D] float
  float* logp_out;                 // [T*n] or null
  float* entropy_out;              // [T*n] or null
  unsigned long long* ls_rows;     // shared log_std: [gridDim.x][D] boxed float64 partial rows (workspace after the slot)
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

template <bool SHARED, typename T>
__global__ void __launch_bounds__(256, 2) ppo_loss_gaussian_kernel(const __grid_constant__ GaussianParams q) {
  // [256 * D] mean of T, [256 * D] action floats (, [256 * D] log_std of T per row), then the mbarrier; every block is a
  // multiple of 16 bytes
  extern __shared__ __align__(128) float sblk[];
  constexpr int kElem = sizeof(T);
  constexpr bool kF32 = std::is_same<T, float>::value;
  __shared__ float s_glp[256], s_gen[256];  // the rows' d loss / d logp and d loss / d H, for the column pass
  __shared__ float s_ls[kMaxD];   // shared log_std: s_d
  __shared__ double s_iv[kMaxD];  // shared log_std: 1 / sigma_d^2 = exp(-2 s_d), in float64 (D exponentials per CTA)
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
  T* sls = reinterpret_cast<T*>(sblk + (64 * kElem + 256) * D);  // per-row log_std only
  uint64_t* bar = reinterpret_cast<uint64_t*>(sblk + (SHARED ? 64 * kElem + 256 : 128 * kElem + 256) * D);
  if (threadIdx.x == 0) {
    tma::mbar_init(bar, 1);
    tma::mbar_fence_init();
  }
  if (SHARED && static_cast<int>(threadIdx.x) < D) {
    const float s = __ldg(static_cast<const float*>(q.log_std) + threadIdx.x);
    s_ls[threadIdx.x] = s;
    s_iv[threadIdx.x] = exp(-2.0 * static_cast<double>(s));
  }
  __syncthreads();
  // row pass: this thread's first column; column pass: this thread's column and first row, K rows apart
  const int d0 = static_cast<int>(threadIdx.x) % D;
  const int K = 256 / D;
  const int kc = static_cast<int>(threadIdx.x) / D;
  const bool col_thread = kc < K;
  double ls_sum = 0.0;  // shared log_std: sum_d s_d
  double iv_cd = 0.0;   // shared log_std: this thread's column's 1 / sigma^2
  if (SHARED) {
    for (int d = 0; d < D; ++d) ls_sum += static_cast<double>(s_ls[d]);
    iv_cd = s_iv[d0];
  }
  const float iv_c = static_cast<float>(iv_cd);
  double g_acc = 0.0;  // shared log_std: this thread's column's gradient terms
  uint32_t parity = 0;
  uintptr_t align_bits = reinterpret_cast<uintptr_t>(q.mean) | reinterpret_cast<uintptr_t>(q.action) |
                         reinterpret_cast<uintptr_t>(q.g_mean);
  if (!SHARED) align_bits |= reinterpret_cast<uintptr_t>(q.log_std) | reinterpret_cast<uintptr_t>(q.g_log_std);
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
        tma::bulk_load(smu, static_cast<const T*>(q.mean) + e0, bytes, bar);
        tma::bulk_load(sac, q.action + e0, abytes, bar);
        if (!SHARED) tma::bulk_load(sls, static_cast<const T*>(q.log_std) + e0, bytes, bar);
      }
    } else {
      stage_in(smu, static_cast<const T*>(q.mean) + e0, total);
      stage_in(sac, q.action + e0, total);
      if (!SHARED) stage_in(sls, static_cast<const T*>(q.log_std) + e0, total);
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
      const long long os = t * p.ld_smp + c;
      vp = to_float(ldg_stream(reinterpret_cast<const T*>(pr.v_pred) + i));
      ol = __ldg(p.old_logp + os), rt = __ldg(p.ret + os), ad = __ldg(p.adv + os);
      ov = h.clip_value ? __ldg(p.old_value + os) : 0.f;
      valid = __ldg(p.reset_next + os) == 0;
    }
    if (bulk) {
      tma::mbar_wait(bar, parity);
      parity ^= 1u;
    } else {
      __syncthreads();
    }
    // ---- row pass: log-prob and entropy of this thread's transition, then the loss element ----
    if (mine) {
      // the two sums in float64, rounded once: the loss sees logp through exp(logp - old_logp), and a float32 sum of
      // D = 64 terms of a |logp| ~ 100 is off by ~1e-5 -- the ratio's whole error budget
      const int rb = static_cast<int>(threadIdx.x) * D;
      double sq = 0.0, ssum = SHARED ? ls_sum : 0.0;
      int d = d0;
      for (int k = 0; k < D; ++k) {
        const double diff = static_cast<double>(sac[rb + d]) - static_cast<double>(to_float(smu[rb + d]));  // exact
        double iv;
        if (SHARED) {
          iv = s_iv[d];
        } else {
          const float s = to_float(sls[rb + d]);
          const float ivf = expf(-2.f * s);
          ssum += static_cast<double>(s);
          if constexpr (kF32) sls[rb + d] = ivf;  // the column pass needs 1 / sigma^2, not log sigma
          iv = static_cast<double>(ivf);
        }
        sq = fma(diff * diff, iv, sq);
        d = (d + 1 == D) ? 0 : d + 1;
      }
      const float logp = static_cast<float>(-0.5 * sq - ssum - D * kLogSqrt2Pi);
      const float ent = static_cast<float>(D * (0.5 + kLogSqrt2Pi) + ssum);
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
    // ---- column pass: d loss / d mean in place of the mean, d loss / d log_std in place of 1 / sigma^2 (per row; a
    // bfloat16 slot still holds log sigma, whose 1 / sigma^2 is the row pass's expression again) ----
    if (col_thread) {
      int idx = static_cast<int>(threadIdx.x);
      for (int r = kc; r < cnt; r += K, idx += K * D) {
        const float a = sac[idx], mu = to_float(smu[idx]);
        const float diff = a - mu;
        float iv = iv_c;
        if constexpr (kF32) {
          if (!SHARED) iv = sls[idx];
        } else {
          if (!SHARED) iv = expf(-2.f * to_float(sls[idx]));
        }
        const float z = diff * iv;
        const float gl = s_glp[r];
        smu[idx] = from_float<T>(gl * z);
        if (SHARED) {
          // formed in float64 too: (a - mu)^2 / sigma^2 - 1 cancels near sigma, and T * n of these terms are summed
          const double dd = static_cast<double>(a) - static_cast<double>(mu);
          g_acc += fma(static_cast<double>(gl), fma(dd * dd, iv_cd, -1.0), static_cast<double>(s_gen[r]));
        } else {
          sls[idx] = from_float<T>(fmaf(gl, fmaf(diff, z, -1.f), s_gen[r]));
        }
      }
    }
    if (bulk) {
      tma::fence_proxy_async_smem();  // the gradients above, before the bulk copies read them
      __syncthreads();
      if (threadIdx.x == 0) {
        const uint32_t bytes = static_cast<uint32_t>(total) * kElem;
        tma::bulk_store(static_cast<T*>(q.g_mean) + e0, smu, bytes);  // read before the next tile
        if (!SHARED) tma::bulk_store(static_cast<T*>(q.g_log_std) + e0, sls, bytes);
      }
      __syncthreads();
    } else {
      __syncthreads();
      stage_out(static_cast<T*>(q.g_mean) + e0, smu, total);
      if (!SHARED) stage_out(static_cast<T*>(q.g_log_std) + e0, sls, total);
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
    static_cast<float*>(q.g_log_std)[threadIdx.x] = static_cast<float>(g);
  }
}

// one resident wave of ppo_loss_gaussian_kernel<SHARED, T> over the T * n transitions of q
template <typename T>
int launch_gaussian(const GaussianParams& q, bool shared, size_t smem, cudaStream_t stream) {
  int rc;
  auto kern = shared ? ppo_loss_gaussian_kernel<true, T> : ppo_loss_gaussian_kernel<false, T>;
  if ((rc = opt_in_smem<ppo_loss_gaussian_kernel<true, T>>(200 * 1024)) != SRL_OK) return rc;
  if ((rc = opt_in_smem<ppo_loss_gaussian_kernel<false, T>>(200 * 1024)) != SRL_OK) return rc;
  const long long tiles = (static_cast<long long>(q.s.T) * q.s.n + 255) / 256;
  // ONE resident wave, as srl_ppo_loss_from_logits sizes its grid: as many CTAs as the SMs hold at once with this much
  // shared memory, at most kMaxGrid.  With a shared log_std this is also what makes CTA 0's wait for the other CTAs' rows
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

// srl_ppo_loss_from_gaussian (elem_bytes = 4) and srl_ppo_loss_from_gaussian_bf16 (elem_bytes = 2: mean, v_pred, g_mean,
// g_value and a per-row log_std / g_log_std are bfloat16; a shared log_std and its gradient are float either way)
int ppo_loss_from_gaussian(const char* fn, size_t elem_bytes, const void* mean, const void* log_std, int log_std_shared,
                           const float* action, int D, const void* v_pred, const float* old_logp, const float* old_value,
                           const float* ret, const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                           const int32_t* lane_idx, int T, int n, const double* norm_stats, const double* local_stats,
                           const double* popart_mean_std, const srl_ppo_hyper* hyper, void* g_mean, void* g_log_std,
                           void* g_value, float* logp_out, float* entropy_out, double* out, float* out_f32,
                           void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  SRL_REQUIRE(T >= 1 && n >= 1, SRL_ERR_INVALID_ARG, "%s: need T >= 1 and n >= 1 (got %d, %d)", fn, T, n);
  SRL_REQUIRE(D >= 1 && D <= kMaxD, SRL_ERR_INVALID_ARG, "%s: D=%d action dimensions outside [1, %d]", fn, D, kMaxD);
  const struct {
    const void* p;
    const char* name;
  } required[] = {{mean, "mean"},         {log_std, "log_std"},     {action, "action"},     {v_pred, "v_pred"},
                  {old_logp, "old_logp"}, {ret, "ret"},             {adv, "adv"},           {on_reset_next, "on_reset_next"},
                  {norm_stats, "norm_stats"}, {local_stats, "local_stats"}, {g_mean, "g_mean"}, {g_log_std, "g_log_std"},
                  {g_value, "g_value"},   {workspace, "workspace"}};
  for (const auto& r : required) SRL_REQUIRE(r.p != nullptr, SRL_ERR_INVALID_ARG, "%s: null pointer %s", fn, r.name);
  SRL_REQUIRE(ld_smp >= (lane_idx ? 1 : n), SRL_ERR_INVALID_ARG, "%s: ld_smp=%lld smaller than the row", fn,
              static_cast<long long>(ld_smp));
  const bool shared = log_std_shared != 0;
  const size_t need = srl_ppo_loss_gaussian_workspace_bytes(T, n, D, log_std_shared);
  SRL_REQUIRE(workspace_bytes >= need, SRL_ERR_INVALID_ARG, "%s: workspace too small (%zu bytes, need %zu)", fn,
              workspace_bytes, need);
  GaussianParams q;
  int rc = fill_loss_hyper(hyper, popart_mean_std, q.s.h);
  if (rc != SRL_OK) return rc;
  SRL_REQUIRE(!(q.s.h.clip_value && old_value == nullptr), SRL_ERR_INVALID_ARG, "%s: clip_value needs old_value", fn);
  const size_t blk_bytes = static_cast<size_t>(256) * D * elem_bytes;  // one dense [256, D] block of the element type
  const size_t act_bytes = static_cast<size_t>(256) * D * sizeof(float);  // the [256, D] action block
  const size_t smem = (shared ? 1 : 2) * blk_bytes + act_bytes + 16;     // + the mbarrier of the bulk copies
  SRL_REQUIRE(smem <= 200 * 1024, SRL_ERR_UNSUPPORTED, "%s: D = %d too wide for shared memory", fn, D);
  q.mean = mean;
  q.log_std = log_std;
  q.action = action;
  q.g_mean = g_mean;
  q.g_log_std = g_log_std;
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
  if (elem_bytes == sizeof(__nv_bfloat16)) return launch_gaussian<__nv_bfloat16>(q, shared, smem, stream);
  return launch_gaussian<float>(q, shared, smem, stream);
}

}  // namespace
}  // namespace loss
}  // namespace srl

extern "C" size_t srl_ppo_loss_gaussian_workspace_bytes(int T, int n, int D, int log_std_shared) {
  const size_t slot = srl_ppo_loss_workspace_bytes(T, n);
  if (!log_std_shared || D < 1) return slot;
  return slot + static_cast<size_t>(srl::loss::kMaxGrid) * static_cast<size_t>(D) * sizeof(double);
}

extern "C" int srl_ppo_loss_from_gaussian(const float* mean, const float* log_std, int log_std_shared, const float* action,
                                          int D, const float* v_pred, const float* old_logp, const float* old_value,
                                          const float* ret, const float* adv, const uint8_t* on_reset_next, int64_t ld_smp,
                                          const int32_t* lane_idx, int T, int n, const double* norm_stats,
                                          const double* local_stats, const double* popart_mean_std,
                                          const srl_ppo_hyper* hyper, float* g_mean, float* g_log_std, float* g_value,
                                          float* logp_out, float* entropy_out, double* out, float* out_f32, void* workspace,
                                          size_t workspace_bytes, srl_stream_t stream) {
  return srl::loss::ppo_loss_from_gaussian("srl_ppo_loss_from_gaussian", sizeof(float), mean, log_std, log_std_shared,
                                           action, D, v_pred, old_logp, old_value, ret, adv, on_reset_next, ld_smp,
                                           lane_idx, T, n, norm_stats, local_stats, popart_mean_std, hyper, g_mean,
                                           g_log_std, g_value, logp_out, entropy_out, out, out_f32, workspace,
                                           workspace_bytes, static_cast<cudaStream_t>(stream));
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
  return srl::loss::ppo_loss_from_gaussian("srl_ppo_loss_from_gaussian_bf16", sizeof(__nv_bfloat16), mean, log_std,
                                           log_std_shared, action, D, v_pred, old_logp, old_value, ret, adv,
                                           on_reset_next, ld_smp, lane_idx, T, n, norm_stats, local_stats,
                                           popart_mean_std, hyper, g_mean, g_log_std, g_value, logp_out, entropy_out, out,
                                           out_f32, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}
