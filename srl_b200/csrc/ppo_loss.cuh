// K4 device code shared by the loss translation units (ppo_loss.cu: C-ABI, logits variant, finaliser;
// ppo_loss_dense.cu / ppo_loss_gather.cu / ppo_loss_pack.cu: the kernel instantiated per sample-side form, one file
// each so nvcc builds them in parallel).  See ppo_loss.cu for the design notes.
#pragma once
#include <float.h>

#include "common.cuh"
#include "xchg.cuh"

namespace srl {
namespace loss {

#ifndef SRL_LOSS_MIN_BLOCKS
#define SRL_LOSS_MIN_BLOCKS 3  // CTAs of 256 threads per SM the register allocator must leave room for
#endif
constexpr int kMaxGrid = 2048;                // partial rows per workspace slot
constexpr int kNumSums = 8;
constexpr size_t kPartialsOffset = 64;
constexpr int kMaxBatch = SRL_MAX_LOSS_BATCH;
constexpr int kFlushRows = 8;  // rows whose masked terms are summed in fp32 before they enter the float64 sums

// First 64 bytes of a workspace slot; the partial rows [n_rows][8] f64 follow.
struct SlotHeader {
  unsigned int ticket;  // immediate mode only; zero between launches
  unsigned int n_rows;  // CTAs that wrote a partial row
  double mask_sum;      // this rank's sum(mask) for the minibatch
  double wv, we;        // loss weights, so the finaliser needs nothing but the slot
  // pair kernel, immediate mode: the minibatch's normalisation sums {count, sum, sum of squares} over all ranks and this
  // rank's count, computed by ONE CTA of the problem and read by the others.  Each word is the float64's bit pattern XOR
  // kBoxKey: 0 (the workspace's initial state, restored by the last CTA with the ticket) means "not there yet", every
  // word validates itself, and neither side needs a fence -- a release behind the exchange's stores into the peers'
  // mailboxes would wait for their acknowledgement over NVLink.
  unsigned long long bc[4];
};
// A signalling-NaN pattern no arithmetic produces (sums are finite, or the canonical quiet NaN of a failed exchange).
constexpr unsigned long long kBoxKey = 0x7ff4deadbeef0001ull;
__device__ __forceinline__ unsigned long long box(double x) { return static_cast<unsigned long long>(__double_as_longlong(x)) ^ kBoxKey; }
__device__ __forceinline__ double unbox(unsigned long long w) { return __longlong_as_double(static_cast<long long>(w ^ kBoxKey)); }
static_assert(sizeof(SlotHeader) == kPartialsOffset, "slot header must stay 64 bytes");

// A policy-side element of K4b / K4c as the arithmetic reads it (bfloat16 -> float is exact), and a result stored back in
// the element type (bfloat16: rounded to nearest even, once, where the float result is final).
__device__ __forceinline__ float to_float(float x) { return x; }
__device__ __forceinline__ float to_float(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T>
__device__ __forceinline__ T from_float(float x);
template <>
__device__ __forceinline__ float from_float<float>(float x) { return x; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

struct LossHyperDev {
  float clip_lo, clip_hi;  // (float)(1 -/+ eps_clip)
  float veps;
  float c_clip;
  float wv, we;
  float vl_param;
  double adv_eps;
  int value_loss, clip_value, dual_clip, normalize_old_value;
};

// Per-minibatch pointers.
struct Problem {
  const float* new_logp;
  const float* v_pred;
  const float* entropy;
  const int32_t* lane_idx;
  const double* norm_stats;
  const double* local_stats;
  float* g_logp;
  float* g_value;
  float* g_entropy;
  double* out;
  float* out_f32;
  SlotHeader* slot;
};

// What every problem of a launch shares.
struct LossShared {
  const float* old_logp;
  const float* old_value;
  const float* ret;
  const float* adv;
  const uint8_t* reset_next;
  const float4* pack;        // K2's pair-interleaved pack (base of the buffer, absolute row 0), or null
  const double* popart;
  const double* lane_aos;    // [N][4] float64 per-lane sums from K2 (ppo_loss_pair.cu: self-computed statistics), or null
  const double* part;        // [slot][part_ctas][4] float64: K2's per-CTA shares of every minibatch's sums, or null
  int part_ctas, part_first; // problem k of the launch is table slot part_first + k
  long long ld_pol, ld_grad;
  long long ld_smp;          // sample-side row stride in elements; pack form: lanes N of the pack
  int T, n;
  int row_lo;                // pack form: absolute row of loss row 0
  int rows_per_tile, col_tiles, n_tiles;
  int smp_vec_ok;  // sample-side leaves allow 128-bit loads at 4-aligned lanes (alignment + row stride)
  LossHyperDev h;
};

struct LossBatch {
  LossShared s;
  Problem prob[kMaxBatch];
  XchgView xv;  // world <= 1: none.  Else the pair kernel adds every problem's sums over the ranks itself (xchg.cuh)
};

// Sample-side forms
constexpr int kDense = 0;   // separate leaves, lanes in policy order, 128-bit loads
constexpr int kGather = 1;  // separate leaves through lane_idx (or any alignment)
constexpr int kPack = 2;    // K2's pack through lane_idx (or in order): pack2[t / 2][lane][t % 2] of float4

// Hyper-parameter configuration of the element math.  The hot kernels are instantiated per configuration
// (StaticCfg): ncu showed ~25 % of the executed instructions of the first batched kernel were uniform branches,
// constant-bank reloads and reconvergence barriers around `if (h.clip_value)`-style tests inside the element loop
// (profiles/r1c_notes.md).  RuntimeCfg keeps one general instantiation for the rare combinations.
template <int VL, bool CLIP, bool DUAL, bool POPART>
struct StaticCfg {
  __device__ static __forceinline__ int vl(const LossHyperDev&) { return VL; }
  __device__ static __forceinline__ bool clip(const LossHyperDev&) { return CLIP; }
  __device__ static __forceinline__ bool dual(const LossHyperDev&) { return DUAL; }
  __device__ static __forceinline__ bool popart(bool) { return POPART; }
};
struct RuntimeCfg {
  __device__ static __forceinline__ int vl(const LossHyperDev& h) { return h.value_loss; }
  __device__ static __forceinline__ bool clip(const LossHyperDev& h) { return h.clip_value != 0; }
  __device__ static __forceinline__ bool dual(const LossHyperDev& h) { return h.dual_clip != 0; }
  __device__ static __forceinline__ bool popart(bool have) { return have; }
};

// torch.nn.{MSELoss,HuberLoss,SmoothL1Loss}(reduction='none'): value and derivative wrt the input, separately (the clipped
// value loss needs the value of ONE difference and the derivative of both, see element()).  Inside a kind both branches
// are evaluated and selected (the quadratic / linear choice is per element, and a divergent branch costs more than the
// spare flops).
__device__ __forceinline__ float pointwise_value(int kind, float prm, float d) {
  if (kind == SRL_VL_MSE) return d * d;
  const float z = fabsf(d);
  const bool quad = z < prm;
  if (kind == SRL_VL_HUBER) {
    const float lq = 0.5f * z * z, ll = prm * (z - 0.5f * prm);
    return quad ? lq : ll;
  }
  const float lq = 0.5f * z * z / prm, ll = z - 0.5f * prm;
  return quad ? lq : ll;
}
__device__ __forceinline__ float pointwise_grad(int kind, float prm, float d) {
  if (kind == SRL_VL_MSE) return 2.f * d;
  const bool quad = fabsf(d) < prm;
  if (kind == SRL_VL_HUBER) return quad ? d : copysignf(prm, d);  // d != 0 in the linear branch (|d| >= prm > 0)
  return quad ? d / prm : copysignf(1.f, d);
}
__device__ __forceinline__ void pointwise_loss(int kind, float prm, float d, float& l, float& dl) {
  l = pointwise_value(kind, prm, d);
  dl = pointwise_grad(kind, prm, d);
}

struct Uniforms {
  double mean, denom, rdenom;   // advantage normalisation: (x - mean) / denom, rdenom = 1 / denom
  double pa_mu, pa_sd, pa_rsd;  // popart: (x - mu) / sd
  float inv_m;                  // 1 / local sum(mask)
  bool popart;
};

__device__ __forceinline__ Uniforms load_uniforms(const double* norm_stats, const double* local_stats,
                                                  const double* popart, double adv_eps, double& mask_sum) {
  Uniforms u;
  const double cnt = __ldg(norm_stats), s1 = __ldg(norm_stats + 1), s2 = __ldg(norm_stats + 2);
  mask_sum = __ldg(local_stats);
  u.popart = popart != nullptr;
  u.pa_mu = u.popart ? __ldg(popart) : 0.0;
  u.pa_sd = u.popart ? __ldg(popart + 1) : 1.0;
  u.pa_rsd = 1.0 / u.pa_sd;
  u.mean = s1 / cnt;
  const double var = s2 / cnt - u.mean * u.mean;  // biased variance, utils.py:62-64
  u.denom = sqrt(var) + adv_eps;                  // eps outside the sqrt, utils.py:67
  u.rdenom = 1.0 / u.denom;
  u.inv_m = 1.f / static_cast<float>(mask_sum);
  return u;
}

__device__ __forceinline__ Uniforms uniforms_from(double cnt, double s1, double s2, double m_local, const double* popart,
                                                  double adv_eps) {
  Uniforms u;
  u.popart = popart != nullptr;
  u.pa_mu = u.popart ? __ldg(popart) : 0.0;
  u.pa_sd = u.popart ? __ldg(popart + 1) : 1.0;
  u.pa_rsd = 1.0 / u.pa_sd;
  u.mean = s1 / cnt;
  const double var = s2 / cnt - u.mean * u.mean;
  u.denom = sqrt(var) + adv_eps;
  u.rdenom = 1.0 / u.denom;
  u.inv_m = 1.f / static_cast<float>(m_local);
  return u;
}

// a / d in float64 given rd = 1 / d (correctly rounded): product, exact residual, one correction.  This is the
// tail of the IEEE division sequence without its reciprocal refinement and special-case handling; d is a
// positive finite scale here (sqrt(var) + eps, or PopArt's sigma >= 0.1).
__device__ __forceinline__ double div_by(double a, double d, double rd) {
  const double q = __dmul_rn(a, rd);
  const double r = __fma_rn(-d, q, a);
  return __fma_rn(r, rd, q);
}

__device__ __forceinline__ float popart_normalize(float x, const Uniforms& u) {
  // RunningMeanStd.normalize: ((x.double() - mean) / std).clip(-5, 5).float()   utils.py:139-144
  // (clipping after the cast gives the same float: +-5 are exact and rounding is monotonic)
  const float z = static_cast<float>(div_by(__dsub_rn(static_cast<double>(x), u.pa_mu), u.pa_sd, u.pa_rsd));
  return fminf(fmaxf(z, -5.f), 5.f);
}

// fp32 partial sums of a few rows (kFlushRows x 4 lanes); folded into the thread's float64 accumulators in blocks.
struct RowSums {
  float pl = 0.f, vl = 0.f, en = 0.f, adv = 0.f, ratio = 0.f, vt = 0.f, ret = 0.f;
  int clip = 0;
};

struct Acc {
  double pl = 0, vl = 0, en = 0, adv = 0, ratio = 0, vt = 0, ret = 0;
  int clip = 0;
  __device__ __forceinline__ void add(const RowSums& r) {
    pl += static_cast<double>(r.pl);
    vl += static_cast<double>(r.vl);
    en += static_cast<double>(r.en);
    adv += static_cast<double>(r.adv);
    ratio += static_cast<double>(r.ratio);
    vt += static_cast<double>(r.vt);
    ret += static_cast<double>(r.ret);
    clip += r.clip;
  }
};

// One transition.  Masked transitions (valid == false) produce zero gradients and enter no sum: in the reference
// every term is multiplied by mask before it is summed (mappo.py:184,197,199) and the stats go through
// masked_select (mappo.py:206-216).
template <class CFG>
__device__ __forceinline__ void element(const LossHyperDev& h, const Uniforms& u, float nl, float vp, float en,
                                        float ol, float ov, float rt, float ad, bool valid, float& g_lp,
                                        float& g_v, float& g_en, RowSums& rs) {
  const float mk = valid ? 1.f : 0.f;
  const float scale = valid ? u.inv_m : 0.f;  // d(masked mean)/d(element) = mask / M
  ad = valid ? ad : 0.f;                      // the pack marks masked transitions with a NaN advantage

  // ---- critic: mappo.py:172-184, utils.py:228-239 ---------------------------------------------
  const float vt = CFG::popart(u.popart) ? popart_normalize(rt, u) : rt;
  const float da = vp - vt;
  float vl, gv;
  if (CFG::clip(h)) {
    // max(loss(v - vt), loss(vc - vt)) with vc = old + clamp(v - old, +-eps).  All three pointwise losses are even and
    // strictly increasing in |d|, so the larger loss is the loss of the larger |difference|: ONE loss evaluation instead of
    // two, and torch.max's gradient rule (the larger operand's, ties split evenly) is decided on |d| -- no data-dependent
    // branch (the round-1 form compared the two losses and branched; ncu showed the reconvergence barriers in the loop).
    const float ovn = (CFG::popart(u.popart) && h.normalize_old_value) ? popart_normalize(ov, u) : ov;
    const float dv = vp - ovn;
    const float vc = ovn + fminf(fmaxf(dv, -h.veps), h.veps);
    const float db = vc - vt;
    const bool in = fabsf(dv) <= h.veps;  // clamp passes grad on the closed interval
    const float za = fabsf(da), zb = fabsf(db);
    const float ga = pointwise_grad(CFG::vl(h), h.vl_param, da);
    const float gb = in ? pointwise_grad(CFG::vl(h), h.vl_param, db) : 0.f;
    vl = pointwise_value(CFG::vl(h), h.vl_param, za >= zb ? da : db);
    gv = za > zb ? ga : gb;
    gv = za == zb ? 0.5f * (ga + gb) : gv;  // torch.max splits ties evenly
  } else {
    pointwise_loss(CFG::vl(h), h.vl_param, da, vl, gv);
  }
  g_v = h.wv * scale * gv;

  // ---- actor: mappo.py:157-158,186-197 ---------------------------------------------------------
  const float ratio = expf(nl - ol);
  // masked_normalization (utils.py:38-67) in float64, cast to float at the end; masked entries are centred
  // zeros there (x = adv * mask) and here
  const float nadv = static_cast<float>(div_by(__dsub_rn(static_cast<double>(ad), u.mean), u.denom, u.rdenom));
  const float cr = fminf(fmaxf(ratio, h.clip_lo), h.clip_hi);
  const float s1 = ratio * nadv;
  const float s2 = cr * nadv;
  // d min(s1, s2) / d new_logp = ratio * nadv (= s1) where s1 is the smaller or the clamp passes (cr == ratio, then
  // s1 == s2 and torch.min's even split adds up to the whole); 0 where the clamped branch is the smaller.  (s1 == s2
  // outside the clip range needs nadv == 0 or an underflow: the reference's half gradient is then a half of ~0.)
  float obj = fminf(s1, s2);
  float gsum = (cr == ratio || s1 < s2) ? s1 : 0.f;
  if (CFG::dual(h)) {
    const float s3 = -h.c_clip * fabsf(nadv);  // -sign(nadv) * c * nadv
    gsum = obj > s3 ? gsum : (obj < s3 ? 0.f : 0.5f * gsum);
    obj = fmaxf(obj, s3);
  }
  g_lp = -scale * gsum;
  g_en = -h.we * scale;  // entropy_loss = -sum(entropy * mask) / M   mappo.py:199

  // masked sums: multiply by the mask as the reference does (mappo.py:184,197,199).  Like there, a non-finite
  // term of a masked transition would poison the sum; the inputs of masked transitions are finite in practice
  // (dead agents carry new_logp = -inf, i.e. ratio = 0).
  rs.pl -= mk * obj;
  rs.vl += mk * vl;
  rs.en += mk * en;
  rs.adv += mk * ad;
  rs.ratio += mk * ratio;
  rs.vt += mk * vt;
  if (CFG::popart(u.popart)) rs.ret += mk * rt;  // only reported with PopArt (mappo.py:215-216)
  rs.clip += (valid && s2 < s1) ? 1 : 0;
}

// Folds n_rows partial rows (fixed order: lane-strided, then the warp-shuffle tree) and writes the results.
// Called by one CTA; sred is [kNumSums][8] shared scratch.
// The rows are cleared behind the fold: between launches a slot's rows are all zero, whichever kernel used it last (the
// pair kernel's immediate mode reads "zero" as "this CTA's row is not there yet").
__device__ __forceinline__ void fold_rows_and_write(double* __restrict__ partials, int n_rows, double M, double wv,
                                                    double we, double (*sred)[8], double* __restrict__ o,
                                                    float* __restrict__ o32) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int k = warp; k < kNumSums; k += nwarps) {
    double s = 0.0;
    for (int b = lane; b < n_rows; b += 32) {
      s += __ldcg(partials + static_cast<size_t>(b) * kNumSums + k);
      partials[static_cast<size_t>(b) * kNumSums + k] = 0.0;
    }
    s = warp_sum(s);
    if (lane == 0) sred[k][0] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNumSums) sred[threadIdx.x][1] = sred[threadIdx.x][0] / M;  // the eight divisions side by side
  __syncthreads();
  if (threadIdx.x == 0) {
    const double pl = sred[0][1], vl = sred[1][1], el = -sred[2][1];
    const double loss = pl + wv * vl + we * el;
    o[SRL_OUT_LOSS] = loss;
    o[SRL_OUT_POLICY_LOSS] = pl;
    o[SRL_OUT_VALUE_LOSS] = vl;
    o[SRL_OUT_ENTROPY_LOSS] = el;
    o[SRL_OUT_ADVANTAGE] = sred[3][1];
    o[SRL_OUT_IMPORTANCE_WEIGHT] = sred[4][1];
    o[SRL_OUT_CLIP_RATIO] = sred[5][1];
    o[SRL_OUT_VALUE_TARGETS] = sred[6][1];
    o[SRL_OUT_DENORM_VALUE] = sred[7][1];
    o[SRL_OUT_MASK_SUM] = M;
    for (int k = SRL_OUT_MASK_SUM + 1; k < SRL_LOSS_OUT_LEN; ++k) o[k] = 0.0;
    if (o32) {
      o32[0] = static_cast<float>(loss);
      o32[1] = static_cast<float>(pl);
      o32[2] = static_cast<float>(vl);
      o32[3] = static_cast<float>(el);
    }
  }
}

// Block reduction of the 8 masked sums -> this CTA's partial row; then either done (deferred) or ticket.
// `row` / `n_rows`: this CTA's row and the number of CTAs working on the same problem.
__device__ __forceinline__ void reduce_and_finalize(const Problem& pr, const LossHyperDev& h, const Acc& acc,
                                                    double mask_sum, int row, int n_rows) {
  __shared__ double sred[kNumSums][8];
  __shared__ bool is_last;
  double* partials = reinterpret_cast<double*>(reinterpret_cast<char*>(pr.slot) + kPartialsOffset);
  double v[kNumSums] = {acc.pl, acc.vl, acc.en, acc.adv, acc.ratio, static_cast<double>(acc.clip), acc.vt, acc.ret};
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  // butterfly level by level over all 8 sums: 8 independent shuffle+add chains per level hide each other's latency
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double w[kNumSums];
#pragma unroll
    for (int k = 0; k < kNumSums; ++k) w[k] = __shfl_xor_sync(0xffffffffu, v[k], o);
#pragma unroll
    for (int k = 0; k < kNumSums; ++k) v[k] += w[k];
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < kNumSums; ++k) sred[k][warp] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < kNumSums) {
    double s = 0.0;
    for (int w = 0; w < nwarps; ++w) s += sred[threadIdx.x][w];
    partials[static_cast<size_t>(row) * kNumSums + threadIdx.x] = s;
  }
  if (pr.out == nullptr) {  // deferred: publish what the finaliser needs and leave
    if (row == 0 && threadIdx.x == 0) {
      pr.slot->n_rows = n_rows;
      pr.slot->mask_sum = mask_sum;
      pr.slot->wv = static_cast<double>(h.wv);
      pr.slot->we = static_cast<double>(h.we);
    }
    return;
  }
  if (threadIdx.x < kNumSums) __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int done = atomicAdd(&pr.slot->ticket, 1u);
    is_last = (done == static_cast<unsigned int>(n_rows) - 1u);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  fold_rows_and_write(partials, n_rows, mask_sum, static_cast<double>(h.wv), static_cast<double>(h.we), sred, pr.out,
                      pr.out_f32);
  if (threadIdx.x == 0) pr.slot->ticket = 0u;  // ready for the next launch on this slot
}

__device__ __forceinline__ void unpack4(const float4 v, float (&a)[4]) { a[0] = v.x, a[1] = v.y, a[2] = v.z, a[3] = v.w; }

// Work decomposition of the row-tile kernel (dense leaves, leaves through lane_idx, odd shapes of the pack form): grid =
// (column tiles, row groups, problems).  A CTA owns `blockDim * LANES` adjacent policy-side lanes and the rows [r0, r1) of
// one problem: its gather indices are loaded once, and it walks its rows in order.  LANES = 4: a thread owns four adjacent
// lanes (n % 4 == 0, 16-byte aligned rows); LANES = 1: any shape.  Permuted minibatches of even width run the pair kernel
// (ppo_loss_pair.cu) instead.
template <int LANES, int MODE, class CFG>
__global__ void __launch_bounds__(256, SRL_LOSS_MIN_BLOCKS) ppo_loss_kernel(const __grid_constant__ LossBatch b) {
  const LossShared& s = b.s;
  const LossHyperDev& h = s.h;
  const Problem& pr = b.prob[blockIdx.z];
  const int T = s.T, n = s.n;
  const int r0 = blockIdx.y * s.rows_per_tile;
  const int r1 = min(T, r0 + s.rows_per_tile);
  Acc acc;
  RowSums rs;
  int pending = 0;
  double mask_sum = 0.0;
  Uniforms u;
  bool have_u = false;

  pdl_wait();  // launched programmatically behind the scan / the statistics kernel (common.cuh)

  // normally one column tile per CTA (gridDim.x == col_tiles); only batches wider than kMaxGrid tiles loop here
  for (int ct = blockIdx.x; ct < s.col_tiles; ct += gridDim.x) {
    const int j = (ct * blockDim.x + threadIdx.x) * LANES;
    const bool active = j < n;
    // gather indices of this thread's lanes: once per column tile
    int c[LANES];
    if (pr.lane_idx && active) {
      if constexpr (LANES == 4) {
        const int4 q = __ldg(reinterpret_cast<const int4*>(pr.lane_idx + j));
        c[0] = q.x, c[1] = q.y, c[2] = q.z, c[3] = q.w;
      } else {
        c[0] = __ldg(pr.lane_idx + j);
      }
    } else {
#pragma unroll
      for (int q = 0; q < LANES; ++q) c[q] = j + q;
    }
    // a run of four consecutive, 4-aligned lanes (agents of one environment, sector-aligned environment blocks) is
    // fetched with one 128-bit load per leaf
    bool run4 = false;
    if constexpr (LANES == 4 && MODE == kGather)
      run4 = s.smp_vec_ok && (c[1] == c[0] + 1) && (c[2] == c[0] + 2) && (c[3] == c[0] + 3) && ((c[0] & 3) == 0);
    // row base pointers are warp-uniform (64-bit, advanced once per row); per-thread offsets stay 32-bit
    const float* nl_row = pr.new_logp + static_cast<long long>(r0) * s.ld_pol;
    const float* vp_row = pr.v_pred + static_cast<long long>(r0) * s.ld_pol;
    const float* en_row = pr.entropy + static_cast<long long>(r0) * s.ld_pol;
    float* glp_row = pr.g_logp + static_cast<long long>(r0) * s.ld_grad;
    float* gv_row = pr.g_value + static_cast<long long>(r0) * s.ld_grad;
    float* ge_row = pr.g_entropy + static_cast<long long>(r0) * s.ld_grad;
    long long ob = static_cast<long long>(r0) * s.ld_smp;  // sample-side row base (elements)
    float nl[LANES], vp[LANES], en[LANES], ol[LANES], ov[LANES], rt[LANES], ad[LANES];
    bool valid[LANES];
    // every global load of loss row t at (nl_row, vp_row, en_row, ob)
    auto load_row = [&](int t) {
      if constexpr (LANES == 4) {
        unpack4(ldg_stream(reinterpret_cast<const float4*>(nl_row + j)), nl);
        unpack4(ldg_stream(reinterpret_cast<const float4*>(vp_row + j)), vp);
        unpack4(ldg_stream(reinterpret_cast<const float4*>(en_row + j)), en);
      } else {
        nl[0] = ldg_stream(nl_row + j);
        vp[0] = ldg_stream(vp_row + j);
        en[0] = ldg_stream(en_row + j);
      }
      if constexpr (MODE == kPack) {
        // pack2[ta / 2][lane][ta % 2], ta = absolute row: items of lane c at (ta / 2) * 2N + 2c + (ta % 2)
        const int ta = s.row_lo + t;
        const float4* pack_row = s.pack + static_cast<long long>(ta >> 1) * (2 * s.ld_smp) + (ta & 1);
#pragma unroll
        for (int q = 0; q < LANES; ++q) {
          const float4 k = __ldg(pack_row + 2 * c[q]);
          ol[q] = k.x;
          ov[q] = k.y;
          rt[q] = k.z;
          ad[q] = k.w;
          valid[q] = (k.w == k.w);  // K2 stores NaN in the advantage slot of masked transitions
        }
      } else if (run4) {
        if constexpr (LANES == 4) {
          unpack4(ldg_stream(reinterpret_cast<const float4*>(s.old_logp + ob + c[0])), ol);
          unpack4(ldg_stream(reinterpret_cast<const float4*>(s.ret + ob + c[0])), rt);
          unpack4(ldg_stream(reinterpret_cast<const float4*>(s.adv + ob + c[0])), ad);
          float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
          if (CFG::clip(h)) o = ldg_stream(reinterpret_cast<const float4*>(s.old_value + ob + c[0]));
          unpack4(o, ov);
          const uint32_t m = ldg_stream(reinterpret_cast<const uint32_t*>(s.reset_next + ob + c[0]));
#pragma unroll
          for (int q = 0; q < LANES; ++q) valid[q] = ((m >> (8 * q)) & 0xffu) == 0u;
        }
      } else {
        const float* ol_row = s.old_logp + ob;
        const float* rt_row = s.ret + ob;
        const float* ad_row = s.adv + ob;
        const float* ov_row = CFG::clip(h) ? s.old_value + ob : nullptr;
        const uint8_t* rs_row = s.reset_next + ob;
#pragma unroll
        for (int q = 0; q < LANES; ++q) {
          ol[q] = __ldg(ol_row + c[q]);
          rt[q] = __ldg(rt_row + c[q]);
          ad[q] = __ldg(ad_row + c[q]);
          ov[q] = CFG::clip(h) ? __ldg(ov_row + c[q]) : 0.f;
          valid[q] = __ldg(rs_row + c[q]) == 0;
        }
      }
    };
    // (Issuing the first row's loads here, ahead of the statistics prologue, and each later row right after the stores of
    // the row before it was built and measured in round 1: it loses -- profiles/r1d_notes.md.)
    if (!have_u) {
      u = load_uniforms(pr.norm_stats, pr.local_stats, s.popart, h.adv_eps, mask_sum);
      have_u = true;
    }
    if (active) {
      for (int t = r0; t < r1; ++t) {
        load_row(t);
        float glp[LANES], gv[LANES], ge[LANES];
#pragma unroll
        for (int q = 0; q < LANES; ++q)
          element<CFG>(h, u, nl[q], vp[q], en[q], ol[q], ov[q], rt[q], ad[q], valid[q], glp[q], gv[q], ge[q], rs);
        if (++pending == kFlushRows) {
          acc.add(rs);
          rs = RowSums();
          pending = 0;
        }
        if constexpr (LANES == 4) {
          stg_stream(reinterpret_cast<float4*>(glp_row + j), make_float4(glp[0], glp[1], glp[2], glp[3]));
          stg_stream(reinterpret_cast<float4*>(gv_row + j), make_float4(gv[0], gv[1], gv[2], gv[3]));
          stg_stream(reinterpret_cast<float4*>(ge_row + j), make_float4(ge[0], ge[1], ge[2], ge[3]));
        } else {
          stg_stream(glp_row + j, glp[0]);
          stg_stream(gv_row + j, gv[0]);
          stg_stream(ge_row + j, ge[0]);
        }
        nl_row += s.ld_pol, vp_row += s.ld_pol, en_row += s.ld_pol;
        glp_row += s.ld_grad, gv_row += s.ld_grad, ge_row += s.ld_grad;
        ob += s.ld_smp;
      }
    }
  }  // column tiles
  acc.add(rs);
  const int row = blockIdx.y * gridDim.x + blockIdx.x;
  reduce_and_finalize(pr, h, acc, mask_sum, row, static_cast<int>(gridDim.x * gridDim.y));
}

template <int LANES, int MODE, class CFG>
struct LossLauncher {
  // CTAs of `threads` threads one SM holds (registers / shared memory), asked once per device and block size
  static int resident(int threads) {
    static int cached[64][2] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 2;
    int& c = cached[dev][threads >= 256 ? 1 : 0];
    if (c == 0) {
      auto kern = ppo_loss_kernel<LANES, MODE, CFG>;
      int n = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, 0) != cudaSuccess || n < 1) n = 1;
      c = n;
    }
    return c;
  }

  static int launch(LossBatch& b, int n_problems, cudaStream_t st) {
    LossShared& s = b.s;
    const int per_row = (s.n + LANES - 1) / LANES;  // threads one row needs
    const int threads = per_row <= 128 ? 128 : 256;
    s.col_tiles = (per_row + threads - 1) / threads;
    const long long capacity = static_cast<long long>(sm_count()) * resident(threads);  // CTAs resident at once
    // row groups: as many as keep the whole grid resident in ONE wave (a second, partial wave would double the
    // kernel's duration); every CTA then walks ceil(T / groups) consecutive rows of its column tile
    long long groups = capacity / (static_cast<long long>(s.col_tiles) * n_problems);
    if (groups < 1) groups = 1;
    if (groups > s.T) groups = s.T;
    int rows = static_cast<int>((s.T + groups - 1) / groups);
    groups = (s.T + rows - 1) / rows;
    long long gx = s.col_tiles;  // CTAs along the lanes; wider batches loop over column tiles inside the kernel
    if (gx * groups > kMaxGrid) gx = kMaxGrid / groups;  // one partial row per CTA in the workspace slot
    s.rows_per_tile = rows;
    s.n_tiles = static_cast<int>(groups);
    const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>(groups), static_cast<unsigned>(n_problems));
    SRL_CUDA(launch_pdl(ppo_loss_kernel<LANES, MODE, CFG>, grid, dim3(threads), 0, st, b));
    return SRL_OK;
  }
};

// Picks the instantiation for the launch's hyper-parameters.  Static configurations: {mse, huber} x clip_value x
// dual_clip x popart with four lanes per thread; everything else (smoothl1, odd shapes) runs the general instantiation.
template <int LANES, int MODE>
int launch_loss_static(LossBatch& b, int n_problems, cudaStream_t st) {
  const LossHyperDev& h = b.s.h;
  const bool popart = b.s.popart != nullptr;
  const int key = (h.value_loss == SRL_VL_MSE ? 0 : h.value_loss == SRL_VL_HUBER ? 1 : 2) * 8 + (h.clip_value ? 4 : 0) +
                  (h.dual_clip ? 2 : 0) + (popart ? 1 : 0);
#define SRL_LOSS_CASE(k, vl, clip, dual, pa) \
  case k:                                    \
    return LossLauncher<LANES, MODE, StaticCfg<vl, clip, dual, pa>>::launch(b, n_problems, st)
  switch (key) {
    SRL_LOSS_CASE(0, SRL_VL_MSE, false, false, false);
    SRL_LOSS_CASE(1, SRL_VL_MSE, false, false, true);
    SRL_LOSS_CASE(2, SRL_VL_MSE, false, true, false);
    SRL_LOSS_CASE(3, SRL_VL_MSE, false, true, true);
    SRL_LOSS_CASE(4, SRL_VL_MSE, true, false, false);
    SRL_LOSS_CASE(5, SRL_VL_MSE, true, false, true);
    SRL_LOSS_CASE(6, SRL_VL_MSE, true, true, false);
    SRL_LOSS_CASE(7, SRL_VL_MSE, true, true, true);
    SRL_LOSS_CASE(8, SRL_VL_HUBER, false, false, false);
    SRL_LOSS_CASE(9, SRL_VL_HUBER, false, false, true);
    SRL_LOSS_CASE(10, SRL_VL_HUBER, false, true, false);
    SRL_LOSS_CASE(11, SRL_VL_HUBER, false, true, true);
    SRL_LOSS_CASE(12, SRL_VL_HUBER, true, false, false);
    SRL_LOSS_CASE(13, SRL_VL_HUBER, true, false, true);
    SRL_LOSS_CASE(14, SRL_VL_HUBER, true, true, false);
    SRL_LOSS_CASE(15, SRL_VL_HUBER, true, true, true);
    default:
      return LossLauncher<LANES, MODE, RuntimeCfg>::launch(b, n_problems, st);
  }
#undef SRL_LOSS_CASE
}

template <int MODE>
int launch_loss_mode(LossBatch& b, int n_problems, bool lanes4, cudaStream_t st) {
  if (!lanes4) {
    if constexpr (MODE == kDense)
      return SRL_ERR_INVALID_ARG;  // the dense form needs 128-bit rows; callers route odd shapes to kGather
    else
      return LossLauncher<1, MODE, RuntimeCfg>::launch(b, n_problems, st);
  }
  return launch_loss_static<4, MODE>(b, n_problems, st);
}

// ppo_loss.cu: the host-side check of the hyper-parameters, shared by every loss entry point
int fill_loss_hyper(const srl_ppo_hyper* hyper, const double* popart_mean_std, LossHyperDev& h);
// defined in ppo_loss_dense.cu / ppo_loss_gather.cu / ppo_loss_pack.cu
int launch_loss_dense(LossBatch& b, int n_problems, bool lanes4, cudaStream_t st);
int launch_loss_gather(LossBatch& b, int n_problems, bool lanes4, cudaStream_t st);
int launch_loss_pack(LossBatch& b, int n_problems, bool lanes4, cudaStream_t st);
// ppo_loss_pair.cu: the pack form for permuted minibatches of even width (two lanes x two rows per thread and step, the
// loads of the next step in flight under the arithmetic of this one, units dealt evenly over a persistent grid)
bool loss_pair_eligible(const LossShared& s, bool aligned8);
int launch_loss_pair(LossBatch& b, int n_problems, cudaStream_t st);

}  // namespace loss
}  // namespace srl
