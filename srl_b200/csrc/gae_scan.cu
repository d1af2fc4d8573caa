// K2: GAE / value-target reverse-time scan (see include/srl_b200.h for the contract and the
// reference lines it replaces: mappo.py:118-144,254-256; gae.py:8-97; utils.py:54-57,113-120).
//
// Design (one CTA = a tile of LW adjacent lanes x all L rows, staged in shared memory):
//   phase A1  all 256 threads: every global load of the tile (coalesced row segments, 4 rows in flight
//             per thread); v' = (popart-denormalised) value * (1 - done) -> smem (fp32) + flag byte
//   phase A2  all threads, shared memory only: delta_t (fp64, explicit mul/add roundings, no FMA
//             contraction -- the reference evaluates each torch op separately) and the carry factor m_t
//   phase B   one warp: the only truly sequential part, A_t = delta_t + m_t * A_{t+1} in fp64 out of
//             shared memory (loads do not depend on the chain, so they pipeline)
//   phase C   all threads: ret = adv + v', coalesced stores of adv/ret (padding row zeroed) and the
//             per-lane float64 partial sums that masked_normalization / PopArt need
// Every global byte is read once and written once: 11 B in + 8 B out per scanned row-lane.
#include <stdlib.h>

#include "common.cuh"
#include "gae_common.cuh"

namespace srl {
namespace {

constexpr int kThreads = 256;
constexpr size_t kSmemBudget = 200 * 1024;

// (delta, m) (2 x f64, interleaved) + adv (f32) + v' (f32) + flags (u8) per cell; with the loss pack also old_logp and
// the raw value (2 x f32)
__host__ __device__ constexpr size_t gae_cell_bytes(bool pack) { return 16 + 4 + 4 + 1 + (pack ? 8 : 0); }

__host__ __device__ constexpr size_t gae_smem_bytes(int L, int LW, bool pack) {
  // the tile is [L][LW] cells (the per-lane reduction scratch [kThreads/LW][7][LW] f64 = 14 KB aliases the same bytes)
  const size_t tile = static_cast<size_t>(L) * LW * gae_cell_bytes(pack);
  const size_t scratch = static_cast<size_t>(kThreads) * 7 * 8;
  return tile > scratch ? tile : scratch;
}

// UN = rows per thread whose global loads are issued back to back.  (UN = 8 -- the whole cfg2 trajectory in one
// batch -- was measured: the 40 loads in flight spill at 64 registers and phase A1 got slower, 13.6 K vs 8.6 K
// cycles; profiles/r1c_notes.md.)
template <int LW, bool VTRACE, bool PACK, int UN>
__global__ void __launch_bounds__(kThreads, 4) gae_scan_kernel(const GaeParams p) {
  constexpr int kUnroll = UN;
  constexpr int RPP = kThreads / LW;  // rows handled per pass of the CTA
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int L = p.L, N = p.N;
  const size_t cells = static_cast<size_t>(L) * LW;
  double2* __restrict__ sdm = reinterpret_cast<double2*>(smem_raw);   // [L][LW] .x = reward -> delta -> A_t, .y = m
  float* __restrict__ sa = reinterpret_cast<float*>(sdm + cells);      // [L][LW] vtrace importance ratio
  float* __restrict__ sv = sa + cells;                                 // [L][LW] v'
  float* __restrict__ sol = sv + cells;                                // [L][LW] old_logp   (PACK only)
  float* __restrict__ svr = sol + (PACK ? cells : 0);                  // [L][LW] raw value  (PACK only)
  uint8_t* __restrict__ sf = reinterpret_cast<uint8_t*>(svr + (PACK ? cells : 0));  // [L][LW] done|trunc|reset bits

  const int tid = threadIdx.x;
  pdl_launch_dependents();  // see gae_scan_ws.cu: the loss kernel behind this one may become resident
  const int lane = tid % LW;
  const int trow = tid / LW;
  const int col = blockIdx.x * LW + lane;
  const bool live = col < N;

  const bool popart = p.popart != nullptr;
  double pa_mean = 0.0, pa_std = 1.0;
  if (popart) {
    pa_mean = p.popart[0];
    pa_std = p.popart[1];
  }

#ifdef SRL_DEBUG_PHASES
  long long ck[6];
  ck[0] = clock64();
#define SRL_STAMP(i) ck[i] = clock64()
#else
#define SRL_STAMP(i)
#endif
  // ---- A1: every global load of the tile, kUnroll rows in flight per thread -------------------------
  for (int t0 = trow; t0 < L; t0 += kUnroll * RPP) {
    float v[kUnroll], rw[kUnroll], nl[kUnroll], ol[kUnroll];
    uint32_t dn[kUnroll], tr[kUnroll], rs[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int t = t0 + u * RPP;
      v[u] = rw[u] = nl[u] = ol[u] = 0.f;
      dn[u] = tr[u] = rs[u] = 0u;
      if (live && t < L) {
        const size_t g = static_cast<size_t>(t) * N + col;
        v[u] = ldg_stream(p.value + g);
        dn[u] = ldg_stream(p.done + g);
        tr[u] = ldg_stream(p.truncated + g);
        rs[u] = ldg_stream(p.on_reset + g);
        if (PACK && !VTRACE) ol[u] = ldg_stream(p.old_logp + g);
        if (t < L - 1) {
          rw[u] = ldg_stream(p.reward + g);
          if (VTRACE) {
            nl[u] = ldg_stream(p.vt_new_logp + g);
            ol[u] = ldg_stream(p.vt_old_logp + g);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int t = t0 + u * RPP;
      if (t < L) {
        const float vv = v[u];
        if (PACK) {
          svr[t * LW + lane] = vv;
          sol[t * LW + lane] = ol[u];
        }
        sv[t * LW + lane] = gae_vprime(vv, dn[u] != 0, popart, pa_mean, pa_std);
        sf[t * LW + lane] = static_cast<uint8_t>((dn[u] != 0 ? 1u : 0u) | (tr[u] != 0 ? 2u : 0u) | (rs[u] != 0 ? 4u : 0u));
        sdm[t * LW + lane].x = static_cast<double>(rw[u]);
        if (VTRACE) sa[t * LW + lane] = expf(nl[u] - ol[u]);  // importance ratio, fp32   mappo.py:129-132
      }
    }
  }
  __syncthreads();
  SRL_STAMP(1);

  // ---- A2: delta_t and m_t for t in [0, L-1), shared memory only -----------------------------------
  for (int t = trow; t < L - 1; t += RPP) {
    const uint32_t f1 = sf[(t + 1) * LW + lane];
    const bool reset1 = (f1 & 4u) != 0, trunc1 = (f1 & 2u) != 0;
    const double v1 = static_cast<double>(sv[(t + 1) * LW + lane]);
    const double v0 = static_cast<double>(sv[t * LW + lane]);
    double d = gae_delta(&sdm[t * LW + lane].x, v0, v1, reset1, p.gamma);
    double m = gae_carry_product(p.gamma_lmbda, reset1, trunc1);
    if (VTRACE) gae_vtrace_scale(d, m, static_cast<double>(sa[t * LW + lane]), p.rho, p.c);
    sdm[t * LW + lane] = make_double2(d, m);
  }
  __syncthreads();
  SRL_STAMP(2);

  // ---- B: the sequential scan, one (partial) warp -----------------------------------------------------
  // A_t = delta_t + m_t * A_{t+1} (gae_step).  Software-pipelined: the (delta, m) pairs of the next 4 steps are already
  // in registers while the dependent DMUL/DADD chain of the current 4 runs, so shared-memory latency is off the chain.
  if (tid < LW) {
    constexpr int CH = 4;
    double g = 0.0;
    int t = L - 2;
    double2 q[CH];
    if (t >= CH - 1) {
#pragma unroll
      for (int u = 0; u < CH; ++u) q[u] = sdm[(t - u) * LW + lane];
    }
    for (; t >= CH - 1; t -= CH) {
      double2 nq[CH];
      const bool more = (t - CH) >= CH - 1;
      if (more) {
#pragma unroll
        for (int u = 0; u < CH; ++u) nq[u] = sdm[(t - CH - u) * LW + lane];
      }
      // the float64 results go back to shared memory as they are: converting here would put a 17-cycle F2F
      // (profiles/microbench/f2f.cu) behind every 16-cycle DMUL+DADD link; phase C converts in parallel instead
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        g = gae_step(q[u].x, q[u].y, g);
        sdm[(t - u) * LW + lane].x = g;
      }
      if (more) {
#pragma unroll
        for (int u = 0; u < CH; ++u) q[u] = nq[u];
      }
    }
    for (; t >= 0; --t) {
      const double2 dm = sdm[t * LW + lane];
      g = gae_step(dm.x, dm.y, g);
      sdm[t * LW + lane].x = g;
    }
  }
  __syncthreads();
  SRL_STAMP(3);

  // ---- C: ret, stores, per-lane partial sums ------------------------------------------------------------
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0, s5 = 0, s6 = 0;
  for (int t = trow; t < L; t += RPP) {
    float a = 0.f, r = 0.f;
    if (t < L - 1) {
      a = static_cast<float>(sdm[t * LW + lane].x);  // adv.float(), gae.py:97
      r = gae_value_target(a, sv[t * LW + lane]);
      if (t >= p.row_lo && t < p.row_hi) {
        const uint32_t f0 = sf[t * LW + lane], f1 = sf[(t + 1) * LW + lane];
        const double mk = (f1 & 4u) ? 0.0 : 1.0;  // loss mask = 1 - on_reset[t+1]   mappo.py:260-261
        const double x = __dmul_rn(static_cast<double>(a), mk);
        const double y = __dmul_rn(static_cast<double>(r), mk);
        s0 += mk;
        s1 += x;
        s2 = __dadd_rn(s2, __dmul_rn(x, x));
        s3 += y;
        s4 = __dadd_rn(s4, __dmul_rn(y, y));
        s5 += (f0 & 1u) ? 1.0 : 0.0;
        s6 += (f0 & 2u) ? 1.0 : 0.0;
      }
    }
    if (live) {  // row L-1 is the zero padding row of mappo.py:254-256
      const size_t g = static_cast<size_t>(t) * N + col;
      stg_stream(p.adv + g, a);
      stg_stream(p.ret + g, r);
      if (PACK) {  // sample side of the loss as one 16-byte item (see include/srl_b200.h)
        const bool keep = t < L - 1 && (sf[(t + 1) * LW + lane] & 4u) == 0u;
        __stcg(reinterpret_cast<float4*>(p.pack) + pack_index(t, N, col),
               pack_item(sol[t * LW + lane], svr[t * LW + lane], r, a, keep));
      }
    }
  }
  SRL_STAMP(4);
  if (p.lane_part != nullptr) {
    __syncthreads();  // the tile is dead; reuse its bytes as [RPP][7][LW] f64
    double* red = reinterpret_cast<double*>(smem_raw);
    red[(trow * 7 + 0) * LW + lane] = s0;
    red[(trow * 7 + 1) * LW + lane] = s1;
    red[(trow * 7 + 2) * LW + lane] = s2;
    red[(trow * 7 + 3) * LW + lane] = s3;
    red[(trow * 7 + 4) * LW + lane] = s4;
    red[(trow * 7 + 5) * LW + lane] = s5;
    red[(trow * 7 + 6) * LW + lane] = s6;
    __syncthreads();
    fold_lane_sums<LW, RPP, kThreads>(p, red, [](int, int, double) {});
  }
  if (tid == 0) pdl_wait();  // scan complete => permutation kernel complete (see gae_scan_ws.cu)
#ifdef SRL_DEBUG_PHASES
  SRL_STAMP(5);
  if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2 || blockIdx.x == gridDim.x - 1))
    printf("gae block %d: A1 %lld  A2 %lld  B %lld  C %lld  red %lld  total %lld cycles\n", blockIdx.x, ck[1] - ck[0],
           ck[2] - ck[1], ck[3] - ck[2], ck[4] - ck[3], ck[5] - ck[4], ck[5] - ck[0]);
#endif
}

template <int LW, bool VTRACE, bool PACK, int UN>
int launch_un(const GaeParams& p, cudaStream_t st) {
  const size_t smem = gae_smem_bytes(p.L, LW, PACK);
  constexpr auto kern = gae_scan_kernel<LW, VTRACE, PACK, UN>;
  const int rc = opt_in_smem<kern>(kSmemBudget);
  if (rc != SRL_OK) return rc;
  const int grid = (p.N + LW - 1) / LW;
  SRL_CUDA(launch_pdl_scan(kern, dim3(grid), dim3(kThreads), smem, st, p));
  return SRL_OK;
}

template <int LW, bool VTRACE>
int launch(const GaeParams& p, cudaStream_t st) {
  // with V-trace the pack's old_logp is the V-trace leaf [L-1, N]: the general phase-A load of that leaf is
  // reused, so row L-1 of the pack carries old_logp = 0 there (never read by the loss)
  constexpr int RPP = kThreads / LW;
  const int rows_per_thread = (p.L + RPP - 1) / RPP;
  // 5 or 6 rows per thread (cfg2: L = 129 over 32 rows per pass): all loads of the tile in ONE batch, i.e. one exposed
  // DRAM round trip in phase A1 instead of two
  if (!VTRACE && rows_per_thread == 5)
    return p.pack != nullptr ? launch_un<LW, false, true, 5>(p, st) : launch_un<LW, false, false, 5>(p, st);
  if (!VTRACE && rows_per_thread == 6)
    return p.pack != nullptr ? launch_un<LW, false, true, 6>(p, st) : launch_un<LW, false, false, 6>(p, st);
  if (p.pack != nullptr) return launch_un<LW, VTRACE, true, 4>(p, st);
  return launch_un<LW, VTRACE, false, 4>(p, st);
}

}  // namespace
}  // namespace srl

namespace srl {
namespace {
int gae_scan_impl(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                  const uint8_t* on_reset, const float* vtrace_new_logp, const float* vtrace_old_logp,
                  const double* popart_mean_std, const float* old_logp, int L, int N, int row_lo, int row_hi, double gamma,
                  double lmbda, double rho, double c, float* adv, float* ret, double* lane_part, double* lane_aos, float* pack,
                  const PermJob* job, int* fused, srl_stream_t stream);
}
}  // namespace srl

extern "C" int srl_gae_scan(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                            const uint8_t* on_reset, const float* vtrace_new_logp, const float* vtrace_old_logp,
                            const double* popart_mean_std, const float* old_logp, int L, int N, int row_lo,
                            int row_hi, double gamma, double lmbda, double rho, double c, float* adv, float* ret,
                            double* lane_part, double* lane_aos, float* pack, srl_stream_t stream) {
  return srl::gae_scan_impl(reward, value, done, truncated, on_reset, vtrace_new_logp, vtrace_old_logp, popart_mean_std,
                            old_logp, L, N, row_lo, row_hi, gamma, lmbda, rho, c, adv, ret, lane_part, lane_aos, pack, nullptr,
                            nullptr, stream);
}

extern "C" int srl_gae_scan_perm(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                                 const uint8_t* on_reset, const float* vtrace_new_logp, const float* vtrace_old_logp,
                                 const double* popart_mean_std, const float* old_logp, int L, int N, int row_lo,
                                 int row_hi, double gamma, double lmbda, double rho, double c, float* adv, float* ret,
                                 double* lane_part, double* lane_aos, float* pack, uint64_t perm_seed, uint32_t perm_epoch,
                                 int perm_n_epochs, int perm_n_env, int perm_group, int32_t* perm_out,
                                 int perm_minibatches, double* minibatch_part, int* fused, srl_stream_t stream) {
  using namespace srl;
  SRL_REQUIRE(perm_out != nullptr && perm_n_env >= 1 && perm_group >= 1 && perm_n_epochs >= 1 && perm_n_epochs <= 65535,
              SRL_ERR_INVALID_ARG, "srl_gae_scan_perm: need a permutation output, n_env >= 1, group >= 1, 1 <= n_epochs <= 65535");
  SRL_REQUIRE(static_cast<long long>(perm_n_env) * perm_group < (1ll << 31), SRL_ERR_UNSUPPORTED,
              "srl_gae_scan_perm: n_env * group must fit int32");
  PermJob job;
  job.seed_lo = static_cast<uint32_t>(perm_seed & 0xffffffffull);
  job.seed_hi = static_cast<uint32_t>(perm_seed >> 32);
  job.epoch0 = perm_epoch;
  job.n_epochs = perm_n_epochs;
  job.n_env = perm_n_env;
  job.group = perm_group;
  job.bits = perm_bits(perm_n_env);
  job.out = perm_out;
  job.minibatches = 1;
  job.per_mb = perm_n_env * perm_group;
  job.part = nullptr;
  if (minibatch_part != nullptr) {
    SRL_REQUIRE(perm_minibatches >= 1 && (static_cast<long long>(perm_n_env) * perm_group) % perm_minibatches == 0 &&
                    perm_n_env * perm_group == N && lane_part != nullptr && aligned(minibatch_part, 32),
                SRL_ERR_INVALID_ARG,
                "srl_gae_scan_perm: minibatch_part needs lane_part, n_env * group == N lanes split evenly into the minibatches "
                "and a 32-byte aligned table");
    if (perm_n_epochs <= kPartEpochs && perm_n_epochs * perm_minibatches <= kPartSlots) {  // else: not produced (*fused = 0)
      job.minibatches = perm_minibatches;
      job.per_mb = perm_n_env * perm_group / perm_minibatches;
      job.part = minibatch_part;
    }
  }
  int did = 0;
  const int rc = gae_scan_impl(reward, value, done, truncated, on_reset, vtrace_new_logp, vtrace_old_logp, popart_mean_std,
                               old_logp, L, N, row_lo, row_hi, gamma, lmbda, rho, c, adv, ret, lane_part, lane_aos, pack, &job,
                               &did, stream);
  if (rc != SRL_OK) return rc;
  // 1: permutations from the scan kernel; 2: and the minibatch partial sums
  if (fused != nullptr) *fused = did ? (job.part != nullptr ? 2 : 1) : 0;
  if (did) return SRL_OK;
  // the scan kernel chosen for this shape does not compute permutations: the stand-alone kernel, behind the scan
  return srl_philox_perm(perm_seed, perm_epoch, perm_n_epochs, perm_n_env, perm_group, perm_out, stream);
}

namespace srl {
namespace {
int gae_scan_impl(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                  const uint8_t* on_reset, const float* vtrace_new_logp, const float* vtrace_old_logp,
                  const double* popart_mean_std, const float* old_logp, int L, int N, int row_lo, int row_hi, double gamma,
                  double lmbda, double rho, double c, float* adv, float* ret, double* lane_part, double* lane_aos, float* pack,
                  const PermJob* job, int* fused, srl_stream_t stream) {

  SRL_REQUIRE(L >= 2 && N >= 1, SRL_ERR_INVALID_ARG, "srl_gae_scan: need L >= 2 and N >= 1 (got L=%d N=%d)", L, N);
  SRL_REQUIRE(reward && value && done && truncated && on_reset && adv && ret, SRL_ERR_INVALID_ARG,
              "srl_gae_scan: null tensor pointer");
  SRL_REQUIRE((vtrace_new_logp == nullptr) == (vtrace_old_logp == nullptr), SRL_ERR_INVALID_ARG,
              "srl_gae_scan: vtrace needs both log-prob tensors");
  SRL_REQUIRE(row_lo >= 0 && row_lo <= row_hi && row_hi <= L - 1, SRL_ERR_INVALID_ARG,
              "srl_gae_scan: loss rows [%d, %d) must lie inside [0, L-1=%d]", row_lo, row_hi, L - 1);
  SRL_REQUIRE(pack == nullptr || (old_logp != nullptr && aligned(pack, 32)), SRL_ERR_INVALID_ARG,
              "srl_gae_scan: the pack needs old_logp and a 32-byte aligned destination");
  SRL_REQUIRE(lane_aos == nullptr || (lane_part != nullptr && aligned(lane_aos, 32)), SRL_ERR_INVALID_ARG,
              "srl_gae_scan: lane_aos needs lane_part and a 32-byte aligned destination");
  const bool vtrace = vtrace_new_logp != nullptr;
  GaeParams p;
  p.reward = reward;
  p.value = value;
  p.done = done;
  p.truncated = truncated;
  p.on_reset = on_reset;
  p.vt_new_logp = vtrace_new_logp;
  p.vt_old_logp = vtrace_old_logp;
  p.popart = popart_mean_std;
  p.old_logp = old_logp;
  p.pack = pack;
  p.adv = adv;
  p.ret = ret;
  p.lane_part = lane_part;
  p.lane_aos = lane_aos;
  p.L = L;
  p.N = N;
  p.row_lo = row_lo;
  p.row_hi = row_hi;
  p.gamma = gamma;
  p.gamma_lmbda = gamma * lmbda;  // python evaluates gamma * lmbda first (gae.py:87)
  p.rho = rho;
  p.c = c;
  p.perm.out = nullptr;
  p.perm.part = nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  // Three kernels, picked by how many 32-lane groups the batch has:
  //   >= 2 groups per SM : one warp per lane group, TMA ring (gae_scan_tma.cu): fewest instructions per row
  //   fewer              : warp-specialised CTA per lane group (gae_scan_ws.cu): the chain runs in its own warp and 16
  //                        worker warps keep a lone CTA's latency per chunk short (measured at mid sizes -- cfg3, cfg4 --
  //                        it only ties or loses: there the machine is issue-bound and it executes more instructions)
  //   ragged / unaligned / V-trace on few lanes: the shared-memory tile kernel below
  const int groups = (N + 31) / 32;
  if (groups >= 2 * sm_count() && gae_tma_eligible(p)) return launch_gae_tma(p, st);
  if (groups >= 8 && gae_ws_eligible(p)) {  // a handful of lanes: the tile kernel's many short CTAs win
    if (job != nullptr) {  // the warp-specialised kernel's workers compute the permutation while they wait for data
      p.perm = *job;
      *fused = 1;
    }
    return launch_gae_ws(p, st);
  }

  // General path (any N, any alignment): shared-memory tile kernel below.
  // Lane-tile width: the widest tile that (a) fits shared memory and (b) still gives every SM work.
  const int sms = sm_count();
  int lw = 32;
  const bool with_pack = pack != nullptr;
  while (lw > 8 && (gae_smem_bytes(L, lw, with_pack) > kSmemBudget || (N + lw - 1) / lw < 2 * sms)) lw >>= 1;
#ifdef SRL_DEBUG_PHASES
  if (const char* e = getenv("SRL_GAE_LW")) lw = atoi(e);  // tuning knob of the instrumented build only
#endif
  SRL_REQUIRE(gae_smem_bytes(L, lw, with_pack) <= kSmemBudget, SRL_ERR_UNSUPPORTED,
              "srl_gae_scan: L=%d does not fit the shared-memory tile (max L = %d%s)", L,
              static_cast<int>(kSmemBudget / (8 * gae_cell_bytes(with_pack))), with_pack ? " with the loss pack" : "");
  if (vtrace) {
    if (lw == 32) return launch<32, true>(p, st);
    if (lw == 16) return launch<16, true>(p, st);
    return launch<8, true>(p, st);
  }
  if (lw == 32) return launch<32, false>(p, st);
  if (lw == 16) return launch<16, false>(p, st);
  return launch<8, false>(p, st);
}
}  // namespace
}  // namespace srl
