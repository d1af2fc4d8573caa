// K2, fast path: TMA-pipelined GAE scan.  One warp owns 32 adjacent lanes for the whole trajectory, so
// EVERY thread is a scanning thread (the tile kernel in gae_scan.cu idles most warps during the scan and
// exposes one DRAM round trip per load batch).  Rows are processed in stages of 8 rows, newest first; each
// stage is five 2-D TMA tile loads ([8 rows x 32 lanes] boxes of reward, value, done, truncated, on_reset;
// six with the loss pack, seven with V-trace) landing in a 4-deep shared-memory ring, completion tracked
// with one mbarrier per slot.  The warp that consumes a slot re-arms it, so there is no CTA-level barrier
// anywhere; 32 rows x 352 B = 11 KB are in flight per warp and 14+ warps fit per SM (all 2048 warps of a
// 65536-lane batch are resident at once), which is what it takes to cover HBM latency at 6.5 TB/s.  Outputs
// leave straight from registers as 128-byte coalesced stores (512-byte for the pack); the per-lane float64
// statistics never leave the thread until the end.
//
// r1c: the kernel was issue-bound (ncu: 91 warp instructions per row, 61 % of issue slots busy, DRAM at 33 %;
// profiles/r1b_ncu_cfg5_before.txt).  Now stages that lie entirely inside the loss rows run a specialised body
// with no per-row range tests, masks are selects instead of fp64 multiplies, the mask / done / truncated counts
// are integers, and squares accumulate with one DFMA.
//
// The per-cell arithmetic is gae_common.cuh's, shared with the other scan kernels.
#include "gae_common.cuh"
#include "tma_util.cuh"

namespace srl {
namespace {

using namespace srl::tma;

#ifndef SRL_TMA_ROWS
#define SRL_TMA_ROWS 8
#endif
#ifndef SRL_TMA_STAGES
#define SRL_TMA_STAGES 4
#endif
constexpr int kRows = SRL_TMA_ROWS;      // rows per stage
constexpr int kStages = SRL_TMA_STAGES;  // ring depth
constexpr int kMaxLanes = 32;            // lanes per CTA (LPW below): one full warp

struct alignas(64) GaeTmaMaps {
  CUtensorMap reward, value, done, truncated, on_reset, old_logp, vt_new;
};

struct GaeTmaParams {
  GaeParams p;
  GaeTmaMaps maps;
};

// OLDLP: the stage also carries old_logp (needed by the pack and by V-trace)
template <bool VTRACE, bool OLDLP, int LPW>
struct StageLayout {
  // byte offsets inside one stage; every sub-buffer is 128-byte aligned
  static constexpr int value = 0;
  static constexpr int reward = value + kRows * LPW * 4;
  static constexpr int old_logp = reward + kRows * LPW * 4;
  static constexpr int vt_new = old_logp + (OLDLP ? kRows * LPW * 4 : 0);
  static constexpr int done = vt_new + (VTRACE ? kRows * LPW * 4 : 0);
  static constexpr int truncated = done + kRows * LPW;
  static constexpr int on_reset = truncated + kRows * LPW;
  static constexpr int bytes = on_reset + kRows * LPW;  // payload = what the mbarrier expects
  static constexpr int stride = (bytes + 127) / 128 * 128;
};

template <bool VTRACE, bool OLDLP, int LPW>
__device__ __forceinline__ void issue_stage(const GaeTmaParams& q, unsigned char* slot, uint64_t* bar, int col0, int row0) {
  using SL = StageLayout<VTRACE, OLDLP, LPW>;
  mbar_expect_tx(bar, SL::bytes);
  tma_load_2d(slot + SL::value, &q.maps.value, col0, row0, bar);
  tma_load_2d(slot + SL::reward, &q.maps.reward, col0, row0, bar);
  tma_load_2d(slot + SL::done, &q.maps.done, col0, row0, bar);
  tma_load_2d(slot + SL::truncated, &q.maps.truncated, col0, row0, bar);
  tma_load_2d(slot + SL::on_reset, &q.maps.on_reset, col0, row0, bar);
  if (OLDLP) tma_load_2d(slot + SL::old_logp, &q.maps.old_logp, col0, row0, bar);
  if (VTRACE) tma_load_2d(slot + SL::vt_new, &q.maps.vt_new, col0, row0, bar);
}

// What a lane carries from row t+1 into row t, and its running statistics.
struct Carry {
  double vd_next = 0.0;  // float64 image of v'[t+1]
  double g = 0.0;        // A[t+1]
  bool reset_next = false, trunc_next = false;
};

// One stage of kRows rows.  EDGE = false: every row t of the stage satisfies row_lo <= t < row_hi (<= L-1), so all
// rows are scanned, stored and counted -- no per-row range tests.  EDGE = true: the general body.
// Straight-line code on purpose: the 8 rows of a stage are independent except for the two-instruction chain in
// pass 2, so the scheduler can overlap their shared-memory, conversion and fp64 latencies.
template <bool VTRACE, bool PACK, bool EDGE, int LPW>
__device__ __forceinline__ void run_stage(const GaeParams& p, const unsigned char* slot, int tbase, int lane, int col,
                                          bool live, bool popart, double pa_mean, double pa_std, Carry& cy,
                                          LaneStats& st) {
  // `live` and `popart` are compile-time constants in the specialised instantiations (FULL / POPART below)
  using SL = StageLayout<VTRACE, PACK || VTRACE, LPW>;
  const float* sv = reinterpret_cast<const float*>(slot + SL::value);
  const float* sr = reinterpret_cast<const float*>(slot + SL::reward);
  const uint8_t* sdn = slot + SL::done;
  const uint8_t* str_ = slot + SL::truncated;
  const uint8_t* srs = slot + SL::on_reset;
  const int L = p.L, N = p.N;
  const double gamma = p.gamma, gl = p.gamma_lmbda;

  // ---- pass 1: v', flags, delta_t, m_t for the 8 rows (independent) -----------------------------------------
  float v[kRows];
  double vd[kRows], dl[kRows], mm[kRows];
  bool dnf[kRows], trf[kRows], rsf[kRows];
#pragma unroll
  for (int r = 0; r < kRows; ++r) {
    const float x = sv[r * LPW + lane];
    dnf[r] = sdn[r * LPW + lane] != 0;
    trf[r] = str_[r * LPW + lane] != 0;
    rsf[r] = srs[r * LPW + lane] != 0;
    v[r] = gae_vprime(x, dnf[r], popart, pa_mean, pa_std);
    vd[r] = static_cast<double>(v[r]);
  }
#pragma unroll
  for (int r = 0; r < kRows; ++r) {
    const double vn = (r == kRows - 1) ? cy.vd_next : vd[r + 1];
    const bool rn = (r == kRows - 1) ? cy.reset_next : rsf[r + 1];
    const bool tn = (r == kRows - 1) ? cy.trunc_next : trf[r + 1];
    double d = gae_delta(&sr[r * LPW + lane], vd[r], vn, rn, gamma);
    double m = gae_carry(!rn && !tn, gl);
    if (VTRACE) {
      const float* snl = reinterpret_cast<const float*>(slot + SL::vt_new);
      const float* sol = reinterpret_cast<const float*>(slot + SL::old_logp);
      const double rd = static_cast<double>(expf(snl[r * LPW + lane] - sol[r * LPW + lane]));  // mappo.py:129-132
      gae_vtrace_scale(d, m, rd, p.rho, p.c);
    }
    if (EDGE) {
      const bool scanned = tbase + r < L - 1;  // rows L-1 (padding row) and beyond carry no advantage
      d = scanned ? d : 0.0;
      m = scanned ? m : 0.0;
    }
    dl[r] = d;
    mm[r] = m;
  }
  // ---- pass 2: the only sequential part, A_t = delta_t + m_t * A_{t+1} ----------------------------------------------
  float a[kRows];
  double g = cy.g;
#pragma unroll
  for (int r = kRows - 1; r >= 0; --r) {
    g = gae_step(dl[r], mm[r], g);
    a[r] = static_cast<float>(g);  // adv.float(), gae.py:97
  }
  cy.g = g;
  // ---- pass 3: value target, stores, per-lane statistics (independent) ------------------------------------------
  size_t gi = static_cast<size_t>(tbase + kRows - 1) * N + col;
#pragma unroll
  for (int r = kRows - 1; r >= 0; --r, gi -= N) {
    const int t = tbase + r;
    const bool rn = (r == kRows - 1) ? cy.reset_next : rsf[r + 1];
    float rt = gae_value_target(a[r], v[r]);
    if (EDGE) rt = (t < L - 1) ? rt : 0.f;
    const bool store = EDGE ? (live && t < L) : live;  // row L-1 is the zero padding row of mappo.py:254-256
    // loss rows [row_lo, row_hi), mask = 1 - on_reset[t+1]   mappo.py:259-261
    const bool in_rows = EDGE ? (t >= p.row_lo && t < p.row_hi) : true;
    const bool mk = in_rows && !rn;
#ifndef SRL_DEBUG_NO_STORES
    if (store) {
      stg_stream(p.adv + gi, a[r]);
      stg_stream(p.ret + gi, rt);
      if (PACK) {
        const float* sol = reinterpret_cast<const float*>(slot + SL::old_logp);
        const bool keep = EDGE ? (!rn && t < L - 1) : !rn;
        __stcg(reinterpret_cast<float4*>(p.pack) + pack_index(t, N, col),
               pack_item(sol[r * LPW + lane], sv[r * LPW + lane], rt, a[r], keep));
      }
    }
#endif
    st.add(in_rows, mk, a[r], rt, dnf[r], trf[r]);
  }
  cy.vd_next = vd[0];
  cy.reset_next = rsf[0];
  cy.trunc_next = trf[0];
}

// SPEC = true: the hot instantiations, N % 32 == 0 (no dead lanes, so no per-row store predicate and no
// reconvergence barrier around the stores) and PopArt known at compile time (POPART); SPEC = false: general.
template <bool VTRACE, bool PACK, bool SPEC, bool POPART, int LPW>
__global__ void __launch_bounds__(LPW) gae_scan_tma_kernel(const __grid_constant__ GaeTmaParams q) {
  constexpr bool OLDLP = PACK || VTRACE;
  using SL = StageLayout<VTRACE, OLDLP, LPW>;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * SL::stride);
  const GaeParams& p = q.p;
  const int lane = threadIdx.x;
  const int col0 = blockIdx.x * LPW;
  const int col = col0 + lane;
  const bool live = SPEC ? true : col < p.N;
  const int L = p.L, N = p.N;
  const int n_stages = (L + kRows - 1) / kRows;  // stage k covers rows [k*kRows, (k+1)*kRows); rows >= L read as 0
  pdl_launch_dependents();  // see gae_scan_ws.cu: the loss kernel behind this one may become resident

  if (lane == 0) {
    const CUtensorMap* maps[] = {&q.maps.value, &q.maps.reward, &q.maps.done, &q.maps.truncated, &q.maps.on_reset};
    for (const CUtensorMap* m : maps) prefetch_map(m);
    for (int s = 0; s < kStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncwarp();
  if (lane == 0) {  // prologue: fill the ring, newest rows first
    for (int i = 0; i < kStages && i < n_stages; ++i)
      issue_stage<VTRACE, OLDLP, LPW>(q, smem + i * SL::stride, &bars[i], col0, (n_stages - 1 - i) * kRows);
  }

  const bool popart = SPEC ? POPART : p.popart != nullptr;
  double pa_mean = 0.0, pa_std = 1.0;
  if (popart) {
    pa_mean = p.popart[0];
    pa_std = p.popart[1];
  }
  Carry cy;
  LaneStats st;

#ifdef SRL_DEBUG_PHASES
  long long dbg_wait = 0;
  const long long dbg_t0 = clock64();
#endif
  for (int it = 0; it < n_stages; ++it) {
    const int k = n_stages - 1 - it;
    const int slot_i = it % kStages;
    unsigned char* slot = smem + slot_i * SL::stride;
#ifdef SRL_DEBUG_PHASES
    const long long w0 = clock64();
#endif
    mbar_wait(&bars[slot_i], (it / kStages) & 1);
#ifdef SRL_DEBUG_PHASES
    dbg_wait += clock64() - w0;
#endif
    const int tbase = k * kRows;
    const bool interior = !VTRACE && tbase >= p.row_lo && tbase + kRows <= p.row_hi;
    if (interior)
      run_stage<VTRACE, PACK, false, LPW>(p, slot, tbase, lane, col, live, popart, pa_mean, pa_std, cy, st);
    else
      run_stage<VTRACE, PACK, true, LPW>(p, slot, tbase, lane, col, live, popart, pa_mean, pa_std, cy, st);
    __syncwarp();  // every lane is done reading this slot
    if (lane == 0 && it + kStages < n_stages)
      issue_stage<VTRACE, OLDLP, LPW>(q, slot, &bars[slot_i], col0, (n_stages - 1 - (it + kStages)) * kRows);
  }
#ifdef SRL_DEBUG_PHASES
  if (lane == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2 || blockIdx.x == gridDim.x - 1))
    printf("gae_tma block %d: loop %lld cycles, of which mbarrier wait %lld (%d stages of %d rows)\n", blockIdx.x,
           clock64() - dbg_t0, dbg_wait, n_stages, kRows);
#endif
  if (p.lane_part != nullptr && live) {
    double* o = p.lane_part + col;
    o[0] = static_cast<double>(st.cnt);
    o[static_cast<size_t>(1) * N] = st.s1;
    o[static_cast<size_t>(2) * N] = st.s2;
    o[static_cast<size_t>(3) * N] = st.s3;
    o[static_cast<size_t>(4) * N] = st.s4;
    o[static_cast<size_t>(5) * N] = static_cast<double>(st.dn);
    o[static_cast<size_t>(6) * N] = static_cast<double>(st.tr);
    o[static_cast<size_t>(7) * N] = 0.0;
    if (p.lane_aos != nullptr) {
      double* a4 = p.lane_aos + static_cast<size_t>(col) * 4;
      a4[0] = static_cast<double>(st.cnt);
      a4[1] = st.s1;
      a4[2] = st.s2;
      a4[3] = 0.0;
    }
  }
  if (lane == 0) pdl_wait();  // scan complete => permutation kernel complete (see gae_scan_ws.cu)
}

template <bool VTRACE, bool PACK, bool SPEC, bool POPART, int LPW>
int launch(const GaeTmaParams& q, cudaStream_t st) {
  using SL = StageLayout<VTRACE, PACK || VTRACE, LPW>;
  const size_t smem = static_cast<size_t>(kStages) * SL::stride + kStages * sizeof(uint64_t);
  constexpr auto kern = gae_scan_tma_kernel<VTRACE, PACK, SPEC, POPART, LPW>;
  const int rc = opt_in_smem<kern>(smem);
  if (rc != SRL_OK) return rc;
  const int grid = (q.p.N + LPW - 1) / LPW;
  SRL_CUDA(launch_pdl_scan(kern, dim3(grid), dim3(LPW), smem, st, q));
  return SRL_OK;
}

}  // namespace

bool gae_tma_eligible(const GaeParams& p) {
  // TMA needs 16-byte aligned bases and row pitches: N % 16 == 0 covers the uint8 flag tensors (and N*4 for fp32)
  if (p.N % 16 != 0 || tma::encode_fn() == nullptr) return false;
  const void* ptrs[] = {p.reward, p.value, p.done, p.truncated, p.on_reset};
  for (const void* q : ptrs)
    if (!aligned(q, 16)) return false;
  if (p.vt_new_logp && (!aligned(p.vt_new_logp, 16) || !aligned(p.vt_old_logp, 16))) return false;
  if (p.pack && !aligned(p.old_logp, 16)) return false;
  return true;
}

// Lanes per CTA: always a full warp.  Half-warp CTAs (LPW = 16: twice the CTAs for mid-size batches such as cfg3's
// 432 lane groups on 148 SMs) were measured and LOST -- cfg3 K2 41 -> 53 us, cfg4 31 -> 39 us: the kernel is bound by
// instruction issue, and a half-empty warp instruction costs a full issue slot (profiles/r1c_notes.md).
template <int LPW>
int launch_gae_tma_lpw(const GaeParams& p, cudaStream_t st) {
  GaeTmaParams q;
  q.p = p;
  int rc;
  if ((rc = make_map(&q.maps.value, p.value, p.L, p.N, 4, LPW, kRows)) != SRL_OK) return rc;
  if ((rc = make_map(&q.maps.reward, p.reward, p.L, p.N, 4, LPW, kRows)) != SRL_OK) return rc;
  if ((rc = make_map(&q.maps.done, p.done, p.L, p.N, 1, LPW, kRows)) != SRL_OK) return rc;
  if ((rc = make_map(&q.maps.truncated, p.truncated, p.L, p.N, 1, LPW, kRows)) != SRL_OK) return rc;
  if ((rc = make_map(&q.maps.on_reset, p.on_reset, p.L, p.N, 1, LPW, kRows)) != SRL_OK) return rc;
  const bool vtrace = p.vt_new_logp != nullptr;
  const bool pack = p.pack != nullptr;
  if (vtrace) {  // [L-1, N]: the last row of the top stage reads as zero and is never used
    if ((rc = make_map(&q.maps.vt_new, p.vt_new_logp, p.L - 1, p.N, 4, LPW, kRows)) != SRL_OK) return rc;
    if ((rc = make_map(&q.maps.old_logp, p.vt_old_logp, p.L - 1, p.N, 4, LPW, kRows)) != SRL_OK) return rc;
    // the pack's old_logp is the sample leaf the V-trace ratio uses as well
    return pack ? launch<true, true, false, false, LPW>(q, st) : launch<true, false, false, false, LPW>(q, st);
  }
  const bool full = p.N % LPW == 0, popart = p.popart != nullptr;
  if (pack) {
    if ((rc = make_map(&q.maps.old_logp, p.old_logp, p.L, p.N, 4, LPW, kRows)) != SRL_OK) return rc;
    if (!full) return launch<false, true, false, false, LPW>(q, st);
    return popart ? launch<false, true, true, true, LPW>(q, st) : launch<false, true, true, false, LPW>(q, st);
  }
  if (!full) return launch<false, false, false, false, LPW>(q, st);
  return popart ? launch<false, false, true, true, LPW>(q, st) : launch<false, false, true, false, LPW>(q, st);
}

int launch_gae_tma(const GaeParams& p, cudaStream_t st) {
  return launch_gae_tma_lpw<32>(p, st);
}

}  // namespace srl
