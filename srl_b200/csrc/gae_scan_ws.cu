// K2, warp-specialised path for small and mid-size batches (a few dozen to ~1000 lane groups).
//
// The one-warp-per-32-lanes TMA kernel (gae_scan_tma.cu) runs all ~75 instructions of a row in the warp that also carries
// the sequential chain A_t = delta_t + m_t * A_{t+1}; with only a few warps per SM (cfg3: 432 lane groups on 148 SMs) it
// is bound by that single warp's latency: 41 us for 105 MB.  Here a CTA still owns 32 lanes for the whole trajectory, but
// its warps have roles:
//   warp 0        producer: TMA loads of the next chunks (16 rows + 1 overlap row, newest first) into a 3-slot ring
//   warp 1        scanner : ONLY the dependent chain, 2 fp64 instructions per row, out of shared memory
//   warps 2..5    workers : per cell -- v', delta_t, the carry flag (before the scan); value target, stores, pack and
//                 per-lane statistics (after it); 4 rows of every chunk each
// handing chunks over through mbarriers (tma_full -> pass1_done -> scanned -> empty), so the scan of chunk k overlaps the
// loads of chunk k+2, the delta pass of k+1 and the store pass of k-1, and the chain runs at ~22 cycles per row instead
// of ~200.  The extra row of every box (row t+16) gives each chunk its own copy of the next-row inputs: no state crosses
// chunks except the scanner's A.  The per-cell arithmetic is gae_common.cuh's, shared with the other scan kernels.
// V-trace is not handled here (the other two kernels do).
#include "gae_common.cuh"
#include "tma_util.cuh"

namespace srl {
namespace {

using namespace srl::tma;

__device__ __forceinline__ void st_cg256(float4* p, float4 a, float4 b) {
  asm volatile("st.global.cg.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w),
               "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w)
               : "memory");
}

constexpr int kR = 16;  // rows per chunk
// Ring depth kS (template parameter): 3 slots when several CTAs share an SM; kDeep when the batch has at most one CTA per
// SM anyway (cfg2: 128 lane groups) -- the whole trajectory of up to kDeep * kR rows is requested from HBM at once (one
// exposed DRAM round trip instead of one per ring turn), and the workers run the delta pass of all resident chunks ahead
// of the scanner.
constexpr int kDeep = 9;
// W = worker warps per CTA (kR / W rows of every chunk each).  The kernel serves batches with fewer CTAs than the SMs can
// hold (cfg2: 128 lane groups), where a CTA's time per chunk is the latency of one worker's rows: W = 16, one row per
// worker warp.  (W = 4 was measured on mid-size batches -- cfg3: 38 us, 129 warp instructions per row-lane, issue slots
// 59 % busy -- no better than the one-warp kernel, which therefore keeps those.)

struct alignas(64) WsMaps {
  CUtensorMap value, reward, done, truncated, on_reset, old_logp;  // value / flags: boxes of kR + 1 rows
};
struct WsParams {
  GaeParams p;
  WsMaps maps;
};

template <bool PACK>
struct Slot {
  static constexpr int value = 0;                                   // f32 [kR + 1][32]
  static constexpr int reward = value + (kR + 1) * 128;             // f32 [kR][32]
  static constexpr int old_logp = reward + kR * 128;                // f32 [kR][32]   (PACK)
  static constexpr int done = old_logp + (PACK ? kR * 128 : 0);     // u8  [kR + 1][32], padded to 640 B
  static constexpr int truncated = done + 640;
  static constexpr int on_reset = truncated + 640;
  static constexpr int tx_bytes = (kR + 1) * 128 + kR * 128 + (PACK ? kR * 128 : 0) + 3 * (kR + 1) * 32;
  static constexpr int delta = on_reset + 640;                      // f64 [kR][32]
  static constexpr int mflag = delta + kR * 256;                    // u8  [kR][32]
  static constexpr int adv = mflag + kR * 32;                       // f32 [kR][32]
  static constexpr int vprime = adv + kR * 128;                     // f32 [kR][32]
  static constexpr int bytes = vprime + kR * 128;
  static_assert(bytes % 128 == 0, "slots stay 128-byte aligned");
};

template <int kS>
struct Bars {
  uint64_t tma_full[kS], pass1[kS], scanned[kS], empty[kS];
};

template <bool PACK, int kW, int kS>
__global__ void __launch_bounds__(32 * (2 + kW)) gae_scan_ws_kernel(const __grid_constant__ WsParams q) {
  constexpr int kRowsPerWorker = kR / kW;
  constexpr int kAhead = kS > 3 ? kS - 1 : 1;  // chunks the workers' delta pass runs ahead of their store pass
  constexpr int kStatsOff = (sizeof(Bars<kS>) + 255) / 256 * 256;
  constexpr int kPartOff = kStatsOff + kW * 7 * 32 * static_cast<int>(sizeof(double));  // [3][32] f64 lane sums, [kPartEpochs][32] u8 map
  constexpr int kThreads = 32 * (2 + kW);
  using SL = Slot<PACK>;
  extern __shared__ __align__(128) unsigned char smem[];
  Bars<kS>* bars = reinterpret_cast<Bars<kS>*>(smem + kS * SL::bytes);
  if (threadIdx.x == 0) SRL_TL(1, blockIdx.x, 0);
  // the kernel behind this one on the stream (the loss) may become resident now; it waits for this grid's completion
  // before it reads anything written here
  pdl_launch_dependents();
  const GaeParams& p = q.p;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = blockIdx.x * 32, col = col0 + lane;
  const bool live = col < p.N;
  const int L = p.L, N = p.N;
  const int n_chunks = (L + kR - 1) / kR;  // chunk c (processing order) covers rows [(n_chunks-1-c)*kR, +kR)

  if (threadIdx.x == 0) {
    for (int s = 0; s < kS; ++s) {
      mbar_init(&bars->tma_full[s], 1);
      mbar_init(&bars->pass1[s], kW);
      mbar_init(&bars->scanned[s], 1);
      mbar_init(&bars->empty[s], kW);
    }
    mbar_fence_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) SRL_TL(1, blockIdx.x, 1);

  if (warp == 0) {
    // ---- producer ----------------------------------------------------------------------------------------------
    if (lane == 0) {
      prefetch_map(&q.maps.value);
      prefetch_map(&q.maps.reward);
      prefetch_map(&q.maps.done);
      prefetch_map(&q.maps.truncated);
      prefetch_map(&q.maps.on_reset);
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % kS;
        if (c >= kS) mbar_wait(&bars->empty[s], ((c / kS) - 1) & 1);  // every worker is done with chunk c - kS
        unsigned char* slot = smem + s * SL::bytes;
        const int row0 = (n_chunks - 1 - c) * kR;
        mbar_expect_tx(&bars->tma_full[s], SL::tx_bytes);
        tma_load_2d(slot + SL::value, &q.maps.value, col0, row0, &bars->tma_full[s]);
        tma_load_2d(slot + SL::reward, &q.maps.reward, col0, row0, &bars->tma_full[s]);
        tma_load_2d(slot + SL::done, &q.maps.done, col0, row0, &bars->tma_full[s]);
        tma_load_2d(slot + SL::truncated, &q.maps.truncated, col0, row0, &bars->tma_full[s]);
        tma_load_2d(slot + SL::on_reset, &q.maps.on_reset, col0, row0, &bars->tma_full[s]);
        if (PACK) tma_load_2d(slot + SL::old_logp, &q.maps.old_logp, col0, row0, &bars->tma_full[s]);
      }
      SRL_TL(1, blockIdx.x, 2);
    }
  } else if (warp == 1) {
    // ---- scanner: A_t = delta_t + m_t * A_{t+1} ---------------------------------------------------------------------
    const double gl = p.gamma_lmbda;
    double g = 0.0;
    for (int c = 0; c < n_chunks; ++c) {
      const int s = c % kS;
      unsigned char* slot = smem + s * SL::bytes;
      mbar_wait(&bars->pass1[s], (c / kS) & 1);
      const double* sd = reinterpret_cast<const double*>(slot + SL::delta);
      const uint8_t* sm = slot + SL::mflag;
      float* sa = reinterpret_cast<float*>(slot + SL::adv);
      // (Leaving out the chain steps of the rows behind the trajectory's end -- 15 of cfg2's 144 -- was measured twice:
      // with a per-row predicate it put two selects on the chain, +1.0 us per step; as one uniform branch around the first
      // chunk it changed nothing, 30.41 -> 30.55 us: the scanner waits for the workers there.  profiles/r2_notes.md)
      double d[kR];
      double m[kR];
#pragma unroll
      for (int r = 0; r < kR; ++r) {
        d[r] = sd[r * 32 + lane];
        m[r] = gae_carry(sm[r * 32 + lane] != 0, gl);
      }
#pragma unroll
      for (int r = kR - 1; r >= 0; --r) {
        g = gae_step(d[r], m[r], g);
        sa[r * 32 + lane] = static_cast<float>(g);  // adv.float(), gae.py:97
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->scanned[s]);
    }
    if (lane == 0) SRL_TL(1, blockIdx.x, 4);
  } else {
    // ---- workers ---------------------------------------------------------------------------------------------------
    const int w = warp - 2;
    const bool popart = p.popart != nullptr;
    double pa_mean = 0.0, pa_std = 1.0;
    if (popart) {
      pa_mean = p.popart[0];
      pa_std = p.popart[1];
    }
    const double gamma = p.gamma;
    // srl_gae_scan_perm: the step's minibatch permutations, computed by the worker threads of all CTAs while their first
    // chunk is in flight (~1.3 us in which they would only wait).  One launch and one completion hop less between the scan
    // and the loss than with the permutation kernel beside the scan; bit-identical to srl_philox_perm (perm.cuh).
    if (p.perm.out != nullptr) {
      const long long total = static_cast<long long>(p.perm.n_epochs) * p.perm.n_env;
      const int wt = w * 32 + lane;
      uint32_t have_epoch = 0xffffffffu;
      PermKeys keys;
      for (long long g = static_cast<long long>(blockIdx.x) * (32 * kW) + wt; g < total;
           g += static_cast<long long>(gridDim.x) * (32 * kW)) {
        const uint32_t ep = static_cast<uint32_t>(g / p.perm.n_env);
        const uint32_t e = static_cast<uint32_t>(g - static_cast<long long>(ep) * p.perm.n_env);
        if (ep != have_epoch) {
          keys = perm_keys(p.perm.seed_lo, p.perm.seed_hi, p.perm.epoch0 + ep, p.perm.bits);
          have_epoch = ep;
        }
        const uint32_t x = perm_at(e, static_cast<uint32_t>(p.perm.n_env), keys);
        int32_t* o = p.perm.out + (static_cast<size_t>(ep) * p.perm.n_env + e) * p.perm.group;
        for (int a = 0; a < p.perm.group; ++a) o[a] = static_cast<int32_t>(x) * p.perm.group + a;
      }
    }
    // ... and, for the loss kernel's minibatch statistics, the minibatch of each of THIS CTA's 32 lanes in every epoch (the
    // inverse permutation: a Feistel network runs backwards as well), kept in shared memory for the end of the kernel
    if (p.perm.out != nullptr && p.perm.part != nullptr) {
      uint8_t* s_mb = smem + kS * SL::bytes + kPartOff + 3 * 32 * sizeof(double);
      for (int i = w * 32 + lane; i < p.perm.n_epochs * 32; i += 32 * kW) {
        const int ep = i >> 5, c2 = col0 + (i & 31);
        int slot = 255;
        if (c2 < N) {
          const PermKeys keys = perm_keys(p.perm.seed_lo, p.perm.seed_hi, p.perm.epoch0 + ep, p.perm.bits);
          const uint32_t env = static_cast<uint32_t>(c2 / p.perm.group);
          const long long pos = static_cast<long long>(perm_pos_of(env, static_cast<uint32_t>(p.perm.n_env), keys)) * p.perm.group +
                                (c2 - static_cast<int>(env) * p.perm.group);
          slot = ep * p.perm.minibatches + static_cast<int>(pos / p.perm.per_mb);
        }
        s_mb[i] = static_cast<uint8_t>(slot);
      }
    }
    LaneStats st;
    // pass 1 of chunk c: v', delta_t and the carry flag of this warp's rows
    auto pass1 = [&](int c) {
      const int s = c % kS;
      unsigned char* slot = smem + s * SL::bytes;
      mbar_wait(&bars->tma_full[s], (c / kS) & 1);
      if (c == 0 && w == 0 && lane == 0) SRL_TL(1, blockIdx.x, 3);
      const float* sv = reinterpret_cast<const float*>(slot + SL::value);
      const float* sr = reinterpret_cast<const float*>(slot + SL::reward);
      const uint8_t* sdn = slot + SL::done;
      const uint8_t* str_ = slot + SL::truncated;
      const uint8_t* srs = slot + SL::on_reset;
      double* sd = reinterpret_cast<double*>(slot + SL::delta);
      uint8_t* sm = slot + SL::mflag;
      float* svp = reinterpret_cast<float*>(slot + SL::vprime);
      const int tbase = (n_chunks - 1 - c) * kR;
#pragma unroll
      for (int i = 0; i < kRowsPerWorker; ++i) {
        const int r = w * kRowsPerWorker + i;
        const int t = tbase + r;
        const float v0 = gae_vprime(sv[r * 32 + lane], sdn[r * 32 + lane] != 0, popart, pa_mean, pa_std);
        const float v1 = gae_vprime(sv[(r + 1) * 32 + lane], sdn[(r + 1) * 32 + lane] != 0, popart, pa_mean, pa_std);
        const bool rn = srs[(r + 1) * 32 + lane] != 0, tn = str_[(r + 1) * 32 + lane] != 0;
        const double dlt = gae_delta(&sr[r * 32 + lane], v0, v1, rn, gamma);
        const bool scanned = t < L - 1;  // row L-1 (padding row) and the zero-filled rows beyond carry no advantage
        sd[r * 32 + lane] = scanned ? dlt : 0.0;
        sm[r * 32 + lane] = (scanned && !rn && !tn) ? 1 : 0;  // the scanner's gae_carry flag
        svp[r * 32 + lane] = v0;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->pass1[s]);
    };
    // pass 3 of chunk c: value target, stores, pack, per-lane statistics
    auto pass3 = [&](int c) {
      const int s = c % kS;
      unsigned char* slot = smem + s * SL::bytes;
      mbar_wait(&bars->scanned[s], (c / kS) & 1);
      const float* sv = reinterpret_cast<const float*>(slot + SL::value);
      const float* sol = reinterpret_cast<const float*>(slot + SL::old_logp);
      const uint8_t* sdn = slot + SL::done;
      const uint8_t* str_ = slot + SL::truncated;
      const uint8_t* srs = slot + SL::on_reset;
      const float* sa = reinterpret_cast<const float*>(slot + SL::adv);
      const float* svp = reinterpret_cast<const float*>(slot + SL::vprime);
      const int tbase = (n_chunks - 1 - c) * kR;
#pragma unroll
      for (int i = 0; i < kRowsPerWorker; ++i) {
        const int r = w * kRowsPerWorker + i;
        const int t = tbase + r;
        const float a = sa[r * 32 + lane];
        const float rt = (t < L - 1) ? gae_value_target(a, svp[r * 32 + lane]) : 0.f;
        const bool rn = srs[(r + 1) * 32 + lane] != 0;
        if (live && t < L) {  // row L-1 is the zero padding row of mappo.py:254-256
          const size_t gi = static_cast<size_t>(t) * N + col;
          stg_stream(p.adv + gi, a);
          stg_stream(p.ret + gi, rt);
          if (PACK && (r & 1) == 0) {
            // the pack's row pair (t, t + 1) as ONE 32-byte store: chunks start at even rows, and everything row t + 1
            // needs (its advantage, v', flags) is in this chunk's slot once the scanner has signalled it
            const float a1 = sa[(r + 1) * 32 + lane];
            const float rt1 = (t + 1 < L - 1) ? gae_value_target(a1, svp[(r + 1) * 32 + lane]) : 0.f;
            const bool keep1 = t + 1 < L - 1 && srs[(r + 2) * 32 + lane] == 0;
            st_cg256(reinterpret_cast<float4*>(p.pack) + pack_index(t, N, col),
                     pack_item(sol[r * 32 + lane], sv[r * 32 + lane], rt, a, !rn && t < L - 1),
                     pack_item(sol[(r + 1) * 32 + lane], sv[(r + 1) * 32 + lane], rt1, a1, keep1));
          }
        }
        // loss rows [row_lo, row_hi), mask = 1 - on_reset[t+1]   mappo.py:259-261
        const bool in_rows = t >= p.row_lo && t < p.row_hi;
        st.add(in_rows, in_rows && !rn, a, rt, sdn[r * 32 + lane] != 0, str_[r * 32 + lane] != 0);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->empty[s]);
    };

    for (int c = 0; c < kAhead && c < n_chunks; ++c) pass1(c);
    for (int c = 0; c < n_chunks; ++c) {
      if (c + kAhead < n_chunks) pass1(c + kAhead);  // stay ahead of the scanner
      pass3(c);
    }
    if (w == 0 && lane == 0) SRL_TL(1, blockIdx.x, 5);
    // per-lane statistics of this worker -> shared memory; the workers' tables are added in worker order below (fixed)
    if (p.lane_part != nullptr) {
      double* red = reinterpret_cast<double*>(smem + kS * SL::bytes + kStatsOff) + (w * 7) * 32;  // [kW][7][32] f64, own region
      red[0 * 32 + lane] = static_cast<double>(st.cnt);
      red[1 * 32 + lane] = st.s1;
      red[2 * 32 + lane] = st.s2;
      red[3 * 32 + lane] = st.s3;
      red[4 * 32 + lane] = st.s4;
      red[5 * 32 + lane] = static_cast<double>(st.dn);
      red[6 * 32 + lane] = static_cast<double>(st.tr);
    }
  }
  __syncthreads();
  if (p.lane_part != nullptr) {
    const double* red = reinterpret_cast<const double*>(smem + kS * SL::bytes + kStatsOff);
    double* lsum = reinterpret_cast<double*>(smem + kS * SL::bytes + kPartOff);  // the minibatch shares' lane sums
    fold_lane_sums<32, kW, kThreads>(p, red, [&](int k, int ln, double sum) {
      if (k < 3) lsum[k * 32 + ln] = sum;
    });
    if (p.perm.out != nullptr && p.perm.part != nullptr) {
      // this CTA's share of every minibatch's {count, sum, sum of squares}, part[slot][cta][4]: the loss kernel adds
      // gridDim.x shares per minibatch (one coalesced round of loads) instead of gathering the minibatch's lane items
      // through the permutation (two dependent rounds).  Four threads per output, 8 lanes each in lane order, then
      // (q0 + q1) + (q2 + q3): a fixed order.
      __syncthreads();
      const uint8_t* s_mb = smem + kS * SL::bytes + kPartOff + 3 * 32 * sizeof(double);
      const int outs = p.perm.n_epochs * p.perm.minibatches * 4;
      for (int i = threadIdx.x; i < ((outs * 4 + 31) & ~31); i += kThreads) {  // whole warps iterate together
        const int o = i >> 2, qr = i & 3;
        const int slot = o >> 2, k = o & 3;
        double acc = 0.0;
        if (o < outs && k < 3) {
          const uint8_t* mb = s_mb + (slot / p.perm.minibatches) * 32 + qr * 8;
          const double* ls = lsum + k * 32 + qr * 8;
#pragma unroll
          for (int ln = 0; ln < 8; ++ln) acc += mb[ln] == slot ? ls[ln] : 0.0;
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (o < outs && qr == 0) p.perm.part[(static_cast<size_t>(slot) * gridDim.x + blockIdx.x) * 4 + k] = acc;
      }
    }
  }
  // Launched programmatically behind the permutation kernel, this grid never waited for it (it does not read the
  // permutation).  Waiting here, before the grid completes, makes "scan complete" imply "permutation complete and
  // visible" for the loss kernel, whose own griddepcontrol.wait only covers this grid.
  if (threadIdx.x == 0) {
    SRL_TL(1, blockIdx.x, 6);
    pdl_wait();
    SRL_TL(1, blockIdx.x, 7);
  }
}

template <bool PACK, int kW, int kS>
int launch_ws(const WsParams& q, cudaStream_t st) {
  const size_t smem = 3 * 32 * sizeof(double) + kPartEpochs * 32 +  // lane sums + lane -> minibatch map (srl_gae_scan_perm)
                      static_cast<size_t>(kS) * Slot<PACK>::bytes + (sizeof(Bars<kS>) + 255) / 256 * 256 +
                      static_cast<size_t>(kW) * 7 * 32 * sizeof(double);
  constexpr auto kern = gae_scan_ws_kernel<PACK, kW, kS>;
  const int rc = opt_in_smem<kern>(smem);
  if (rc != SRL_OK) return rc;
  const int grid = (q.p.N + 31) / 32;
  SRL_CUDA(launch_pdl_scan(kern, dim3(grid), dim3(32 * (2 + kW)), smem, st, q));
  return SRL_OK;
}

}  // namespace
}  // namespace srl
SRL_TL_SETTER(srl_tl_set_gae)
namespace srl {

bool gae_ws_eligible(const GaeParams& p) { return p.vt_new_logp == nullptr && gae_tma_eligible(p); }

int launch_gae_ws(const GaeParams& p, cudaStream_t st) {
  WsParams q;
  q.p = p;
  int rc;
  // at most one CTA per SM anyway: spend the SM's shared memory on a ring that holds the whole trajectory
  const bool deep = (p.N + 31) / 32 <= sm_count();
  if ((rc = tma::make_map(&q.maps.value, p.value, p.L, p.N, 4, 32, kR + 1)) != SRL_OK) return rc;
  if ((rc = tma::make_map(&q.maps.reward, p.reward, p.L, p.N, 4, 32, kR)) != SRL_OK) return rc;
  if ((rc = tma::make_map(&q.maps.done, p.done, p.L, p.N, 1, 32, kR + 1)) != SRL_OK) return rc;
  if ((rc = tma::make_map(&q.maps.truncated, p.truncated, p.L, p.N, 1, 32, kR + 1)) != SRL_OK) return rc;
  if ((rc = tma::make_map(&q.maps.on_reset, p.on_reset, p.L, p.N, 1, 32, kR + 1)) != SRL_OK) return rc;
  if (p.pack != nullptr) {
    if ((rc = tma::make_map(&q.maps.old_logp, p.old_logp, p.L, p.N, 4, 32, kR)) != SRL_OK) return rc;
    return deep ? launch_ws<true, 16, kDeep>(q, st) : launch_ws<true, 16, 3>(q, st);
  }
  return deep ? launch_ws<false, 16, kDeep>(q, st) : launch_ws<false, 16, 3>(q, st);
}

}  // namespace srl
