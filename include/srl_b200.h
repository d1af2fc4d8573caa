/* srl_b200.h -- C-ABI of the B200-native SRL trainer hot path (libsrl_b200.so).
 *
 * Every entry point takes raw DEVICE pointers, plain sizes and a cudaStream_t (as void*), launches
 * asynchronously on that stream and returns an int status (SRL_OK == 0).  Nothing here aborts: the
 * Python plugin turns a non-zero status into an exception, which is the reference's error
 * convention at this boundary (exceptions propagate out of Trainer.step, api/trainer.py:117 /
 * distributed/system/trainer_worker.py:171,496-498).  No torch types appear in any signature.
 *
 * Layout contract (reference: base/buffer.py:118-126): every per-transition leaf is TIME-MAJOR
 * [L, N] with the N = B * n_agents lanes contiguous (the trailing size-1 dim of the reference's
 * [L, B, (A,) 1] leaves is dropped).  Values are float32; flags are uint8 as the actor workers
 * emit them (distributed/system/actor_worker.py:278-281) -- the reference inflates them to float32
 * on device (api/trainer.py:217), this library does not.
 *
 * Each function names the reference code it replaces (paths relative to the SRL repo root).
 */
#ifndef SRL_B200_H_
#define SRL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRL_B200_ABI_VERSION 12

typedef void* srl_stream_t; /* cudaStream_t */

enum srl_status {
  SRL_OK = 0,
  SRL_ERR_INVALID_ARG = 1, /* null pointer, negative size, misaligned pointer ... */
  SRL_ERR_UNSUPPORTED = 2, /* valid request this build cannot serve (e.g. L too long for smem) */
  SRL_ERR_CUDA = 3,        /* a CUDA runtime call failed; see srl_last_error() */
  SRL_ERR_NO_DEVICE = 4    /* no sm_100 device visible */
};

/* Thread-local, NUL-terminated description of the last non-OK status returned on this thread. */
const char* srl_last_error(void);
int srl_abi_version(void);
/* Programmatic dependent launch between the kernels of a step (default on; SRL_PDL=0 in the environment or
 * srl_set_pdl(0) turns it off; srl_set_pdl returns the previous setting).  On: srl_gae_scan and the loss kernels are
 * launched with cudaLaunchAttributeProgrammaticStreamSerialization, so that on ONE stream the order
 * srl_philox_perm -> srl_gae_scan -> srl_ppo_loss_* overlaps: the scan starts beside the permutation kernel, and the loss
 * kernel's CTAs become resident and pull their policy-side rows into L2 while the scan still runs; each kernel waits
 * (griddepcontrol.wait) before it touches anything an earlier kernel writes, so results do not change.
 * The scan is launched programmatically ONLY directly behind srl_philox_perm on the same stream and thread (the library
 * notes that launch): it waits for its predecessor only at its end, which is correct exactly when the predecessor writes
 * nothing the scan reads.  Behind any other kernel it is an ordinary launch.  The loss kernels wait first and are always
 * launched programmatically. */
int srl_pdl_enabled(void);
int srl_set_pdl(int on);
/* Fills SM count and compute capability of the current device. */
int srl_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * K2  GAE / value-target reverse-time scan.
 * Replaces MultiAgentPPO._compute_adv_and_value_target (legacy/algorithm/ppo/mappo.py:118-144),
 * modules.gae_trace (legacy/algorithm/modules/gae.py:8-97, float64 scan, float32 result), the
 * zero-row padding at mappo.py:254-256 and, for the statistics, the reductions inside
 * masked_normalization (legacy/algorithm/modules/utils.py:54-57) and RunningMeanStd.update
 * (utils.py:113-120).
 *
 *   v'[t]  = (popart ? float(double(value)*std + mean) : value) * (1 - done[t])        (fp32)
 *   d[t]   = reward[t] + gamma * v'[t+1] * (1 - on_reset[t+1]) - v'[t]                  (fp64, no FMA)
 *   m[t]   = gamma * lmbda * (1 - on_reset[t+1]) * (1 - truncated[t+1])                 (fp64)
 *   vtrace: rho_t = exp(new_logp - old_logp); d *= min(rho_t, rho); m *= min(rho_t, c)
 *   A[t]   = d[t] + m[t] * A[t+1], A[L-1] = 0 ;  adv = float(A) ;  ret = adv + v'[t]   (fp32 add)
 *   adv[L-1] = ret[L-1] = 0 (padding row).
 *
 * pack (optional, may be NULL; needs old_logp): the sample side of the loss as ONE 16-byte item per transition,
 * {old_logp[t], value[t] (as stored in the sample), ret[t], mask[t] ? adv[t] : NaN} with mask[t] = 1 - on_reset[t+1]
 * (row L-1: NaN).  With V-trace the first column is vtrace_old_logp[t] for rows 0..L-2 and 0 in row L-1, and old_logp is
 * not read (it must still be non-NULL).  The two rows of a row pair sit next to each other: item (t, lane) is float4 number
 * ((t / 2) * N + lane) * 2 + t % 2, i.e. float32 [ceil(L / 2), N, 2, 4] (so the buffer holds L + L % 2 rows), 32-byte
 * aligned.  A minibatch that gathers lanes through a permutation (srl_ppo_loss_fwd_bwd_batched, `pack`) then issues one
 * 256-bit load per lane and ROW PAIR -- every 32-byte sector it touches is used whole -- instead of five narrow loads per
 * transition.
 *
 * lane_part (optional, may be NULL): [SRL_LANE_PART][N] float64 per-lane sums over the loss rows
 * t in [row_lo, row_hi) with mask[t] = 1 - on_reset[t+1] (mappo.py:259-261):
 *   0: sum mask   1: sum adv*mask   2: sum (adv*mask)^2   3: sum ret*mask   4: sum (ret*mask)^2
 *   5: sum done[t]   6: sum truncated[t]   7: reserved (0)
 * lane_aos (optional, may be NULL; needs lane_part): [N][4] float64, 32-byte aligned: rows 0..2 of lane_part once more, one
 * 32-byte item per lane {sum mask, sum adv*mask, sum (adv*mask)^2, 0} -- the form in which the loss kernel adds the
 * statistics of a permuted minibatch itself (one 256-bit gather per lane; srl_ppo_loss_fwd_bwd_batched, `lane_aos`).
 * ------------------------------------------------------------------------------------------ */
#define SRL_LANE_PART 8

int srl_gae_scan(const float* reward,          /* [L, N]; row L-1 is ignored                    */
                 const float* value,           /* [L, N]                                        */
                 const uint8_t* done,          /* [L, N]                                        */
                 const uint8_t* truncated,     /* [L, N]                                        */
                 const uint8_t* on_reset,      /* [L, N]                                        */
                 const float* vtrace_new_logp, /* [L-1, N] or NULL (vtrace off)                 */
                 const float* vtrace_old_logp, /* [L-1, N] or NULL                              */
                 const double* popart_mean_std, /* device {mean, std} or NULL (popart off)      */
                 const float* old_logp,        /* [L, N] or NULL (only read when pack != NULL)  */
                 int L, int N, int row_lo, int row_hi, double gamma, double lmbda, double rho, double c,
                 float* adv,        /* [L, N] out */
                 float* ret,        /* [L, N] out */
                 double* lane_part, /* [SRL_LANE_PART, N] out or NULL */
                 double* lane_aos,  /* [N, 4] out or NULL */
                 float* pack,       /* [ceil(L/2), N, 2, 4] out or NULL */
                 srl_stream_t stream);

/* srl_gae_scan + the step's minibatch permutations (== srl_philox_perm(perm_seed, perm_epoch, perm_n_epochs, perm_n_env,
 * perm_group, perm_out), bit for bit) in the same launch where the scan kernel chosen for this shape can: its worker
 * threads compute them while they wait for their first tile (the warp-specialised kernel of small batches -- the shape
 * whose step is latency-bound).  Otherwise the stand-alone permutation kernel is launched behind the scan.
 * minibatch_part (optional, device [SRL_MAX_LOSS_BATCH][ceil(N / 32)][4] float64, 32-byte aligned; needs lane_part and
 * n_env * group == N): every scan CTA also adds ITS 32 lanes' {sum mask, sum adv*mask, sum (adv*mask)^2, 0} per minibatch
 * -- minibatch j of epoch e = positions [j * N / perm_minibatches, ...) of epoch e's permuted lane list, table slot
 * e * perm_minibatches + j, item [slot][scan CTA] -- so that the loss kernel adds ceil(N / 32) partial sums per minibatch
 * (one coalesced round of loads) instead of gathering the minibatch's lanes through the permutation (two dependent
 * rounds): srl_ppo_loss_fwd_bwd_batched, `minibatch_part`.
 * *fused (host, may be NULL): 0 = two launches and no partial sums, 1 = one launch (permutations only: more than 8
 * epochs or SRL_MAX_LOSS_BATCH minibatches), 2 = one launch with the partial sums.  New capability, like
 * srl_philox_perm (SURVEY.md F2). */
int srl_gae_scan_perm(const float* reward, const float* value, const uint8_t* done, const uint8_t* truncated,
                      const uint8_t* on_reset, const float* vtrace_new_logp, const float* vtrace_old_logp,
                      const double* popart_mean_std, const float* old_logp, int L, int N, int row_lo, int row_hi,
                      double gamma, double lmbda, double rho, double c, float* adv, float* ret, double* lane_part,
                      double* lane_aos, float* pack, uint64_t perm_seed, uint32_t perm_epoch, int perm_n_epochs,
                      int perm_n_env, int perm_group, int32_t* perm_out, int perm_minibatches, double* minibatch_part,
                      int* fused, srl_stream_t stream);

/* The general form of the same scan: everything modules.gae_trace (legacy/algorithm/modules/gae.py:8-97) accepts
 * beyond what MultiAgentPPO passes -- vector critics (reward / value / adv / ret are [.., N, critic_dim], the flags stay
 * [.., N] and broadcast over the critic axis, gae.py:26-30), per-element discount / lambda tensors (gamma_t, lmbda_t:
 * [L-1, N] float32 or NULL = the scalar; gae.py:31-34,51-60: gamma_t * lmbda_t is a float64 product per element) and a
 * ready-made importance ratio (imp_ratio [L-1, N] or NULL; gae.py:36,64-65,88-89).
 *   done == NULL : `value` is used as it is (plain gae_trace); else v' = value * (1 - done) in float32 (mappo.py:120-124)
 *   ret  == NULL : advantages only (gae_trace's return value); else ret = adv + v' in float32 (mappo.py:143)
 *   pad_last_row : adv / ret have L rows and row L-1 is zeroed (mappo.py:254-256); else they have L-1 rows.
 * Same float64 rounding sequence as srl_gae_scan (bit-identical where both apply); no statistics, no pack. */
int srl_gae_trace(const float* reward,       /* [>= L-1, N, critic_dim]                    */
                  const float* value,        /* [L, N, critic_dim]                         */
                  const uint8_t* done,       /* [L, N] or NULL                             */
                  const uint8_t* truncated,  /* [L, N]                                     */
                  const uint8_t* on_reset,   /* [L, N]                                     */
                  const float* gamma_t,      /* [L-1, N] or NULL                           */
                  const float* lmbda_t,      /* [L-1, N] or NULL                           */
                  const float* imp_ratio,    /* [L-1, N] or NULL (V-trace off)             */
                  int L, int N, int critic_dim, double gamma, double lmbda, double rho, double c, int pad_last_row,
                  float* adv, float* ret, srl_stream_t stream);

/* GAE along whole episodes: replaces TrajGAE.process (legacy/algorithm/modules/gae.py:100-139, the 'gae' trajectory
 * post-processor of api/trainer.py:84-99,249-262) for MANY episodes in one launch.  Episode k occupies steps
 * [offsets[k], offsets[k+1]) of reward / value / adv / ret, each [total_steps, width] in the arrays' own dtype
 * (float32, or float64 when is_float64 != 0 -- numpy semantics: the python scalars gamma and gamma * lmbda are rounded
 * to the array dtype, every operation rounds in that dtype).  For steps s = len-2 .. 0 of an episode:
 *   boot  = s == len-2 ? (final_has_value[k] ? value[last] * final_truncated[k] : 0) : value[s+1]
 *   delta = reward[s] + gamma * boot - value[s];  gae = gamma * lmbda * gae + delta
 *   adv[s] = gae;  ret[s] = gae + value[s]
 * The last step of every episode is left untouched, as in the reference. */
int srl_traj_gae(const void* reward, const void* value, const int64_t* offsets /* device [n_traj + 1] */,
                 const uint8_t* final_truncated /* device [n_traj, width] */,
                 const uint8_t* final_has_value /* device [n_traj] */, int n_traj, int width, int is_float64,
                 double gamma, double lmbda, void* adv, void* ret, srl_stream_t stream);

/* n-step return on the same [rows, N] layout (rows = n + T - 1): replaces modules.n_step_return
 * (legacy/algorithm/modules/n_step_return.py:11-50; the return estimator of the DQN / QMIX trainers), float64 with the
 * reference's operation order, float32 result out[T, N]:
 *   ret += reward[t+i] * disc;  ret += disc * gamma * nex_truncated[t+i] * nex_value[t+i];
 *   disc *= gamma * (1 - nex_done[t+i]) * (1 - nex_truncated[t+i])   for i in [0, n);  out[t] = ret + disc * nex_value[t+n-1] */
int srl_n_step_return(const float* reward, const float* nex_value, const uint8_t* nex_done,
                      const uint8_t* nex_truncated, int n, int rows, int N, double gamma, float* out,
                      srl_stream_t stream);

/* The same [SRL_LANE_PART][N] table from adv / ret that already exist: a sample re-served by the buffer carries
 * them in its host copy and MultiAgentPPO.step skips GAE for it (mappo.py:224-225,249 with
 * recompute_adv_on_reuse=False; base/buffer.py:142-162 re-serves a ReplayEntry `reuses` times). */
int srl_lane_stats(const float* adv, const float* ret, const uint8_t* done, const uint8_t* truncated,
                   const uint8_t* on_reset, int L, int N, int row_lo, int row_hi, double* lane_part,
                   srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Group statistics: out[g][k] = sum over the lanes of group g of lane_part[k][lane].
 * Group g holds the `per` lanes idx[g*per .. (g+1)*per) (idx == NULL: identity).  One group per
 * minibatch; with G == 1 and per == N this is the whole-batch reduction of utils.py:54-57 /
 * utils.py:113-120.  The [G, SRL_LANE_PART] float64 table is what gets all-reduced (SUM) across
 * ranks in place of the 3 + 3 one-element all-reduces of utils.py:58-61,121-124.
 * whole_first != 0: out has G + 1 rows and row 0 is the sum over ALL N lanes (the batch statistics PopArt
 * needs), rows 1..G are the groups -- one launch for the whole table.
 * Summation order is fixed (deterministic for a given G, per).
 * Rows longer than 512 lanes are summed by several CTAs through `workspace` (srl_group_stats_workspace_bytes()
 * bytes, 8-byte aligned, zero before its FIRST use; the kernel leaves it zeroed); shorter rows need none (NULL).
 * ------------------------------------------------------------------------------------------ */
size_t srl_group_stats_workspace_bytes(int G, int whole_first);
int srl_group_stats(const double* lane_part, int N, const int32_t* idx, int G, int per, int whole_first,
                    double* out, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3  PopArt / RunningMeanStd update for a scalar critic (critic_dim == 1).
 * Replaces RunningMeanStd.update + mean_std (utils.py:106-137) as called from
 * PopArtValueHead.update (legacy/algorithm/modules/popart.py:42-47).
 *   state = {mean, mean_sq, debias, update_count} (float64, device, updated in place)
 *   batch_stats: one row of the group-stats table; uses [0] = sum mask, [3] = sum x, [4] = sum x^2.
 *   mean_std_out = {mu, sigma, mu_before, sigma_before} (float64[4]): mu = mean/max(debias,eps),
 *   sigma = sqrt(max(mean_sq/max(debias,eps) - mu^2, 1e-2)); the "before" pair is what PopArtValueHead.update
 *   needs to rescale the head (popart.py:43,49-51).
 * ------------------------------------------------------------------------------------------ */
int srl_popart_update(const double* batch_stats, double* state, double beta, double eps, double* mean_std_out,
                      srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4  Fused PPO / MAPPO loss, forward + backward to (new_logp, state_values, entropy).
 * Replaces MultiAgentPPO._compute_loss (mappo.py:146-217) + masked_normalization (utils.py:10-67)
 * + get_clip_value_loss_fn / init_value_loss_fn (utils.py:228-265) + loss.backward() down to the
 * three differentiable inputs (mappo.py:274) + the eleven .mean().item() stats (mappo.py:293-299).
 * ------------------------------------------------------------------------------------------ */
enum srl_value_loss { SRL_VL_MSE = 0, SRL_VL_HUBER = 1, SRL_VL_SMOOTHL1 = 2 };

typedef struct srl_ppo_hyper {
  double eps_clip;             /* mappo.py:75 */
  double value_eps_clip;       /* mappo.py:90 */
  double c_clip;               /* mappo.py:78 */
  double value_loss_weight;    /* mappo.py:91 */
  double entropy_bonus_weight; /* mappo.py:93 */
  double vl_param;             /* HuberLoss delta / SmoothL1Loss beta (value_loss_config) */
  double adv_eps;              /* masked_normalization eps, 1e-5 (utils.py:17) */
  int32_t value_loss;          /* enum srl_value_loss */
  int32_t clip_value;          /* mappo.py:76 */
  int32_t dual_clip;           /* mappo.py:77 */
  int32_t normalize_old_value; /* mappo.py:86 (needs popart_mean_std) */
} srl_ppo_hyper;

/* indices into the float64 result vector written by srl_ppo_loss_fwd_bwd */
enum srl_loss_out {
  SRL_OUT_LOSS = 0,
  SRL_OUT_POLICY_LOSS = 1,
  SRL_OUT_VALUE_LOSS = 2,
  SRL_OUT_ENTROPY_LOSS = 3,
  SRL_OUT_ADVANTAGE = 4,         /* mean(adv[mask])                    mappo.py:206 */
  SRL_OUT_IMPORTANCE_WEIGHT = 5, /* mean(ratio[mask])                  mappo.py:212 */
  SRL_OUT_CLIP_RATIO = 6,        /* mean((s2 < s1)[mask])              mappo.py:213 */
  SRL_OUT_VALUE_TARGETS = 7,     /* mean(normalised target[mask])      mappo.py:214 */
  SRL_OUT_DENORM_VALUE = 8,      /* mean(ret[mask]) (popart only)      mappo.py:215-216 */
  SRL_OUT_MASK_SUM = 9,          /* local sum(mask)                                 */
  SRL_LOSS_OUT_LEN = 16
};

/* Bytes of one device scratch "slot" for a [T, n] problem: a 64-byte header + one float64[8] partial row per
 * CTA.  A slot must be ALL ZERO before its first use; every kernel that uses it leaves its state zero again (ticket
 * counter in bytes 0-3, published statistics in bytes 32-63, partial rows from byte 64: "zero" means "not there yet" to
 * the kernels that wait for a word; bytes 4-31 hand n_rows / sum(mask) / the weights from a deferred launch to
 * srl_ppo_loss_finalize and keep their last values), so a deferred launch must be followed by srl_ppo_loss_finalize
 * before the slot is used again.  Launches that may overlap in time need distinct slots. */
size_t srl_ppo_loss_workspace_bytes(int T, int n);

/* Deferred finalisation: when srl_ppo_loss_fwd_bwd / srl_ppo_loss_from_logits(_masked)(_bf16)(_pack) are called with out == NULL they
 * stop after writing gradients and partial rows.  This folds n_slots consecutive slots (slot k at
 * workspace + k * slot_bytes) into out[k][SRL_LOSS_OUT_LEN] (and out_f32[k][4] if not NULL) in one launch, and
 * clears the rows it folded. */
int srl_ppo_loss_finalize(void* workspace, size_t slot_bytes, int n_slots, double* out, float* out_f32,
                          srl_stream_t stream);

int srl_ppo_loss_fwd_bwd(
    /* policy side: dense [T, n], row stride ld_pol elements (analyze() output, mappo.py:244-246) */
    const float* new_logp, const float* v_pred, const float* entropy, int64_t ld_pol,
    /* sample side: row t of the loss = row (row_lo + t) of the [L, N] leaves; the caller passes
     * pointers already offset to row_lo (on_reset_next to row_lo + 1), row stride ld_smp.
     * lane_idx (int32[n]) selects columns (minibatch gather fused into the load) or NULL. */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats,      /* device [>=3]: GLOBAL (all-reduced) sum mask, sum x, sum x^2   */
    const double* local_stats,     /* device [>=1]: this rank's sum mask (== norm_stats if 1 rank) */
    const double* popart_mean_std, /* device {mu, sigma} or NULL                                  */
    const srl_ppo_hyper* hyper,    /* HOST pointer, copied by value into the launch              */
    float* g_logp, float* g_value, float* g_entropy, int64_t ld_grad, /* [T, n] out */
    double* out,      /* device [SRL_LOSS_OUT_LEN] out, or NULL = deferred (srl_ppo_loss_finalize) */
    float* out_f32,   /* device [4] out: loss, policy_loss, value_loss, entropy_loss, or NULL */
    void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* Several minibatches of ONE shape in one launch (a PPO step runs epochs x minibatches of them; launched one by
 * one each is a ~3 MB kernel that cannot fill 148 SMs).  Every problem carries its own policy-side tensors,
 * permutation slice, statistics rows, gradient tensors, outputs and workspace slot; the sample side is shared.
 * The sample side is either the five leaves of srl_ppo_loss_fwd_bwd (pack == NULL) or K2's pack (the BASE of the buffer
 * srl_gae_scan wrote, ld_smp = its N lanes, pack_row_lo = the absolute row of loss row 0; the leaf pointers may then be
 * NULL).  Either every problem has a lane_idx or none has.  n_problems > SRL_MAX_LOSS_BATCH is split into several launches.
 * lane_aos != NULL (K2's [N][4] table; pack form with lane indices, one GPU, no PopArt, even n <= 1024): every CTA adds the
 * per-lane sums of ITS minibatch's lanes itself and the problems' norm_stats / local_stats are ignored (may be NULL) --
 * no srl_group_stats launch between K2 and the loss.
 * minibatch_part != NULL (with lane_aos; the table srl_gae_scan_perm wrote when it reported *fused == 2, part_ctas =
 * ceil(N / 32) of that scan): problem k's sums are the part_ctas items of table slot part_first + k, added in a fixed order
 * -- problem k's lane_idx MUST be that slot's minibatch of the permutation the same scan wrote.
 * xchg != NULL (with lane_aos, several ranks): the kernel also adds every problem's three sums over the RANKS itself -- the
 * problem's first CTA stores this rank's sums into every rank's mailbox (NVLink peer memory, the srl_xchg_* protocol
 * below; capacity >= 3 * SRL_MAX_LOSS_BATCH doubles), every CTA collects them in rank order -- so the statistics
 * all-reduce of utils.py:58-61 costs one NVLink latency inside the loss kernel's prologue instead of two kernels between
 * the scan and the loss.  Every rank must launch the same sequence of calls on this srl_xchg; it must not be the object
 * srl_group_stats_xchg / srl_xchg_allreduce_sum use.
 * Gradient tensors must not alias the policy-side inputs (the kernels prefetch inputs of later rows before they store). */
#define SRL_MAX_LOSS_BATCH 32
struct srl_xchg; /* the peer-memory exchange handle, declared with its functions at the end of this header */
typedef struct srl_loss_problem {
  const float* new_logp;     /* [T, n], row stride ld_pol */
  const float* v_pred;
  const float* entropy;
  const int32_t* lane_idx;   /* device int32[n] or NULL */
  const double* norm_stats;  /* device [>=3] */
  const double* local_stats; /* device [>=1] */
  float* g_logp;             /* [T, n] out, row stride ld_grad */
  float* g_value;
  float* g_entropy;
  double* out;               /* device [SRL_LOSS_OUT_LEN] or NULL = deferred */
  float* out_f32;            /* device [4] or NULL */
  void* workspace;           /* one slot of srl_ppo_loss_workspace_bytes() bytes, zero before first use */
} srl_loss_problem;

int srl_ppo_loss_fwd_bwd_batched(const srl_loss_problem* problems_host, int n_problems, int64_t ld_pol,
                                 int64_t ld_grad, const float* old_logp, const float* old_value, const float* ret,
                                 const float* adv, const uint8_t* on_reset_next, int64_t ld_smp, const float* pack,
                                 int pack_row_lo, const double* lane_aos, const double* minibatch_part, int part_ctas,
                                 int part_first, int T, int n,
                                 const double* popart_mean_std, const srl_ppo_hyper* hyper,
                                 size_t workspace_bytes_per_slot, struct srl_xchg* xchg /* or NULL */, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4b  Same loss, but starting from the actor head's logits: also replaces
 * ActorCriticPolicy.__get_log_prob_and_entropy / get_action_distribution
 * (legacy/algorithm/ppo/actor_critic_policies/actor_critic_policy.py:303-324): per head h with K_h
 * logits z: lp = z - logsumexp(z); logp = sum_h lp[a_h]; H = sum_h -sum_k softmax(z)_k lp_k.
 * Writes d loss / d logits ([T, n, sumK]) and d loss / d v_pred.  sumK above SRL_K4B_MAX_SUM_K is SRL_ERR_UNSUPPORTED.
 * ------------------------------------------------------------------------------------------ */
#define SRL_MAX_HEADS 8
#define SRL_K4B_MAX_SUM_K 199
#define SRL_K4B_MAX_SUM_K_MASKED 159
int srl_ppo_loss_from_logits(
    const float* logits,   /* [T, n, sumK] dense */
    const int32_t* action, /* [T, n, heads]      */
    const int32_t* head_sizes_host, int heads, const float* v_pred, /* [T, n] dense */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, float* g_logits, /* [T, n, sumK] out */
    float* g_value,                               /* [T, n] out */
    float* logp_out, float* entropy_out,          /* [T, n] out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* The same with an availability mask (SMAC's available_action): the reference's categorical policy replaces unavailable
 * logits before it builds the distributions, logits.masked_fill(available_action == 0, -1e10)
 * (legacy/algorithm/ppo/actor_critic_policies/actor_critic_policy.py:135-136).  available is one byte per logit, aligned
 * with the logits across all heads; 0 = unavailable: that logit is float32(-1e10) for the log-prob, the entropy and the ten
 * outputs, and its g_logits entry is exactly 0 (masked_fill passes no gradient), also where it is the chosen action (logp
 * about -1e10, ratio 0, everything finite).  A head with no available action adds 0 to logp and to the entropy, as in torch
 * (its log-sum-exp rounds to -1e10).  available must not be NULL; sumK above SRL_K4B_MAX_SUM_K_MASKED (the mask is staged
 * in shared memory beside the logits) is SRL_ERR_UNSUPPORTED.  Everything else, the deferred mode included, is
 * srl_ppo_loss_from_logits'. */
int srl_ppo_loss_from_logits_masked(
    const float* logits,      /* [T, n, sumK] dense */
    const uint8_t* available, /* [T, n, sumK] dense, non-zero = available */
    const int32_t* action,    /* [T, n, heads]      */
    const int32_t* head_sizes_host, int heads, const float* v_pred, /* [T, n] dense */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, float* g_logits, /* [T, n, sumK] out */
    float* g_value,                               /* [T, n] out */
    float* logp_out, float* entropy_out,          /* [T, n] out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* The two entries above with a bfloat16 policy side, for policies trained under torch.autocast(dtype=torch.bfloat16), whose
 * last nn.Linear layers produce bfloat16 logits and values.  Same arguments in the same order; logits, v_pred, g_logits and
 * g_value are bfloat16 bit patterns (uint16_t, the upper half of the float32 pattern), everything else is as above:
 * logp_out / entropy_out, the sample side and the ten outputs stay float32.  Each logit and v_pred is widened to float32
 * exactly where it is read and all arithmetic is float32, as torch runs logsumexp / log_softmax / softmax on upcast bfloat16
 * values; each g_logits and g_value entry is the float32 result rounded to bfloat16 once (round to nearest even).  So the
 * results are the float32 entry's on the widened values, with the gradients rounded, wherever the two make the same
 * choice of caching exponentials (sum K <= 99 without a mask and <= 88 with one; the bfloat16 entries cache them up to 133
 * and 114).  The widest rows are the float32 entries' limits, SRL_K4B_MAX_SUM_K and SRL_K4B_MAX_SUM_K_MASKED; wider rows
 * are SRL_ERR_UNSUPPORTED.  The masked entry rejects a NULL mask.  Deferred finalisation works as above. */
int srl_ppo_loss_from_logits_bf16(
    const uint16_t* logits, /* [T, n, sumK] dense bfloat16 */
    const int32_t* action,  /* [T, n, heads]               */
    const int32_t* head_sizes_host, int heads, const uint16_t* v_pred, /* [T, n] dense bfloat16 */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, uint16_t* g_logits, /* [T, n, sumK] bfloat16 out */
    uint16_t* g_value,                               /* [T, n] bfloat16 out */
    float* logp_out, float* entropy_out,             /* [T, n] float32 out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);
int srl_ppo_loss_from_logits_masked_bf16(
    const uint16_t* logits,   /* [T, n, sumK] dense bfloat16 */
    const uint8_t* available, /* [T, n, sumK] dense, non-zero = available */
    const int32_t* action,    /* [T, n, heads]               */
    const int32_t* head_sizes_host, int heads, const uint16_t* v_pred, /* [T, n] dense bfloat16 */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, uint16_t* g_logits, /* [T, n, sumK] bfloat16 out */
    uint16_t* g_value,                               /* [T, n] bfloat16 out */
    float* logp_out, float* entropy_out,             /* [T, n] float32 out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* srl_ppo_loss_from_logits(_masked)(_bf16) with the sample side read from K2's loss pack (srl_gae_scan's `pack`: the BASE of
 * the buffer, pack_lanes = its N lanes, pack_row_lo = the absolute sample row of loss row 0) instead of the five leaves:
 * transition (t, j) reads ONE 16-byte item {old_logp, value, ret, mask ? adv : NaN} at lane c = lane_idx ? lane_idx[j] : j
 * and row pack_row_lo + t -- what a permuted minibatch of the trainer has.  elem_bytes = 4 (float32) or 2 (bfloat16)
 * selects the policy side's element type with the rules of the _bf16 entries; available may be NULL (no mask) or the mask
 * of srl_ppo_loss_from_logits_masked.  Same grid, same per-element arithmetic and the same fold order as the leaf entry
 * with the same lane_idx: the results are bit-identical to it on the leaves the pack was written from.  Invalid arguments
 * besides the leaf entries': a NULL or not 16-byte aligned pack, pack_row_lo < 0, lane_idx == NULL with pack_lanes < n,
 * elem_bytes other than 2 or 4.  Deferred finalisation works as above. */
int srl_ppo_loss_from_logits_pack(
    const void* logits, int elem_bytes, /* [T, n, sumK] dense, float32 or bfloat16 */
    const uint8_t* available,           /* [T, n, sumK] dense or NULL               */
    const int32_t* action,              /* [T, n, heads]                            */
    const int32_t* head_sizes_host, int heads, const void* v_pred, /* [T, n] dense, the logits' type */
    const float* pack, int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, void* g_logits, /* [T, n, sumK] out, the logits' type */
    void* g_value,                               /* [T, n] out, the logits' type */
    float* logp_out, float* entropy_out,         /* [T, n] float32 out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4b-wide  K4b for wide rows: 1 .. SRL_MAX_HEADS heads of sum K = 1 .. SRL_K4B_WIDE_MAX_SUM_K logits per transition
 * (Go's 362 actions, chess's 4672 with a legal-move mask, a language model's vocabulary in bfloat16), where the entries
 * above stage a [256, sum K] tile in shared memory and stop at SRL_K4B_MAX_SUM_K / SRL_K4B_MAX_SUM_K_MASKED.  A warp walks
 * one transition's row instead.  Same contract as K4b: per head h with K_h logits z, lp = z - logsumexp(z),
 * logp = sum_h lp[a_h], H = sum_h -sum_k softmax(z)_k lp_k; K4's loss, its ten outputs, masking and statistics; writes
 * d loss / d logits (g_lp ([k == a] - p_k) - g_en p_k (lp_k + H_h)) and d loss / d v_pred.  Correct at every width from 1
 * up, the narrow ones included, though ops.ppo_loss_from_logits only routes rows the entries above refuse here.
 *  - elem_bytes = 4 (float32) or 2 (bfloat16) selects the policy side's element type (logits, v_pred, g_logits, g_value),
 *    with the rules of the _bf16 entries: each input widened where it is read, float32 arithmetic, each gradient rounded
 *    once.  Every logit goes to the same lane in the same order for both types, so the bfloat16 launch returns exactly the
 *    float32 launch's logp and entropy on the widened values and its gradients rounded, and the same `out` / `out_f32`.
 *  - available: NULL or the mask of srl_ppo_loss_from_logits_masked.  An unavailable logit is float32(-1e10) and gets
 *    exactly 0 gradient, also where it is the chosen action.  A head with no available action adds exactly 0 to logp and
 *    to the entropy, as in torch: its entropy is computed as (l - m) - w / s with l = fl(m + log s) already rounded (m the
 *    head's max, s = sum e^{z-m}, w = sum e^{z-m} (z - m)), not as log s - w / s, which would give log K.
 *  - -inf logits of an unmasked policy (dead agents) give finite entropies and gradients (lp is clamped at -FLT_MAX as
 *    torch's Categorical.entropy clamps it); a chosen -inf action gives logp -inf and ratio 0.
 *  - The grid has at most as many CTAs as one workspace slot has partial rows, so srl_ppo_loss_workspace_bytes and the
 *    deferred mode (out == NULL, then srl_ppo_loss_finalize) work as for the entries above.
 * srl_ppo_loss_from_logits_wide takes the leaves of srl_ppo_loss_from_logits; srl_ppo_loss_from_logits_wide_pack takes
 * srl_ppo_loss_from_logits_pack's arguments in its order and makes its checks.  Argument checks and error texts are the K4b
 * entries'; elem_bytes other than 2 or 4 is SRL_ERR_INVALID_ARG, sum K above SRL_K4B_WIDE_MAX_SUM_K SRL_ERR_UNSUPPORTED.
 * ------------------------------------------------------------------------------------------ */
#define SRL_K4B_WIDE_MAX_SUM_K 262144
int srl_ppo_loss_from_logits_wide(
    const void* logits, int elem_bytes, /* [T, n, sumK] dense, float32 or bfloat16 */
    const uint8_t* available,           /* [T, n, sumK] dense or NULL               */
    const int32_t* action,              /* [T, n, heads]                            */
    const int32_t* head_sizes_host, int heads, const void* v_pred, /* [T, n] dense, the logits' type */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, void* g_logits, /* [T, n, sumK] out, the logits' type */
    void* g_value,                               /* [T, n] out, the logits' type */
    float* logp_out, float* entropy_out,         /* [T, n] float32 out or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);
int srl_ppo_loss_from_logits_wide_pack(
    const void* logits, int elem_bytes, const uint8_t* available, const int32_t* action,
    const int32_t* head_sizes_host, int heads, const void* v_pred,
    const float* pack, int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper, void* g_logits, void* g_value, float* logp_out, float* entropy_out,
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4c Same loss, but starting from a diagonal-Gaussian actor head (continuous actions, D = 1 .. 64 dimensions).
 * NEW capability: the reference's policies are categorical, so no reference line pins this head; the definition is
 * torch.distributions.Normal(mean, exp(log_std)), summed over the action dimensions, as any PyTorch Gaussian policy
 * computes it (sigma = exp(s)):
 *   logp = sum_d [ -(a_d - mu_d)^2 / (2 sigma_d^2) - log sigma_d - log sqrt(2 pi) ]     (.log_prob(a).sum(-1))
 *   H    = sum_d [ 0.5 + 0.5 log(2 pi) + log sigma_d ]                                    (.entropy().sum(-1))
 * The loss, the ten outputs and the masking are K4's.  Writes
 *   g_mean[i, d]    = g_lp (a_d - mu_d) / sigma_d^2
 *   g_log_std[i, d] = g_lp ((a_d - mu_d)^2 / sigma_d^2 - 1) + g_en
 * with (g_lp, g_en) = d loss / d (logp, H) of transition i, and d loss / d v_pred.  log_std_shared != 0: log_std is ONE
 * [D] vector for every transition (a state-independent parameter) and g_log_std[d] is the sum of the expression above
 * over the T * n transitions, added in float64 in a fixed order (deterministic for a given launch shape) and complete
 * when the launch completes, in both finalisation modes.
 * The workspace (zero before first use, left zero) starts with a K4 slot of srl_ppo_loss_workspace_bytes(T, n) bytes, so
 * out == NULL followed by srl_ppo_loss_finalize(workspace, srl_ppo_loss_gaussian_workspace_bytes(...), 1, ...) works as
 * for srl_ppo_loss_fwd_bwd; with a shared log_std the float64 partial rows of its gradient follow the slot.
 * D outside [1, 64] is an invalid argument.
 * ------------------------------------------------------------------------------------------ */
size_t srl_ppo_loss_gaussian_workspace_bytes(int T, int n, int D, int log_std_shared);
int srl_ppo_loss_from_gaussian(
    const float* mean, const float* log_std, int log_std_shared, /* [T,n,D]; log_std [T,n,D] or [D] */
    const float* action, int D,                                    /* [T,n,D] float32                    */
    const float* v_pred,                                           /* [T,n]                              */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    float* g_mean, float* g_log_std /* [T,n,D] or [D] */, float* g_value,
    float* logp_out, float* entropy_out,                           /* [T,n] or NULL                      */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);
/* The entry above with a bfloat16 policy side, for Gaussian policies trained under torch.autocast(dtype=torch.bfloat16),
 * whose last nn.Linear layers produce bfloat16 means and values.  Same arguments in the same order; mean, v_pred, g_mean
 * and g_value are bfloat16 bit patterns (uint16_t).  log_std and g_log_std are untyped because their element type follows
 * log_std_shared: bfloat16 [T,n,D] per transition (the output of a head), float32 [D] when shared (an nn.Parameter, which
 * autocast leaves float32; its gradient, a sum over the minibatch, feeds float32 master weights and is not rounded).
 * action stays float32: old_logp was computed on the sampled float32 action, and a rounded one would bias every ratio.
 * logp_out / entropy_out, the sample side and the ten outputs stay float32.  Each bfloat16 input is widened to float32
 * exactly where it is read and all arithmetic is the entry above's, so logp and entropy are bit-identical to
 * srl_ppo_loss_from_gaussian's on the widened values, and each bfloat16 gradient is that entry's float32 result rounded
 * to bfloat16 once (round to nearest even).  out, out_f32 and a shared g_log_std are float64 sums added in an order the
 * launch grid fixes; they are bit-identical too whenever both entries launch the same grid, which is always the case
 * for T * n <= 256 * (number of SMs), and at any size unless the smaller bfloat16 blocks fit 2 CTAs per SM where the
 * float32 ones fit 1 (on a B200: D = 37 .. 55 per transition, D = 54 .. 64 shared).  D is 1 .. 64, the workspace is the
 * one srl_ppo_loss_gaussian_workspace_bytes sizes, and deferred finalisation works as above. */
int srl_ppo_loss_from_gaussian_bf16(
    const uint16_t* mean, const void* log_std, int log_std_shared, /* [T,n,D] bf16; log_std [T,n,D] bf16 or [D] f32 */
    const float* action, int D,                                      /* [T,n,D] float32                              */
    const uint16_t* v_pred,                                          /* [T,n] bfloat16                               */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    uint16_t* g_mean, void* g_log_std /* [T,n,D] bf16 or [D] f32 */, uint16_t* g_value, /* bfloat16 out */
    float* logp_out, float* entropy_out,                             /* [T,n] float32 or NULL                        */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* srl_ppo_loss_from_gaussian(_bf16) with the sample side read from K2's loss pack, as srl_ppo_loss_from_logits_pack reads
 * it (pack_lanes, pack_row_lo, lane_idx: see there).  elem_bytes = 4 or 2 selects the float32 or bfloat16 policy side with
 * the rules of the _bf16 entry (a shared [D] log_std and its gradient are float32 either way).  Bit-identical to the leaf
 * entry with the same lane_idx on the leaves the pack was written from; the same argument checks as
 * srl_ppo_loss_from_logits_pack besides the leaf entries' (D, workspace size, deferred mode). */
int srl_ppo_loss_from_gaussian_pack(
    const void* mean, const void* log_std, int log_std_shared, /* [T,n,D]; log_std [T,n,D] (mean's type) or [D] f32 */
    const float* action, int D,                                  /* [T,n,D] float32                                   */
    int elem_bytes, const void* v_pred,                          /* [T,n], mean's type                                */
    const float* pack, int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    void* g_mean, void* g_log_std /* [T,n,D] or [D] f32 */, void* g_value,
    float* logp_out, float* entropy_out,                         /* [T,n] float32 or NULL                             */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4d  Same loss, but starting from a Beta actor head (actions bounded to an interval, D = 1 .. 64 dimensions).
 * NEW capability: no reference line pins this head; the definition is torch.distributions.Beta(c1, c0) with
 * c1 = concentration1 (alpha) and c0 = concentration0 (beta), summed over the action dimensions, as any PyTorch Beta
 * policy computes it (x in (0, 1), psi = digamma):
 *   logp = sum_d [ (c1-1) log x + (c0-1) log(1-x) + lgamma(c1+c0) - lgamma(c1) - lgamma(c0) ]      (.log_prob(x).sum(-1))
 *   H    = sum_d [ lgamma(c1) + lgamma(c0) - lgamma(c1+c0) - (c1-1) psi(c1) - (c0-1) psi(c0)
 *                  + (c1+c0-2) psi(c1+c0) ]                                                          (.entropy().sum(-1))
 * The loss, the ten outputs and the masking are K4's.  Writes
 *   g_concentration1[i, d] = g_lp (log x - psi(c1) + psi(c1+c0)) + g_en ((c1+c0-2) psi'(c1+c0) - (c1-1) psi'(c1))
 *   g_concentration0[i, d] = g_lp (log(1-x) - psi(c0) + psi(c1+c0)) + g_en ((c1+c0-2) psi'(c1+c0) - (c0-1) psi'(c0))
 * with (g_lp, g_en) = d loss / d (logp, H) of transition i, and d loss / d v_pred.  The per-dimension terms and their
 * sums over d are float64 (lgamma(c1+c0) - lgamma(c1) - lgamma(c0) cancels for large concentrations); logp and H are
 * rounded to float32 once, each gradient once.  The actions are the float32 samples in the open interval (0, 1) (a
 * policy maps them to its action bounds itself) and the concentrations are positive; neither is checked on the device.
 * An action outside (0, 1) gives what torch's formula gives; a concentration that is not positive (or NaN) gives NaN
 * psi / psi' terms, so that transition's entropy and gradients are NaN (torch's digamma would evaluate a negative
 * argument) -- the launch ends either way, and a NaN transition makes the statistics NaN.  The workspace (zero before first use, left zero) is one
 * K4 slot of srl_ppo_loss_workspace_bytes(T, n) bytes, so out == NULL followed by srl_ppo_loss_finalize works as for
 * srl_ppo_loss_fwd_bwd.  D outside [1, 64] is an invalid argument.
 * ------------------------------------------------------------------------------------------ */
int srl_ppo_loss_from_beta(
    const float* concentration1, const float* concentration0, /* [T,n,D] */
    const float* action, int D,                                 /* [T,n,D] float32, in (0, 1) */
    const float* v_pred,                                        /* [T,n]   */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    float* g_concentration1, float* g_concentration0, float* g_value, /* [T,n,D], [T,n,D], [T,n] */
    float* logp_out, float* entropy_out,                                /* [T,n] or NULL          */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);
/* The entry above with a bfloat16 policy side (a Beta policy under torch.autocast(dtype=torch.bfloat16)): same arguments
 * in the same order; concentration1, concentration0, v_pred and their gradients are bfloat16 bit patterns (uint16_t).
 * action, logp_out / entropy_out, the sample side and the ten outputs stay float32.  Each bfloat16 input is widened to
 * float32 where it is read and all arithmetic is the entry above's, so logp and entropy are bit-identical to
 * srl_ppo_loss_from_beta's on the widened values and each gradient is that entry's float32 result rounded to bfloat16
 * once (round to nearest even); out and out_f32 are too whenever both entries launch the same grid (as for
 * srl_ppo_loss_from_gaussian_bf16). */
int srl_ppo_loss_from_beta_bf16(
    const uint16_t* concentration1, const uint16_t* concentration0, /* [T,n,D] bfloat16 */
    const float* action, int D,                                       /* [T,n,D] float32  */
    const uint16_t* v_pred,                                           /* [T,n] bfloat16   */
    const float* old_logp, const float* old_value, const float* ret, const float* adv,
    const uint8_t* on_reset_next, int64_t ld_smp, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    uint16_t* g_concentration1, uint16_t* g_concentration0, uint16_t* g_value, /* bfloat16 out */
    float* logp_out, float* entropy_out,                                        /* [T,n] float32 or NULL */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);
/* srl_ppo_loss_from_beta(_bf16) with the sample side read from K2's loss pack, as srl_ppo_loss_from_gaussian_pack reads
 * it; elem_bytes = 4 or 2 selects the float32 or bfloat16 policy side.  Bit-identical to the leaf entry with the same
 * lane_idx on the leaves the pack was written from; the same argument checks as srl_ppo_loss_from_gaussian_pack. */
int srl_ppo_loss_from_beta_pack(
    const void* concentration1, const void* concentration0, /* [T,n,D], float32 or bfloat16 */
    const float* action, int D,                               /* [T,n,D] float32              */
    int elem_bytes, const void* v_pred,                       /* [T,n], the concentrations' type */
    const float* pack, int64_t pack_lanes, int pack_row_lo, const int32_t* lane_idx, int T, int n,
    const double* norm_stats, const double* local_stats, const double* popart_mean_std,
    const srl_ppo_hyper* hyper,
    void* g_concentration1, void* g_concentration0, void* g_value,
    float* logp_out, float* entropy_out,                      /* [T,n] float32 or NULL        */
    double* out, float* out_f32, void* workspace, size_t workspace_bytes, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K5a  Philox-keyed permutation of the environment axis (NEW capability: the reference has no
 * minibatching, SURVEY.md F2; nearest relative SimpleReplayBuffer.get, base/buffer.py:262-277).
 * out is [n_epochs][n_env * group]; row r holds epoch (epoch + r):
 * out[r][e*group + a] = perm_r[e] * group + a for e in [0, n_env), a in [0, group): an 8-round Feistel
 * bijection on ceil(log2 n_env) bits, round keys from Philox4x32-10(key = seed, counter =
 * (block, epoch, 'SRLP', 0)), cycle-walked into [0, n_env).  Spec: oracle/ref_math.py:philox_perm_ref.
 * ------------------------------------------------------------------------------------------ */
int srl_philox_perm(uint64_t seed, uint32_t epoch, int n_epochs, int n_env, int group, int32_t* out,
                    srl_stream_t stream);
/* Raw Philox4x32-10 blocks (for known-answer tests): out[i] = philox(counter[i], key[i]). */
int srl_philox4x32_10(const uint32_t* counter, const uint32_t* key, int n_blocks, uint32_t* out,
                      srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K1 / K5b  Batch assembly and minibatch gather over many leaves in one launch.
 * For every leaf: dst[t, j, :] = src[t, idx[j], :] for t in [0, L), j in [0, B), rows of `row_bytes`.
 * Replaces recursive_aggregate(samples, np.stack(axis=1)) in PriorityQueueBuffer.put
 * (base/buffer.py:118-126, base/namedarray.py:598-633) when src is a slot slab, and
 * SharedMemoryDock.get = buf[:, sorted(idx)] (base/shared_memory.py:85-99); bit-exact byte copy.
 * ------------------------------------------------------------------------------------------ */
#define SRL_MAX_LEAVES 32
typedef struct srl_leaf_desc {
  const void* src;         /* item (t, slot) at src + t * src_t_stride + slot * src_slot_stride                      */
  void* dst;               /* [L, B, row_bytes]                                                                       */
  int64_t row_bytes;       /* bytes per (t, slot) item                                                                */
  int64_t src_slots;       /* slots addressable in src                                                                */
  int64_t src_t_stride;    /* 0 = row_bytes * src_slots: src is [L, src_slots, row] (SharedMemoryDock's slab layout)  */
  int64_t src_slot_stride; /* 0 = row_bytes; L * row_bytes with src_t_stride = row_bytes: src is [slots, L, row],
                              i.e. whole samples staged one after another -- the gather is np.stack(axis=1)           */
} srl_leaf_desc;

int srl_batch_gather(const srl_leaf_desc* leaves_host, int n_leaves, const int32_t* idx /* device [B] or NULL */,
                     int L, int B, srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (f)4  What a recurrent policy needs from a minibatch besides the chunked leaves, in one launch.  Replaces, for the
 * reset flags and the hidden states, recursive_apply(sample, to_chunk) + x[0].transpose(0, 1)
 * (legacy/algorithm/ppo/actor_critic_policies/actor_critic_policy.py:348-363) and the reset handling of
 * AutoResetRNN.forward (legacy/algorithm/modules/autoreset_rnn.py:42-60): the rows in which any lane resets
 * ((masks[1:] == 0).any(dim=1).nonzero(), a host synchronisation in the reference) and `hxs * masks[0]`.
 *   on_reset    uint8  [T, B]                (the sample's rows from burn_in on)
 *   hx          float32 [T, B, layers, H]    per-step hidden states, or NULL (then hx0 NULL)
 *   env_idx     int32  [n]                   the minibatch's lanes (srl_philox_perm slice)
 *   reset_chunk uint8  [T/C, C*n]  out       = to_chunk(on_reset[:, env_idx], C): column c*n + j = chunk c, lane env_idx[j]
 *   row_any     uint8  [T/C]       out       1 where some column of that chunk-row resets (row 0 included)
 *   hx0         float32 [layers, C*n, H] out = hx[c*T/C, env_idx[j]] layer-major, times (1 - reset_chunk[0])
 * T % num_chunks != 0 is SRL_ERR_INVALID_ARG (the reference raises IndexError, utils.py:176-179). */
int srl_rnn_chunk_prep(const uint8_t* on_reset, const float* hx, const int32_t* env_idx, int T, int B, int n,
                       int num_chunks, int layers, int H, uint8_t* reset_chunk, uint8_t* row_any, float* hx0,
                       srl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (f)2  HOST decoders of the compressed sample-wire payloads (no CUDA call; host pointers): what blosc.decompress does
 * for the frames blosc.compress(payload, typesize=4, cname='lz4') writes (base/namedarray.py:126,150,184-185,203), decoded
 * straight into the destination the caller names -- the buffer's pinned staging block -- with up to `threads`
 * participants over the frame's blocks.  Byte-shuffled or plain, split or unsplit, LZ4 / LZ4HC streams and stored
 * (memcpyed) frames; other codec families and bit-shuffle are SRL_ERR_UNSUPPORTED.  Malformed input is SRL_ERR_INVALID_ARG.
 * srl_blosc1_info reads the 16-byte header (any pointer may be NULL); srl_lz4_block_decompress decodes one raw LZ4 block. */
int srl_blosc1_info(const void* src, size_t src_bytes, size_t* nbytes, size_t* cbytes, size_t* blocksize, int* typesize,
                    int* flags);
int srl_blosc1_decompress(const void* src, size_t src_bytes, void* dst, size_t dst_bytes, int threads);
int srl_lz4_block_decompress(const void* src, size_t src_bytes, void* dst, size_t dst_capacity, size_t* written);

/* HOST helper of the device sample buffer (no CUDA call; host pointers): copies `bytes` bytes with up to `threads`
 * participants (a persistent pool inside the library + the caller; small copies fall back to one memcpy).  It replaces the
 * single-threaded copy into the staging block that bounded the per-sample `put` -- in the reference that copy is the
 * np.stack of PriorityQueueBuffer.put (base/buffer.py:118-126), also on one thread.  Calls are serialised. */
int srl_host_copy(void* dst, const void* src, size_t bytes, int threads);

/* ------------------------------------------------------------------------------------------
 * One-shot SUM all-reduce of a small float64 table over NVLink peer memory (one process per GPU of ONE node).
 * Replaces the dist.all_reduce calls of masked_normalization / RunningMeanStd.update
 * (legacy/algorithm/modules/utils.py:58-61,121-124) for the step's statistics table: every rank stores its table into
 * every peer's mailbox, publishes a sequence number, waits for the peers' numbers in its own memory and adds the tables
 * in rank order (bit-identical result on every rank).  One kernel launch, capturable in a CUDA graph.
 *   create  : allocates this rank's mailbox (cudaMalloc on the CURRENT device) for tables of <= capacity doubles
 *   handle  : 64-byte IPC handle of the local mailbox, to be sent to every peer (any host channel)
 *   connect : `handles` = world * 64 bytes, rank-major; opens the peers' mailboxes
 *   allreduce_sum : global[i] = sum over ranks of local[i], i < n; every rank must call it the same number of times
 *   status  : 0, or 1 when a wait timed out (a peer never arrived); synchronises the device.  status_async copies the
 *             same word into PINNED host memory on `stream` (read it after the caller's own synchronisation).
 *   set_timeout : how long a rank waits for its peers' words (default ~10 minutes: a late peer is late, not gone).  When
 *             the wait does expire NO sums are produced: the whole output table is NaN and the status is sticky, so
 *             nothing downstream can silently train on stale statistics; callers check the status every step and raise.
 * ------------------------------------------------------------------------------------------ */
#define SRL_XCHG_HANDLE_BYTES 64
typedef struct srl_xchg srl_xchg;
/* srl_group_stats with the exchange fused in: the CTA that completes the table's last row sends it to the peers at once
 * (local_out = this rank's table, global_out = the sum over ranks); always needs the workspace. */
int srl_group_stats_xchg(const double* lane_part, int N, const int32_t* idx, int G, int per, int whole_first,
                         double* local_out, double* global_out, void* workspace, size_t workspace_bytes, srl_xchg* x,
                         srl_stream_t stream);
int srl_xchg_create(int world, int rank, int capacity_doubles, srl_xchg** out);
int srl_xchg_local_handle(srl_xchg* x, void* handle_out);
int srl_xchg_connect(srl_xchg* x, const void* handles);
int srl_xchg_allreduce_sum(srl_xchg* x, const double* local, double* global, int n, srl_stream_t stream);
int srl_xchg_status(srl_xchg* x, int* status_out);
int srl_xchg_status_async(srl_xchg* x, int* pinned_status_out, srl_stream_t stream);
int srl_xchg_set_timeout(srl_xchg* x, double seconds);
int srl_xchg_destroy(srl_xchg* x);

#ifdef __cplusplus
}
#endif
#endif /* SRL_B200_H_ */
