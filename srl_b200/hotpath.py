"""Device-resident executor of the trainer hot path for one batch shape.

Owns every HBM buffer the path needs (allocated once, reused every step), the pinned host staging
buffers for the host-facing entry point, the statistics tables and -- optionally -- a CUDA graph of the
whole step.  `srl_b200.trainer.MultiAgentPPOB200` and `bench.py` both drive this class.

Step structure (reference: MultiAgentPPO.step, legacy/algorithm/ppo/mappo.py:219-328):

    load_sample        H2D of the six scalar leaves                      (api/trainer.py:215-217)
    advantages         K2 GAE scan -> adv, ret, loss pack, per-lane sums (mappo.py:252-257)
                       K5a Philox permutations for all epochs, launched behind the scan and running beside it
                       (programmatic dependent launch; a parallel branch without it)   (new, SURVEY F2)
                       group statistics for the batch and every minibatch -- lazily when the batched loss adds its own;
                       with several ranks the same kernel exchanges the table over NVLink peer memory
                                                                          (utils.py:58-61,121-124)
    per epoch          PopArt update                                      (mappo.py:263-264)
      all minibatches  K4 fused loss forward+backward in ONE launch, gather fused in   (mappo.py:270-274)
                       (one GPU, no PopArt, minibatches <= 1024 lanes: K4 adds its own minibatch statistics and the
                       table is produced on a side branch; the trainer's per-minibatch launches read the table)

HBM layout: every leaf is time-major [L, N], lanes contiguous; N = B * n_agents; flags stay uint8.
Statistics table: float64 [1 + E*M, 8]; row 0 = whole batch, row 1 + e*M + j = minibatch j of epoch e.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import numpy as np
import torch

from srl_b200 import ops
from srl_b200._lib import SRL_LANE_PART, SRL_LOSS_OUT_LEN

SAMPLE_F32 = ("reward", "value", "old_logp")
SAMPLE_U8 = ("done", "truncated", "on_reset")


def exchange_stats(local: torch.Tensor, out: torch.Tensor, group=None) -> torch.Tensor:
    """The one data-path collective of the step: SUM all-reduce of the float64 statistics table
    [1 + E*M, 8] (row 0 = batch, row 1 + e*M + j = minibatch (e, j)).  It replaces the 3 one-element all-reduces
    per loss call of masked_normalization (utils.py:58-61) and the 3 per PopArt update (utils.py:121-124);
    the masked means of the loss stay rank-local, as in the reference (SURVEY.md F4).  Works on any backend
    (nccl on the GPUs, gloo in the CPU tests)."""
    out.copy_(local)
    torch.distributed.all_reduce(out, op=torch.distributed.ReduceOp.SUM, group=group)
    return out


class HotPath:

    def __init__(self, L: int, B: int, A: int = 1, *, gamma: float, lmbda: float, hyper: ops.LossHyper,
                 bootstrap_steps: int = 1, burn_in_steps: int = 0, epochs: int = 1, minibatches: int = 1, seed: int = 0,
                 popart: bool = False, popart_beta: float = 0.99999, popart_eps: float = 1e-5,
                 device: Optional[torch.device] = None, process_group=None, fuse_gather: bool = True,
                 graph_branches: int = 16, shuffle_block: int = 1, use_pack: bool = True, batch_losses: bool = True,
                 stats_exchange: str = "auto", fuse_stats: bool = True, exchange_timeout_s: Optional[float] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("srl_b200.HotPath needs a CUDA device (there is no CPU path)")
        if bootstrap_steps < 1:
            # mappo.py:259-261 slices on_reset[1 + burn_in : 1 + L - bootstrap]; with bootstrap_steps == 0 the
            # reference's mask is one row short of the data and the loss raises.  Same restriction here.
            raise ValueError("bootstrap_steps must be >= 1")
        # Minibatches are drawn by permuting blocks of `shuffle_block` consecutive environments (1 = every
        # environment on its own, the textbook shuffle).  Blocks of 8 single-agent environments are exactly one
        # 32-byte sector of every float32 leaf, which turns the gather-on-load into full-sector 128-bit loads.
        if shuffle_block < 1 or B % shuffle_block != 0 or (B // shuffle_block) % minibatches != 0:
            raise ValueError(f"B={B} environments do not split into {minibatches} equal minibatches of "
                             f"{shuffle_block}-environment blocks")
        self.shuffle_block = int(shuffle_block)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.L, self.B, self.A, self.N = L, B, A, B * A
        self.gamma, self.lmbda, self.hyper = float(gamma), float(lmbda), hyper
        self.row_lo, self.row_hi = burn_in_steps, L - bootstrap_steps
        self.T = self.row_hi - self.row_lo
        if self.T < 1:
            raise ValueError(f"no loss rows: L={L}, burn_in={burn_in_steps}, bootstrap={bootstrap_steps}")
        self.epochs, self.minibatches, self.seed = epochs, minibatches, int(seed)
        self.n_mb = self.N // minibatches  # lanes per minibatch
        self.popart, self.popart_beta, self.popart_eps = popart, popart_beta, popart_eps
        self.pg = process_group
        # the statistics exchange: "p2p" = one-kernel NVLink peer-memory mailbox exchange (srl_b200/xchg.py), "nccl" =
        # torch.distributed all-reduce (also gloo in the CPU tests); "auto" tries p2p on an NCCL group and falls back
        self.peer = None
        self.exchange_kind = "none" if process_group is None else "nccl"
        if process_group is not None and stats_exchange in ("auto", "p2p") and \
                torch.distributed.get_backend(process_group) == "nccl":
            from srl_b200.xchg import PeerExchange, PeerExchangeUnavailable
            try:  # collective: every rank ends up with the exchange, or every rank falls back (xchg.py)
                self.peer = PeerExchange(process_group, (1 + epochs * minibatches) * SRL_LANE_PART,
                                         torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device),
                                         timeout_s=exchange_timeout_s)
                self.exchange_kind = "p2p"
            except PeerExchangeUnavailable:
                if stats_exchange == "p2p":
                    raise
        # A second mailbox for the loss kernel's own exchange of each minibatch's three sums (ppo_loss_pair.cu): with it the
        # multi-GPU step keeps the single-GPU critical path K2 -> K4 -- the statistics table (still exchanged, for PopArt-less
        # reporting and the parity checks) moves to the side branch.  Collective, like the first one.
        self.peer_loss = None
        fusable = bool(fuse_stats) and not popart and batch_losses and minibatches > 1 and fuse_gather and use_pack and \
            (self.N // minibatches) <= 1024 and (self.N // minibatches) % 2 == 0
        if self.peer is not None and fusable:
            from srl_b200.xchg import PeerExchange, PeerExchangeUnavailable
            try:
                self.peer_loss = PeerExchange(process_group, 4 * 32, self.device, timeout_s=exchange_timeout_s)
            except PeerExchangeUnavailable:
                self.peer_loss = None
        self.fuse_gather = fuse_gather
        self.graph_branches = max(1, int(graph_branches))
        self.batch_losses = bool(batch_losses)
        # batched launches finalise their loss scalars themselves (last CTA of each minibatch); the per-minibatch
        # launches of the trainer path defer to finalize()
        self._immediate = self.batch_losses and (fuse_gather or minibatches == 1)
        self.pack_valid = False
        # One GPU, no PopArt, minibatches of <= 1024 lanes: the batched loss kernel adds K2's per-lane sums over its own
        # minibatch (its indices are in registers anyway), so the statistics table is no longer on the critical path
        # K2 -> K4; it is still produced (the trainer reports done / truncated from its batch row), on a side branch.
        self.fuse_stats = fusable and self._immediate and (process_group is None or self.peer_loss is not None)
        self._stats_pending = False
        self._lazy_table, self._table_valid = False, False
        self.step_count = 0

        dev, N = self.device, self.N
        f32 = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        u8 = lambda *s: torch.empty(s, dtype=torch.uint8, device=dev)
        self.leaf: Dict[str, torch.Tensor] = {k: f32(L, N) for k in SAMPLE_F32}
        self.leaf.update({k: u8(L, N) for k in SAMPLE_U8})
        self.adv, self.ret = f32(L, N), f32(L, N)
        self.lane_part = torch.empty((SRL_LANE_PART, N), dtype=torch.float64, device=dev)
        # the same per-lane sums as one 32-byte item per lane: what the pair loss kernel gathers for its own statistics
        self.lane_aos = torch.empty((N, 4), dtype=torch.float64, device=dev) if self.fuse_stats else None
        # ... and, where the scan kernel computes the permutations itself, every scan CTA's share of every minibatch's
        # sums: the loss kernel then adds N / 32 contiguous items per minibatch instead of gathering the minibatch's lanes
        # (SRL_MB_PART=0: an A/B knob for profiles/)
        self.mb_part = ops.new_minibatch_part(N, dev) if (self.fuse_stats and epochs <= 8 and epochs * minibatches <= 32 and
                                                          os.environ.get("SRL_MB_PART", "1") != "0") else None
        self._part_valid = False
        G = 1 + epochs * minibatches
        self.local_stats = torch.zeros((G, SRL_LANE_PART), dtype=torch.float64, device=dev)
        self.global_stats = self.local_stats if process_group is None else torch.zeros_like(self.local_stats)
        self.perm = torch.empty((epochs, N), dtype=torch.int32, device=dev) if minibatches > 1 else None
        # K2's pack: the loss's sample side as one 16-byte item per transition (only a permuted minibatch gathers
        # lane by lane, so only then is it worth its extra 16 B/transition of GAE writes)
        self.pack = ops.new_pack(L, N, dev) if (minibatches > 1 and fuse_gather and use_pack) else None
        self._perm_stream = torch.cuda.Stream(device=dev) if minibatches > 1 else None
        self.popart_state = torch.zeros(4, dtype=torch.float64, device=dev)
        self.popart_ms = torch.tensor([0.0, 0.1, 0.0, 0.1], dtype=torch.float64, device=dev)  # sqrt(1e-2) floor
        n = self.n_mb
        # gradients of every (epoch, minibatch) in one allocation so the host-facing call moves them with one copy
        self.grads_all = f32(epochs, minibatches, 3, self.T, n)
        self.grads = [[tuple(self.grads_all[e, j, q] for q in range(3)) for j in range(minibatches)]
                      for e in range(epochs)]
        self.out = torch.zeros((epochs * minibatches, SRL_LOSS_OUT_LEN), dtype=torch.float64, device=dev)
        self.out_f32 = torch.zeros((epochs * minibatches, 4), dtype=torch.float32, device=dev)
        self.workspace = ops.new_loss_workspace(dev, slots=epochs * minibatches)  # one slot per (epoch, minibatch)
        self.stats_ws = ops.group_stats_workspace(dev, epochs * minibatches if minibatches > 1 else 1, minibatches > 1)
        if not fuse_gather and minibatches > 1:  # explicit K5 gather into contiguous minibatch leaves
            self.mb_leaf = {k: f32(L, n) for k in ("old_logp", "value", "ret", "adv")}
            self.mb_leaf["on_reset"] = u8(L, n)
        # pinned host mirrors for the host-facing call
        self._pin: Dict[str, torch.Tensor] = {}
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_a: Optional[torch.cuda.CUDAGraph] = None
        self._graph_pol = None
        self._perm_fused = False
        self.launches_per_step = 0

    # ------------------------------------------------------------------------------------------
    def popart_mean_std(self) -> Optional[torch.Tensor]:
        return self.popart_ms if self.popart else None

    def _pinned(self, key: str, like: np.ndarray) -> torch.Tensor:
        t = self._pin.get(key)
        if t is None or t.numel() != like.size or t.dtype != torch.from_numpy(like.reshape(-1)[:1]).dtype:
            t = torch.empty(like.size, dtype=torch.from_numpy(like.reshape(-1)[:1]).dtype).pin_memory()
            self._pin[key] = t
        return t

    def load_sample(self, sample: Dict[str, np.ndarray], non_blocking: bool = True) -> int:
        """Host -> HBM copy of the scalar leaves (reward, value, old_logp float32; done, truncated,
        on_reset uint8, each [L, B, (A,) 1] or [L, N]).  Float flags are narrowed to uint8 on the host:
        the reference's device representation is float32 (api/trainer.py:217), ours is one byte.
        Returns the bytes moved."""
        moved = 0
        for k in SAMPLE_F32 + SAMPLE_U8:
            x = sample[k]
            want = np.float32 if k in SAMPLE_F32 else np.uint8
            if isinstance(x, torch.Tensor) and x.is_cuda:  # device-resident batch: a device copy (+ dtype narrowing)
                if x.numel() != self.L * self.N:
                    raise ValueError(f"{k}: {tuple(x.shape)} does not hold L*N = {self.L}*{self.N} elements")
                self.leaf[k].view(-1).copy_(x.reshape(-1), non_blocking=True)
                continue
            if isinstance(x, torch.Tensor):
                if x.is_pinned() and x.dtype == (torch.float32 if k in SAMPLE_F32 else torch.uint8) and \
                        x.numel() == self.L * self.N and x.is_contiguous():
                    self.leaf[k].view(-1).copy_(x.view(-1), non_blocking=non_blocking)  # already page-locked
                    moved += x.numel() * x.element_size()
                    continue
                x = x.numpy()
            if x.size != self.L * self.N:
                raise ValueError(f"{k}: {x.shape} does not hold L*N = {self.L}*{self.N} elements")
            if x.dtype != want:
                x = x.astype(want)
            pin = self._pinned(k, x)
            pin.numpy()[:] = x.reshape(-1)
            self.leaf[k].view(-1).copy_(pin, non_blocking=non_blocking)
            moved += x.nbytes
        return moved

    # ------------------------------------------------------------------------------------------
    def advantages(self, cached: bool = False, vtrace_new_logp: Optional[torch.Tensor] = None,
                   permute: bool = True) -> None:
        """K2 (or, for cached adv/ret already in self.adv / self.ret, only their per-lane sums), then all epochs'
        permutations in one launch, then the whole statistics table in one launch (+ the one small all-reduce
        when distributed)."""
        lf = self.leaf
        main = torch.cuda.current_stream()
        # The permutations do not depend on the scan.  With programmatic dependent launch the order K2 -> K5a -> K4 on
        # ONE stream already overlaps (K5a is launched beside K2 and only completes when K2 has; K4 becomes resident under
        # both): no fork / join, three nodes in a line in the step graph.  Without it: a parallel branch.
        inline_perm = self.minibatches > 1 and permute and ops.pdl_enabled() and not cached
        fork_perm = self.minibatches > 1 and permute and not inline_perm
        perm_first = inline_perm and os.environ.get("SRL_PERM_FIRST") == "1"  # A/B knob: round 1's order K5a -> K2 -> K4
        if perm_first:
            self.permute()
        if fork_perm:
            self._perm_stream.wait_stream(main)
            with torch.cuda.stream(self._perm_stream):
                self.permute()
        self.pack_valid = False
        job = None
        if cached:
            ops.lane_stats(self.adv, self.ret, lf["done"], lf["truncated"], lf["on_reset"], self.row_lo, self.row_hi,
                           lane_part=self.lane_part)
        else:
            kw = {}
            if vtrace_new_logp is not None:  # V-trace: rho_t from the current policy (mappo.py:129-132)
                kw = dict(vtrace_new_logp=vtrace_new_logp, vtrace_old_logp=lf["old_logp"])
            elif self.pack is not None:
                kw = dict(old_logp=lf["old_logp"], pack=self.pack, lane_aos=self.lane_aos)
                self.pack_valid = True
            if inline_perm and not perm_first and os.environ.get("SRL_PERM_FUSED", "1") != "0":
                # the scan kernel's own idle threads compute the permutations (one launch and one completion hop less
                # between the scan and the loss); where the scan kernel for this shape cannot, the stand-alone kernel runs
                # behind the scan as before
                job = self.perm_job(with_part="lane_aos" in kw)
                kw["perm_job"] = job
            ops.gae_scan(lf["reward"], lf["value"], lf["done"], lf["truncated"], lf["on_reset"], self.gamma, self.lmbda,
                         row_lo=self.row_lo, row_hi=self.row_hi, popart_mean_std=self.popart_mean_std(), adv=self.adv,
                         ret=self.ret, lane_part=self.lane_part, **kw)
            self._perm_fused = bool(job and job.get("fused"))
        self._part_valid = bool(job and job.get("part_valid"))
        if inline_perm and not perm_first and job is None:
            # K2 -> K5a -> K4 on one stream: the scan is the long pole and starts first; the permutation kernel starts beside
            # it (programmatic launch) and only completes once the scan has, so the loss kernel behind it waits for both
            self.permute()
        if fork_perm:
            main.wait_stream(self._perm_stream)
        # The statistics table (row 0 = batch, row 1 + e*M + j = minibatch (e, j); summed over the ranks).  When the batched
        # loss kernel adds its minibatches' sums itself (fuse_stats) nothing on the step's critical path reads the table: it
        # is then produced LAZILY (ensure_table(): the per-minibatch launches of the trainer, the reports, the parity checks).
        # Round 1 put it on a side stream instead; but the loss kernel's one-wave grid takes every CTA slot of the machine,
        # so the side branch only ever ran AFTER the loss kernel and the step waited for it (N = 2: 44 us against 41.4 us with
        # the table between K2 and K4, profiles/r2_notes.md).
        self._lazy_table = self.fuse_stats and not cached
        self._stats_pending = self._lazy_table  # the batched loss adds its own statistics from lane_aos
        self._table_valid = False
        if not self._lazy_table:
            self.ensure_table()

    def perm_job(self, with_part: bool = True) -> dict:
        """The permutation job advantages() hands to the scan (ops.gae_scan, `perm_job`): this step's seed, every epoch, and
        -- where the loss adds its own statistics -- the table of per-CTA minibatch shares."""
        blk = self.shuffle_block
        job = dict(seed=self.seed + self.step_count, epoch=0, n_epochs=self.epochs, n_env=self.B // blk,
                   group=self.A * blk, out=self.perm)
        if self.mb_part is not None and with_part:
            job.update(minibatches=self.minibatches, part=self.mb_part)
        return job

    def ensure_table(self) -> None:
        """Produces local_stats / global_stats for the current sample if advantages() left them for later."""
        if self._table_valid:
            return
        # with the peer-memory exchange the table is sent from the kernel that produces it (fused), see stats.cu
        xk = dict(exchange=self.peer, global_out=self.global_stats) if (self.peer is not None and self.pg is not None) else {}
        if self.minibatches > 1:
            ops.group_stats(self.lane_part, idx=self.perm.view(-1), groups=self.epochs * self.minibatches,
                            per=self.n_mb, out=self.local_stats, whole_first=True, workspace=self.stats_ws, **xk)
        else:
            ops.group_stats(self.lane_part, groups=1, per=self.N, out=self.local_stats[0:1], workspace=self.stats_ws,
                            **xk)
        self._table_valid = True
        if not xk and self.pg is not None:
            self.exchange()

    def exchange(self) -> None:
        """The step's one data-path collective: SUM of the statistics table over the ranks."""
        if self.peer is not None:
            self.peer.allreduce_sum(self.local_stats, self.global_stats)
        else:
            exchange_stats(self.local_stats, self.global_stats, self.pg)

    def check_exchange(self) -> None:
        """Synchronises and raises when a rank never arrived at a statistics exchange (the table is NaN then)."""
        peers = [p for p in (self.peer, self.peer_loss) if p is not None]
        for p in peers:
            p.check_async()
        if peers:
            torch.cuda.current_stream().synchronize()
        for p in peers:
            p.raise_if_failed()

    def _join_stats(self) -> None:
        """Before anything reads the table (kept under its round-1 name for the callers)."""
        self.ensure_table()

    def permute(self) -> None:
        """K5a: the environment(-block) permutations of every epoch of this step, one launch."""
        blk = self.shuffle_block
        ops.philox_perm(self.seed + self.step_count, 0, self.B // blk, self.A * blk, out=self.perm, n_epochs=self.epochs)

    def stats_row(self, e: int, j: int) -> int:
        return 0 if self.minibatches == 1 else 1 + e * self.minibatches + j

    def minibatch_lanes(self, e: int, j: int) -> Optional[torch.Tensor]:
        """int32 lane indices of minibatch j in epoch e (None = the whole batch in order)."""
        if self.minibatches == 1:
            return None
        return self.perm[e, j * self.n_mb:(j + 1) * self.n_mb]

    def update_popart(self) -> None:
        """Once per epoch before the loss (mappo.py:263-264), on the whole-batch (all-reduced) row."""
        ops.popart_update(self.global_stats[0], self.popart_state, self.popart_beta, self.popart_eps, self.popart_ms)

    def loss(self, e: int, j: int, new_logp: torch.Tensor, v_pred: torch.Tensor, entropy: torch.Tensor):
        """K4 for minibatch (e, j) in deferred mode: gradients now, loss scalars + stats at finalize().
        Policy outputs are [T, n_mb] float32.  Returns (g_logp, g_value, g_entropy, None, None)."""
        self._join_stats()  # the per-minibatch launch reads its statistics from the table
        lo, hi = self.row_lo, self.row_hi
        row = self.stats_row(e, j)
        k = e * self.minibatches + j
        idx = self.minibatch_lanes(e, j)
        lf = self.leaf
        if idx is not None and not self.fuse_gather:
            m = self.mb_leaf
            ops.batch_gather([(lf["old_logp"].unsqueeze(-1), m["old_logp"].unsqueeze(-1)),
                              (lf["value"].unsqueeze(-1), m["value"].unsqueeze(-1)),
                              (self.ret.unsqueeze(-1), m["ret"].unsqueeze(-1)),
                              (self.adv.unsqueeze(-1), m["adv"].unsqueeze(-1)),
                              (lf["on_reset"].unsqueeze(-1), m["on_reset"].unsqueeze(-1))], idx)
            olp, ov, rt, ad, rs, idx = m["old_logp"], m["value"], m["ret"], m["adv"], m["on_reset"], None
        elif idx is not None and self.pack is not None and self.pack_valid:
            ops.ppo_loss_batched([self._problem(e, j, new_logp, v_pred, entropy, deferred=True)], None, None, None, None,
                                 None, self.hyper, popart_mean_std=self.popart_mean_std(), pack=self.pack, pack_row_lo=lo)
            return self.grads[e][j] + (None, None)
        else:
            olp, ov, rt, ad, rs = lf["old_logp"], lf["value"], self.ret, self.adv, lf["on_reset"]
        return ops.ppo_loss_fwd_bwd(new_logp, v_pred, entropy, olp[lo:hi], ov[lo:hi], rt[lo:hi], ad[lo:hi],
                                    rs[lo + 1:hi + 1], self.global_stats[row], self.hyper,
                                    local_stats=self.local_stats[row], popart_mean_std=self.popart_mean_std(),
                                    lane_idx=idx, grads=self.grads[e][j], workspace=self.workspace[k], defer=True)

    def loss_from_logits(self, e: int, j: int, logits: torch.Tensor, action: torch.Tensor, head_sizes, v_pred: torch.Tensor,
                         available: Optional[torch.Tensor] = None):
        """K4b for minibatch (e, j) in deferred mode, the head twin of loss(): the categorical head's logits
        `[T, n_mb, sum K]`, int32 actions `[T, n_mb, heads]` and v_pred `[T, n_mb]` (float32 or bfloat16, both the same),
        optionally SMAC's availability mask.  Gradients now, loss scalars + stats at finalize().  Returns (g_logits,
        g_value) in the inputs' dtype."""
        g_logits, g_value, _, _, _, _ = ops.ppo_loss_from_logits(
            logits, action, head_sizes, v_pred, hyper=self.hyper, available=available, defer=True,
            workspace=self.workspace[e * self.minibatches + j], **self._head_common(e, j))
        return g_logits, g_value

    def loss_from_gaussian(self, e: int, j: int, mean: torch.Tensor, log_std: torch.Tensor, action: torch.Tensor,
                           v_pred: torch.Tensor):
        """K4c for minibatch (e, j) in deferred mode, the head twin of loss(): mean and float32 actions `[T, n_mb, D]`,
        log_std `[D]` (shared) or `[T, n_mb, D]`, v_pred `[T, n_mb]`.  Gradients now, loss scalars + stats at finalize().
        Returns (g_mean, g_log_std, g_value) in the inputs' dtypes."""
        shared = log_std.dim() == 1
        self._gaussian_slots(mean.shape[-1], shared)
        g_mean, g_log_std, g_value, _, _, _, _ = ops.ppo_loss_from_gaussian(
            mean, log_std, action, v_pred, hyper=self.hyper, defer=True, workspace=self.workspace[e * self.minibatches + j],
            **self._head_common(e, j))
        return g_mean, g_log_std, g_value

    def loss_from_beta(self, e: int, j: int, concentration1: torch.Tensor, concentration0: torch.Tensor,
                       action: torch.Tensor, v_pred: torch.Tensor):
        """K4d for minibatch (e, j) in deferred mode, the head twin of loss(): concentration1, concentration0 and float32
        actions in (0, 1) `[T, n_mb, D]`, v_pred `[T, n_mb]`.  Gradients now, loss scalars + stats at finalize().
        Returns (g_concentration1, g_concentration0, g_value) in the inputs' dtype."""
        g_c1, g_c0, g_value, _, _, _, _ = ops.ppo_loss_from_beta(
            concentration1, concentration0, action, v_pred, hyper=self.hyper, defer=True,
            workspace=self.workspace[e * self.minibatches + j], **self._head_common(e, j))
        return g_c1, g_c0, g_value

    def _head_common(self, e: int, j: int) -> dict:
        """Statistics rows and sample side of a head loss for minibatch (e, j): K2's pack where this step's scan wrote it
        and the minibatch is permuted, the leaves through lane_idx otherwise (one minibatch, cached advantages,
        fuse_gather=False)."""
        self._join_stats()  # the per-minibatch launch reads its statistics from the table
        lo, hi = self.row_lo, self.row_hi
        row = self.stats_row(e, j)
        idx = self.minibatch_lanes(e, j)
        kw = dict(norm_stats=self.global_stats[row], local_stats=self.local_stats[row],
                  popart_mean_std=self.popart_mean_std(), lane_idx=idx)
        if idx is not None and self.pack is not None and self.pack_valid:
            kw.update(old_logp=None, old_value=None, ret=None, adv=None, on_reset_next=None, pack=self.pack, pack_row_lo=lo)
        else:
            lf = self.leaf
            kw.update(old_logp=lf["old_logp"][lo:hi], old_value=lf["value"][lo:hi], ret=self.ret[lo:hi],
                      adv=self.adv[lo:hi], on_reset_next=lf["on_reset"][lo + 1:hi + 1])
        return kw

    def _gaussian_slots(self, D: int, shared: bool) -> None:
        """A shared log_std's partial rows follow the K4 slot (srl_ppo_loss_gaussian_workspace_bytes): widen every slot once
        so that one loss_finalize still folds them all.  Slots already written keep their bytes."""
        need = ops.gaussian_loss_workspace_bytes(self.T, self.n_mb, D, shared)
        old = self.workspace
        if need > old.shape[1]:
            self.workspace = torch.zeros((old.shape[0], need), dtype=torch.uint8, device=self.device)
            self.workspace[:, :old.shape[1]].copy_(old)

    def _problem(self, e: int, j: int, new_logp, v_pred, entropy, deferred: bool) -> dict:
        row = self.stats_row(e, j)
        k = e * self.minibatches + j
        q = dict(new_logp=new_logp, v_pred=v_pred, entropy=entropy, lane_idx=self.minibatch_lanes(e, j),
                 norm_stats=self.global_stats[row], local_stats=self.local_stats[row], grads=self.grads[e][j],
                 workspace=self.workspace[k])
        if not deferred:
            q.update(out=self.out[k], out_f32=self.out_f32[k])
        return q

    def loss_batch(self, pairs, pol) -> None:
        """K4 for several (epoch, minibatch) pairs in ONE launch, loss scalars + stats finalised by the last CTA of
        each minibatch (no separate finalize launch).  pol[e][j] = (new_logp, v_pred, entropy)."""
        lo, hi = self.row_lo, self.row_hi
        lf = self.leaf
        probs = [self._problem(e, j, *pol[e][j], deferred=False) for e, j in pairs]
        if self.minibatches > 1 and self.pack is not None and self.pack_valid:
            own = self.lane_aos if (self.fuse_stats and self._stats_pending) else None
            # the scan's per-CTA shares serve a run of consecutive minibatches (table slot = e * minibatches + j)
            slots = [e * self.minibatches + j for e, j in pairs]
            part = self.mb_part if (own is not None and self._part_valid and
                                    slots == list(range(slots[0], slots[0] + len(slots)))) else None
            ops.ppo_loss_batched(probs, None, None, None, None, None, self.hyper,
                                 popart_mean_std=self.popart_mean_std(), pack=self.pack, pack_row_lo=lo, lane_aos=own,
                                 exchange=self.peer_loss if own is not None else None, minibatch_part=part,
                                 part_first=slots[0] if part is not None else 0)
        else:
            ops.ppo_loss_batched(probs, lf["old_logp"][lo:hi], lf["value"][lo:hi], self.ret[lo:hi], self.adv[lo:hi],
                                 lf["on_reset"][lo + 1:hi + 1], self.hyper, popart_mean_std=self.popart_mean_std())

    def finalize(self) -> None:
        """One launch: fold every minibatch's partial rows into self.out / self.out_f32 (loss scalars + stats)."""
        ops.loss_finalize(self.workspace, self.out, self.out_f32)

    # ------------------------------------------------------------------------------------------
    def _run_losses(self, pol, branches: int = 1) -> None:
        """Every (epoch, minibatch) loss launch, then finalize().  With branches > 1 the launches of one epoch are
        spread round-robin over side streams (fork/join around each epoch): under CUDA-graph capture this
        becomes parallel graph branches, so the small per-minibatch kernels overlap instead of queueing.
        (PopArt re-normalises between epochs, hence the join per epoch.)"""
        if self._immediate:
            if self.popart:  # K3 re-normalises between epochs: one launch per epoch
                for e in range(self.epochs):
                    self.update_popart()
                    self.loss_batch([(e, j) for j in range(self.minibatches)], pol)
            else:  # every (epoch, minibatch) is independent: one launch
                self.loss_batch([(e, j) for e in range(self.epochs) for j in range(self.minibatches)], pol)
            return
        main = torch.cuda.current_stream()
        if branches > 1 and not hasattr(self, "_side"):
            self._side = [torch.cuda.Stream(device=self.device) for _ in range(branches)]
        if branches <= 1:
            for e in range(self.epochs):
                if self.popart:
                    self.update_popart()
                for j in range(self.minibatches):
                    self.loss(e, j, *pol[e][j])
        elif self.popart:  # fork / join around every epoch: K3 re-normalises between epochs
            used = self._side[:min(branches, self.minibatches)]
            for e in range(self.epochs):
                self.update_popart()
                for st in used:
                    st.wait_stream(main)
                for j in range(self.minibatches):
                    with torch.cuda.stream(used[j % len(used)]):
                        self.loss(e, j, *pol[e][j])
                for st in used:
                    main.wait_stream(st)
        else:  # all E*M launches are independent: fork once, join once
            used = self._side[:min(branches, self.epochs * self.minibatches)]
            for st in used:
                st.wait_stream(main)
            for k in range(self.epochs * self.minibatches):
                e, j = divmod(k, self.minibatches)
                with torch.cuda.stream(used[k % len(used)]):
                    self.loss(e, j, *pol[e][j])
            for st in used:
                main.wait_stream(st)
        self.finalize()

    def run_device(self, pol, use_graph: bool = True, plan: bool = False) -> None:
        """The whole step on resident inputs: advantages() then every (epoch, minibatch) loss.
        pol[e][j] = (new_logp, v_pred, entropy), each [T, n_mb] float32 on device.  With use_graph the
        launches are captured once into a CUDA graph (two graphs around the all-reduce when distributed).
        plan=True: the step's C-ABI calls are recorded once (on the first call: an ordinary eager step) and from then on
        issued again as they are -- plain stream launches of the same kernels on the same buffers, without the Python-side
        argument checking of `ops` (tens of microseconds per launch) and without a graph launch."""
        if plan:
            self._run_plan(pol)
            return
        if not use_graph:
            self.advantages()
            self._run_losses(pol)
            self.step_count += 1
            return
        if self._graph is None or self._graph_pol is not pol:
            self._capture(pol)
        if self._graph_a is None:
            self._graph.replay()  # the whole step, the statistics all-reduce included when distributed
        else:
            self._graph_a.replay()
            self.exchange()
            self._graph.replay()
        self._table_valid = not self._lazy_table  # a replay does not run ensure_table()'s python side
        self.step_count += 1

    def plan_supported(self) -> bool:
        """A recorded plan holds this library's launches only: every kernel of the step must be one (no torch.distributed
        collective between them, no side streams)."""
        return (self.pg is None or self.peer is not None) and self._immediate and \
            (self.minibatches == 1 or ops.pdl_enabled())

    def _run_plan(self, pol) -> None:
        from srl_b200 import _lib
        st = torch.cuda.current_stream().cuda_stream
        if getattr(self, "_plan", None) is None or self._plan_pol is not pol or self._plan_stream != st:
            if not self.plan_supported():
                raise RuntimeError("HotPath.run_device(plan=True): the step holds launches that are not this library's (a "
                                   "torch.distributed exchange, side streams); use the CUDA graph")
            # like a captured graph, the plan re-uses the launch arguments of step_count == 0 (its permutations) every step
            saved, self.step_count = self.step_count, 0
            calls = []
            try:
                with _lib.record_calls(calls):
                    self.advantages()
                    self._run_losses(pol)
            finally:
                self.step_count = saved
            self._plan, self._plan_pol, self._plan_stream = _lib.bind_calls(calls), pol, st
            self.plan_launch_calls = len(calls)
        else:
            _lib.replay_calls(self._plan)
            self._table_valid = not self._lazy_table
        self.step_count += 1

    def run_trainer_order(self, pol, use_graph: bool = True) -> None:
        """The step in the order a trainer must issue it (mappo.py:240-299 with minibatches): GAE once, then ONE loss launch
        per (epoch, minibatch), each behind the previous one on the same stream -- minibatch j+1's policy outputs do not exist
        before the optimizer step on minibatch j, so the launches cannot be batched.  With use_graph the chain is a linear
        CUDA graph (what `bench.py` reports as step_trainer_order); `MultiAgentPPOB200.step` issues the same launches
        eagerly between its policy calls."""
        if not use_graph:
            self._trainer_order_launches(pol)
            self.step_count += 1
            return
        if getattr(self, "_graph_to", None) is None or self._graph_to_pol is not pol:
            saved = self.step_count
            self.step_count = 0
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._trainer_order_launches(pol)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._trainer_order_launches(pol)
            self._graph_to, self._graph_to_pol = g, pol
            self.step_count = saved
        self._graph_to.replay()
        self.step_count += 1

    def _trainer_order_launches(self, pol) -> None:
        self.advantages()
        self._join_stats()  # per-minibatch launches read their statistics rows from the table
        for e in range(self.epochs):
            if self.popart:
                self.update_popart()
            for j in range(self.minibatches):
                self.loss(e, j, *pol[e][j])
        self.finalize()

    def loss_chain_graph(self, pol) -> torch.cuda.CUDAGraph:
        """Only the E*M dependent per-minibatch loss launches of run_trainer_order, as a graph (bench.py: time per launch)."""
        def chain():
            for e in range(self.epochs):
                for j in range(self.minibatches):
                    self.loss(e, j, *pol[e][j])
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            chain()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            chain()
        return g

    def _capture(self, pol) -> None:
        # NOTE: launch arguments are frozen at capture, so a replayed graph re-uses the permutations of
        # step_count == 0 every step (what a benchmark wants); the trainer launches eagerly and reseeds per step.
        # warm-up on a side stream (allocations, module loading, NCCL channel set-up) before capture
        saved = self.step_count
        self.step_count = 0
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.advantages()
            self._run_losses(pol)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self._graph_a = None
        if self.pg is None or self.peer is not None:
            # one graph for the whole step; the peer-memory exchange is an ordinary kernel, so it is just a node
            # between K2 and the loss launches
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.advantages()
                self._run_losses(pol, self.graph_branches)
            self._graph = g
        else:
            # torch.distributed all-reduce (NCCL without peer access, gloo): kept BETWEEN two graphs -- a captured NCCL
            # collective measured faster (64 vs 66 us per step at 2 GPUs) but the process then hung at teardown
            pg, self.pg = self.pg, None
            try:
                ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(ga):
                    self.advantages()
                with torch.cuda.graph(gb):
                    self._run_losses(pol, self.graph_branches)
                self._graph_a, self._graph = ga, gb
            finally:
                self.pg = pg
        self.step_count = saved
        self._graph_pol = pol
        self.launches_per_step = self.count_launches()

    def count_launches(self) -> int:
        """Kernels of this library launched by one step (the claim behind bench.py's gpu_launches)."""
        n = 1 if self.fuse_stats else 2  # gae_scan (+ group_stats unless the batched loss adds its own statistics)
        if self.minibatches > 1 and not self._perm_fused:
            n += 1  # all epochs' permutations (computed inside the scan kernel when it can: advantages())
        if self._immediate:
            per_launch = 32  # SRL_MAX_LOSS_BATCH
            if self.popart:
                n += self.epochs * (1 + -(-self.minibatches // per_launch))
            else:
                n += -(-(self.epochs * self.minibatches) // per_launch)
            return n
        per_loss = 1 if (self.fuse_gather or self.minibatches == 1) else 2
        n += self.epochs * self.minibatches * per_loss
        n += 1  # loss_finalize
        if self.popart:
            n += self.epochs
        return n

    # ------------------------------------------------------------------------------------------
    def run_host(self, sample: Dict[str, np.ndarray], pol_host: torch.Tensor, out_host: Dict[str, torch.Tensor],
                 use_graph: bool = True, pol_device: Optional[torch.Tensor] = None) -> Dict[str, int]:
        """Host buffers in, host buffers out -- the call a host-side user of the path makes.

        sample: the six scalar leaves (pinned tensors are copied directly, numpy arrays are staged through pinned
        memory); pol_host: pinned float32 [E, M, 3, T, n_mb] = (new_logp, v_pred, entropy) of every minibatch;
        out_host: pinned destinations 'adv', 'ret' [L, N] (the reference mirrors them into the host sample,
        mappo.py:254-257), 'out' [E*M, 16] (loss scalars + stats) and optionally 'grads' [E, M, 3, T, n_mb] (the
        gradients otherwise stay in HBM, where the policy's backward pass consumes them).

        Three streams: copy-in (sample, then one epoch of policy outputs at a time), compute (advantages, then each
        epoch as soon as its inputs have landed) and copy-out (adv/ret while epoch 0 computes, each epoch's gradients
        while the next epoch computes), so H2D, kernels and D2H overlap on the full-duplex link.  With use_graph the
        whole choreography -- copies, kernels, cross-stream dependencies -- is ONE CUDA graph keyed by the host buffer
        addresses (the ~40 host-side launches of the eager version cost more wall clock than the kernels).
        `pol_device` (float32 [E, M, 3, T, n_mb] already in HBM, where the policy network produces it in production):
        the policy outputs are taken from there and only the sample crosses PCIe (pol_host is ignored).
        Returns the bytes moved each way."""
        E, Mb = self.epochs, self.minibatches
        if not hasattr(self, "_pol_dev_all"):
            self._pol_dev_all = torch.empty((E, Mb, 3, self.T, self.n_mb), dtype=torch.float32, device=self.device)
            self._pol_dev = [[tuple(self._pol_dev_all[e, j, q] for q in range(3)) for j in range(Mb)] for e in range(E)]
            self._s_in, self._s_out = torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device)
            self._host_graph, self._host_graph_key = None, None
        pinned = self._stage_sample(sample)
        pol_src = pol_host if pol_device is None else pol_device
        if use_graph and (self.pg is None or self.peer is not None):  # see _capture about captured NCCL collectives
            key = tuple(pinned[k].data_ptr() for k in SAMPLE_F32 + SAMPLE_U8) + (pol_src.data_ptr(),) + \
                tuple(out_host[k].data_ptr() for k in ("adv", "ret", "grads", "out") if k in out_host)
            if self._host_graph is None or self._host_graph_key != key:
                self._capture_host(pinned, pol_src, out_host)
                self._host_graph_key = key
            self._host_graph.replay()
            self._table_valid = not self._lazy_table
        else:
            self._host_pipeline(pinned, pol_src, out_host, 1)
        self.step_count += 1
        torch.cuda.current_stream().synchronize()
        h2d = sum(pinned[k].numel() * pinned[k].element_size() for k in pinned) + \
            (pol_host.numel() * 4 if pol_device is None else 0)
        d2h = 2 * self.adv.numel() * 4 + self.out.numel() * 8
        if "grads" in out_host:
            d2h += self.grads_all.numel() * 4
        return dict(h2d_bytes=h2d, d2h_bytes=d2h)

    def _stage_sample(self, sample) -> Dict[str, torch.Tensor]:
        """Pinned float32 / uint8 [L*N] images of the six leaves: pinned tensors of the right type pass through,
        anything else is converted and copied into this object's own pinned staging buffers (host work)."""
        out = {}
        seen = self.__dict__.setdefault("_pinned_seen", {})  # leaf -> (tensor object, flat view): is_pinned() asks the driver
        for k in SAMPLE_F32 + SAMPLE_U8:                       # (~10 us per leaf): a tensor OBJECT is asked once
            x = sample[k]
            c = seen.get(k)
            if c is not None and c[0] is x:
                out[k] = c[1]
                continue
            want_t = torch.float32 if k in SAMPLE_F32 else torch.uint8
            if isinstance(x, torch.Tensor) and x.is_pinned() and x.dtype == want_t and x.is_contiguous() and \
                    x.numel() == self.L * self.N:
                out[k] = x.view(-1)
                seen[k] = (x, out[k])
                continue
            if isinstance(x, torch.Tensor):
                x = x.numpy()
            if x.size != self.L * self.N:
                raise ValueError(f"{k}: {x.shape} does not hold L*N = {self.L}*{self.N} elements")
            want = np.float32 if k in SAMPLE_F32 else np.uint8
            if x.dtype != want:
                x = x.astype(want)
            pin = self._pinned(k, x)
            pin.numpy()[:] = x.reshape(-1)
            out[k] = pin
        return out

    def _host_pipeline(self, pinned, pol_host, out_host, branches: int) -> None:
        """The three-stream choreography of run_host (run eagerly, or under capture into one graph)."""
        E = self.epochs
        main = torch.cuda.current_stream()
        s_in, s_out = self._s_in, self._s_out
        s_in.wait_stream(main)
        with torch.cuda.stream(s_in):
            for k in SAMPLE_F32 + SAMPLE_U8:
                self.leaf[k].view(-1).copy_(pinned[k], non_blocking=True)
            ev_sample = torch.cuda.Event()
            ev_sample.record(s_in)
            ev_pol = []
            resident = pol_host.is_cuda  # policy outputs already in HBM: used in place
            self._pol_run = [[tuple(pol_host[e, j, q] for q in range(3)) for j in range(self.minibatches)]
                             for e in range(E)] if resident else self._pol_dev
            for e in range(E):
                if not resident:
                    self._pol_dev_all[e].copy_(pol_host[e], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
                ev_pol.append(ev)
        main.wait_event(ev_sample)
        self.advantages()
        ev_adv = torch.cuda.Event()
        ev_adv.record(main)
        s_out.wait_event(ev_adv)
        with torch.cuda.stream(s_out):
            out_host["adv"].copy_(self.adv, non_blocking=True)
            out_host["ret"].copy_(self.ret, non_blocking=True)
        for e in range(E):
            main.wait_event(ev_pol[e])
            self._run_epoch(e, branches)
            if "grads" in out_host:  # optional: the gradients normally stay in HBM for the policy's backward pass
                ev = torch.cuda.Event()
                ev.record(main)
                s_out.wait_event(ev)
                with torch.cuda.stream(s_out):
                    out_host["grads"][e].copy_(self.grads_all[e], non_blocking=True)
        if not self._immediate:
            self.finalize()
        out_host["out"].copy_(self.out, non_blocking=True)
        main.wait_stream(s_out)

    def _capture_host(self, pinned, pol_host, out_host) -> None:
        saved = self.step_count
        self.step_count = 0
        try:
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):  # warm-up outside capture (allocations, NCCL channels)
                self._host_pipeline(pinned, pol_host, out_host, 1)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._host_pipeline(pinned, pol_host, out_host, self.graph_branches)
            self._host_graph = g
        finally:
            self.step_count = saved

    def _run_epoch(self, e: int, branches: int) -> None:
        main = torch.cuda.current_stream()
        if self.popart:
            self.update_popart()
        if self._immediate:
            self.loss_batch([(e, j) for j in range(self.minibatches)], self._pol_run)
            return
        if branches <= 1:
            for j in range(self.minibatches):
                self.loss(e, j, *self._pol_run[e][j])
            return
        if not hasattr(self, "_side") or len(self._side) < branches:
            self._side = [torch.cuda.Stream(device=self.device) for _ in range(branches)]
        used = self._side[:min(branches, self.minibatches)]
        for st in used:
            st.wait_stream(main)
        for j in range(self.minibatches):
            with torch.cuda.stream(used[j % len(used)]):
                self.loss(e, j, *self._pol_run[e][j])
        for st in used:
            main.wait_stream(st)
