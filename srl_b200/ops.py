"""Tensor-level entry points: torch CUDA tensors in, C-ABI calls on the current stream, tensors out.

torch is plumbing here (device memory, streams); every computation happens inside libsrl_b200.so.
All functions raise (never fall back) when the library is missing or a tensor is not a contiguous
CUDA tensor of the expected dtype.  Reference lines each op replaces are in include/srl_b200.h.
"""
from __future__ import annotations

import ctypes
import dataclasses
from typing import List, Optional, Sequence, Tuple

import torch

from srl_b200 import _lib
from srl_b200._lib import (SRL_LANE_PART, SRL_LOSS_OUT_LEN, SRL_MAX_HEADS, SRL_MAX_LEAVES, SRL_MAX_LOSS_BATCH, LeafDesc, LossProblem,
                           PpoHyper, VALUE_LOSS_CODES)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _check(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (srl_b200 has no CPU path), got {type(t).__name__}"
                         f"{'' if not isinstance(t, torch.Tensor) else ' on ' + str(t.device)}")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor, got strides {t.stride()} for shape {tuple(t.shape)}")
    return t


def _check_view(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    """Like _check but for row-offset views (not necessarily contiguous as a whole)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (srl_b200 has no CPU path)")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t


def _rows_lanes(t: torch.Tensor) -> Tuple[int, int]:
    """[L, B, (A,) 1] or [L, N] -> (L, N)."""
    if t.dim() < 2:
        raise ValueError(f"expected a time-major [L, N, ...] tensor, got shape {tuple(t.shape)}")
    return t.shape[0], t[0].numel()


def pdl_enabled() -> bool:
    """Programmatic dependent launch between perm -> scan -> loss on one stream (include/srl_b200.h: srl_set_pdl)."""
    return bool(_lib.load_library().srl_pdl_enabled())


def set_pdl(on: bool) -> bool:
    """Switches programmatic dependent launch for later launches; returns the previous setting."""
    return bool(_lib.load_library().srl_set_pdl(int(bool(on))))


# ------------------------------------------------------------------------------------------------
# K2
# ------------------------------------------------------------------------------------------------
def gae_scan(reward, value, done, truncated, on_reset, gamma: float, lmbda: float, row_lo: int = 0,
             row_hi: Optional[int] = None, popart_mean_std: Optional[torch.Tensor] = None,
             vtrace_new_logp: Optional[torch.Tensor] = None, vtrace_old_logp: Optional[torch.Tensor] = None,
             rho: float = 1.0, c: float = 1.0, adv: Optional[torch.Tensor] = None,
             ret: Optional[torch.Tensor] = None, lane_part: Optional[torch.Tensor] = None, want_stats: bool = True,
             old_logp: Optional[torch.Tensor] = None, pack: Optional[torch.Tensor] = None,
             lane_aos: Optional[torch.Tensor] = None, perm_job: Optional[dict] = None):
    """GAE + value target + zero padding row + per-lane statistics in one launch.

    reward/value float32 and done/truncated/on_reset uint8, all `[L, N(, 1)]`; returns
    (adv, ret) shaped like `value` and lane_part float64 `[8, N]` (or None).
    `pack` (float32 `[ceil(L/2), N, 2, 4]` = `new_pack(L, N)`, needs `old_logp` `[L, N]`): additionally writes the loss's
    sample side as one 16-byte item per transition, {old_logp, value, ret, mask ? adv : NaN}, the two rows of a row pair
    next to each other (see include/srl_b200.h; `unpack_rows` gives the `[L, N, 4]` view back).
    `lane_aos` (float64 `[N, 4]`): rows 0..2 of lane_part once more as one 32-byte item per lane.
    `perm_job` (dict: seed, epoch, n_epochs, n_env, group, out int32 `[n_epochs, n_env * group]`): the step's minibatch
    permutations (== `philox_perm` with the same arguments, bit for bit) computed by the scan kernel's own idle threads where
    the kernel chosen for this shape can (srl_gae_scan_perm), by the stand-alone kernel behind the scan otherwise; the
    dict's key "fused" says which (True / False).  Optional keys `minibatches` and `part` (float64
    `new_minibatch_part(N)` = `[32, ceil(N / 32), 4]`): every scan CTA also leaves its 32 lanes' share of every minibatch's
    {count, sum, sum of squares} -- what `ppo_loss_batched(minibatch_part=...)` adds instead of gathering lane items; the
    key "part_valid" says whether the table was written (only by the fused kernel, <= 8 epochs, <= 32 minibatches per step).
    Reference: MultiAgentPPO._compute_adv_and_value_target (mappo.py:118-144) + F.pad (mappo.py:254-256).
    """
    L, N = _rows_lanes(value)
    for name, t in (("reward", reward), ("value", value)):
        _check(t, torch.float32, name)
    for name, t in (("done", done), ("truncated", truncated), ("on_reset", on_reset)):
        _check(t, torch.uint8, name)
    for name, t in (("reward", reward), ("done", done), ("truncated", truncated), ("on_reset", on_reset)):
        if _rows_lanes(t) != (L, N):
            raise ValueError(f"{name}: shape {tuple(t.shape)} does not match value {tuple(value.shape)}")
    if row_hi is None:
        row_hi = L - 1
    if (vtrace_new_logp is None) != (vtrace_old_logp is None):
        raise ValueError("vtrace needs both new and old log-probs")
    for name, t in (("vtrace_new_logp", vtrace_new_logp), ("vtrace_old_logp", vtrace_old_logp)):
        if t is not None:
            _check(t, torch.float32, name)
            if t.shape[0] < L - 1 or t[0].numel() != N:
                raise ValueError(f"{name}: need at least L-1={L - 1} rows of {N} lanes, got {tuple(t.shape)}")
    if popart_mean_std is not None:
        _check(popart_mean_std, torch.float64, "popart_mean_std")
    adv = torch.empty_like(value) if adv is None else _check(adv, torch.float32, "adv")
    ret = torch.empty_like(value) if ret is None else _check(ret, torch.float32, "ret")
    if want_stats and lane_part is None:
        lane_part = torch.empty((SRL_LANE_PART, N), dtype=torch.float64, device=value.device)
    if lane_part is not None:
        _check(lane_part, torch.float64, "lane_part")
        if tuple(lane_part.shape) != (SRL_LANE_PART, N):
            raise ValueError(f"lane_part: expected shape {(SRL_LANE_PART, N)}, got {tuple(lane_part.shape)}")
    if pack is not None:
        _check(pack, torch.float32, "pack")
        if old_logp is None:
            raise ValueError("pack needs old_logp")
        _check(old_logp, torch.float32, "old_logp")
        if pack.numel() != pack_rows(L) * N * 4 or _rows_lanes(old_logp) != (L, N):
            raise ValueError(f"pack must hold [ceil(L/2), N, 2, 4] = {pack_rows(L) * N * 4} floats and old_logp [L, N]; got "
                             f"{tuple(pack.shape)} and {tuple(old_logp.shape)}")
    if lane_aos is not None:
        _check(lane_aos, torch.float64, "lane_aos")
        if lane_part is None or tuple(lane_aos.shape) != (N, 4):
            raise ValueError(f"lane_aos needs lane_part and shape {(N, 4)}, got {tuple(lane_aos.shape)}")
    args = (_ptr(reward), _ptr(value), _ptr(done), _ptr(truncated), _ptr(on_reset),
            _ptr(vtrace_new_logp), _ptr(vtrace_old_logp), _ptr(popart_mean_std),
            _ptr(old_logp) if pack is not None else None, L, N, int(row_lo), int(row_hi),
            float(gamma), float(lmbda), float(rho), float(c), _ptr(adv), _ptr(ret), _ptr(lane_part), _ptr(lane_aos),
            _ptr(pack))
    if perm_job is None:
        _lib.call("srl_gae_scan", *args, _stream())
    else:
        out = _check(perm_job["out"], torch.int32, "perm_job['out']")
        n_ep, n_env, group = int(perm_job["n_epochs"]), int(perm_job["n_env"]), int(perm_job.get("group", 1))
        if out.numel() != n_ep * n_env * group:
            raise ValueError(f"perm_job['out'] must hold [n_epochs, n_env * group] = {n_ep * n_env * group} int32")
        part = perm_job.get("part")
        if part is not None:
            _check(part, torch.float64, "perm_job['part']")
            if tuple(part.shape) != (SRL_MAX_LOSS_BATCH, (N + 31) // 32, 4):
                raise ValueError(f"perm_job['part']: expected new_minibatch_part(N) = {(SRL_MAX_LOSS_BATCH, (N + 31) // 32, 4)}, "
                                 f"got {tuple(part.shape)}")
        fused = ctypes.c_int(0)
        _lib.call("srl_gae_scan_perm", *args, ctypes.c_uint64(int(perm_job["seed"]) & (2 ** 64 - 1)),
                  ctypes.c_uint32(int(perm_job.get("epoch", 0))), n_ep, n_env, group, _ptr(out),
                  int(perm_job.get("minibatches", 1)), _ptr(part), ctypes.byref(fused), _stream())
        perm_job["fused"] = fused.value >= 1
        perm_job["part_valid"] = fused.value == 2
    return adv, ret, lane_part


def new_minibatch_part(N: int, device) -> torch.Tensor:
    """The table srl_gae_scan_perm's `minibatch_part` writes: [minibatch slot][scan CTA = 32-lane group][4] float64."""
    return torch.zeros((SRL_MAX_LOSS_BATCH, (N + 31) // 32, 4), dtype=torch.float64, device=device)


def pack_rows(L: int) -> int:
    """Rows the pair-interleaved loss pack holds for an L-row sample (L rounded up to even)."""
    return L + (L & 1)


def new_pack(L: int, N: int, device) -> torch.Tensor:
    """K2's loss pack for an `[L, N]` sample: float32 `[ceil(L/2), N, 2, 4]` (include/srl_b200.h, srl_gae_scan)."""
    return torch.empty((pack_rows(L) // 2, N, 2, 4), dtype=torch.float32, device=device)


def unpack_rows(pack: torch.Tensor) -> torch.Tensor:
    """`[rows, N, 4]` view-copy of a pair-interleaved pack (tests, debugging): row t = pack[t // 2, :, t % 2]."""
    P, N = pack.shape[0], pack.shape[1]
    return pack.permute(0, 2, 1, 3).reshape(2 * P, N, 4)


def gae_trace(reward, value, truncated, done, on_reset, gamma, lmbda, vtrace: bool = False, imp_ratio=None,
              rho: float = 1.0, c: float = 1.0, high_precision: bool = True, apply_done: bool = False,
              want_ret: bool = False, pad_last_row: bool = False):
    """Same signature and meaning as modules.gae_trace (legacy/algorithm/modules/gae.py:8-97), on device:
    reward float32 `[T, bs, Nc]`, value `[T+1, bs, Nc]`, truncated / done / on_reset uint8 `[T+1, bs, 1]`; `gamma` /
    `lmbda` a python float or a float32 tensor `[T, bs, 1]`; `imp_ratio` float32 `[T, bs, 1]` with `vtrace`.
    Returns adv float32 `[T, bs, Nc]` (`[T+1, ..]` with a zero row when `pad_last_row`, mappo.py:254-256).
    `apply_done` multiplies value by (1 - done) first and `want_ret` also returns the value target -- together they are
    MultiAgentPPO._compute_adv_and_value_target (mappo.py:118-144) for vector critics and per-element discounts.
    `done` is otherwise only shape-checked: the reference reads it in its data asserts alone (gae.py:69-77)."""
    if not high_precision:
        raise NotImplementedError("gae_trace: only the float64 scan (high_precision=True, the reference's default)")
    for name, t in (("reward", reward), ("value", value)):
        _check(t, torch.float32, name)
    for name, t in (("truncated", truncated), ("done", done), ("on_reset", on_reset)):
        _check(t, torch.uint8, name)
    L = value.shape[0]
    if L < 2 or reward.shape[0] < L - 1:
        raise ValueError(f"value needs >= 2 rows and reward >= L-1 rows; got {tuple(value.shape)}, {tuple(reward.shape)}")
    N = on_reset[0].numel()
    if value[0].numel() % N != 0:
        raise ValueError(f"value {tuple(value.shape)} is not on_reset {tuple(on_reset.shape)} x critic_dim")
    Nc = value[0].numel() // N
    if reward[0].numel() != N * Nc:
        raise ValueError(f"reward {tuple(reward.shape)} does not match value {tuple(value.shape)}")
    for name, t in (("truncated", truncated), ("done", done)):
        if t.shape[0] != L or t[0].numel() != N:
            raise ValueError(f"{name}: shape {tuple(t.shape)} does not match on_reset {tuple(on_reset.shape)}")
    per = {}
    for name, x in (("gamma", gamma), ("lmbda", lmbda)):
        if isinstance(x, torch.Tensor):
            _check(x, torch.float32, name)
            if x.shape[0] != L - 1 or x[0].numel() != N:  # gae.py:53,58: same shape as on_reset[:-1]
                raise AssertionError(tuple(x.shape))
            per[name] = x
        elif not isinstance(x, float):
            raise AssertionError(type(x))  # gae.py:52,57
    if vtrace:
        if imp_ratio is None:
            raise ValueError("vtrace needs imp_ratio")
        _check(imp_ratio, torch.float32, "imp_ratio")
        if imp_ratio.shape[0] < L - 1 or imp_ratio[0].numel() != N:
            raise ValueError(f"imp_ratio: need [>= {L - 1}, {N}], got {tuple(imp_ratio.shape)}")
    rows = L if pad_last_row else L - 1
    adv = torch.empty((rows,) + tuple(value.shape[1:]), dtype=torch.float32, device=value.device)
    ret = torch.empty_like(adv) if want_ret else None
    _lib.call("srl_gae_trace", _ptr(reward), _ptr(value), _ptr(done) if apply_done else None, _ptr(truncated),
              _ptr(on_reset), _ptr(per.get("gamma")), _ptr(per.get("lmbda")), _ptr(imp_ratio) if vtrace else None, L, N,
              Nc, 0.0 if "gamma" in per else float(gamma), 0.0 if "lmbda" in per else float(lmbda), float(rho), float(c),
              int(bool(pad_last_row)), _ptr(adv), _ptr(ret), _stream())
    return (adv, ret) if want_ret else adv


def traj_gae(reward, value, offsets, final_truncated, final_has_value, gamma: float, lmbda: float):
    """GAE along whole episodes laid out one after another (TrajGAE.process, gae.py:100-139, for many episodes):
    reward / value `[total_steps, W]` float32 or float64 (one dtype), offsets int64 `[n + 1]`, final_truncated uint8
    `[n, W]`, final_has_value uint8 `[n]`.  Returns (adv, ret) like reward; the last step of each episode is left 0."""
    if reward.dtype not in (torch.float32, torch.float64):
        raise ValueError(f"reward: expected float32 or float64, got {reward.dtype}")
    _check(reward, reward.dtype, "reward")
    _check(value, reward.dtype, "value")
    _check(offsets, torch.int64, "offsets")
    _check(final_truncated, torch.uint8, "final_truncated")
    _check(final_has_value, torch.uint8, "final_has_value")
    if reward.dim() != 2 or value.shape != reward.shape:
        raise ValueError(f"reward / value: expected equal [total_steps, W] shapes, got {tuple(reward.shape)}, "
                         f"{tuple(value.shape)}")
    n = offsets.numel() - 1
    W = reward.shape[1]
    if n < 0 or final_has_value.numel() != n or final_truncated.numel() != n * W:
        raise ValueError("offsets / final_truncated / final_has_value disagree on the number of episodes")
    adv = torch.zeros_like(reward)
    ret = torch.zeros_like(reward)
    _lib.call("srl_traj_gae", _ptr(reward), _ptr(value), _ptr(offsets), _ptr(final_truncated), _ptr(final_has_value), n,
              W, int(reward.dtype == torch.float64), float(gamma), float(lmbda), _ptr(adv), _ptr(ret), _stream())
    return adv, ret


def n_step_return(n: int, reward, nex_value, nex_done, nex_truncated, gamma: float,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """n-step return: reward / nex_value float32 and nex_done / nex_truncated uint8, all `[n+T-1, N(, 1)]`; returns
    float32 `[T, N(, 1)]`.  Reference: modules.n_step_return (legacy/algorithm/modules/n_step_return.py:11-50)."""
    rows, N = _rows_lanes(reward)
    for name, t in (("reward", reward), ("nex_value", nex_value)):
        _check(t, torch.float32, name)
    for name, t in (("nex_done", nex_done), ("nex_truncated", nex_truncated)):
        _check(t, torch.uint8, name)
    for name, t in (("nex_value", nex_value), ("nex_done", nex_done), ("nex_truncated", nex_truncated)):
        if _rows_lanes(t) != (rows, N):
            raise ValueError(f"{name}: shape {tuple(t.shape)} does not match reward {tuple(reward.shape)}")
    if not 1 <= n <= rows:
        raise ValueError(f"need 1 <= n <= rows = {rows}, got n = {n}")
    T = rows - n + 1
    if out is None:
        out = torch.empty((T,) + tuple(reward.shape[1:]), dtype=torch.float32, device=reward.device)
    _check(out, torch.float32, "out")
    if out.numel() != T * N:
        raise ValueError(f"out holds {out.numel()} elements, expected T*N = {T * N}")
    _lib.call("srl_n_step_return", _ptr(reward), _ptr(nex_value), _ptr(nex_done), _ptr(nex_truncated), int(n), rows, N,
              float(gamma), _ptr(out), _stream())
    return out


def lane_stats(adv, ret, done, truncated, on_reset, row_lo: int, row_hi: int,
               lane_part: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-lane partial sums [8, N] from existing adv / ret (cached advantages of a re-served sample)."""
    L, N = _rows_lanes(adv)
    for name, t in (("adv", adv), ("ret", ret)):
        _check(t, torch.float32, name)
    for name, t in (("done", done), ("truncated", truncated), ("on_reset", on_reset)):
        _check(t, torch.uint8, name)
        if _rows_lanes(t) != (L, N):
            raise ValueError(f"{name}: shape {tuple(t.shape)} does not match adv {tuple(adv.shape)}")
    if lane_part is None:
        lane_part = torch.empty((SRL_LANE_PART, N), dtype=torch.float64, device=adv.device)
    _check(lane_part, torch.float64, "lane_part")
    _lib.call("srl_lane_stats", _ptr(adv), _ptr(ret), _ptr(done), _ptr(truncated), _ptr(on_reset), L, N, int(row_lo),
              int(row_hi), _ptr(lane_part), _stream())
    return lane_part


_stats_ws = {}


def group_stats_workspace(device, groups: int, whole_first: bool) -> torch.Tensor:
    """Zeroed scratch for group_stats (ticket counters + per-chunk partial rows); one per concurrent stream."""
    nbytes = int(_lib.load_library().srl_group_stats_workspace_bytes(int(groups), int(bool(whole_first))))
    return torch.zeros(nbytes, dtype=torch.uint8, device=device)


def group_stats(lane_part: torch.Tensor, idx: Optional[torch.Tensor] = None, groups: int = 1,
                per: Optional[int] = None, out: Optional[torch.Tensor] = None, whole_first: bool = False,
                workspace: Optional[torch.Tensor] = None, exchange=None,
                global_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[g, k] = sum of lane_part[k, lane] over the lanes of group g (fixed summation order).
    whole_first: out gets groups + 1 rows, row 0 = the sum over all N lanes (one launch for the whole table)."""
    _check(lane_part, torch.float64, "lane_part")
    N = lane_part.shape[1]
    if per is None:
        per = (idx.numel() if idx is not None else N) // groups
    if idx is not None:
        _check(idx, torch.int32, "idx")
        if idx.numel() < groups * per:
            raise ValueError(f"idx has {idx.numel()} entries, need groups*per = {groups * per}")
    rows = groups + (1 if whole_first else 0)
    out = torch.empty((rows, SRL_LANE_PART), dtype=torch.float64, device=lane_part.device) if out is None else out
    _check(out, torch.float64, "out")
    if out.numel() < rows * SRL_LANE_PART:
        raise ValueError(f"out has {out.numel()} entries, need {rows * SRL_LANE_PART}")
    if workspace is None:  # default scratch: one per (device, stream, table shape)
        key = (lane_part.device.index, _stream(), int(groups), bool(whole_first))
        workspace = _stats_ws.get(key)
        if workspace is None:
            workspace = _stats_ws[key] = group_stats_workspace(lane_part.device, groups, whole_first)
    _check(workspace, torch.uint8, "workspace")
    if exchange is not None:  # srl_b200.xchg.PeerExchange: the table goes to the peers from this very kernel
        if global_out is None:
            raise ValueError("a fused exchange needs global_out")
        _check(global_out, torch.float64, "global_out")
        if global_out.numel() < rows * SRL_LANE_PART:
            raise ValueError(f"global_out has {global_out.numel()} entries, need {rows * SRL_LANE_PART}")
        _lib.call("srl_group_stats_xchg", _ptr(lane_part), N, _ptr(idx), int(groups), int(per), int(bool(whole_first)),
                  _ptr(out), _ptr(global_out), _ptr(workspace), workspace.numel(), exchange._h, _stream())
        return out
    _lib.call("srl_group_stats", _ptr(lane_part), N, _ptr(idx), int(groups), int(per), int(bool(whole_first)), _ptr(out),
              _ptr(workspace), workspace.numel(), _stream())
    return out


def popart_update(batch_stats: torch.Tensor, state: torch.Tensor, beta: float, eps: float,
                  mean_std: torch.Tensor) -> None:
    """RunningMeanStd.update + mean_std (utils.py:106-137) on device; state/mean_std float64 [4]."""
    _check(batch_stats, torch.float64, "batch_stats")
    _check(state, torch.float64, "state")
    _check(mean_std, torch.float64, "mean_std")
    if batch_stats.numel() < 5 or state.numel() < 4 or mean_std.numel() < 4:
        raise ValueError("popart_update: batch_stats needs >= 5, state and mean_std >= 4 float64 entries")
    _lib.call("srl_popart_update", _ptr(batch_stats), _ptr(state), float(beta), float(eps), _ptr(mean_std), _stream())


# ------------------------------------------------------------------------------------------------
# K4
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class LossHyper:
    """The hyper-parameters of mappo.py:71-112 that enter the loss."""
    eps_clip: float = 0.2
    clip_value: bool = False
    value_eps_clip: Optional[float] = None  # defaults to eps_clip (mappo.py:90)
    dual_clip: bool = True
    c_clip: float = 3.0
    value_loss: str = "mse"
    value_loss_config: Optional[dict] = None
    value_loss_weight: float = 0.5
    entropy_bonus_weight: float = 0.01
    normalize_old_value: bool = False
    adv_eps: float = 1e-5

    def to_c(self) -> PpoHyper:
        if self.value_loss not in VALUE_LOSS_CODES:
            # same failure the reference raises at utils.py:246-249
            raise AssertionError(f"Value loss name {self.value_loss} does not match any implemented loss functions "
                                 f"({list(VALUE_LOSS_CODES)})")
        cfg = dict(self.value_loss_config or {})
        if self.value_loss == "huber":
            prm = cfg.pop("delta", 1.0)
        elif self.value_loss == "smoothl1":
            prm = cfg.pop("beta", 1.0)
        else:
            prm = 0.0
        cfg.pop("reduction", None)
        if cfg:
            raise TypeError(f"unsupported value_loss_config keys for {self.value_loss}: {sorted(cfg)}")
        veps = self.eps_clip if self.value_eps_clip is None else self.value_eps_clip
        return PpoHyper(float(self.eps_clip), float(veps), float(self.c_clip), float(self.value_loss_weight),
                        float(self.entropy_bonus_weight), float(prm), float(self.adv_eps),
                        VALUE_LOSS_CODES[self.value_loss], int(bool(self.clip_value)), int(bool(self.dual_clip)),
                        int(bool(self.normalize_old_value)))


_workspaces = {}


def loss_slot_bytes() -> int:
    return int(_lib.load_library().srl_ppo_loss_workspace_bytes(1, 1))


def new_loss_workspace(device, slots: int = 1) -> torch.Tensor:
    """Zero-initialised scratch for the loss kernels, uint8 [slots, slot_bytes] (the ticket counter must start at
    0; the kernel re-zeroes it).  Launches that may overlap in time must use different slots."""
    return torch.zeros((slots, loss_slot_bytes()), dtype=torch.uint8, device=device)


def loss_finalize(workspace: torch.Tensor, out: torch.Tensor, out_f32: Optional[torch.Tensor] = None) -> None:
    """Folds every slot of a deferred-mode workspace [slots, slot_bytes] into out [slots, 16] (float64) and
    out_f32 [slots, 4] in one launch."""
    _check(workspace, torch.uint8, "workspace")
    _check(out, torch.float64, "out")
    slots = workspace.shape[0]
    if out.numel() < slots * SRL_LOSS_OUT_LEN or (out_f32 is not None and out_f32.numel() < slots * 4):
        raise ValueError("loss_finalize: output tensors smaller than the number of slots")
    _lib.call("srl_ppo_loss_finalize", _ptr(workspace), workspace.shape[1], slots, _ptr(out), _ptr(out_f32), _stream())


def loss_workspace(device) -> torch.Tensor:
    """Default scratch: one buffer per (device, stream)."""
    key = (torch.device(device).index, _stream())
    ws = _workspaces.get(key)
    if ws is None:
        ws = _workspaces[key] = new_loss_workspace(device)
    return ws


def _sample_side(old_logp, old_value, ret, adv, on_reset_next, lane_idx, T, n, clip_value):
    """Validates the sample-side views: row stride = stride(0), unit lane stride, >= T rows."""
    ld = None
    for name, t, dt in (("old_logp", old_logp, torch.float32), ("old_value", old_value, torch.float32),
                        ("ret", ret, torch.float32), ("adv", adv, torch.float32),
                        ("on_reset_next", on_reset_next, torch.uint8)):
        if t is None:
            if name == "old_value" and not clip_value:
                continue
            raise ValueError(f"{name} is required")
        if not t.is_cuda or t.dtype != dt:
            raise ValueError(f"{name}: expected CUDA {dt}, got {t.dtype} on {t.device}")
        if t.dim() != 2 or t.stride(1) != 1 or t.shape[0] < T:
            raise ValueError(f"{name}: expected a [>=T, N] view with unit lane stride, got shape {tuple(t.shape)} "
                             f"strides {t.stride()}")
        this_ld = t.stride(0) if t.shape[0] > 1 else t.shape[1]
        if ld is None:
            ld = this_ld
        elif this_ld != ld:
            raise ValueError(f"{name}: row stride {this_ld} differs from the other sample leaves ({ld})")
        if lane_idx is None and t.shape[1] != n:
            raise ValueError(f"{name}: {t.shape[1]} lanes but the policy side has {n}")
    if lane_idx is not None:
        _check(lane_idx, torch.int32, "lane_idx")
        if lane_idx.numel() != n:
            raise ValueError(f"lane_idx has {lane_idx.numel()} entries, policy side has {n} lanes")
    return ld


def ppo_loss_fwd_bwd(new_logp, v_pred, entropy, old_logp, old_value, ret, adv, on_reset_next, norm_stats, hyper: LossHyper,
                     local_stats=None, popart_mean_std=None, lane_idx=None, grads=None, out=None, out_f32=None,
                     workspace=None, defer: bool = False):
    """One launch: loss, stats and d loss / d (new_logp, v_pred, entropy).

    Policy side `[T, n]` float32 contiguous; sample side `[>=T, N]` row views already offset to the
    first loss row (`on_reset_next` offset by one more row, mappo.py:260-261); `lane_idx` int32 `[n]`
    fuses the minibatch gather into the loads.  norm_stats: float64 `[>=3]` = (sum mask, sum adv*mask,
    sum (adv*mask)^2), all-reduced across ranks; local_stats: this rank's (defaults to norm_stats).
    Returns (g_logp, g_value, g_entropy, out float64[16], out_f32 float32[4]).
    """
    T, n = _rows_lanes(new_logp)
    for name, t in (("new_logp", new_logp), ("v_pred", v_pred), ("entropy", entropy)):
        _check(t, torch.float32, name)
        if _rows_lanes(t) != (T, n):
            raise ValueError(f"{name}: shape {tuple(t.shape)} does not match new_logp {tuple(new_logp.shape)}")
    ld_smp = _sample_side(old_logp, old_value, ret, adv, on_reset_next, lane_idx, T, n, hyper.clip_value)
    _check(norm_stats, torch.float64, "norm_stats")
    local_stats = norm_stats if local_stats is None else _check(local_stats, torch.float64, "local_stats")
    if popart_mean_std is not None:
        _check(popart_mean_std, torch.float64, "popart_mean_std")
    dev = new_logp.device
    if grads is None:
        grads = tuple(torch.empty_like(new_logp) for _ in range(3))
    if defer:  # gradients + partial rows only; loss_finalize() folds the slot(s) later
        if workspace is None:
            raise ValueError("deferred finalisation needs an explicit workspace slot")
        out = out_f32 = None
    else:
        out = torch.empty(SRL_LOSS_OUT_LEN, dtype=torch.float64, device=dev) if out is None else out
        out_f32 = torch.empty(4, dtype=torch.float32, device=dev) if out_f32 is None else out_f32
    ws = loss_workspace(dev) if workspace is None else workspace
    hc = hyper.to_c()
    _lib.call("srl_ppo_loss_fwd_bwd", _ptr(new_logp), _ptr(v_pred), _ptr(entropy), n, _ptr(old_logp), _ptr(old_value),
              _ptr(ret), _ptr(adv), _ptr(on_reset_next), ld_smp, _ptr(lane_idx), T, n, _ptr(norm_stats),
              _ptr(local_stats), _ptr(popart_mean_std), ctypes.byref(hc), _ptr(grads[0]), _ptr(grads[1]),
              _ptr(grads[2]), n, _ptr(out), _ptr(out_f32), _ptr(ws), ws.numel(), _stream())
    return grads[0], grads[1], grads[2], out, out_f32


def ppo_loss_batched(problems: Sequence[dict], old_logp, old_value, ret, adv, on_reset_next, hyper: LossHyper,
                     popart_mean_std=None, pack: Optional[torch.Tensor] = None, pack_row_lo: int = 0,
                     lane_aos: Optional[torch.Tensor] = None, exchange=None,
                     minibatch_part: Optional[torch.Tensor] = None, part_first: int = 0) -> None:
    """Several minibatches of one shape in ONE launch (srl_ppo_loss_fwd_bwd_batched).

    Each problem is a dict with `new_logp`, `v_pred`, `entropy` (`[T, n]` float32), `norm_stats`, `local_stats`
    (float64), `grads` (three `[T, n]` float32 outputs), `workspace` (one uint8 slot row), optional `lane_idx`
    (int32 `[n]`), `out` (float64 `[16]`) and `out_f32` (float32 `[4]`); without `out` the problem is deferred
    (loss_finalize folds its slot later).  The sample side is shared: the five leaf views of ppo_loss_fwd_bwd, or
    `pack` = the whole pair-interleaved pack K2 wrote (`new_pack`) with `pack_row_lo` = the sample row of loss row 0.
    `lane_aos` (K2's `[N, 4]` float64 table; pack form with lane indices, one GPU, no PopArt, even n <= 1024): the kernel
    adds the minibatch statistics itself and `norm_stats` / `local_stats` of the problems are not read (may be omitted).
    `minibatch_part` (with `lane_aos`; the table `gae_scan`'s perm_job wrote, "part_valid"): problem k's sums are table slot
    `part_first + k`'s per-CTA shares -- its `lane_idx` must be that slot's minibatch of the same scan's permutation.
    `exchange` (a srl_b200.xchg.PeerExchange of its own, with `lane_aos`, several ranks): the kernel adds every problem's sums
    over the ranks itself (NVLink peer memory) -- no statistics kernels between the scan and the loss.
    The gradient tensors must not alias the policy-side inputs."""
    if not problems:
        return
    T, n = _rows_lanes(problems[0]["new_logp"])
    has_idx = problems[0].get("lane_idx") is not None
    arr = (LossProblem * len(problems))()
    slot_bytes = None
    for k, q in enumerate(problems):
        for name in ("new_logp", "v_pred", "entropy"):
            _check(q[name], torch.float32, f"problem {k} {name}")
            if _rows_lanes(q[name]) != (T, n):
                raise ValueError(f"problem {k} {name}: shape {tuple(q[name].shape)}, expected [T, n] = [{T}, {n}]")
        for g in q["grads"]:
            _check(g, torch.float32, f"problem {k} gradient")
            if g.numel() != T * n:
                raise ValueError(f"problem {k}: gradient tensor holds {g.numel()} elements, expected {T * n}")
        ns = q.get("norm_stats")
        if ns is None and lane_aos is None:
            raise ValueError(f"problem {k}: norm_stats is required unless lane_aos is given")
        if ns is not None:
            _check(ns, torch.float64, f"problem {k} norm_stats")
        ls = q.get("local_stats")
        ls = ns if ls is None else _check(ls, torch.float64, f"problem {k} local_stats")
        li = q.get("lane_idx")
        if (li is not None) != has_idx:
            raise ValueError("either every problem has a lane_idx or none has")
        if li is not None:
            _check(li, torch.int32, f"problem {k} lane_idx")
            if li.numel() != n:
                raise ValueError(f"problem {k}: lane_idx has {li.numel()} entries, policy side has {n} lanes")
        ws = _check(q["workspace"], torch.uint8, f"problem {k} workspace")
        slot_bytes = ws.numel() if slot_bytes is None else min(slot_bytes, ws.numel())
        out, out_f32 = q.get("out"), q.get("out_f32")
        if out is not None:
            _check(out, torch.float64, f"problem {k} out")
        if out_f32 is not None:
            _check(out_f32, torch.float32, f"problem {k} out_f32")
        arr[k] = LossProblem(_ptr(q["new_logp"]), _ptr(q["v_pred"]), _ptr(q["entropy"]), _ptr(li), _ptr(ns),
                             _ptr(ls), _ptr(q["grads"][0]), _ptr(q["grads"][1]), _ptr(q["grads"][2]), _ptr(out),
                             _ptr(out_f32), _ptr(ws))
    if pack is not None:
        _check(pack, torch.float32, "pack")
        if pack.dim() != 4 or pack.shape[2:] != (2, 4) or 2 * pack.shape[0] < pack_row_lo + T or pack_row_lo < 0:
            raise ValueError(f"pack: expected K2's [ceil(L/2), N, 2, 4] float32 pack holding rows [{pack_row_lo}, "
                             f"{pack_row_lo + T}), got shape {tuple(pack.shape)}")
        ld_smp = pack.shape[1]
        if not has_idx and pack.shape[1] != n:
            raise ValueError(f"pack has {pack.shape[1]} lanes but the policy side has {n}")
        old_logp = old_value = ret = adv = on_reset_next = None
    else:
        ld_smp = _sample_side(old_logp, old_value, ret, adv, on_reset_next, problems[0].get("lane_idx"), T, n,
                              hyper.clip_value)
    if popart_mean_std is not None:
        _check(popart_mean_std, torch.float64, "popart_mean_std")
    if lane_aos is not None:
        _check(lane_aos, torch.float64, "lane_aos")
        if pack is None or lane_aos.dim() != 2 or tuple(lane_aos.shape) != (pack.shape[1], 4):
            raise ValueError(f"lane_aos: expected [N, 4] float64 beside the pack, got {tuple(lane_aos.shape)}")
    part_ctas = 0
    if minibatch_part is not None:
        _check(minibatch_part, torch.float64, "minibatch_part")
        if lane_aos is None or minibatch_part.dim() != 3 or \
                tuple(minibatch_part.shape) != (SRL_MAX_LOSS_BATCH, (lane_aos.shape[0] + 31) // 32, 4):
            raise ValueError(f"minibatch_part: expected new_minibatch_part(N) beside lane_aos, got {tuple(minibatch_part.shape)}")
        part_ctas = minibatch_part.shape[1]
    hc = hyper.to_c()
    _lib.call("srl_ppo_loss_fwd_bwd_batched", arr, len(problems), n, n, _ptr(old_logp), _ptr(old_value), _ptr(ret),
              _ptr(adv), _ptr(on_reset_next), ld_smp, _ptr(pack), int(pack_row_lo), _ptr(lane_aos), _ptr(minibatch_part),
              part_ctas, int(part_first), T, n,
              _ptr(popart_mean_std), ctypes.byref(hc), slot_bytes, None if exchange is None else exchange._h, _stream())


def _availability(available, logits) -> torch.Tensor:
    """The availability mask as the kernel reads it: one byte per logit, non-zero = available."""
    if not isinstance(available, torch.Tensor):
        raise ValueError(f"available: expected a tensor, got {type(available).__name__}")
    if tuple(available.shape) != tuple(logits.shape):
        raise ValueError(f"available: shape {tuple(available.shape)} does not match logits {tuple(logits.shape)}")
    if any(st == 0 and sz > 1 for st, sz in zip(available.stride(), available.shape)):
        raise ValueError(f"available: a stride-0 expand (strides {available.stride()}); the mask is read per logit, pass "
                         f"a dense [T, n, sum K] tensor")
    if not available.is_contiguous():
        raise ValueError(f"available: expected a contiguous tensor, got strides {available.stride()}")
    if available.dtype.is_floating_point:
        available = available != 0  # the reference's `available_action == 0` test, negated
    elif available.dtype not in (torch.uint8, torch.bool):
        raise ValueError(f"available: expected dtype torch.uint8, torch.bool or a floating dtype, got {available.dtype}")
    if not available.is_cuda or available.device != logits.device:
        raise ValueError(f"available: expected a CUDA tensor on {logits.device}, got one on {available.device}")
    return available


def ppo_loss_from_logits(logits, action, head_sizes: Sequence[int], v_pred, old_logp, old_value, ret, adv, on_reset_next,
                         norm_stats, hyper: LossHyper, local_stats=None, popart_mean_std=None, lane_idx=None,
                         want_logp_entropy: bool = False, available=None, workspace=None, defer: bool = False):
    """Loss starting from the actor head's logits `[T, n, sum K]` and int32 actions `[T, n, heads]`
    (actor_critic_policy.py:303-324 fused in).  Returns (g_logits, g_value, out, out_f32, logp, entropy).

    `logits` and `v_pred` are torch.float32 or torch.bfloat16, the same for both (a bfloat16 policy under
    torch.autocast passes its outputs as they are); g_logits and g_value come back in that dtype, logp / entropy and the
    statistics are float32.  bfloat16 inputs are widened exactly and the arithmetic is float32; each gradient is rounded
    to bfloat16 once (nearest even).
    `available` (SMAC's available_action, the logits' shape): where it is 0 the logit is replaced by -1e10 before the
    Categorical (actor_critic_policy.py:135-136) and its gradient is 0.  torch.uint8 and torch.bool are read in place; a
    floating mask costs one extra pass (`available != 0`).  At most 159 logits per transition with a mask, 199 without.
    `defer` (needs an explicit `workspace` slot): out / out_f32 are None and loss_finalize folds the slot later."""
    if available is not None:
        available = _availability(available, logits)
    dtype = logits.dtype if isinstance(logits, torch.Tensor) else torch.float32
    if dtype not in (torch.float32, torch.bfloat16):
        raise ValueError(f"logits: expected dtype torch.float32 or torch.bfloat16, got {dtype}")
    if isinstance(v_pred, torch.Tensor) and v_pred.dtype != dtype:
        raise ValueError(f"v_pred has dtype {v_pred.dtype} but logits have {dtype}; both must have the same dtype, cast "
                         f"one of them")
    _check(logits, dtype, "logits")
    _check(action, torch.int32, "action")
    _check(v_pred, dtype, "v_pred")
    heads = len(head_sizes)
    if not 1 <= heads <= SRL_MAX_HEADS:
        raise ValueError(f"between 1 and {SRL_MAX_HEADS} action heads are supported, got {heads}")
    SK = int(sum(head_sizes))
    if logits.shape[-1] != SK or action.shape[-1] != heads:
        raise ValueError(f"logits last dim {logits.shape[-1]} / action last dim {action.shape[-1]} do not match "
                         f"head sizes {list(head_sizes)}")
    T = logits.shape[0]
    n = logits[0].numel() // SK
    if _rows_lanes(v_pred) != (T, n) or action.numel() != T * n * heads:
        raise ValueError("logits, action and v_pred disagree on [T, n]")
    ld_smp = _sample_side(old_logp, old_value, ret, adv, on_reset_next, lane_idx, T, n, hyper.clip_value)
    _check(norm_stats, torch.float64, "norm_stats")
    local_stats = norm_stats if local_stats is None else _check(local_stats, torch.float64, "local_stats")
    dev = logits.device
    g_logits = torch.empty_like(logits)
    g_value = torch.empty_like(v_pred)
    logp = torch.empty_like(v_pred, dtype=torch.float32) if want_logp_entropy else None
    ent = torch.empty_like(v_pred, dtype=torch.float32) if want_logp_entropy else None
    if defer:
        if workspace is None:
            raise ValueError("deferred finalisation needs an explicit workspace slot")
        out = out_f32 = None
    else:
        out = torch.empty(SRL_LOSS_OUT_LEN, dtype=torch.float64, device=dev)
        out_f32 = torch.empty(4, dtype=torch.float32, device=dev)
    ws = loss_workspace(dev) if workspace is None else _check(workspace, torch.uint8, "workspace")
    hc = hyper.to_c()
    hs = (ctypes.c_int32 * heads)(*[int(k) for k in head_sizes])
    tail = (hs, heads, _ptr(v_pred), _ptr(old_logp), _ptr(old_value), _ptr(ret), _ptr(adv), _ptr(on_reset_next), ld_smp,
            _ptr(lane_idx), T, n, _ptr(norm_stats), _ptr(local_stats), _ptr(popart_mean_std), ctypes.byref(hc),
            _ptr(g_logits), _ptr(g_value), _ptr(logp), _ptr(ent), _ptr(out), _ptr(out_f32), _ptr(ws), ws.numel(), _stream())
    suffix = "_bf16" if dtype == torch.bfloat16 else ""
    if available is None:
        _lib.call("srl_ppo_loss_from_logits" + suffix, _ptr(logits), _ptr(action), *tail)
    else:
        _lib.call("srl_ppo_loss_from_logits_masked" + suffix, _ptr(logits), _ptr(available), _ptr(action), *tail)
    return g_logits, g_value, out, out_f32, logp, ent


GAUSSIAN_MAX_D = 64
_gaussian_workspaces = {}


def gaussian_loss_workspace_bytes(T: int, n: int, D: int, log_std_shared: bool) -> int:
    return int(_lib.load_library().srl_ppo_loss_gaussian_workspace_bytes(int(T), int(n), int(D), int(bool(log_std_shared))))


def new_gaussian_loss_workspace(device, T: int = 1, n: int = 1, D: int = GAUSSIAN_MAX_D,
                                log_std_shared: bool = True) -> torch.Tensor:
    """Zero-initialised scratch for ppo_loss_from_gaussian (uint8); the default size serves every shape.  Its first
    bytes are a loss slot, so a deferred launch is folded by loss_finalize(ws.view(1, -1), out)."""
    return torch.zeros(gaussian_loss_workspace_bytes(T, n, D, log_std_shared), dtype=torch.uint8, device=device)


def gaussian_loss_workspace(device) -> torch.Tensor:
    """Default scratch of ppo_loss_from_gaussian: one buffer per (device, stream)."""
    key = (torch.device(device).index, _stream())
    ws = _gaussian_workspaces.get(key)
    if ws is None:
        ws = _gaussian_workspaces[key] = new_gaussian_loss_workspace(device)
    return ws


def ppo_loss_from_gaussian(mean, log_std, action, v_pred, old_logp, old_value, ret, adv, on_reset_next, norm_stats,
                           hyper: LossHyper, local_stats=None, popart_mean_std=None, lane_idx=None,
                           want_logp_entropy: bool = False, workspace=None, defer: bool = False):
    """Loss starting from a diagonal-Gaussian actor head: `mean` and float32 `action` `[T, n, D]`, `log_std` either
    `[T, n, D]` (one per transition) or `[D]` (one parameter shared by every transition), D <= 64.  The head's log-prob
    and entropy are torch.distributions.Normal(mean, log_std.exp()).log_prob(action).sum(-1) / .entropy().sum(-1); the
    loss is ppo_loss_fwd_bwd's.  Returns (g_mean, g_log_std, g_value, out, out_f32, logp, entropy): g_log_std has
    log_std's shape (a shared log_std gets the sum over the minibatch); logp / entropy `[T, n]` only with
    want_logp_entropy.  `defer` (needs an explicit `workspace`): out / out_f32 are None and loss_finalize folds the
    slot later; the gradients are complete either way.

    `mean`, `v_pred` and a per-transition `log_std` are torch.float32 or torch.bfloat16, the same for all three (a Gaussian
    policy under torch.autocast passes its bfloat16 outputs as they are); their gradients come back in that dtype, logp /
    entropy and the statistics are float32.  bfloat16 inputs are widened exactly and the arithmetic is the float32
    entry's; each bfloat16 gradient is the float32 one rounded once (nearest even).  A shared `[D]` log_std is float32
    (an nn.Parameter, which autocast leaves alone) or bfloat16 (a module cast with .bfloat16()) with either mean dtype:
    it is widened (D elements), its gradient is summed in float64 as always, and comes back float32 or rounded to
    bfloat16 once, in log_std's dtype.  `action` is float32 always: the actions the actors sampled, on which old_logp
    was computed."""
    dtype = mean.dtype if isinstance(mean, torch.Tensor) else torch.float32
    if dtype not in (torch.float32, torch.bfloat16):
        raise ValueError(f"mean: expected dtype torch.float32 or torch.bfloat16, got {dtype}")
    if isinstance(v_pred, torch.Tensor) and v_pred.dtype != dtype:
        raise ValueError(f"v_pred has dtype {v_pred.dtype} but mean has {dtype}; both must have the same dtype, cast "
                         f"one of them")
    if isinstance(log_std, torch.Tensor):
        if log_std.dim() > 1 and log_std.dtype != dtype:
            raise ValueError(f"log_std has dtype {log_std.dtype} but mean has {dtype}; a per-transition log_std must have "
                             f"mean's dtype, cast one of them")
        if log_std.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f"log_std: expected dtype torch.float32 or torch.bfloat16, got {log_std.dtype}")
    if isinstance(action, torch.Tensor) and action.dtype != torch.float32:
        raise ValueError(f"action: expected dtype torch.float32, got {action.dtype}; pass the float32 actions the actors "
                         f"sampled (old_logp was computed on them, and a rounded action would bias every ratio)")
    _check(v_pred, dtype, "v_pred")
    T, n = _rows_lanes(v_pred)
    _check(mean, dtype, "mean")
    _check(action, torch.float32, "action")
    D = mean.shape[-1] if mean.dim() >= 2 else 0
    if mean.dim() < 2 or mean.shape[0] != T or mean.numel() != T * n * D:
        raise ValueError(f"mean: expected [T, n, D] with [T, n] = [{T}, {n}] (v_pred), got shape {tuple(mean.shape)}")
    if not 1 <= D <= GAUSSIAN_MAX_D:
        raise ValueError(f"mean: D = {D} action dimensions, supported are 1 .. {GAUSSIAN_MAX_D}")
    if tuple(action.shape) != tuple(mean.shape):
        raise ValueError(f"action: shape {tuple(action.shape)} does not match mean {tuple(mean.shape)}")
    if not isinstance(log_std, torch.Tensor):
        raise ValueError("log_std: expected a CUDA tensor")
    if tuple(log_std.shape) == (D,):
        shared = True
    elif tuple(log_std.shape) == tuple(mean.shape):
        shared = False
        if 0 in log_std.stride():
            raise ValueError("log_std: a stride-0 expand of a [D] parameter; pass the [D] tensor itself (a shared log_std "
                             "gets its gradient summed over the minibatch in the kernel)")
    else:
        raise ValueError(f"log_std: expected [D] = [{D}] (shared) or mean's shape {tuple(mean.shape)} (per transition), "
                         f"got {tuple(log_std.shape)}")
    _check(log_std, log_std.dtype, "log_std")
    # a shared bfloat16 [D] log_std: the kernel reads float32 [D] for both policy dtypes
    ls_dtype = log_std.dtype
    if shared and ls_dtype == torch.bfloat16:
        log_std = log_std.float()
    ld_smp = _sample_side(old_logp, old_value, ret, adv, on_reset_next, lane_idx, T, n, hyper.clip_value)
    _check(norm_stats, torch.float64, "norm_stats")
    local_stats = norm_stats if local_stats is None else _check(local_stats, torch.float64, "local_stats")
    if popart_mean_std is not None:
        _check(popart_mean_std, torch.float64, "popart_mean_std")
    dev = mean.device
    g_mean = torch.empty_like(mean)
    g_log_std = torch.empty_like(log_std)
    g_value = torch.empty_like(v_pred)
    logp = torch.empty_like(v_pred, dtype=torch.float32) if want_logp_entropy else None
    ent = torch.empty_like(v_pred, dtype=torch.float32) if want_logp_entropy else None
    if defer:
        if workspace is None:
            raise ValueError("deferred finalisation needs an explicit workspace")
        out = out_f32 = None
    else:
        out = torch.empty(SRL_LOSS_OUT_LEN, dtype=torch.float64, device=dev)
        out_f32 = torch.empty(4, dtype=torch.float32, device=dev)
    ws = gaussian_loss_workspace(dev) if workspace is None else _check(workspace, torch.uint8, "workspace")
    hc = hyper.to_c()
    suffix = "_bf16" if dtype == torch.bfloat16 else ""
    _lib.call("srl_ppo_loss_from_gaussian" + suffix, _ptr(mean), _ptr(log_std), int(shared), _ptr(action), D,
              _ptr(v_pred), _ptr(old_logp), _ptr(old_value), _ptr(ret), _ptr(adv), _ptr(on_reset_next), ld_smp,
              _ptr(lane_idx), T, n, _ptr(norm_stats), _ptr(local_stats), _ptr(popart_mean_std), ctypes.byref(hc),
              _ptr(g_mean), _ptr(g_log_std), _ptr(g_value), _ptr(logp), _ptr(ent), _ptr(out), _ptr(out_f32), _ptr(ws),
              ws.numel(), _stream())
    if g_log_std.dtype != ls_dtype:
        g_log_std = g_log_std.to(ls_dtype)  # what autograd's cast hands a bfloat16 parameter through .float()
    return g_mean, g_log_std, g_value, out, out_f32, logp, ent


class PPOGaussianLossFunction(torch.autograd.Function):
    """Autograd node for a continuous-action policy: forward returns the scalar loss (float32) and the float64 stats
    vector of ppo_loss_from_gaussian; backward hands the gradients the same launch produced to mean, log_std ([D]
    parameter or [T, n, D]) and v_pred.  A policy under torch.autocast("cuda", dtype=torch.bfloat16) passes its bfloat16
    mean, value and per-transition log_std as they are, with no casts, and a float32 (or, in a module cast with
    .bfloat16(), bfloat16) [D] log_std parameter; the action stays float32.  Each input gets a gradient of its own dtype:
    the launch's bfloat16 gradients (the float32 ones rounded once) for the bfloat16 inputs, the float32 [D] gradient for
    a float32 parameter, rounded once for a bfloat16 one.

        loss, out = PPOGaussianLossFunction.apply(mean, log_std, action, v_pred, old_logp, old_value, ret, adv,
                                                  on_reset_next, norm_stats, local_stats, popart_mean_std, lane_idx, hyper)
        loss.backward()
    """

    @staticmethod
    def forward(ctx, mean, log_std, action, v_pred, old_logp, old_value, ret, adv, on_reset_next, norm_stats, local_stats,
                popart_mean_std, lane_idx, hyper):
        g_mean, g_ls, g_v, out, out_f32, _, _ = ppo_loss_from_gaussian(
            mean.detach(), log_std.detach(), action, v_pred.detach(), old_logp, old_value, ret, adv, on_reset_next,
            norm_stats, hyper, local_stats=local_stats, popart_mean_std=popart_mean_std, lane_idx=lane_idx)
        ctx.save_for_backward(g_mean, g_ls, g_v.view(v_pred.shape))
        ctx.mark_non_differentiable(out)
        return out_f32[0], out

    @staticmethod
    def backward(ctx, grad_loss, _grad_out):
        g_mean, g_ls, g_v = ctx.saved_tensors
        return (g_mean * grad_loss, g_ls * grad_loss, None, g_v * grad_loss) + (None,) * 10


class PPOCategoricalLossFunction(torch.autograd.Function):
    """Autograd node for a categorical policy (K4b): forward returns the scalar loss (float32) and the float64 stats
    vector of ppo_loss_from_logits; backward hands the gradients the same launch produced to the logits (exactly 0 where
    `available` is 0) and v_pred.  `available` is the availability mask or None.  A bfloat16 policy (torch.autocast(
    "cuda", dtype=torch.bfloat16)) passes its bfloat16 logits and value as they are, with no casts: the launch reads
    bfloat16, and backward hands the launch's bfloat16 gradients (the float32 ones rounded once) times the incoming
    gradient to the bfloat16 inputs.

        loss, out = PPOCategoricalLossFunction.apply(logits, available, action, head_sizes, v_pred, old_logp, old_value,
                                                     ret, adv, on_reset_next, norm_stats, local_stats, popart_mean_std,
                                                     lane_idx, hyper)
        loss.backward()
    """

    @staticmethod
    def forward(ctx, logits, available, action, head_sizes, v_pred, old_logp, old_value, ret, adv, on_reset_next,
                norm_stats, local_stats, popart_mean_std, lane_idx, hyper):
        g_logits, g_v, out, out_f32, _, _ = ppo_loss_from_logits(
            logits.detach(), action, head_sizes, v_pred.detach(), old_logp, old_value, ret, adv, on_reset_next, norm_stats,
            hyper, local_stats=local_stats, popart_mean_std=popart_mean_std, lane_idx=lane_idx, available=available)
        ctx.save_for_backward(g_logits, g_v)
        ctx.mark_non_differentiable(out)
        return out_f32[0], out

    @staticmethod
    def backward(ctx, grad_loss, _grad_out):
        g_logits, g_v = ctx.saved_tensors
        return (g_logits * grad_loss, None, None, None, g_v * grad_loss) + (None,) * 10


class PPOLossFunction(torch.autograd.Function):
    """Autograd node at the SampleAnalyzedResult boundary (mappo.py:21-33): forward returns the scalar
    loss (float32) and the float64 stats vector; the gradients were already produced by the same launch."""

    @staticmethod
    def forward(ctx, new_logp, v_pred, entropy, old_logp, old_value, ret, adv, on_reset_next, norm_stats, local_stats,
                popart_mean_std, lane_idx, hyper):
        shape = new_logp.shape
        g_lp, g_v, g_en, out, out_f32 = ppo_loss_fwd_bwd(new_logp.detach(), v_pred.detach(), entropy.detach(), old_logp,
                                                        old_value, ret, adv, on_reset_next, norm_stats, hyper,
                                                        local_stats=local_stats, popart_mean_std=popart_mean_std,
                                                        lane_idx=lane_idx)
        ctx.save_for_backward(g_lp.view(shape), g_v.view(shape), g_en.view(shape))
        ctx.mark_non_differentiable(out)
        return out_f32[0], out

    @staticmethod
    def backward(ctx, grad_loss, _grad_out):
        g_lp, g_v, g_en = ctx.saved_tensors
        return (g_lp * grad_loss, g_v * grad_loss, g_en * grad_loss) + (None,) * 10


# ------------------------------------------------------------------------------------------------
# K5 / K1
# ------------------------------------------------------------------------------------------------
def philox_perm(seed: int, epoch: int, n_env: int, group: int = 1, out: Optional[torch.Tensor] = None,
                device="cuda", n_epochs: Optional[int] = None) -> torch.Tensor:
    """Lane indices of a Philox-keyed permutation of the n_env environments: int32 [n_env * group], or
    [n_epochs, n_env * group] for epochs epoch .. epoch + n_epochs - 1 in one launch."""
    rows = 1 if n_epochs is None else int(n_epochs)
    if out is None:
        shape = (n_env * group,) if n_epochs is None else (rows, n_env * group)
        out = torch.empty(shape, dtype=torch.int32, device=device)
    _check(out, torch.int32, "out")
    if out.numel() < rows * n_env * group:
        raise ValueError(f"out has {out.numel()} entries, need {rows * n_env * group}")
    _lib.call("srl_philox_perm", int(seed) & 0xFFFFFFFFFFFFFFFF, int(epoch) & 0xFFFFFFFF, rows, int(n_env), int(group),
              _ptr(out), _stream())
    return out


def stack_samples(descs: Sequence[LeafDesc], idx: Optional[torch.Tensor], L: int, B: int) -> None:
    """Raw form of batch_gather for callers that build their own leaf descriptors (srl_b200.buffer: samples staged
    one after another, [slots, L, row], gathered into [L, B, row] = np.stack(axis=1))."""
    if idx is not None:
        _check(idx, torch.int32, "idx")
        if idx.numel() != B:
            raise ValueError(f"idx has {idx.numel()} entries, expected B = {B}")
    for i in range(0, len(descs), SRL_MAX_LEAVES):
        chunk = list(descs[i:i + SRL_MAX_LEAVES])
        arr = (LeafDesc * len(chunk))(*chunk)
        _lib.call("srl_batch_gather", arr, len(chunk), _ptr(idx), int(L), int(B), _stream())


def philox4x32_10(counter: torch.Tensor, key: torch.Tensor) -> torch.Tensor:
    """Raw Philox blocks for known-answer tests: counter int32-viewed uint32 [n, 4], key [n, 2]."""
    _check(counter, torch.int32, "counter")
    _check(key, torch.int32, "key")
    n = counter.shape[0]
    out = torch.empty_like(counter)
    _lib.call("srl_philox4x32_10", _ptr(counter), _ptr(key), n, _ptr(out), _stream())
    return out


def batch_gather(pairs: List[Tuple[torch.Tensor, torch.Tensor]], idx: Optional[torch.Tensor]) -> None:
    """For every (src `[L, slots, ...]`, dst `[L, B, ...]`) pair: dst[:, j] = src[:, idx[j]] (bit-exact).
    One call handles up to 32 leaves per launch group; longer lists are split."""
    if not pairs:
        return
    L, B = pairs[0][1].shape[0], pairs[0][1].shape[1]
    if idx is not None:
        _check(idx, torch.int32, "idx")
        if idx.numel() != B:
            raise ValueError(f"idx has {idx.numel()} entries but dst has {B} columns")
    descs = []
    for k, (src, dst) in enumerate(pairs):
        for name, t in (("src", src), ("dst", dst)):
            if not t.is_cuda or not t.is_contiguous():
                raise ValueError(f"leaf {k} {name}: expected a contiguous CUDA tensor")
        if src.dtype != dst.dtype or src.shape[0] != L or dst.shape[:2] != (L, B) or src.shape[2:] != dst.shape[2:]:
            raise ValueError(f"leaf {k}: src {tuple(src.shape)}/{src.dtype} and dst {tuple(dst.shape)}/{dst.dtype} "
                             f"are not a [L, slots, ...] -> [L, B, ...] pair")
        row_bytes = dst[0, 0].numel() * dst.element_size() if dst.dim() > 2 else dst.element_size()
        descs.append(LeafDesc(src.data_ptr(), dst.data_ptr(), row_bytes, src.shape[1], 0, 0))
    for i in range(0, len(descs), SRL_MAX_LEAVES):
        chunk = descs[i:i + SRL_MAX_LEAVES]
        arr = (LeafDesc * len(chunk))(*chunk)
        _lib.call("srl_batch_gather", arr, len(chunk), _ptr(idx), L, B, _stream())


_chunk_idx = {}


def _row_split(row_bytes: int, items: int) -> int:
    """Pieces a moved row is cut into so that a reshape of a few huge rows (an observation leaf: B x 28 KB per time
    step) still spreads over every SM: pieces of >= 16 KB, 16-byte granules kept, at most ~64 K items."""
    want = min(row_bytes // 16384, max(1, 65536 // max(items, 1)))
    for cand in range(int(want), 1, -1):
        if row_bytes % cand == 0 and (row_bytes // cand) % 16 == 0:
            return cand
    return 1


def _split_index(device, outer: int, outer_stride: int, split: int) -> torch.Tensor:
    """int32 [outer * split]: idx[o * split + k] = o * outer_stride + k (cached per shape and device)."""
    key = (torch.device(device).index, outer, outer_stride, split)
    idx = _chunk_idx.get(key)
    if idx is None:
        o = torch.arange(outer, dtype=torch.int32, device=device).view(-1, 1) * outer_stride
        idx = _chunk_idx[key] = (o + torch.arange(split, dtype=torch.int32, device=device).view(1, -1)).reshape(-1)
    return idx


def to_chunk(x: torch.Tensor, num_chunks: int) -> torch.Tensor:
    """modules.to_chunk (legacy/algorithm/modules/utils.py:164-180): `[T, B, *D]` -> `[T//C, B*C, *D]`, chunk c of the
    time axis becomes columns [c*B, (c+1)*B) -- one K1 launch (dst[t', c] = src row c*(T//C) + t'), bit-exact."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise ValueError("to_chunk: expected a CUDA tensor (srl_b200 has no CPU path)")
    T = x.shape[0]
    if T % num_chunks != 0:  # same error as the reference (utils.py:176-179)
        raise IndexError(f"The first dimension(usually the step/time) {T} must be a multiple of "
                         f"num_chunks {num_chunks}. This usually means the sample_steps(config:AgentSpec) "
                         f"is not dividable by chunk_len(config:Policy).")
    Tc = T // num_chunks
    B = x.shape[1]
    x = x if x.is_contiguous() else x.contiguous()
    out = torch.empty((Tc, B * num_chunks) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
    if x.numel() == 0:
        return out
    row_bytes = x[0].numel() * x.element_size()
    split = _row_split(row_bytes, T)
    piece = row_bytes // split
    # item (t', j = c*split + k): piece k of source row c*Tc + t' -> slot c*Tc*split + k, time stride = one row
    idx = _split_index(x.device, num_chunks, Tc * split, split)
    d = LeafDesc(x.data_ptr(), out.data_ptr(), piece, T * split, row_bytes, piece)
    _lib.call("srl_batch_gather", (LeafDesc * 1)(d), 1, _ptr(idx), Tc, num_chunks * split, _stream())
    return out


def gather_to_chunk(x: torch.Tensor, env_idx: torch.Tensor, num_chunks: int) -> torch.Tensor:
    """`to_chunk(x[:, env_idx], num_chunks)` in ONE K1 launch: the minibatch gather (K5) and the RNN-chunk reshape
    (modules.to_chunk, legacy/algorithm/modules/utils.py:164-180) fused -- `[T, B, *D]` and int32 `env_idx [n]` ->
    `[T//C, n*C, *D]` with chunk c of the time axis in columns [c*n, (c+1)*n); bit-exact.  What an RNN policy does to
    every leaf of a minibatch before its recurrent core (actor_critic_policy.py: `recursive_apply(sample, to_chunk)`): two
    full copies of the minibatch become one."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise ValueError("gather_to_chunk: expected a CUDA tensor (srl_b200 has no CPU path)")
    _check(env_idx, torch.int32, "env_idx")
    T, B = x.shape[0], x.shape[1]
    if T % num_chunks != 0:  # same error as the reference (utils.py:176-179)
        raise IndexError(f"The first dimension(usually the step/time) {T} must be a multiple of "
                         f"num_chunks {num_chunks}. This usually means the sample_steps(config:AgentSpec) "
                         f"is not dividable by chunk_len(config:Policy).")
    Tc, n = T // num_chunks, env_idx.numel()
    x = x if x.is_contiguous() else x.contiguous()
    out = torch.empty((Tc, n * num_chunks) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
    if x.numel() == 0 or n == 0:
        return out
    row_bytes = x[0, 0].numel() * x.element_size() if x.dim() > 2 else x.element_size()
    # destination item (t', c*n + j) = source item (row c*Tc + t', slot env_idx[j]): with a time stride of one source row
    # ([B] items) that is slot c*Tc*B + env_idx[j] of row t'
    base = torch.arange(num_chunks, dtype=torch.int32, device=x.device).view(-1, 1) * (Tc * B)
    idx = (base + env_idx.view(1, -1)).reshape(-1).contiguous()
    d = LeafDesc(x.data_ptr(), out.data_ptr(), row_bytes, T * B, B * row_bytes, row_bytes)
    _lib.call("srl_batch_gather", (LeafDesc * 1)(d), 1, _ptr(idx), Tc, num_chunks * n, _stream())
    return out


def rnn_chunk_prep(on_reset: torch.Tensor, env_idx: torch.Tensor, num_chunks: int, hx: Optional[torch.Tensor] = None):
    """What a recurrent policy needs from a minibatch's reset flags and hidden states, in ONE launch (srl_rnn_chunk_prep):

      reset_chunk uint8 `[T//C, C*n]`        == `to_chunk(on_reset[:, env_idx], C)`
      row_any     uint8 `[T//C]`             1 where any column of that chunk-row resets -- `reset_segments(row_any)` gives
                                             AutoResetRNN's segment boundaries (autoreset_rnn.py:46-47) from ONE small
                                             device-to-host read instead of `(masks[1:] == 0).any(dim=1).nonzero()`
      hx0         float32 `[layers, C*n, H]` == `to_chunk(hx[:, env_idx], C)[0].transpose(0, 1) * (1 - reset_chunk[0])`
                                             (actor_critic_policy.py:362-363 + the first segment's `hxs * masks[0]`), or None

    `on_reset` uint8 `[T, B]` or `[T, B, 1]`, `hx` float32 `[T, B, layers, H]`, `env_idx` int32 `[n]`.  Bit-exact."""
    _check(on_reset, torch.uint8, "on_reset")
    _check(env_idx, torch.int32, "env_idx")
    T, B = _rows_lanes(on_reset)
    if T % num_chunks != 0:  # same error as the reference (utils.py:176-179)
        raise IndexError(f"The first dimension(usually the step/time) {T} must be a multiple of "
                         f"num_chunks {num_chunks}. This usually means the sample_steps(config:AgentSpec) "
                         f"is not dividable by chunk_len(config:Policy).")
    n, Tc = env_idx.numel(), T // num_chunks
    dev = on_reset.device
    reset_chunk = torch.empty((Tc, num_chunks * n), dtype=torch.uint8, device=dev)
    row_any = torch.zeros((Tc,), dtype=torch.uint8, device=dev)
    hx0, layers, H = None, 0, 0
    if hx is not None:
        _check(hx, torch.float32, "hx")
        if hx.dim() != 4 or tuple(hx.shape[:2]) != (T, B):
            raise ValueError(f"hx: expected [T, B, layers, H] = [{T}, {B}, layers, H], got {tuple(hx.shape)}")
        layers, H = int(hx.shape[2]), int(hx.shape[3])
        hx0 = torch.empty((layers, num_chunks * n, H), dtype=torch.float32, device=dev)
    _lib.call("srl_rnn_chunk_prep", _ptr(on_reset), _ptr(hx), _ptr(env_idx), T, B, n, int(num_chunks), layers, H,
              _ptr(reset_chunk), _ptr(row_any), _ptr(hx0), _stream())
    return reset_chunk, row_any, hx0


def reset_segments(row_any: torch.Tensor) -> list:
    """AutoResetRNN's `has_zeros` (autoreset_rnn.py:46-47) from `rnn_chunk_prep`'s row_any: `[0] + (rows >= 1 in which some
    lane resets) + [T']` -- the RNN runs each segment [a, b) in one call and masks its hidden state at every boundary."""
    flags = row_any.cpu()
    return [0] + [int(t) + 1 for t in torch.nonzero(flags[1:]).view(-1)] + [int(flags.shape[0])]


def back_to_trajectory(x: torch.Tensor, num_chunks: int) -> torch.Tensor:
    """modules.back_to_trajectory (utils.py:183-195), the inverse of to_chunk: `[T//C, B*C, *D]` -> `[T, B, *D]`."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise ValueError("back_to_trajectory: expected a CUDA tensor (srl_b200 has no CPU path)")
    Tc, BC = x.shape[0], x.shape[1]
    if BC % num_chunks != 0:
        raise IndexError(f"The second dimension {BC} must be a multiple of num_chunks {num_chunks}.")
    B = BC // num_chunks
    x = x if x.is_contiguous() else x.contiguous()
    out = torch.empty((Tc * num_chunks, B) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
    if x.numel() == 0:
        return out
    blk = (x[0].numel() // num_chunks) * x.element_size()  # one [B, *D] block
    split = _row_split(blk, Tc * num_chunks)
    piece = blk // split
    # destination row c*Tc + t' is item (t = c, j = t'*split + k): piece k of source block t'*C + c
    idx = _split_index(x.device, Tc, num_chunks * split, split)
    d = LeafDesc(x.data_ptr(), out.data_ptr(), piece, Tc * num_chunks * split, blk, piece)
    _lib.call("srl_batch_gather", (LeafDesc * 1)(d), 1, _ptr(idx), num_chunks, Tc * split, _stream())
    return out
