"""`MultiAgentPPOB200` -- drop-in for SRL's `MultiAgentPPO` trainer (legacy/algorithm/ppo/mappo.py:50-331).

Same constructor keywords and defaults (mappo.py:68-116), same `step(sample) -> TrainerStepResult`
contract (api/trainer.py:101-136), same checkpoint dict (mappo.py:58-66), same stats keys (mappo.py:293-326),
same one-call prefetch delay (api/trainer.py:199-228) and the same host write-back of adv / ret into the
sample (mappo.py:254-257).  What changes is who does the work between `policy.analyze` and `loss.backward`:

  reference                                              here
  ---------------------------------------------------------------------------------------------------------
  per-leaf pageable H2D + .float() of EVERY leaf          one pinned H2D per leaf in its own dtype; float views only for
                                                         what the policy reads, of the gathered minibatch when minibatched
  gae_trace: python loop, 3 kernels per time step        K2, one launch, float64 scan bit-identical to it
  masked_normalization + 3 all-reduces per loss          statistics table from K2's per-lane sums, 1 all-reduce/step
  PopArt update: ~10 kernels + 3 all-reduces             K3, one thread, state stays on device
  _compute_loss + autograd: ~70 kernels, 5 masked_select K4, one launch: loss terms + the three gradients
  11 .item() syncs per epoch                             one D2H of the stats table per step
  (no minibatching)                                      Philox env permutation + gather (K5), `num_minibatches`

The policy network, its optimizer, gradient clipping and DDP stay PyTorch (cuBLAS / cuDNN / NCCL).
"""
from __future__ import annotations

from collections import defaultdict
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist
import torch.nn as nn

from srl_b200 import ops
from srl_b200.api import PPOHeadAnalyzedResult, PytorchTrainer, TrainerStepResult, register
from srl_b200.hotpath import HotPath
from srl_b200.namedarray import flatten, from_flattened, record_class, recursive_apply


def init_optimizer(parameters, name: str, config: Dict):
    """legacy/algorithm/modules/utils.py:268-286."""
    table = dict(adam=torch.optim.Adam, rmsprop=torch.optim.RMSprop, sgd=torch.optim.SGD, adamw=torch.optim.AdamW)
    assert name in table, f"Optimizer name {name} does not match any implemented optimizers ({list(table)})."
    return table[name](parameters, **config)


class _PopArtBridge:
    """Keeps the policy's PopArtValueHead (legacy/algorithm/modules/popart.py:8-59) and the device-resident
    statistics of the hot path in step: the head's float64 running statistics are nn.Parameters inside the
    policy's state_dict (utils.py:80-82), which is what policy workers load, so K3's result is written back
    into them after every update, and the head is rescaled exactly as popart.py:49-51 does."""

    def __init__(self, policy):
        head = getattr(policy, "popart_head", None)
        rms = getattr(head, "_PopArtValueHead__rms", None) if head is not None else None
        if rms is None:
            raise ValueError("popart=True needs a policy whose `popart_head` is a PopArtValueHead "
                             "(legacy/algorithm/modules/popart.py) or the test double tests/doubles.py::PopArtValueHead")
        self.head, self.rms = head, rms
        g = lambda obj, cls, name: getattr(obj, f"_{cls}__{name}")
        self.mean, self.mean_sq = g(rms, "RunningMeanStd", "mean"), g(rms, "RunningMeanStd", "mean_sq")
        self.debias = g(rms, "RunningMeanStd", "debiasing_term")
        self.beta, self.eps = float(g(rms, "RunningMeanStd", "beta")), float(g(rms, "RunningMeanStd", "eps"))
        if self.mean.numel() != 1:
            raise ValueError(f"only scalar critics (critic_dim == 1) are supported, got {tuple(self.mean.shape)}")
        self.weight, self.bias = g(head, "PopArtValueHead", "weight"), g(head, "PopArtValueHead", "bias")
        self.burn_in = g(head, "PopArtValueHead", "burn_in_updates")

    def pull(self, hp: HotPath) -> None:
        """policy -> hot path (start of a step; the statistics may have been loaded from a checkpoint)."""
        st = hp.popart_state
        st[0:1].copy_(self.mean.data.view(-1))
        st[1:2].copy_(self.mean_sq.data.view(-1))
        st[2:3].copy_(self.debias.data.view(-1))
        with torch.no_grad():  # utils.py:132-137 on device, no host round trip
            d = st[2].clamp(min=self.eps)
            mu = st[0] / d
            hp.popart_ms[0] = mu
            hp.popart_ms[1] = (st[1] / d - mu * mu).clamp(min=1e-2).sqrt()

    def push(self, hp: HotPath) -> None:
        """hot path -> policy after K3 (popart.py:42-51)."""
        st, ms = hp.popart_state, hp.popart_ms
        self.mean.data.view(-1).copy_(st[0:1])
        self.mean_sq.data.view(-1).copy_(st[1:2])
        self.debias.data.view(-1).copy_(st[2:3])
        cnt = getattr(self.head, "_PopArtValueHead__update_cnt") + 1
        setattr(self.head, "_PopArtValueHead__update_cnt", cnt)
        if cnt > self.burn_in:
            with torch.no_grad():
                new_mu, new_sd, old_mu, old_sd = ms[0], ms[1], ms[2], ms[3]
                self.weight.data.mul_((old_sd / new_sd).to(self.weight.dtype))
                self.bias.data.copy_(((old_sd * self.bias.data.double() + old_mu - new_mu) / new_sd).to(self.bias.dtype))


class MultiAgentPPOB200(PytorchTrainer):
    """Multi-agent PPO with the sample-batch hot path on hand-written sm_100a kernels."""

    def get_checkpoint(self):  # mappo.py:58-61
        checkpoint = self.policy.get_checkpoint()
        checkpoint.update({"optimizer_state_dict": self.optimizer.state_dict()})
        return checkpoint

    def load_checkpoint(self, checkpoint, **kwargs):  # mappo.py:63-66
        if "optimizer_state_dict" in checkpoint.keys():
            self.optimizer.load_state_dict(checkpoint["optimizer_state_dict"])
        self.policy.load_checkpoint(checkpoint)

    def __init__(self, policy, **kwargs):
        super().__init__(policy)
        if policy.device == "cpu" or not torch.cuda.is_available():
            raise RuntimeError("MultiAgentPPOB200 needs a CUDA policy device: srl_b200 has no CPU path "
                               "(use SRL's own 'mappo' trainer on CPU)")
        ops._lib.load_library()  # fail at construction, not mid-training, if the CUDA library is missing
        # ---- mappo.py:71-112, same names and defaults ---------------------------------------------------
        self.discount_rate = kwargs.get("discount_rate", 0.99)
        self.gae_lambda = kwargs.get("gae_lambda", 0.97)
        self.eps_clip = kwargs.get("eps_clip", 0.2)
        self.clip_value = kwargs.get("clip_value", False)
        self.dual_clip = kwargs.get("dual_clip", True)
        self.c_clip = kwargs.get("c_clip", 3)
        self.burn_in_steps = kwargs.get("burn_in_steps", 0)
        self.vtrace = kwargs.get("vtrace", False)
        self.recompute_adv_on_reuse = kwargs.get("recompute_adv_on_reuse", True)
        self.recompute_adv_among_epochs = kwargs.get("recompute_adv_among_epochs", False)
        self.normalize_old_value = kwargs.get("normalize_old_value", False)
        if self.clip_value and self.normalize_old_value != getattr(policy, "denormalize_value_during_rollout", False):
            raise ValueError(
                "Trainer `normalize_old_value` and policy `denormalize_value_during_rollout` should be consistent!")
        self.value_eps_clip = kwargs.get("value_eps_clip", self.eps_clip)
        self.value_loss_weight = kwargs.get("value_loss_weight", 0.5)
        self.entropy_bonus_weight = kwargs.get("entropy_bonus_weight", 0.01)
        self.entropy_decay_per_steps = kwargs.get("entropy_decay_per_steps", None)
        self.entropy_bonus_decay = kwargs.get("entropy_bonus_decay", 0.99)
        self.max_grad_norm = kwargs.get("max_grad_norm")
        self.popart = kwargs.get("popart", False)
        self.bootstrap_steps = kwargs.get("bootstrap_steps", 1)
        self.ppo_epochs = kwargs.get("ppo_epochs", 1)
        self.optimizer = init_optimizer(self.policy.parameters(), kwargs.get("optimizer", "adam"),
                                        kwargs.get("optimizer_config", {}))
        self.value_loss = kwargs.get("value_loss", "mse")
        self.value_loss_config = kwargs.get("value_loss_config", {})
        self._hyper().to_c()  # validates value_loss / value_loss_config like utils.py:241-265
        # ---- new capabilities (absent from the reference, SURVEY.md F2) ----------------------------------
        self.num_minibatches = int(kwargs.get("num_minibatches", 1))
        self.shuffle_seed = int(kwargs.get("shuffle_seed", 0))
        self.shuffle_block = int(kwargs.get("shuffle_block", 1))  # environments per shuffled block
        self.prefetch = bool(kwargs.get("prefetch", True))  # one-call delay of api/trainer.py:219-228
        self.copy_threads = int(kwargs.get("copy_threads", 8))  # host threads filling the pinned staging blocks
        if self.vtrace and (self.num_minibatches > 1 or self.recompute_adv_among_epochs):
            raise ValueError("vtrace supports num_minibatches == 1 without recompute_adv_among_epochs")
        # A policy that declares `ppo_head = True` hands over its actor head (api.PPOHeadAnalyzedResult) and trains through
        # the fused head losses K4b / K4c; every other policy takes the `target="ppo"` path.
        self.ppo_head = getattr(policy, "ppo_head", False) is True
        if self.ppo_head and self.vtrace:
            raise ValueError("vtrace=True needs the policy's new log-probabilities before the GAE scan, and a `ppo_head` "
                             "policy returns its actor head instead; train V-trace with target='ppo' (no ppo_head)")
        self.frames = 0
        self._hp: Optional[HotPath] = None
        self._pending = None  # (host sample, device float sample) staged by the previous step() call
        self._copy_stream = torch.cuda.Stream()
        self._mirror_stream = torch.cuda.Stream()
        self._stage_done = torch.cuda.Event()
        self._stage_pin: Dict[str, torch.Tensor] = {}
        self._mirror, self._mirror_key = None, None
        self.h2d_bytes = 0  # bytes this trainer has sent over PCIe (tests: == the host sample's bytes, A2)
        self._popart = _PopArtBridge(policy) if self.popart else None

    # ----------------------------------------------------------------------------------------------------
    def _hyper(self) -> ops.LossHyper:
        return ops.LossHyper(eps_clip=self.eps_clip, clip_value=self.clip_value, value_eps_clip=self.value_eps_clip,
                             dual_clip=self.dual_clip, c_clip=self.c_clip, value_loss=self.value_loss,
                             value_loss_config=dict(self.value_loss_config), value_loss_weight=self.value_loss_weight,
                             entropy_bonus_weight=self.entropy_bonus_weight, normalize_old_value=self.normalize_old_value)

    def _hot_path(self, L: int, B: int, A: int) -> HotPath:
        hp = self._hp
        if hp is None or (hp.L, hp.B, hp.A) != (L, B, A):
            pg = dist.group.WORLD if dist.is_initialized() and dist.get_world_size() > 1 else None
            hp = HotPath(L, B, A, gamma=self.discount_rate, lmbda=self.gae_lambda, hyper=self._hyper(),
                         bootstrap_steps=self.bootstrap_steps, burn_in_steps=self.burn_in_steps, epochs=self.ppo_epochs,
                         minibatches=self.num_minibatches, seed=self.shuffle_seed, popart=self.popart,
                         popart_beta=self._popart.beta if self._popart else 0.99999,
                         popart_eps=self._popart.eps if self._popart else 1e-5, device=torch.device(self.policy.device),
                         process_group=pg, shuffle_block=self.shuffle_block)
            self._hp = hp
        hp.hyper = self._hyper()  # entropy_bonus_weight decays over time (mappo.py:310-311)
        return hp

    # ----------------------------------------------------------------------------------------------------
    # A2: staging.  The reference's prefetcher copies every leaf from pageable memory and inflates ALL of them to float32
    # on the device (api/trainer.py:211-217: 4 x the bytes of a uint8 frame stack, a 4-byte float per 1-byte flag).  Here a
    # leaf crosses PCIe ONCE, in its own dtype, from a pinned staging block (filled by the library's multi-threaded host
    # copy), and stays in that dtype in HBM; `policy.analyze` receives float32 views that are made where they are used --
    # of the gathered minibatch only, when the step is minibatched.
    # ----------------------------------------------------------------------------------------------------
    def _pinned(self, name: str, x: np.ndarray) -> torch.Tensor:
        t = self._stage_pin.get(name)
        if t is None or t.numel() != x.size or t.dtype != torch.from_numpy(x.reshape(-1)[:1]).dtype:
            t = torch.empty(x.size, dtype=torch.from_numpy(x.reshape(-1)[:1]).dtype).pin_memory()
            self._stage_pin[name] = t
        return t

    def _to_device(self, name: str, x):
        if isinstance(x, torch.Tensor):  # a DeviceSlabBuffer batch: already in HBM, in the sample's own dtype
            return x if x.is_cuda else x.cuda(non_blocking=True)
        x = np.ascontiguousarray(x)
        if x.dtype.kind not in "fiub":
            raise TypeError(f"leaf {name}: dtype {x.dtype} cannot live on the device (SRL's trainer worker clears "
                            f"policy_name before step(), trainer_worker.py:169)")
        if x.size == 0:
            return torch.from_numpy(x).cuda()
        pin = self._pinned(name, x)
        if x.nbytes >= (1 << 20) and self.copy_threads > 1:
            ops._lib.call("srl_host_copy", pin.data_ptr(), x.ctypes.data, x.nbytes, self.copy_threads)
        else:
            pin.numpy()[:] = x.reshape(-1)
        self.h2d_bytes += x.nbytes
        return pin.cuda(non_blocking=True).view(x.shape)

    def _stage(self, sample):
        """Host -> device copy of the whole sample on the side stream, every leaf in its own dtype (the reference:
        api/trainer.py:211-217).  Returns (host sample, device sample of the same record family)."""
        self._stage_done.synchronize()  # the pinned staging blocks are free again (the copy ahead of this one has landed)
        self._copy_stream.wait_stream(torch.cuda.current_stream())
        names, leaves = zip(*flatten(sample))
        with torch.cuda.stream(self._copy_stream):
            dev = [None if v is None else self._to_device(k, v) for k, v in zip(names, leaves)]
            self._stage_done.record(self._copy_stream)
        return sample, from_flattened(list(zip(names, dev)), record_class(sample))

    @staticmethod
    def _float_view(rec):
        """What `policy.analyze` is handed: float32 leaves, as the reference's prefetcher produces (api/trainer.py:217)."""
        return recursive_apply(rec, lambda x: x if x.dtype == torch.float32 else x.float())

    @staticmethod
    def _lanes(x) -> tuple:
        """[L, B, 1] -> (B, 1); [L, B, A, 1] -> (B, A)."""
        if x.ndim == 3:
            return x.shape[1], 1
        if x.ndim == 4:
            return x.shape[1], x.shape[2]
        raise ValueError(f"expected [L, B, 1] or [L, B, A, 1] scalar leaves, got shape {tuple(x.shape)}")

    # ----------------------------------------------------------------------------------------------------
    def step(self, sample) -> TrainerStepResult:
        on_device = isinstance(sample.on_reset, torch.Tensor)  # a DeviceSlabBuffer batch: nothing crosses PCIe
        if sample.truncated is None:  # mappo.py:222-223
            sample.truncated = torch.zeros_like(sample.done) if on_device else np.zeros_like(sample.done)
        if self.recompute_adv_on_reuse:  # mappo.py:224-225
            sample.analyzed_result.adv = sample.analyzed_result.ret = None

        if self.prefetch:  # api/trainer.py:219-228: wait for the copy in flight, take it, start the next one
            torch.cuda.current_stream().wait_stream(self._copy_stream)
            staged, self._pending = self._pending, self._stage(sample)
            if staged is None:
                return TrainerStepResult({}, 0)  # api/trainer.py:220-223: the first call only primes the pipeline
        else:
            staged = self._stage(sample)
            torch.cuda.current_stream().wait_stream(self._copy_stream)
        sample, tensor_sample = staged
        on_device = isinstance(sample.on_reset, torch.Tensor)

        L = tensor_sample.on_reset.shape[0]
        B, A = self._lanes(sample.on_reset)
        hp = self._hot_path(L, B, A)
        ar, tar = sample.analyzed_result, tensor_sample.analyzed_result
        # the six scalar leaves go from the staged device sample into the hot path's own [L, N] buffers: a device copy
        # (flags that arrived as floats are narrowed to uint8 there), no second trip over PCIe
        hp.load_sample(dict(reward=tensor_sample.reward, value=tar.value, old_logp=tar.log_probs, done=tensor_sample.done,
                            truncated=tensor_sample.truncated, on_reset=tensor_sample.on_reset))
        if self._popart:
            self._popart.pull(hp)
        # decided from what was STAGED (mappo.py:249): with the prefetch delay the host sample may have gained its
        # adv / ret only after its device copy was made (a buffer entry served twice in a row), and then they are recomputed
        cached_adv = tar.adv is not None
        if cached_adv:  # re-served sample with cached advantages (recompute_adv_on_reuse=False)
            hp.adv.copy_(tar.adv.reshape(L, hp.N))
            hp.ret.copy_(tar.ret.reshape(L, hp.N))

        lo, hi, T = hp.row_lo, hp.row_hi, hp.T
        lead = tuple(sample.on_reset.shape[1:])  # (B, 1) or (B, A, 1)
        whole = self._float_view(tensor_sample) if self.num_minibatches == 1 else None
        have_adv = False
        mirrored = False
        grad_norm_sum = torch.zeros((), device=hp.device)
        for e in range(self.ppo_epochs):
            for j in range(self.num_minibatches):
                idx = hp.minibatch_lanes(e, j) if have_adv else None
                if self.num_minibatches > 1 and not have_adv:
                    # the first analyze of the step needs the permutation before the advantages exist
                    hp.permute()
                    idx = hp.minibatch_lanes(e, j)
                mb = whole if idx is None else self._float_view(self._gather_minibatch(tensor_sample, idx, hp))
                # mappo.py:243-246
                tail_len = 1 if (self.vtrace and not cached_adv and not have_adv) else self.bootstrap_steps
                res = self.policy.analyze(mb[:L - tail_len], target="ppo_head" if self.ppo_head else "ppo",
                                          burn_in_steps=self.burn_in_steps)
                if not have_adv:  # mappo.py:249-257
                    vt = None
                    if self.vtrace and not cached_adv:
                        vt = res.new_action_log_probs.detach().reshape(-1, hp.N).contiguous()
                    hp.advantages(cached=cached_adv, vtrace_new_logp=vt, permute=False)
                    have_adv = True
                    if not on_device and not self.recompute_adv_among_epochs and not mirrored:
                        self._mirror_adv_ret(hp)  # D2H of adv / ret under the epochs' compute (mappo.py:254-257)
                        mirrored = True
                if self._popart and j == 0:  # once per epoch, before the loss (mappo.py:263-264)
                    hp.update_popart()
                    self._popart.push(hp)
                if self.ppo_head:
                    outs = self._head_loss(hp, e, j, res)
                else:
                    nl, vp, en = (x[:T].reshape(T, -1) for x in (res.new_action_log_probs, res.state_values, res.entropy))
                    g_lp, g_v, g_en, _, _ = hp.loss(e, j, nl.detach().contiguous(), vp.detach().contiguous(),
                                                    en.detach().contiguous())
                    outs = [(o, g) for o, g in ((nl, g_lp), (vp, g_v), (en, g_en)) if o.requires_grad]
                self.optimizer.zero_grad(set_to_none=True)  # mappo.py:273-274: loss.backward()
                torch.autograd.backward([o for o, _ in outs], [g for _, g in outs])
                if self.max_grad_norm is not None:  # mappo.py:280-284
                    gn = nn.utils.clip_grad_norm_(self.policy.parameters(), self.max_grad_norm)
                else:
                    gn = torch.sqrt(sum((p.grad.norm()**2 for p in self.policy.parameters() if p.grad is not None),
                                        torch.zeros((), device=hp.device)))
                self.optimizer.step()
                grad_norm_sum = grad_norm_sum + gn.detach()
            if self.recompute_adv_among_epochs and e + 1 < self.ppo_epochs:  # mappo.py:287-289
                have_adv, cached_adv = False, False
        hp.finalize()
        hp.step_count += 1

        # ---- ONE synchronisation for everything the step reports (mappo.py:254-257, 293-303): the loss / stats table,
        # the batch row and the gradient norm follow adv / ret into pinned mirrors, then the stream is waited for once
        n_loss = self.ppo_epochs * self.num_minibatches
        m = self._host_mirror(hp)
        m["out"].copy_(hp.out, non_blocking=True)
        m["whole"].copy_(hp.local_stats[0], non_blocking=True)
        m["gn"].copy_(grad_norm_sum.reshape(1).double(), non_blocking=True)
        self._xchg_check(hp)
        torch.cuda.current_stream().synchronize()
        self._mirror_stream.synchronize()
        if hp.peer is not None:
            hp.peer.raise_if_failed()
        out, whole_row = m["out"].numpy(), m["whole"].numpy()
        if self.recompute_adv_among_epochs:  # mappo.py:287-289 leaves the host copies cleared
            ar.adv = ar.ret = None
        elif on_device:  # the cached copies stay in HBM next to the batch
            ar.adv = hp.adv.reshape((L,) + lead).clone()
            ar.ret = hp.ret.reshape((L,) + lead).clone()
        else:  # mappo.py:254-257: the buffer may serve this sample again and reuse them
            ar.adv = m["adv"].numpy().reshape((L,) + lead).copy()
            ar.ret = m["ret"].numpy().reshape((L,) + lead).copy()
        train_stats = defaultdict(lambda: 0)
        names = dict(advantage=4, entropy=3, policy_loss=1, value_loss=2, clip_ratio=6, importance_weight=5, value_targets=7)
        if self.popart:
            names["denorm_value"] = 8
        for k, slot in names.items():
            v = float(out[:, slot].mean())
            train_stats[k] = -v if k == "entropy" else v  # entropy = -entropy_loss (mappo.py:207)
        valid_count = float(T * hp.N)
        train_stats["done"] = float(whole_row[5]) / valid_count  # unmasked means over the valid rows (mappo.py:210-211)
        train_stats["truncated"] = float(whole_row[6]) / valid_count
        train_stats["grad_norm"] = float(m["gn"][0]) / n_loss

        self.policy.inc_version()  # mappo.py:305-307
        if self.entropy_decay_per_steps and self.policy.version % self.entropy_decay_per_steps == 0:
            self.entropy_bonus_weight *= self.entropy_bonus_decay
        valid = slice(self.burn_in_steps, L - self.bootstrap_steps)
        self.frames += int(np.prod(sample.on_reset[valid].shape))
        info = {}
        if getattr(sample, "info_mask", None) is not None and sample.info is not None:  # mappo.py:317-324
            elapsed = float(sample.info_mask[valid].sum())
            if elapsed != 0:
                info = {k: float((v[valid] * sample.info_mask[valid]).sum() / elapsed) for k, v in flatten(sample.info)
                        if v is not None}
        stats = dict(frames=int(self.frames), **train_stats, **info)
        return TrainerStepResult(stats=stats, step=self.policy.version)

    # ----------------------------------------------------------------------------------------------------
    def _head_loss(self, hp: HotPath, e: int, j: int, res) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        """K4b / K4c for minibatch (e, j) on the head a `ppo_head` policy returned: [(output, d loss / d output)] for the
        outputs that require grad (the loss scalars follow at hp.finalize())."""
        h = _head_fields(res, hp.T, hp.n_mb)
        T, n = hp.T, hp.n_mb
        vp = h.state_values[:T].reshape(T, n)
        if h.logits is not None:
            lg = h.logits[:T].reshape(T, n, -1)
            act = h.action[:T].reshape(T, n, -1).to(torch.int32).contiguous()
            av = None if h.available is None else h.available[:T].reshape(T, n, -1).contiguous()
            g_lg, g_v = hp.loss_from_logits(e, j, lg.detach().contiguous(), act, [int(k) for k in h.head_sizes],
                                            vp.detach().contiguous(), av)
            pairs = ((lg, g_lg), (vp, g_v))
        else:
            mu = h.mean[:T].reshape(T, n, -1)
            ls = h.log_std if h.log_std.dim() == 1 else h.log_std[:T].reshape(T, n, -1)
            act = h.action[:T].reshape(T, n, -1).contiguous()
            g_mu, g_ls, g_v = hp.loss_from_gaussian(e, j, mu.detach().contiguous(), ls.detach().contiguous(), act,
                                                    vp.detach().contiguous())
            pairs = ((mu, g_mu), (ls, g_ls), (vp, g_v))
        return [(o, g) for o, g in pairs if o.requires_grad]

    def _host_mirror(self, hp: HotPath) -> Dict[str, torch.Tensor]:
        """Pinned host images of what a step reports, allocated once per batch shape."""
        key = (hp.L, hp.N, hp.epochs, hp.minibatches)
        if self._mirror_key != key:
            pin = lambda *shape, dtype=torch.float32: torch.empty(shape, dtype=dtype).pin_memory()
            self._mirror = dict(adv=pin(hp.L, hp.N), ret=pin(hp.L, hp.N), out=pin(*hp.out.shape, dtype=torch.float64),
                                whole=pin(hp.local_stats.shape[1], dtype=torch.float64), gn=pin(1, dtype=torch.float64))
            self._mirror_key = key
        return self._mirror

    def _mirror_adv_ret(self, hp: HotPath) -> None:
        """adv / ret -> pinned host mirrors on a side stream, right behind K2 (the reference's blocking `.cpu()` calls at
        mappo.py:254-257; here the copy runs under the epochs' compute and is waited for once, at the end of the step)."""
        m = self._host_mirror(hp)
        self._mirror_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._mirror_stream):
            m["adv"].copy_(hp.adv, non_blocking=True)
            m["ret"].copy_(hp.ret, non_blocking=True)

    def _xchg_check(self, hp: HotPath) -> None:
        """A peer that never arrived at the statistics exchange must fail the step, not feed it stale sums."""
        if hp.peer is not None:
            hp.peer.check_async()

    def _gather_minibatch(self, tensor_sample, idx: torch.Tensor, hp: HotPath):
        """K5: every leaf `[L, B, ...]` of the device sample -> `[L, n_env, ...]` for the environments of this
        minibatch, one C-ABI call for all leaves (bit-exact, in the leaves' own dtypes; numpy equivalent: x[:, env_idx])."""
        env_idx = idx.view(-1, hp.A)[:, 0].contiguous() // hp.A if hp.A > 1 else idx
        env_idx = env_idx.to(torch.int32)
        names, pairs = [], []
        for name, v in flatten(tensor_sample):
            if v is None:
                names.append((name, None))
                continue
            v = v.contiguous()
            dst = torch.empty((v.shape[0], env_idx.numel()) + tuple(v.shape[2:]), dtype=v.dtype, device=v.device)
            if v.numel() > 0:
                pairs.append((v, dst))
            names.append((name, dst))
        ops.batch_gather(pairs, env_idx)
        return from_flattened(names, record_class(tensor_sample))


_HEAD_FLOATS = (torch.float32, torch.bfloat16)


def _head_fields(res, T: int, n: int) -> PPOHeadAnalyzedResult:
    """Checks what analyze(target="ppo_head") returned against the contract of api.PPOHeadAnalyzedResult for T loss rows of
    n lanes; raises TypeError / ValueError naming the field."""
    if not isinstance(res, PPOHeadAnalyzedResult):
        raise TypeError(f"analyze(target='ppo_head') must return srl_b200.api.PPOHeadAnalyzedResult, got {type(res).__name__}")

    def tensor(name, required=True):
        x = getattr(res, name)
        if x is None and not required:
            return None
        if x is None:
            raise ValueError(f"PPOHeadAnalyzedResult.{name} is required")
        if not isinstance(x, torch.Tensor):
            raise TypeError(f"PPOHeadAnalyzedResult.{name}: expected a torch.Tensor, got {type(x).__name__}")
        return x

    sv, act = tensor("state_values"), tensor("action")
    if sv.dtype not in _HEAD_FLOATS:
        raise ValueError(f"PPOHeadAnalyzedResult.state_values: dtype {sv.dtype}, expected torch.float32 or torch.bfloat16")
    if sv.dim() < 2 or sv.shape[-1] != 1 or sv.shape[0] < T or sv[0].numel() != n:
        raise ValueError(f"PPOHeadAnalyzedResult.state_values: expected [T', B, (A,) 1] with T' >= {T} rows of {n} lanes, "
                         f"got shape {tuple(sv.shape)}")
    lead = tuple(sv.shape[:-1])
    if (res.logits is None) == (res.mean is None):
        raise ValueError("PPOHeadAnalyzedResult: set exactly one of `logits` (categorical head) and `mean` (Gaussian head)")
    if res.logits is not None:
        lg = tensor("logits")
        if lg.dtype != sv.dtype:
            raise ValueError(f"PPOHeadAnalyzedResult.logits: dtype {lg.dtype} differs from state_values' {sv.dtype}")
        if res.head_sizes is None:
            raise ValueError("PPOHeadAnalyzedResult.head_sizes is required with logits")
        hs = [int(k) for k in res.head_sizes]
        if tuple(lg.shape[:-1]) != lead or lg.shape[-1] != sum(hs):
            raise ValueError(f"PPOHeadAnalyzedResult.logits: expected {lead + (sum(hs),)} (state_values' rows and lanes, "
                             f"sum of head_sizes {hs}), got {tuple(lg.shape)}")
        if act.dtype == torch.bool or act.dtype.is_complex or tuple(act.shape) != lead + (len(hs),):
            raise ValueError(f"PPOHeadAnalyzedResult.action: expected integer-valued {lead + (len(hs),)}, got "
                             f"{act.dtype} {tuple(act.shape)}")
        av = tensor("available", required=False)
        if av is not None and tuple(av.shape) != tuple(lg.shape):
            raise ValueError(f"PPOHeadAnalyzedResult.available: shape {tuple(av.shape)} differs from logits' "
                             f"{tuple(lg.shape)}")
    else:
        mu, ls = tensor("mean"), tensor("log_std")
        if mu.dtype != sv.dtype:
            raise ValueError(f"PPOHeadAnalyzedResult.mean: dtype {mu.dtype} differs from state_values' {sv.dtype}")
        if mu.dim() != len(lead) + 1 or tuple(mu.shape[:-1]) != lead:
            raise ValueError(f"PPOHeadAnalyzedResult.mean: expected {lead + ('D',)}, got {tuple(mu.shape)}")
        D = mu.shape[-1]
        if tuple(ls.shape) != (D,) and tuple(ls.shape) != tuple(mu.shape):
            raise ValueError(f"PPOHeadAnalyzedResult.log_std: expected [{D}] or the mean's {tuple(mu.shape)}, got "
                             f"{tuple(ls.shape)}")
        if ls.dim() > 1 and ls.dtype != mu.dtype:
            raise ValueError(f"PPOHeadAnalyzedResult.log_std: dtype {ls.dtype} differs from mean's {mu.dtype}")
        if act.dtype != torch.float32 or tuple(act.shape) != tuple(mu.shape):
            raise ValueError(f"PPOHeadAnalyzedResult.action: expected float32 {tuple(mu.shape)}, got {act.dtype} "
                             f"{tuple(act.shape)}")
    return res


register("mappo_b200", MultiAgentPPOB200)
