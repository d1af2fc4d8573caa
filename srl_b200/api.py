"""Stand-alone mirror of the plugin contract the trainer hot path lives behind (SRL `api/trainer.py`).

Inside an SRL checkout, use SRL's own classes: `srl_b200.srl_plugin.register_into_srl()` registers
`MultiAgentPPOB200` with `api.trainer.register("mappo_b200", ...)` and the trainer then receives SRL's own
`SampleBatch`.  Outside (tests, bench, GPU box) these mirrors keep the same names, arguments and behaviour:

  SampleBatch          api/trainer.py:14-82      (a NamedArray with the fixed field set)
  TrainerStepResult    api/trainer.py:101-106
  Trainer              api/trainer.py:109-157
  PytorchTrainer       api/trainer.py:160-193    (policy property, distributed(), device selection)
  register / make      api/trainer.py:231-246
  TrajPostprocessor, register_traj_postprocessor / make_traj_postprocessor   api/trainer.py:84-99,249-262

and one record of this package's own, `PPOHeadAnalyzedResult`: what a policy that declares `ppo_head = True` returns from
`analyze(sample, target="ppo_head", ...)`.
"""
from __future__ import annotations

import dataclasses
from typing import Any, Dict, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist

from srl_b200.namedarray import NamedArray

_SAMPLE_FIELDS = ("obs", "on_reset", "done", "truncated", "action", "reward", "info", "info_mask", "policy_state",
                  "analyzed_result", "policy_name", "policy_version_steps", "send_timestamp", "buffer_recv_timestamp",
                  "actor_worker_post_timestamp", "actor_worker_flush_timestamp", "trainer_worker_recv_timestamp",
                  "trainer_worker_batch_timestamp")


class SampleBatch(NamedArray):
    """Same field set and defaults as api/trainer.py:14-82; unknown keyword arguments are ignored there too."""

    def __init__(self, obs=None, sampling_weight=None, **kwargs):
        fields = {k: kwargs.get(k) for k in _SAMPLE_FIELDS}
        fields["obs"] = obs
        super().__init__(**fields)
        self.register_metadata(sampling_weight=sampling_weight)


class AnalyzedResult(NamedArray):
    """PPO rollout by-products stored in the sample (actor_critic_policy.py:22-25 PPORolloutAnalyzedResult)."""

    def __init__(self, value=None, log_probs=None, adv=None, ret=None, **extra):
        super().__init__(value=value, log_probs=log_probs, adv=adv, ret=ret, **extra)


@dataclasses.dataclass
class PPOHeadAnalyzedResult:
    """The actor head and the value of a policy, for a trainer that computes log-probabilities and entropies itself.

    A policy opts in by declaring the class attribute `ppo_head = True`; `MultiAgentPPOB200` then calls
    `policy.analyze(sample, target="ppo_head", burn_in_steps=...)` instead of `target="ppo"` and trains through the fused
    head losses (K4b / K4c / K4d): the policy builds no torch.distributions object, and the trainer hands the gradients of the
    loss with respect to the fields below to autograd.  Return them as the network produced them (still attached to the
    graph).  Shapes lead with the analyzed rows and lanes `[T', B, (A,)]` of the sample, burn-in rows already dropped, as
    `target="ppo"` returns its tensors; float32 or bfloat16 (torch.autocast) on the policy's device.

    Exactly one head kind:
      categorical (actor_critic_policy.py:303-324): `logits [T', B, (A,) sum K]` -- what the policy would hand to
        `Categorical(logits=...)`, the heads side by side -- `head_sizes` (the K of each head, at most 8 heads, sum K <= 262144;
        rows wider than 199, or 159 with a mask, run the wide kernel K4b-wide) and optionally `available` (SMAC's available_action, the logits' shape, non-zero = available;
        an unavailable logit is treated as masked_fill(-1e10), actor_critic_policy.py:135-136).  `action [T', B, (A,)
        heads]` of any integer dtype or integer-valued floats (SRL stores `action.x` as float32); the trainer converts it
        to int32 once.
      diagonal Gaussian: `mean [T', B, (A,) D]`, `log_std` either one `[D]` parameter shared by every transition or the
        mean's shape, D <= 64; `action` the float32 actions the actors sampled, the mean's shape.
      Beta (bounded actions): `concentration1` (alpha) and `concentration0` (beta), both `[T', B, (A,) D]`, positive, in
        the dtype of `state_values`, D <= 64 -- torch.distributions.Beta(concentration1, concentration0); `action` the
        float32 samples in (0, 1) the actors drew, the concentrations' shape (the policy maps them to its action bounds).
    `state_values [T', B, (A,) 1]` in the head's dtype (a scalar critic; with PopArt, the normalised value).
    """
    state_values: Any
    action: Any
    logits: Any = None
    head_sizes: Optional[Sequence[int]] = None
    available: Any = None
    mean: Any = None
    log_std: Any = None
    concentration1: Any = None
    concentration0: Any = None


@dataclasses.dataclass
class TrainerStepResult:
    stats: Dict  # stats to be logged
    step: int  # current step count of the trainer
    agree_pushing: Optional[bool] = True
    priorities: Optional[np.ndarray] = None


class Trainer:

    @property
    def policy(self):
        raise NotImplementedError()

    def step(self, samples) -> TrainerStepResult:
        raise NotImplementedError()

    def distributed(self, **kwargs):
        raise NotImplementedError()

    def get_checkpoint(self, *args, **kwargs):
        raise NotImplementedError()

    def load_checkpoint(self, checkpoint, **kwargs):
        raise NotImplementedError()


class PytorchTrainer(Trainer):

    @property
    def policy(self):
        return self._policy

    def __init__(self, policy):
        if policy.device != "cpu":
            torch.cuda.set_device(policy.device)  # api/trainer.py:174-176
        self._policy = policy

    def distributed(self, rank, world_size, init_method, **kwargs):
        """api/trainer.py:179-189: nccl when the policy lives on a GPU, gloo otherwise, then wrap the policy."""
        on_gpu = dist.is_nccl_available() and torch.cuda.is_available() and self.policy.device != "cpu"
        dist.init_process_group(backend="nccl" if on_gpu else "gloo", init_method=init_method, rank=rank,
                                world_size=world_size)
        self.policy.distributed()


ALL_TRAINER_CLASSES: Dict[str, Any] = {}


def register(name: str, trainer_class) -> None:
    ALL_TRAINER_CLASSES[name] = trainer_class


def make(cfg, policy):
    """api/trainer.py:238-246 with the policy already built: `cfg` is a name or an object with .type_/.args."""
    type_ = cfg if isinstance(cfg, str) else cfg.type_
    args = {} if isinstance(cfg, str) else (cfg.args or {})
    if hasattr(policy, "train_mode"):
        policy.train_mode()
    return ALL_TRAINER_CLASSES[type_](policy=policy, **args)


class TrajPostprocessor:
    """Post-process trajectories in actor workers before sending to trainers (api/trainer.py:84-91)."""

    def process(self, memory):
        raise NotImplementedError()


class NullTrajPostprocessor(TrajPostprocessor):

    def process(self, memory):
        return memory


ALL_TRAJ_POSTPROCESSOR_CLASSES: Dict[str, Any] = {}


def register_traj_postprocessor(name, cls_) -> None:
    ALL_TRAJ_POSTPROCESSOR_CLASSES[name] = cls_


register_traj_postprocessor("null", NullTrajPostprocessor)


def make_traj_postprocessor(cfg):
    """api/trainer.py:255-262: `cfg` is a name or an object with .type_/.args."""
    type_ = cfg if isinstance(cfg, str) else cfg.type_
    args = {} if isinstance(cfg, str) else (cfg.args or {})
    return ALL_TRAJ_POSTPROCESSOR_CLASSES[type_](**args)
