"""Test doubles for the trainer boundary, in the spirit of SRL's api/testing (NullTrainer, RandomPolicy):
a tiny actor-critic policy with the surface `MultiAgentPPO` calls on a policy (SURVEY.md §8b), and mirrors of
RunningMeanStd / PopArtValueHead (legacy/algorithm/modules/utils.py:70-151, popart.py:8-59) with the same
attribute names, so the trainer's PopArt bridge is exercised without an SRL checkout; and a record family of its own
(NamedArray, SampleBatch, recursive_apply) standing in for SRL's."""
from __future__ import annotations

import dataclasses
import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


class NamedArray:
    """A record family of its own, standing in for SRL's base.namedarray.NamedArray where no SRL checkout is staged: keyword
    construction, keys(), item access by name or by index / slice over every leaf, attribute access and assignment -- what
    the trainer and an SRL policy use of it -- and
    nothing shared with srl_b200.namedarray (duck-typed like SRL's class, not a subclass of the mirror)."""

    def __init__(self, **fields):
        object.__setattr__(self, "_fields", dict(fields))

    def keys(self):
        return self._fields.keys()

    def __getitem__(self, key):
        """A field by name; any other key (an index, a slice) indexes every leaf and gives a record of the same type."""
        if isinstance(key, str):
            return self._fields[key]
        new = object.__new__(type(self))
        object.__setattr__(new, "_fields", {k: None if v is None else v[key] for k, v in self._fields.items()})
        return new

    def __getattr__(self, name):
        fields = object.__getattribute__(self, "_fields")
        if name in fields:
            return fields[name]
        raise AttributeError(name)

    def __setattr__(self, name, value):
        self._fields[name] = value


class SampleBatch(NamedArray):
    """api/trainer.py's SampleBatch in the stand-in family."""


def recursive_apply(x, fn):
    """base/namedarray.py's recursive_apply in the stand-in family: subclasses come back as plain NamedArray records."""
    if x is None:
        return None
    if isinstance(x, NamedArray):
        return NamedArray(**{k: recursive_apply(x[k], fn) for k in x.keys()})
    return fn(x)


@dataclasses.dataclass
class SampleAnalyzedResult:  # legacy/algorithm/ppo/mappo.py:21-33
    old_action_log_probs: torch.Tensor
    new_action_log_probs: torch.Tensor
    state_values: torch.Tensor
    entropy: Optional[torch.Tensor] = None


class RunningMeanStd(nn.Module):
    """float64 debiased EMA statistics held as parameters (they travel in the state_dict)."""

    def __init__(self, input_shape, beta=0.999, epsilon=1e-5):
        super().__init__()
        self.__beta, self.__eps, self.__input_shape = beta, epsilon, tuple(input_shape)
        self.__mean = nn.Parameter(torch.zeros(input_shape, dtype=torch.float64), requires_grad=False)
        self.__mean_sq = nn.Parameter(torch.zeros(input_shape, dtype=torch.float64), requires_grad=False)
        self.__debiasing_term = nn.Parameter(torch.zeros(1, dtype=torch.float64), requires_grad=False)

    @torch.no_grad()
    def update(self, x, mask=None):
        x = x.to(torch.float64)
        dims = tuple(range(x.dim() - len(self.__input_shape)))
        if mask is None:
            factor = torch.tensor(float(math.prod(x.shape[:len(dims)])), dtype=torch.float64, device=x.device)
        else:
            mask = mask.to(torch.float64)
            x = x * mask
            factor = mask.sum()
        s1, s2 = x.sum(dim=dims), x.square().sum(dim=dims)
        if torch.distributed.is_initialized():
            for t in (factor, s1, s2):
                torch.distributed.all_reduce(t)
        b = self.__beta
        self.__mean.data[:] = b * self.__mean.data + (s1 / factor) * (1.0 - b)
        self.__mean_sq.data[:] = b * self.__mean_sq.data + (s2 / factor) * (1.0 - b)
        self.__debiasing_term.data[:] = b * self.__debiasing_term.data + 1.0 - b

    @torch.no_grad()
    def mean_std(self):
        d = self.__debiasing_term.clamp(min=self.__eps)
        m = self.__mean / d
        return m, (self.__mean_sq / d - m**2).clamp(min=1e-2).sqrt()

    @torch.no_grad()
    def normalize(self, x):
        m, s = self.mean_std()
        return ((x.to(torch.float64) - m) / s).clip(-5, 5).float()

    @torch.no_grad()
    def denormalize(self, x):
        m, s = self.mean_std()
        return (x.to(torch.float64) * s + m).float()


class PopArtValueHead(nn.Module):

    def __init__(self, input_dim, critic_dim, beta=0.99999, epsilon=1e-5, burn_in_updates=float("inf")):
        super().__init__()
        self.__rms = RunningMeanStd((critic_dim,), beta=beta, epsilon=epsilon)
        self.__weight = nn.Parameter(torch.zeros(critic_dim, input_dim))
        self.__bias = nn.Parameter(torch.zeros(critic_dim))
        nn.init.kaiming_uniform_(self.__weight, a=math.sqrt(5))
        nn.init.uniform_(self.__bias, -1 / math.sqrt(input_dim), 1 / math.sqrt(input_dim))
        self.__burn_in_updates = burn_in_updates
        self.__update_cnt = 0

    def forward(self, feature):
        return F.linear(feature, self.__weight, self.__bias)

    @torch.no_grad()
    def update(self, x, mask):
        old_mean, old_std = self.__rms.mean_std()
        self.__rms.update(x, mask)
        new_mean, new_std = self.__rms.mean_std()
        self.__update_cnt += 1
        if self.__update_cnt > self.__burn_in_updates:
            self.__weight.data[:] = self.__weight * (old_std / new_std).unsqueeze(-1)
            self.__bias.data[:] = (old_std * self.__bias + old_mean - new_mean) / new_std

    def normalize(self, x):
        return self.__rms.normalize(x)

    def denormalize(self, x):
        return self.__rms.denormalize(x)


class _Net(nn.Module):

    def __init__(self, obs_dim, num_actions, hidden, popart, popart_beta, burn_in_updates, popart_head_cls=None):
        super().__init__()
        self.body = nn.Sequential(nn.Linear(obs_dim, hidden), nn.Tanh())
        self.actor = nn.Linear(hidden, num_actions)
        head = popart_head_cls or PopArtValueHead  # oracle/make_golden.py passes the reference's own class
        self.critic = (head(hidden, 1, beta=popart_beta, burn_in_updates=burn_in_updates) if popart else
                       nn.Linear(hidden, 1))

    def forward(self, x):
        h = self.body(x)
        return self.actor(h), self.critic(h)


class TinyActorCriticPolicy:
    """obs.vec [..., obs_dim] -> Categorical(num_actions) + scalar value.  Implements exactly what the PPO
    trainer touches: device, version, inc_version, parameters, analyze(target='ppo'), train_mode,
    get/load_checkpoint, distributed and the three PopArt hooks."""

    def __init__(self, obs_dim=6, num_actions=5, hidden=16, device="cuda:0", popart=False, popart_beta=0.99,
                 burn_in_updates=float("inf"), seed=0, denormalize_value_during_rollout=False, popart_head_cls=None):
        g = torch.random.get_rng_state()
        torch.manual_seed(seed)
        self._net = _Net(obs_dim, num_actions, hidden, popart, popart_beta, burn_in_updates, popart_head_cls).to(device)
        torch.random.set_rng_state(g)
        self.device = device
        self._version = -1
        self.denormalize_value_during_rollout = denormalize_value_during_rollout
        self._popart = popart

    @property
    def version(self):
        return self._version

    @property
    def net(self):
        return self._net

    def inc_version(self):
        self._version += 1

    def parameters(self):
        return self._net.parameters(recurse=True)

    def train_mode(self):
        self._net.train()

    def distributed(self):
        if torch.distributed.is_initialized():
            from torch.nn.parallel import DistributedDataParallel as DDP
            self._net = DDP(self._net)

    def get_checkpoint(self):
        return {"steps": self._version, "state_dict": {k.replace("module.", ""): v.cpu() for k, v in
                                                       self._net.state_dict().items()}}

    def load_checkpoint(self, checkpoint):
        self._version = checkpoint.get("steps", 0)
        target = self._net.module if hasattr(self._net, "module") else self._net
        target.load_state_dict(checkpoint["state_dict"])

    # PopArt hooks (actor_critic_policy.py:262-274)
    @property
    def popart_head(self):
        net = self._net.module if hasattr(self._net, "module") else self._net
        return net.critic if self._popart else None

    def normalize_value(self, x):
        return self.popart_head.normalize(x)

    def denormalize_value(self, x):
        return self.popart_head.denormalize(x)

    def update_popart(self, x, mask):
        return self.popart_head.update(x, mask)

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        assert target == "ppo"
        obs = sample.obs.vec[burn_in_steps:]
        logits, value = self._net(obs)
        dist = torch.distributions.Categorical(logits=logits)
        action = sample.action.x[burn_in_steps:, ..., 0].long()
        new_lp = dist.log_prob(action).unsqueeze(-1)
        return SampleAnalyzedResult(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                                    new_action_log_probs=new_lp, state_values=value,
                                    entropy=dist.entropy().unsqueeze(-1))
