"""Seeded synthetic sample batches for the trainer hot path (host side, numpy only).

Shapes, distributions and hyper-parameters follow SURVEY.md §8(d); the flag fields satisfy the
data invariants the reference asserts at legacy/algorithm/modules/gae.py:69-77:

    truncated * done == 0;  (truncated + done)[:-1] == on_reset[1:];  reward * on_reset[1:] == 0

Layout mirrors what `PriorityQueueBuffer.put` hands the trainer (base/buffer.py:118-126):
time-major leaves `[L, B, (A,) 1]`, float32 values, uint8 flags (distributed/system/actor_worker.py:278-281).
"""
from __future__ import annotations

import dataclasses
from typing import Dict, Optional, Tuple

import numpy as np


@dataclasses.dataclass(frozen=True)
class PathConfig:
    """One row of BASELINE.json `configs` (SURVEY.md §8d)."""
    name: str
    T: int  # rows entering the loss
    B: int  # environments
    A: int = 1  # agents per environment (lanes N = B * A)
    bootstrap_steps: int = 1
    burn_in_steps: int = 0
    epochs: int = 1
    minibatches: int = 1
    p_end: float = 0.002  # per-step episode end probability
    gamma: float = 0.99
    lmbda: float = 0.97
    eps_clip: float = 0.2
    clip_value: bool = False
    dual_clip: bool = True
    c_clip: float = 3.0
    value_loss: str = "mse"
    value_loss_delta: float = 1.0  # huber delta / smoothl1 beta
    value_loss_weight: float = 0.5
    entropy_bonus_weight: float = 0.01
    popart: bool = False
    num_actions: Tuple[int, ...] = (18,)
    dead_agent_frac: float = 0.0  # SMAC: new_logp = -inf where the agent is dead (smac_rnn.py:311-313)
    obs_shape: Tuple[int, ...] = ()
    obs_dtype: str = "uint8"

    @property
    def L(self) -> int:
        return self.T + self.burn_in_steps + self.bootstrap_steps

    @property
    def N(self) -> int:
        return self.B * self.A

    @property
    def transitions(self) -> int:
        return self.T * self.N


# legacy/experiments/atari.py:952-973 (cfg1/cfg2), smac.py:545-582,630 (cfg3),
# football.py:110-136 (cfg4), hns_reproduce.py:171-212 (cfg5)
_ATARI = dict(p_end=0.002, gamma=0.99, lmbda=0.97, eps_clip=0.2, clip_value=True, dual_clip=False,
              value_loss="huber", value_loss_delta=10.0, value_loss_weight=1.0, entropy_bonus_weight=0.01,
              num_actions=(18,), obs_shape=(4, 84, 84), obs_dtype="uint8")
CONFIGS: Dict[str, PathConfig] = {
    "cfg1_atari_cpu": PathConfig("cfg1_atari_cpu", T=80, B=32, **_ATARI),
    "cfg2_atari_large": PathConfig("cfg2_atari_large", T=128, B=4096, epochs=4, minibatches=8, **_ATARI),
    "cfg3_smac_27m": PathConfig("cfg3_smac_27m", T=400, B=512, A=27, p_end=1 / 180, gamma=0.99, lmbda=0.95,
                                dual_clip=True, c_clip=3.0, clip_value=False, value_loss="huber",
                                value_loss_delta=10.0, value_loss_weight=1.0, popart=True, num_actions=(36,),
                                dead_agent_frac=0.2),
    "cfg4_football_11v11": PathConfig("cfg4_football_11v11", T=200, B=2048, A=10, p_end=0.005, gamma=0.99,
                                      lmbda=0.95, clip_value=True, dual_clip=True, value_loss="huber",
                                      value_loss_delta=10.0, value_loss_weight=1.0, popart=True,
                                      num_actions=(19,)),
    "cfg5_hns_scale": PathConfig("cfg5_hns_scale", T=160, B=65536, A=1, p_end=1 / 240, gamma=0.998, lmbda=0.95,
                                 clip_value=False, dual_clip=False, value_loss="mse", value_loss_weight=0.5,
                                 popart=True, num_actions=(11, 11, 11, 2, 2)),
}


def make_sample_scalars(cfg: PathConfig, seed: int = 0, B: Optional[int] = None) -> Dict[str, np.ndarray]:
    """The scalar leaves of one assembled SampleBatch: reward, value, old_logp float32 and
    done, truncated, on_reset uint8, each `[L, B, (A,) 1]`.  Flags are per environment and shared by
    its agents (legacy/environment/smac/smac_env.py:157-166 emits them as [A,1] copies)."""
    B = cfg.B if B is None else B
    rng = np.random.Generator(np.random.PCG64(seed))
    L, A = cfg.L, cfg.A
    env_shape = (L, B, 1, 1) if A > 1 else (L, B, 1)
    full_shape = (L, B, A, 1) if A > 1 else (L, B, 1)
    done = (rng.random(env_shape) < cfg.p_end).astype(np.uint8)
    truncated = ((rng.random(env_shape) < cfg.p_end) & (done == 0)).astype(np.uint8)
    on_reset = np.zeros(env_shape, dtype=np.uint8)
    on_reset[1:] = done[:-1] + truncated[:-1]
    if A > 1:
        done, truncated, on_reset = (np.ascontiguousarray(np.broadcast_to(x, full_shape))
                                     for x in (done, truncated, on_reset))
    value = rng.standard_normal(full_shape, dtype=np.float32)
    reward = rng.standard_normal(full_shape, dtype=np.float32)
    reward[:-1] *= (1 - on_reset[1:]).astype(np.float32)  # gae.py:72
    old_logp = -rng.standard_exponential(full_shape, dtype=np.float32)
    return dict(reward=reward, value=value, done=done, truncated=truncated, on_reset=on_reset, old_logp=old_logp)


def make_policy_outputs(cfg: PathConfig, sample: Dict[str, np.ndarray], seed: int = 1,
                        epochs: Optional[int] = None) -> Dict[str, np.ndarray]:
    """What `policy.analyze` would return for the loss rows, one set per epoch: new_logp, v_pred, entropy
    `[E, T, B, (A,) 1]` float32 (SURVEY.md §8d: new = old + 0.1 N(0,1); v = value + 0.1 N(0,1); H ~ U(0, log K))."""
    E = cfg.epochs if epochs is None else epochs
    rng = np.random.Generator(np.random.PCG64(seed + 7919))
    lo, hi = cfg.burn_in_steps, cfg.L - cfg.bootstrap_steps
    shape = (E,) + sample["value"][lo:hi].shape
    new_logp = sample["old_logp"][lo:hi][None] + np.float32(0.1) * rng.standard_normal(shape, dtype=np.float32)
    if cfg.dead_agent_frac > 0:
        dead = rng.random(shape) < cfg.dead_agent_frac
        new_logp = np.where(dead, np.float32(-np.inf), new_logp).astype(np.float32)
    v_pred = sample["value"][lo:hi][None] + np.float32(0.1) * rng.standard_normal(shape, dtype=np.float32)
    logk = float(sum(np.log(k) for k in cfg.num_actions))
    entropy = (rng.random(shape, dtype=np.float32) * np.float32(logk)).astype(np.float32)
    return dict(new_logp=new_logp.astype(np.float32), v_pred=v_pred.astype(np.float32), entropy=entropy)


def make_logits_actions(cfg: PathConfig, lead_shape, seed: int = 2):
    """For the from-logits loss variant: logits ~ N(0,1) `[*lead, sum K]` float32 and actions `[*lead, heads]`
    int32 sampled from them (make_masked_logits_actions adds an availability mask)."""
    rng = np.random.Generator(np.random.PCG64(seed + 104729))
    K = int(sum(cfg.num_actions))
    logits = rng.standard_normal(tuple(lead_shape) + (K,), dtype=np.float32)
    actions = np.zeros(tuple(lead_shape) + (len(cfg.num_actions),), dtype=np.int32)
    off = 0
    for h, k in enumerate(cfg.num_actions):
        z = logits[..., off:off + k].astype(np.float64)
        p = np.exp(z - z.max(-1, keepdims=True))
        p /= p.sum(-1, keepdims=True)
        u = rng.random(tuple(lead_shape) + (1,))
        actions[..., h] = np.minimum((p.cumsum(-1) < u).sum(-1), k - 1)
        off += k
    return logits, actions


def make_masked_logits_actions(cfg: PathConfig, lead_shape, seed: int = 2, p_unavailable: float = 0.3):
    """For the from-logits loss with SMAC's availability mask: logits ~ N(0,1) `[*lead, sum K]` float32, `available`
    `[*lead, sum K]` uint8 (each action unavailable with probability p_unavailable, action 0 of every head always
    available, as SMAC's no-op is) and actions `[*lead, heads]` int32 sampled from the masked distribution.
    Returns (logits, actions, available)."""
    rng = np.random.Generator(np.random.PCG64(seed + 1299709))
    lead = tuple(lead_shape)
    K = int(sum(cfg.num_actions))
    logits = rng.standard_normal(lead + (K,), dtype=np.float32)
    available = (rng.random(lead + (K,)) >= p_unavailable).astype(np.uint8)
    actions = np.zeros(lead + (len(cfg.num_actions),), dtype=np.int32)
    off = 0
    for h, k in enumerate(cfg.num_actions):
        available[..., off] = 1
        z = logits[..., off:off + k].astype(np.float64)
        p = np.exp(z - z.max(-1, keepdims=True)) * available[..., off:off + k]
        p /= p.sum(-1, keepdims=True)
        u = rng.random(lead + (1,))
        a = np.minimum((p.cumsum(-1) < u).sum(-1), k - 1)
        # the float64 cumsum can end a hair below u: take the last available action instead of an unavailable one
        last = k - 1 - np.argmax(available[..., off:off + k][..., ::-1], axis=-1)
        actions[..., h] = np.minimum(a, last)
        off += k
    return logits, actions, available


def make_obs(cfg: PathConfig, L: int, B: int, seed: int = 3) -> np.ndarray:
    """Synthetic observations `[L, B, *obs_shape]` (uniform bytes for uint8, N(0,1) otherwise)."""
    rng = np.random.Generator(np.random.PCG64(seed + 15485863))
    shape = (L, B) + tuple(cfg.obs_shape)
    if cfg.obs_dtype == "uint8":
        return rng.integers(0, 256, size=shape, dtype=np.uint8)
    return rng.standard_normal(shape, dtype=np.float32).astype(cfg.obs_dtype)
