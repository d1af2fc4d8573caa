"""Reference of the Beta actor head (K4d, srl_ppo_loss_from_beta) for the tests.

The reference trainer's policies are categorical only, so no reference line pins this head; its definition is
torch.distributions.Beta, what any PyTorch Beta policy computes.  It sits beside the tests rather than in
oracle/ref_math.py, whose functions restate the reference trainer itself.
"""
import torch


def logp_entropy_from_beta_ref(concentration1, concentration0, action):
    """Beta(concentration1, concentration0).log_prob(action).sum(-1) and .entropy().sum(-1).

    All three [..., D], action in (0, 1); the concentrations may require grad; returns (logp, entropy), each [...]."""
    dist = torch.distributions.Beta(concentration1, concentration0)
    return dist.log_prob(action).sum(-1), dist.entropy().sum(-1)
