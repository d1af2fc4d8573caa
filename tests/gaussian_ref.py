"""Reference of the diagonal-Gaussian actor head (K4c, srl_ppo_loss_from_gaussian) for the tests.

The reference trainer's policies are categorical only, so no reference line pins this head; its definition is
torch.distributions.Normal, what any PyTorch Gaussian policy computes.  It sits beside the tests rather than in
oracle/ref_math.py, whose functions restate the reference trainer itself.
"""
import torch


def logp_entropy_from_gaussian_ref(mean, log_std, action):
    """Normal(mean, exp(log_std)).log_prob(action).sum(-1) and .entropy().sum(-1).

    mean, action [..., D]; log_std [..., D] or [D] (broadcast: a shared, state-independent parameter).  Any of them may
    require grad; returns (logp, entropy), each [...]."""
    dist = torch.distributions.Normal(mean, log_std.exp())
    lp = dist.log_prob(action).sum(-1)
    en = dist.entropy().sum(-1)  # the distribution's batch shape is mean's: a [D] log_std is broadcast
    return lp, en
