"""Registration of the B200 trainer inside an SRL checkout.

    # legacy/algorithm/__init__.py  (one added line, next to the existing algorithm imports)
    import srl_b200.srl_plugin  # noqa: F401  -> api.trainer.register("mappo_b200", MultiAgentPPOB200)

After that an experiment selects it exactly like the stock trainer (legacy/experiments/atari.py:952-973):

    trainer=api.config.Trainer(type_="mappo_b200", args=dict(discount_rate=0.99, gae_lambda=0.97, ...))

Nothing else in SRL changes: `api.trainer.make` builds the policy and calls `cls(policy=policy, **cfg.args)`
(api/trainer.py:238-246); `GPUThread` calls `trainer.distributed(...)` once and `trainer.step(sample)` in a loop
(distributed/system/trainer_worker.py:94,171).

A policy trained through the fused head losses declares `ppo_head = True` and returns
`srl_b200.srl_plugin.PPOHeadAnalyzedResult` from `analyze(..., target="ppo_head")` (INTEGRATION.md).
"""
from srl_b200.api import PPOHeadAnalyzedResult  # noqa: F401  (the record a `ppo_head` policy returns)
from srl_b200.postprocess import TrajGAEB200
from srl_b200.trainer import MultiAgentPPOB200


def register_into_srl(name: str = "mappo_b200") -> bool:
    """Registers with SRL's own registry when SRL is importable; returns whether it was."""
    try:
        import api.trainer as srl_trainer  # SRL's module, not srl_b200.api
    except Exception:
        return False
    srl_trainer.register(name, MultiAgentPPOB200)
    # the actor-side sibling: api.config.TrajPostprocessor('gae_b200', args=dict(gamma=..., lmbda=...))
    srl_trainer.register_traj_postprocessor("gae_b200", TrajGAEB200)
    return True


REGISTERED_IN_SRL = register_into_srl()
