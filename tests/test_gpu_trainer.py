"""End-to-end parity of the drop-in trainer: `MultiAgentPPOB200.step` on the GPU against the CPU restatement of
`MultiAgentPPO.step` (oracle/ref_trainer.py, mappo.py:219-328) with the same policy class, optimizer and
samples.  After several steps the network parameters, the logged stats and the adv / ret written back into the
host sample must agree."""
import copy

import numpy as np
import pytest
import torch

from oracle.ref_trainer import RefPPOTrainer
from srl_b200 import api, synth
from srl_b200.namedarray import NamedArray
from tests.doubles import TinyActorCriticPolicy
from tests.util import assert_close_ref

pytestmark = pytest.mark.gpu

OBS_DIM, NUM_ACTIONS = 6, 5


def make_sample(cfg, seed):
    s = synth.make_sample_scalars(cfg, seed)
    rng = np.random.default_rng(seed + 99)
    lead = s["value"].shape[:-1]
    obs = NamedArray(vec=rng.standard_normal(lead + (OBS_DIM,)).astype(np.float32))
    action = NamedArray(x=rng.integers(0, NUM_ACTIONS, lead + (1,)).astype(np.float32))
    info = NamedArray(episode_return=rng.standard_normal(lead + (1,)).astype(np.float32))
    info_mask = (rng.random(lead + (1,)) < 0.1).astype(np.float32)
    return api.SampleBatch(obs=obs, on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"], action=action,
                           reward=s["reward"], info=info, info_mask=info_mask,
                           analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))


def clone_sample(x):
    return copy.deepcopy(x)


CASES = {
    "atari": (synth.PathConfig("t_atari", T=12, B=16, p_end=0.08),
              dict(clip_value=True, dual_clip=False, value_loss="huber", value_loss_config=dict(delta=10.0),
                   value_loss_weight=1.0, ppo_epochs=2)),
    "smac_popart": (synth.PathConfig("t_smac", T=10, B=6, A=3, p_end=0.1, lmbda=0.95),
                    dict(gae_lambda=0.95, dual_clip=True, value_loss="huber", value_loss_config=dict(delta=10.0),
                         popart=True, ppo_epochs=2, max_grad_norm=0.5)),
    "minibatch": (synth.PathConfig("t_mb", T=8, B=16, p_end=0.1),
                  dict(clip_value=True, value_loss="mse", ppo_epochs=2, num_minibatches=4, shuffle_seed=5)),
    "boot_burn": (synth.PathConfig("t_bb", T=9, B=8, bootstrap_steps=3, burn_in_steps=2, p_end=0.1),
                  dict(bootstrap_steps=3, burn_in_steps=2, value_loss="smoothl1", popart=True)),
    "vtrace": (synth.PathConfig("t_vt", T=9, B=8, p_end=0.1), dict(vtrace=True, dual_clip=False)),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_trainer_steps_match_reference_restatement(name):
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES[name]
    kw = dict(kw, discount_rate=cfg.gamma, optimizer="sgd", optimizer_config=dict(lr=0.05))
    popart = kw.get("popart", False)
    pol_gpu = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", popart=popart, seed=3)
    pol_cpu = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cpu", popart=popart, seed=3)
    mine = MultiAgentPPOB200(pol_gpu, prefetch=False, **kw)
    ref = RefPPOTrainer(pol_cpu, **kw)
    for it in range(3):
        s_gpu = make_sample(cfg, seed=10 + it)
        s_cpu = clone_sample(s_gpu)
        got = mine.step(s_gpu)
        want_stats, want_version = ref.step(s_cpu)
        assert got.step == want_version == it
        np.testing.assert_array_equal(s_gpu.analyzed_result.adv, s_cpu.analyzed_result.adv) if name != "vtrace" else \
            assert_close_ref(s_gpu.analyzed_result.adv, s_cpu.analyzed_result.adv, what="adv")
        assert_close_ref(s_gpu.analyzed_result.ret, s_cpu.analyzed_result.ret, what="ret")
        for k, v in want_stats.items():
            assert k in got.stats, k
            assert_close_ref(got.stats[k], v, tol=2e-5, what=f"stat {k} at step {it}")
        assert "info/episode_return" not in got.stats and "episode_return" in got.stats
    for (n1, p1), (n2, p2) in zip(pol_gpu.net.state_dict().items(), pol_cpu.net.state_dict().items()):
        assert n1 == n2
        assert_close_ref(p1.cpu(), p2, tol=2e-5, what=f"parameter {n1}")


def test_prefetch_delay_and_checkpoint_contract():
    """The first step() only primes the pipeline (api/trainer.py:219-223); checkpoints carry the reference's keys."""
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES["atari"]
    pol = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=1)
    tr = api.make(type("Cfg", (), dict(type_="mappo_b200", args=dict(kw)))(), pol)
    assert isinstance(tr, MultiAgentPPOB200) and tr.policy is pol
    first = tr.step(make_sample(cfg, 1))
    assert first.stats == {} and first.step == 0
    second = tr.step(make_sample(cfg, 2))
    assert second.step == 0 and second.stats["frames"] == cfg.T * cfg.N  # trained on sample 1
    for key in ("advantage", "entropy", "policy_loss", "value_loss", "done", "truncated", "clip_ratio",
                "importance_weight", "value_targets", "grad_norm", "frames"):
        assert key in second.stats and np.isfinite(second.stats[key]), key
    ck = tr.get_checkpoint()
    assert set(ck) == {"steps", "state_dict", "optimizer_state_dict"} and ck["steps"] == 0
    pol2 = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=2)
    tr2 = MultiAgentPPOB200(pol2, **kw)
    tr2.load_checkpoint(ck)
    for a, b in zip(pol.net.state_dict().values(), pol2.net.state_dict().values()):
        assert torch.equal(a, b)


def test_cached_advantages_are_reused():
    """recompute_adv_on_reuse=False: a sample served again carries adv/ret in its host copy and GAE is skipped
    (mappo.py:224-225,249; base/buffer.py:142-162)."""
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES["atari"]
    kw = dict(kw, recompute_adv_on_reuse=False, optimizer="sgd", optimizer_config=dict(lr=0.0))
    pol = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=4)
    tr = MultiAgentPPOB200(pol, prefetch=False, **kw)
    s = make_sample(cfg, 7)
    r1 = tr.step(s)
    adv1 = s.analyzed_result.adv.copy()
    s.reward[:] = 0  # would change a recomputed advantage
    r2 = tr.step(s)
    np.testing.assert_array_equal(s.analyzed_result.adv, adv1)
    assert_close_ref(r2.stats["advantage"], r1.stats["advantage"], what="advantage stat with cached adv")


def test_constructor_contract():
    from srl_b200.trainer import MultiAgentPPOB200
    pol = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0")
    with pytest.raises(ValueError, match="should be consistent"):  # mappo.py:85-89
        MultiAgentPPOB200(pol, clip_value=True, normalize_old_value=True)
    with pytest.raises(AssertionError, match="does not match any implemented loss"):
        MultiAgentPPOB200(pol, value_loss="l1")
    with pytest.raises(ValueError, match="popart_head"):
        MultiAgentPPOB200(pol, popart=True)
    tr = MultiAgentPPOB200(pol, unknown_key=123)  # unknown kwargs are ignored, like kwargs.get in mappo.py:71-112
    assert (tr.discount_rate, tr.gae_lambda, tr.eps_clip, tr.c_clip, tr.value_loss_weight, tr.ppo_epochs) == \
        (0.99, 0.97, 0.2, 3, 0.5, 1)
    cpu_pol = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path"):
        MultiAgentPPOB200(cpu_pol)


def test_staging_keeps_wire_dtypes_and_crosses_pcie_once():
    """A2: every leaf is sent to the device ONCE, in its own dtype (the reference inflates all of them to float32 on the
    device, api/trainer.py:215-217; the first drop-in sent the scalar leaves twice).  H2D bytes of a step == the host
    sample's bytes; uint8 frames and flags are uint8 in HBM; what `policy.analyze` sees is float32."""
    from srl_b200.namedarray import size_bytes
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES["minibatch"]
    seen = {}

    class Spy(TinyActorCriticPolicy):

        def analyze(self, sample, **k):
            seen["analyze_dtypes"] = {str(sample.obs.vec.dtype), str(sample.obs.frame.dtype), str(sample.on_reset.dtype)}
            return super().analyze(sample, **k)

    pol = Spy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=3)
    tr = MultiAgentPPOB200(pol, prefetch=False, **dict(kw, optimizer="sgd", optimizer_config=dict(lr=0.01)))
    s = make_sample(cfg, seed=2)
    rng = np.random.default_rng(0)
    s.obs = NamedArray(vec=s.obs.vec, frame=rng.integers(0, 255, s.obs.vec.shape[:2] + (4, 12, 12), dtype=np.uint8))
    host_bytes = size_bytes(s)
    staged_host, staged_dev = tr._stage(s)
    torch.cuda.synchronize()
    assert staged_dev.obs.frame.dtype == torch.uint8 and staged_dev.on_reset.dtype == torch.uint8
    assert staged_dev.obs.vec.dtype == torch.float32 and staged_dev.obs.frame.is_cuda
    assert tr.h2d_bytes == host_bytes
    before = tr.h2d_bytes
    tr.step(s)
    assert tr.h2d_bytes - before == host_bytes  # one more staging of the same sample: again exactly its bytes, once
    assert seen["analyze_dtypes"] == {"torch.float32"}


def test_trainer_accepts_the_references_own_records():
    """Inside an SRL checkout the sample is SRL's `SampleBatch` and SRL policies test `isinstance(x, NamedArray)` against
    SRL's class (e.g. base.namedarray.recursive_apply inside analyze): the records handed to `policy.analyze` must be of
    that family, not of this package's mirror.  Uses the unmodified reference classes (oracle/ref_loader.py) where they are
    staged, and otherwise a record family of the same surface that shares nothing with the mirror (tests/doubles.py)."""
    from oracle import ref_loader
    from srl_b200.trainer import MultiAgentPPOB200
    if ref_loader.available():
        R = ref_loader.load()
        NA, SB, rapply = R.namedarray.NamedArray, R.trainer.SampleBatch, R.namedarray.recursive_apply
    else:
        from tests import doubles
        NA, SB, rapply = doubles.NamedArray, doubles.SampleBatch, doubles.recursive_apply
    assert NA is not NamedArray and not issubclass(NA, NamedArray)
    cfg, kw = CASES["minibatch"]
    a = make_sample(cfg, seed=4)

    class RefStylePolicy(TinyActorCriticPolicy):

        def analyze(self, sample, **k):
            assert isinstance(sample, NA) and isinstance(sample.obs, NA), type(sample)
            sample = rapply(sample, lambda x: x)  # what SRL's _ppo_analyze does first
            assert isinstance(sample, NA)
            return super().analyze(sample, **k)

    sb = SB(obs=NA(vec=a.obs.vec), on_reset=a.on_reset, done=a.done, truncated=a.truncated, action=NA(x=a.action.x),
            reward=a.reward, info=NA(episode_return=a.info.episode_return), info_mask=a.info_mask,
            analyzed_result=NA(value=a.analyzed_result.value, log_probs=a.analyzed_result.log_probs, adv=None, ret=None))
    pol = RefStylePolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=3)
    tr = MultiAgentPPOB200(pol, prefetch=False, **dict(kw, optimizer="sgd", optimizer_config=dict(lr=0.01)))
    res = tr.step(sb)
    assert res.step == 0 and np.isfinite(res.stats["policy_loss"]) and "episode_return" in res.stats
    assert isinstance(sb.analyzed_result.adv, np.ndarray) and sb.analyzed_result.adv.shape == a.on_reset.shape


def test_reused_entry_with_prefetch_recomputes_when_staged_before_adv_existed():
    """recompute_adv_on_reuse=False + prefetch: a buffer entry served on two consecutive calls is staged the second time
    BEFORE the first processing wrote adv / ret into it.  The reference decides from the STAGED copy (mappo.py:249) and
    simply recomputes; the first drop-in looked at the host sample and crashed."""
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES["atari"]
    pol = TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0", seed=4)
    tr = MultiAgentPPOB200(pol, **dict(kw, recompute_adv_on_reuse=False, optimizer="sgd", optimizer_config=dict(lr=0.0)))
    s = make_sample(cfg, 7)
    assert tr.step(s).stats == {}          # primes the pipeline with s
    r1 = tr.step(s)                        # stages s again (adv still None), processes the first copy -> s.adv is set
    assert s.analyzed_result.adv is not None
    r2 = tr.step(s)                        # processes the second copy, staged without adv: recomputed, no crash
    assert_close_ref(r2.stats["advantage"], r1.stats["advantage"], what="advantage stat")
    r3 = tr.step(s)                        # this copy was staged WITH adv: the cached branch
    assert_close_ref(r3.stats["advantage"], r1.stats["advantage"], what="advantage stat (cached)")
