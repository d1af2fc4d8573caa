"""CPU tests of the host-side mirror of the reference interface: NamedArray semantics, the trainer registry,
the test policy, and the CPU restatement of the trainer step."""
import numpy as np
import pytest
import torch

from oracle import ref_math as M
from oracle.ref_trainer import RefPPOTrainer
from srl_b200 import api, namedarray as na, synth
from tests.doubles import PopArtValueHead, TinyActorCriticPolicy
from tests.util import load_golden


def test_namedarray_sorted_keys_slicing_and_flatten():
    x = na.NamedArray(b=np.arange(6).reshape(3, 2), a=na.NamedArray(z=np.ones((3, 1)), y=None), c=None)
    assert list(x.keys()) == ["a", "b", "c"]  # sorted, base/namedarray.py:282
    assert [k for k, _ in na.flatten(x)] == ["a.y", "a.z", "b", "c"]
    s = x[1:]
    assert s.b.shape == (2, 2) and s.a.z.shape == (2, 1) and s.c is None and s.a.y is None
    back = na.from_flattened(na.flatten(x))
    assert [k for k, _ in na.flatten(back)] == [k for k, _ in na.flatten(x)]
    with pytest.raises(AttributeError):
        x.not_a_field = 1
    x.b = np.zeros((3, 2))
    assert x["b"].sum() == 0 and len(x) == 3
    assert na.size_bytes(x) == 3 * 2 * 8 + 3 * 8


def test_recursive_aggregate_matches_reference_fixture():
    """tests/golden/stack.npz was produced by base.namedarray.recursive_aggregate(np.stack(axis=1))."""
    d = load_golden("stack.npz")
    samples = []
    for b in range(6):
        obs = na.NamedArray(frame=d[f"s{b}.obs.frame"], vec=d[f"s{b}.obs.vec"])
        samples.append(api.SampleBatch(obs=obs, reward=d[f"s{b}.reward"], on_reset=d[f"s{b}.on_reset"],
                                       truncated=d.get(f"s{b}.truncated")))
    agg = na.recursive_aggregate(samples, lambda xs: np.stack(xs, axis=1))
    got = {k: v for k, v in na.flatten(agg) if v is not None}
    assert sorted(got) == sorted(str(k) for k in d["out_keys"])
    for k, v in got.items():
        assert np.array_equal(v, d[f"out.{k}"]), k


def test_sample_batch_field_set_and_registry():
    s = api.SampleBatch(obs=None, reward=np.zeros((2, 1)), bogus_field=1)  # unknown kwargs are dropped
    assert "reward" in s and "bogus_field" not in s and s.done is None and s.sampling_weight is None
    assert set(s.keys()) >= {"obs", "on_reset", "done", "truncated", "action", "reward", "info", "info_mask",
                             "policy_state", "analyzed_result", "policy_version_steps"}
    r = api.TrainerStepResult({}, 0)
    assert r.agree_pushing is True and r.priorities is None

    class Dummy(api.Trainer):
        def __init__(self, policy, **kw):
            self.p, self.kw = policy, kw

    api.register("dummy", Dummy)
    t = api.make(type("Cfg", (), dict(type_="dummy", args=dict(a=1)))(), policy=object())
    assert isinstance(t, Dummy) and t.kw == dict(a=1)
    with pytest.raises(NotImplementedError):
        api.Trainer().step(None)


def _sample(cfg, seed):
    s = synth.make_sample_scalars(cfg, seed)
    rng = np.random.default_rng(seed)
    lead = s["value"].shape[:-1]
    return api.SampleBatch(obs=na.NamedArray(vec=rng.standard_normal(lead + (6,)).astype(np.float32)),
                           action=na.NamedArray(x=rng.integers(0, 5, lead + (1,)).astype(np.float32)),
                           on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"], reward=s["reward"],
                           analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))


def test_reference_trainer_restatement_learns_and_writes_back():
    cfg = synth.PathConfig("h", T=8, B=8, A=2, p_end=0.1)
    pol = TinyActorCriticPolicy(device="cpu", popart=True, seed=0)
    assert isinstance(pol.popart_head, PopArtValueHead)
    tr = RefPPOTrainer(pol, popart=True, ppo_epochs=2, num_minibatches=2, optimizer="sgd", optimizer_config=dict(lr=0.1))
    before = [p.detach().clone() for p in pol.parameters()]
    s = _sample(cfg, 0)
    stats, version = tr.step(s)
    assert version == 0 and s.analyzed_result.adv.shape == s.reward.shape and not s.analyzed_result.adv[-1].any()
    assert any(not torch.equal(a, b) for a, b in zip(before, pol.parameters()))
    assert {"advantage", "entropy", "policy_loss", "value_loss", "clip_ratio", "importance_weight", "value_targets",
            "denorm_value", "grad_norm", "done", "truncated", "frames"} <= set(stats)
    # PopArt statistics moved away from their zero initialisation, twice (once per epoch)
    rms = pol.popart_head._PopArtValueHead__rms
    assert float(rms._RunningMeanStd__debiasing_term) == pytest.approx(1 - 0.99**2)


def test_popart_mirror_matches_oracle():
    head = PopArtValueHead(4, 1, beta=0.99)
    ref = M.RunningMeanStdRef((1,), beta=0.99)
    g = torch.Generator().manual_seed(0)
    for _ in range(3):
        x = torch.randn(7, 5, 1, generator=g)
        m = (torch.rand(7, 5, 1, generator=g) < 0.7).float()
        head.update(x, m)
        ref.update(x, m)
    y = torch.randn(9, 1, generator=g)
    assert torch.equal(head.normalize(y), ref.normalize(y)) and torch.equal(head.denormalize(y), ref.denormalize(y))


def test_plugin_registers_into_srl_registry_when_srl_is_importable(monkeypatch):
    """INTEGRATION.md: `import srl_b200.srl_plugin` inside an SRL checkout adds 'mappo_b200' next to 'mappo'.  Where the
    reference files are not staged, SRL's `api.trainer` is a stand-in: its two registries and their register functions
    (api/trainer.py:84-99,231-235, mirrored by srl_b200/api.py), with 'mappo' in it as SRL's own import leaves it."""
    import importlib
    import sys
    import types

    from oracle import ref_loader
    if ref_loader.available():
        srl_trainer = ref_loader.load().trainer
    else:
        srl_trainer = types.ModuleType("api.trainer")
        srl_trainer.ALL_TRAINER_CLASSES = {"mappo": object}
        srl_trainer.ALL_TRAJ_POSTPROCESSOR_CLASSES = {}
        srl_trainer.register = srl_trainer.ALL_TRAINER_CLASSES.__setitem__
        srl_trainer.register_traj_postprocessor = srl_trainer.ALL_TRAJ_POSTPROCESSOR_CLASSES.__setitem__
        srl_api = types.ModuleType("api")
        srl_api.trainer = srl_trainer
        monkeypatch.setitem(sys.modules, "api", srl_api)
        monkeypatch.setitem(sys.modules, "api.trainer", srl_trainer)

    import srl_b200.srl_plugin as plugin
    importlib.reload(plugin)
    assert plugin.REGISTERED_IN_SRL
    assert {"mappo", "mappo_b200"} <= set(srl_trainer.ALL_TRAINER_CLASSES)
    assert srl_trainer.ALL_TRAINER_CLASSES["mappo_b200"] is plugin.MultiAgentPPOB200
    if not ref_loader.available():
        assert srl_trainer.ALL_TRAJ_POSTPROCESSOR_CLASSES == {"gae_b200": plugin.TrajGAEB200}


# ---- chunk reshape descriptors (ops.to_chunk / back_to_trajectory build these for srl_batch_gather) ----------------
def _emulate_gather(src_bytes, piece, t_stride, slot_stride, idx, L, B):
    """What srl_batch_gather does with ONE leaf descriptor (include/srl_b200.h: srl_leaf_desc), in numpy."""
    out = np.empty(L * B * piece, np.uint8)
    for t in range(L):
        for j in range(B):
            o = t * t_stride + int(idx[j]) * slot_stride
            out[(t * B + j) * piece:(t * B + j + 1) * piece] = src_bytes[o:o + piece]
    return out


@pytest.mark.parametrize("T,B,D,C,split", [(24, 8, 1, 8, 1), (24, 8, 4, 4, 2), (12, 6, 8, 3, 4), (6, 5, 2, 1, 1)])
def test_chunk_reshape_descriptors_reproduce_to_chunk(T, B, D, C, split):
    """The (piece, strides, index vector) ops.to_chunk / back_to_trajectory hand to K1 reproduce
    torch.cat(torch.split(...)) (legacy/algorithm/modules/utils.py:180,195) byte for byte, with and without row splitting."""
    import torch
    from srl_b200 import ops
    x = torch.randn(T, B, D)
    ref = torch.cat(torch.split(x, T // C, dim=0), dim=1).contiguous()
    raw = x.numpy().view(np.uint8).reshape(-1)
    Tc, row = T // C, B * D * 4
    piece = row // split
    idx = ops._split_index("cpu", C, Tc * split, split).numpy()
    got = _emulate_gather(raw, piece, row, piece, idx, Tc, C * split)
    assert np.array_equal(got, ref.numpy().view(np.uint8).reshape(-1))
    idx_back = ops._split_index("cpu", Tc, C * split, split).numpy()
    back = _emulate_gather(ref.numpy().view(np.uint8).reshape(-1), piece, row, piece, idx_back, C, Tc * split)
    assert np.array_equal(back, raw)


def test_row_split_keeps_16_byte_granules_and_bounds_items():
    from srl_b200 import ops
    assert ops._row_split(32, 24) == 1  # short rows move whole
    for row_bytes, items in [(4096 * 28224, 128), (1 << 20, 16), (48 * 1024, 4), (16384 * 3 + 16, 8)]:
        s = ops._row_split(row_bytes, items)
        assert s >= 1 and row_bytes % s == 0 and (s == 1 or ((row_bytes // s) % 16 == 0 and row_bytes // s >= 16384))
        assert s * items <= 65536 or s == 1


# ---- device buffer staging layout (host side of srl_b200/buffer.py) -------------------------------------------------
def test_staging_layout_alignment_and_extension():
    from srl_b200.buffer import _ALIGN, _Layout
    leaves = [("a", np.zeros((5, 3), np.float32)), ("b", None), ("c.x", np.zeros((5, 7), np.uint8))]
    lay = _Layout(leaves)
    assert lay.L == 5 and set(lay.spec) == {"a", "c.x"}
    assert all(off % _ALIGN == 0 for off, _, _ in lay.spec.values()) and lay.bytes % _ALIGN == 0
    assert lay.matches("a", np.zeros((5, 3), np.float32)) and not lay.matches("a", np.zeros((5, 3), np.float64))
    ext = lay.extended_with([("a", np.zeros((5, 3), np.float32)), ("b", np.zeros((5, 1), np.int64)), ("c.x", None)])
    assert set(ext.spec) == {"a", "b", "c.x"} and ext.spec["b"][1] == np.int64 and ext.names == sorted(ext.names)
    with pytest.raises(ValueError):
        _Layout([("a", np.zeros((5, 3))), ("z", np.zeros((4, 3)))])
