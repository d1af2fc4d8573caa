"""Training through the fused head losses: K4b / K4c reading K2's loss pack, and `MultiAgentPPOB200` routing a policy that
declares `ppo_head = True` through them.

  kernel : the pack form of srl_ppo_loss_from_logits / _from_gaussian is bit-identical to the leaf form with the same lane_idx
  trainer: a `ppo_head` policy reproduces the reference goldens (tests/golden/trainer_*.npz) and the CPU restatement
           (oracle/ref_trainer.py) driving the same policy through target="ppo"
  bf16   : autocast policies train through the head path with no casts
  errors : the head-result contract and the new C entries' argument checks
"""
import ctypes
import json

import numpy as np
import pytest
import torch
import torch.nn as nn

from srl_b200 import _lib, api, ops, synth
from srl_b200.api import PPOHeadAnalyzedResult
from srl_b200.namedarray import NamedArray
from tests.doubles import SampleAnalyzedResult, TinyActorCriticPolicy
from tests.util import assert_close_ref, load_golden

OBS_DIM, NUM_ACTIONS = 6, 5
HEADS2 = (4, 3)  # the masked two-head double
D = 3            # the Gaussian double's action dimensions


# ---- doubles ---------------------------------------------------------------------------------------------------------
class HeadTiny(TinyActorCriticPolicy):
    """tests/doubles.py's categorical double, opted in: target="ppo_head" returns the logits it hands to Categorical."""
    ppo_head = True

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        if target != "ppo_head":
            return super().analyze(sample, target=target, burn_in_steps=burn_in_steps, **kwargs)
        logits, value = self._net(sample.obs.vec[burn_in_steps:])
        return PPOHeadAnalyzedResult(state_values=value, action=sample.action.x[burn_in_steps:], logits=logits,
                                     head_sizes=[logits.shape[-1]])


class MaskedTwoHead(TinyActorCriticPolicy):
    """Two categorical heads (4 and 3 actions) with SMAC's availability mask in obs.avail (actor_critic_policy.py:135-136,
    303-324): target="ppo" builds the masked Categoricals in torch, target="ppo_head" returns logits + mask."""
    ppo_head = True

    def __init__(self, device, seed=3):
        super().__init__(OBS_DIM, sum(HEADS2), device=device, seed=seed)

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        logits, value = self._net(sample.obs.vec[burn_in_steps:])
        avail = sample.obs.avail[burn_in_steps:]
        action = sample.action.x[burn_in_steps:]
        if target == "ppo_head":
            return PPOHeadAnalyzedResult(state_values=value, action=action, logits=logits, head_sizes=HEADS2,
                                         available=avail)
        lg = logits.masked_fill(avail == 0, -1e10)
        lp, en, off = 0, 0, 0
        for k, K in enumerate(HEADS2):
            d = torch.distributions.Categorical(logits=lg[..., off:off + K])
            lp = lp + d.log_prob(action[..., k].long())
            en = en + d.entropy()
            off += K
        return SampleAnalyzedResult(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                                    new_action_log_probs=lp.unsqueeze(-1), state_values=value, entropy=en.unsqueeze(-1))


class GaussianDouble(TinyActorCriticPolicy):
    """A diagonal Gaussian over D = 3 actions: mean from the actor layer, log_std one shared [D] parameter or a head of its
    own (per transition).  target="ppo" is torch.distributions.Normal."""
    ppo_head = True

    def __init__(self, device, shared, seed=3, hidden=16):
        super().__init__(OBS_DIM, D, hidden=hidden, device=device, seed=seed)
        self.shared = shared
        g = torch.random.get_rng_state()
        torch.manual_seed(seed + 1)
        if shared:
            self._net.log_std = nn.Parameter(torch.full((D,), -0.3, device=device))
        else:
            self._net.log_std_head = nn.Linear(hidden, D).to(device)
        torch.random.set_rng_state(g)

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        net = self._net
        h = net.body(sample.obs.vec[burn_in_steps:])
        mean, value = net.actor(h), net.critic(h)
        log_std = net.log_std if self.shared else net.log_std_head(h)
        action = sample.action.x[burn_in_steps:]
        if target == "ppo_head":
            return PPOHeadAnalyzedResult(state_values=value, action=action, mean=mean, log_std=log_std)
        d = torch.distributions.Normal(mean, log_std.exp())
        return SampleAnalyzedResult(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                                    new_action_log_probs=d.log_prob(action).sum(-1, keepdim=True), state_values=value,
                                    entropy=d.entropy().sum(-1, keepdim=True))


SAMPLE_KIND = {"tiny": "tiny", "masked": "masked", "gauss_shared": "gauss", "gauss_row": "gauss"}


def make_policy(kind, device, popart=False, seed=3):
    if kind == "tiny":
        return HeadTiny(OBS_DIM, NUM_ACTIONS, device=device, popart=popart, seed=seed)
    if kind == "masked":
        return MaskedTwoHead(device, seed=seed)
    return GaussianDouble(device, shared=(kind == "gauss_shared"), seed=seed)


def make_sample(cfg, seed, kind="tiny"):
    s = synth.make_sample_scalars(cfg, seed)
    rng = np.random.default_rng(seed + 99)
    lead = s["value"].shape[:-1]
    obs = dict(vec=rng.standard_normal(lead + (OBS_DIM,)).astype(np.float32))
    if kind == "tiny":
        x = rng.integers(0, NUM_ACTIONS, lead + (1,)).astype(np.float32)
    elif kind == "masked":
        x = np.stack([rng.integers(0, K, lead) for K in HEADS2], -1).astype(np.float32)
        avail = rng.random(lead + (sum(HEADS2),)) < 0.6
        off = 0
        for k, K in enumerate(HEADS2):  # the actors only took available actions
            np.put_along_axis(avail[..., off:off + K], x[..., k:k + 1].astype(np.int64), True, -1)
            off += K
        obs["avail"] = avail.astype(np.float32)
        s["old_logp"] = rng.normal(-2.3, 0.3, s["old_logp"].shape).astype(np.float32)
    else:
        x = rng.standard_normal(lead + (D,)).astype(np.float32)
        s["old_logp"] = rng.normal(-4.5, 0.5, s["old_logp"].shape).astype(np.float32)
    info = NamedArray(episode_return=rng.standard_normal(lead + (1,)).astype(np.float32))
    info_mask = (rng.random(lead + (1,)) < 0.1).astype(np.float32)
    return api.SampleBatch(obs=NamedArray(**obs), on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"],
                           action=NamedArray(x=x), reward=s["reward"], info=info, info_mask=info_mask,
                           analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))


# ---- 1. kernel: the pack form equals the leaf form -------------------------------------------------------------------
# (L, B, A, burn-in, minibatch envs or None = every lane in order): odd n with an odd pack_row_lo; T * n = 468, one full
# tile and a partial one (bulk copy + staging); multi-agent lanes, 576 transitions
SHAPES = {"odd": (10, 7, 1, 1, 5), "tiles": (40, 13, 1, 3, None), "agents": (19, 24, 3, 2, 12)}
HYPER = ops.LossHyper(clip_value=True, dual_clip=True, value_loss="huber", value_loss_config=dict(delta=2.0))


def _scan(shape, seed=0):
    L, B, A, lo, mb_env = SHAPES[shape]
    N = B * A
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = lambda: torch.randn(L, N, device="cuda", generator=g)
    u8 = lambda p: (torch.rand(L, N, device="cuda", generator=g) < p).to(torch.uint8)
    reward, value, old_logp = f(), f(), f() * 0.3 - 1.5
    done, trunc, on_reset = u8(0.05), u8(0.03), u8(0.15)
    pack = ops.new_pack(L, N, "cuda")
    adv, ret, _ = ops.gae_scan(reward, value, done, trunc, on_reset, 0.99, 0.95, row_lo=lo, row_hi=L - 1,
                               old_logp=old_logp, pack=pack)
    hi = L - 1
    leaves = dict(old_logp=old_logp[lo:hi], old_value=value[lo:hi], ret=ret[lo:hi], adv=adv[lo:hi],
                  on_reset_next=on_reset[lo + 1:hi + 1])
    idx = None if mb_env is None else ops.philox_perm(seed + 7, 0, B, A)[:mb_env * A].contiguous()
    n = N if idx is None else idx.numel()
    stats = dict(norm_stats=torch.tensor([float(hi - lo) * n, 3.0, 2.0 * (hi - lo) * n], dtype=torch.float64, device="cuda"),
                 local_stats=torch.tensor([float(hi - lo) * n - 5.0], dtype=torch.float64, device="cuda"))
    return hi - lo, n, lo, idx, pack, leaves, stats


def _same(a, b, what):
    if a is None:
        assert b is None, what
        return
    assert a.dtype == b.dtype and a.shape == b.shape, what
    assert torch.equal(a.view(torch.uint8) if a.dtype == torch.bfloat16 else a,
                       b.view(torch.uint8) if b.dtype == torch.bfloat16 else b), what


def _zero_rows(ws):
    """The slot's ticket and partial rows (bytes 64 on) are zero again; bytes 4-31 keep a deferred launch's header."""
    w = ws.view(-1)
    return int(w[:4].count_nonzero()) == 0 and int(w[32:].count_nonzero()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("masked", [False, True], ids=["plain", "masked"])
@pytest.mark.parametrize("heads", [(18,), (11, 11, 11, 2, 2)], ids=["k18", "k11x3_2x2"])
def test_logits_pack_form_is_bit_identical_to_leaves(shape, dtype, masked, heads):
    T, n, lo, idx, pack, leaves, stats = _scan(shape)
    g = torch.Generator(device="cuda").manual_seed(1)
    SK = sum(heads)
    logits = (torch.randn(T, n, SK, device="cuda", generator=g) * 2).to(dtype)
    v_pred = torch.randn(T, n, device="cuda", generator=g).to(dtype)
    action = torch.stack([torch.randint(0, K, (T, n), device="cuda", generator=g) for K in heads], -1).to(torch.int32)
    avail = None
    if masked:
        avail = (torch.rand(T, n, SK, device="cuda", generator=g) < 0.7).to(torch.uint8)
        avail[..., 0] = 1
    common = dict(hyper=HYPER, lane_idx=idx, want_logp_entropy=True, available=avail, **stats)
    ws = [ops.new_loss_workspace("cuda")[0] for _ in range(3)]
    ref = ops.ppo_loss_from_logits(logits, action, heads, v_pred, workspace=ws[0], **leaves, **common)
    got = ops.ppo_loss_from_logits(logits, action, heads, v_pred, None, None, None, None, None, workspace=ws[1], pack=pack,
                                   pack_row_lo=lo, **common)
    for name, a, b in zip(("g_logits", "g_value", "out", "out_f32", "logp", "entropy"), ref, got):
        _same(a, b, name)
    deferred = ops.ppo_loss_from_logits(logits, action, heads, v_pred, None, None, None, None, None, workspace=ws[2],
                                        defer=True, pack=pack, pack_row_lo=lo, **common)
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    ops.loss_finalize(ws[2].view(1, -1), out)
    _same(deferred[0], ref[0], "g_logits (deferred)")
    _same(out[0], ref[2], "out (deferred)")
    torch.cuda.synchronize()
    assert int(ws[0].count_nonzero()) == 0 and int(ws[1].count_nonzero()) == 0 and _zero_rows(ws[2])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("shared", [True, False], ids=["shared", "per_row"])
def test_gaussian_pack_form_is_bit_identical_to_leaves(shape, dtype, shared):
    T, n, lo, idx, pack, leaves, stats = _scan(shape, seed=2)
    g = torch.Generator(device="cuda").manual_seed(3)
    Dg = 6
    mean = torch.randn(T, n, Dg, device="cuda", generator=g).to(dtype)
    action = torch.randn(T, n, Dg, device="cuda", generator=g)
    log_std = (torch.randn((Dg,) if shared else (T, n, Dg), device="cuda", generator=g) * 0.3)
    log_std = log_std if shared else log_std.to(dtype)
    v_pred = torch.randn(T, n, device="cuda", generator=g).to(dtype)
    common = dict(hyper=HYPER, lane_idx=idx, want_logp_entropy=True, **stats)
    ws = [ops.new_gaussian_loss_workspace("cuda", T, n, Dg, shared) for _ in range(3)]
    ref = ops.ppo_loss_from_gaussian(mean, log_std, action, v_pred, workspace=ws[0], **leaves, **common)
    got = ops.ppo_loss_from_gaussian(mean, log_std, action, v_pred, None, None, None, None, None, workspace=ws[1],
                                     pack=pack, pack_row_lo=lo, **common)
    for name, a, b in zip(("g_mean", "g_log_std", "g_value", "out", "out_f32", "logp", "entropy"), ref, got):
        _same(a, b, name)
    deferred = ops.ppo_loss_from_gaussian(mean, log_std, action, v_pred, None, None, None, None, None, workspace=ws[2],
                                          defer=True, pack=pack, pack_row_lo=lo, **common)
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    ops.loss_finalize(ws[2].view(1, -1), out)
    _same(deferred[1], ref[1], "g_log_std (deferred)")
    _same(out[0], ref[3], "out (deferred)")
    torch.cuda.synchronize()
    assert int(ws[0].count_nonzero()) == 0 and int(ws[1].count_nonzero()) == 0 and _zero_rows(ws[2])


# ---- 2. the trainer against the reference goldens --------------------------------------------------------------------
def _golden_sample(fx, it):
    g = lambda k: fx[f"call{it}/in/{k}"].copy()
    return api.SampleBatch(obs=NamedArray(vec=g("obs_vec")), on_reset=g("on_reset"), done=g("done"), truncated=g("truncated"),
                           action=NamedArray(x=g("action_x")), reward=g("reward"),
                           info=NamedArray(episode_return=g("info_episode_return")), info_mask=g("info_mask"),
                           analyzed_result=api.AnalyzedResult(value=g("value"), log_probs=g("old_logp")))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["plain", "popart", "boot_burn"])
def test_head_path_reproduces_reference_goldens(name):
    from srl_b200.trainer import MultiAgentPPOB200
    fx = load_golden(f"trainer_{name}.npz")
    kw = json.loads(str(fx["kwargs_json"]))
    pol = make_policy("tiny", "cuda:0", popart=kw.get("popart", False))
    pol.net.load_state_dict({k[len("init/"):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith("init/")})
    tr = MultiAgentPPOB200(pol, **kw)
    assert tr.ppo_head
    samples = []
    for it in range(int(fx["n_calls"])):
        samples.append(_golden_sample(fx, it))
        res = tr.step(samples[-1])
        if it == 0:
            assert res.stats == {} and res.step == 0
            continue
        assert res.step == int(fx[f"call{it}/step"])
        assert sorted(res.stats) == list(fx[f"call{it}/stat_keys"])
        for k in res.stats:
            assert_close_ref(res.stats[k], fx[f"call{it}/stat/{k}"], tol=2e-5, what=f"call {it} stat {k}")
        ar = samples[it - 1].analyzed_result
        if bool(fx[f"call{it}/adv_is_none"]):
            assert ar.adv is None and ar.ret is None
        else:
            assert_close_ref(ar.adv, fx[f"call{it}/adv"], what=f"call {it} adv write-back")
            assert_close_ref(ar.ret, fx[f"call{it}/ret"], what=f"call {it} ret write-back")
    for k, v in pol.net.state_dict().items():
        assert_close_ref(v.cpu(), fx[f"final/{k}"], tol=2e-5, what=f"parameter {k} after the last call")


# ---- 3. the trainer against the CPU restatement ----------------------------------------------------------------------
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
}
RUNS = [("tiny", c) for c in sorted(CASES)] + [(k, c) for k in ("masked", "gauss_shared", "gauss_row")
                                                 for c in ("atari", "minibatch")]


def _train_pair(kind, case, steps=3):
    from oracle.ref_trainer import RefPPOTrainer
    from srl_b200.trainer import MultiAgentPPOB200
    cfg, kw = CASES[case]
    kw = dict(kw, discount_rate=cfg.gamma, optimizer="sgd", optimizer_config=dict(lr=0.05))
    popart = kw.get("popart", False)
    pol_gpu, pol_cpu = make_policy(kind, "cuda:0", popart), make_policy(kind, "cpu", popart)
    mine, ref = MultiAgentPPOB200(pol_gpu, prefetch=False, **kw), RefPPOTrainer(pol_cpu, **kw)
    for it in range(steps):
        s_gpu, s_cpu = make_sample(cfg, 10 + it, SAMPLE_KIND[kind]), make_sample(cfg, 10 + it, SAMPLE_KIND[kind])
        got = mine.step(s_gpu)
        want_stats, want_version = ref.step(s_cpu)
        assert got.step == want_version == it
        np.testing.assert_array_equal(s_gpu.analyzed_result.adv, s_cpu.analyzed_result.adv)
        for k, v in want_stats.items():
            assert_close_ref(got.stats[k], v, tol=2e-5, what=f"stat {k} at step {it}")
    return pol_gpu, pol_cpu


@pytest.mark.gpu
@pytest.mark.parametrize("kind,case", RUNS, ids=[f"{k}-{c}" for k, c in RUNS])
def test_head_path_matches_reference_restatement(kind, case):
    pol_gpu, pol_cpu = _train_pair(kind, case)
    for (n1, p1), (n2, p2) in zip(pol_gpu.net.state_dict().items(), pol_cpu.net.state_dict().items()):
        assert n1 == n2
        assert_close_ref(p1.cpu(), p2, tol=2e-5, what=f"parameter {n1}")


# ---- 4. bfloat16 -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["masked", "gauss_shared", "gauss_row"])
def test_autocast_policy_trains_through_the_head_path_without_casts(kind, monkeypatch):
    """The 1e-2 bound is on what bfloat16 rounding of the policy's forward does to the loss and its statistics.  The
    learning rate is small enough that both runs' parameters stay near their common start: at lr = 0.05 the ratios far
    outside the clip range turn the rounding into trajectories that part by several per cent within one step (8 updates),
    whatever the loss kernel does.  256 transitions per minibatch keep one transition crossing the clip boundary (the
    clip_ratio statistic) well inside the bound."""
    from srl_b200.hotpath import HotPath
    from srl_b200.trainer import MultiAgentPPOB200
    cfg = synth.PathConfig("t_bf16", T=16, B=64, p_end=0.1)
    kw = dict(clip_value=True, value_loss="mse", ppo_epochs=2, num_minibatches=4, shuffle_seed=5, discount_rate=cfg.gamma,
              optimizer="sgd", optimizer_config=dict(lr=1e-3))
    seen = []
    for name in ("loss_from_logits", "loss_from_gaussian"):
        orig = getattr(HotPath, name)

        def spy(self, e, j, head, *a, _orig=orig, **k):
            seen.append((head.dtype, a[2].dtype))  # (logits or mean, v_pred): both signatures have v_pred third after it
            return _orig(self, e, j, head, *a, **k)
        monkeypatch.setattr(HotPath, name, spy)
    stats = {}
    for mode in ("f32", "bf16"):
        pol = make_policy(kind, "cuda:0")
        tr = MultiAgentPPOB200(pol, prefetch=False, **kw)
        seen.clear()
        for it in range(2):
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16")):
                stats[mode, it] = tr.step(make_sample(cfg, 20 + it, SAMPLE_KIND[kind])).stats
        want = torch.bfloat16 if mode == "bf16" else torch.float32
        assert seen and all(d == want for pair in seen for d in pair), seen  # the head and the value reach K4b / K4c as is
        for p in pol.parameters():
            assert p.grad is not None and p.grad.dtype == p.dtype
    for it in range(2):
        for k, v in stats["f32", it].items():
            assert_close_ref(stats["bf16", it][k], v, tol=1e-2, what=f"bf16 stat {k} at step {it}")


# ---- 5. contract errors ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vtrace_with_a_head_policy_is_refused():
    from srl_b200.trainer import MultiAgentPPOB200
    with pytest.raises(ValueError, match="ppo_head"):
        MultiAgentPPOB200(make_policy("tiny", "cuda:0"), vtrace=True)
    assert not MultiAgentPPOB200(TinyActorCriticPolicy(OBS_DIM, NUM_ACTIONS, device="cuda:0")).ppo_head


def _head(**over):
    T, B = 4, 3
    f = dict(state_values=torch.zeros(T, B, 1), action=torch.zeros(T, B, 2), logits=torch.zeros(T, B, 7), head_sizes=[4, 3])
    f.update(over)
    return PPOHeadAnalyzedResult(**f)


@pytest.mark.parametrize("res,exc,match", [
    (dict(state_values=1), TypeError, "PPOHeadAnalyzedResult"),
    (_head(action=None), ValueError, "action is required"),
    (_head(state_values=[0.0]), TypeError, "state_values"),
    (_head(state_values=torch.zeros(4, 3, 1, dtype=torch.float64)), ValueError, "state_values"),
    (_head(state_values=torch.zeros(2, 3, 1)), ValueError, "state_values"),
    (_head(logits=None), ValueError, "exactly one"),
    (_head(mean=torch.zeros(4, 3, 2), log_std=torch.zeros(2)), ValueError, "exactly one"),
    (_head(head_sizes=None), ValueError, "head_sizes"),
    (_head(head_sizes=[4, 4]), ValueError, "logits"),
    (_head(logits=torch.zeros(4, 3, 7, dtype=torch.bfloat16)), ValueError, "logits"),
    (_head(action=torch.zeros(4, 3, 1)), ValueError, "action"),
    (_head(available=torch.ones(4, 3, 6)), ValueError, "available"),
    (_head(logits=None, mean=torch.zeros(4, 3, 2), log_std=None), ValueError, "log_std is required"),
    (_head(logits=None, mean=torch.zeros(4, 3, 2), log_std=torch.zeros(3)), ValueError, "log_std"),
    (_head(logits=None, mean=torch.zeros(4, 3, 2), log_std=torch.zeros(2), action=torch.zeros(4, 3, 2, dtype=torch.int64)),
     ValueError, "action"),
], ids=lambda x: None)
def test_malformed_head_results_are_refused(res, exc, match):
    from srl_b200.trainer import _head_fields
    with pytest.raises(exc, match=match):
        _head_fields(res, 4, 3)


def test_well_formed_head_results_pass():
    from srl_b200.trainer import _head_fields
    _head_fields(_head(available=torch.ones(4, 3, 7)), 4, 3)
    _head_fields(_head(logits=None, mean=torch.zeros(4, 3, 2), log_std=torch.zeros(2), action=torch.zeros(4, 3, 2)), 3, 3)
    _head_fields(_head(logits=None, mean=torch.zeros(4, 3, 2), log_std=torch.zeros(4, 3, 2), action=torch.zeros(4, 3, 2)),
                 4, 3)


def _entry_args(name, elem_bytes=4, pack=4096, pack_lanes=8, pack_row_lo=0, lane_idx=None):
    """Arguments of a new C entry with fake, non-null device pointers: every call below is refused before any is used."""
    hc = ops.LossHyper().to_c()
    P = 4096
    rest = (lane_idx, 2, 8, P, P, None, ctypes.byref(hc))
    if name == "srl_ppo_loss_from_logits_pack":
        hs = (ctypes.c_int32 * 1)(5)
        return (P, elem_bytes, None, P, hs, 1, P, pack, pack_lanes, pack_row_lo) + rest + (P, P, None, None, None, None, P,
                                                                                           1 << 20, None)
    return (P, P, 1, P, 3, elem_bytes, P, pack, pack_lanes, pack_row_lo) + rest + (P, P, P, None, None, None, None, P,
                                                                                   1 << 20, None)


@pytest.mark.parametrize("name", ["srl_ppo_loss_from_logits_pack", "srl_ppo_loss_from_gaussian_pack"])
@pytest.mark.parametrize("bad,match", [
    (dict(pack=None), b"pack is null"),
    (dict(pack=4096 + 8), b"16-byte aligned"),
    (dict(pack_row_lo=-1), b"pack_row_lo=-1"),
    (dict(pack_lanes=7), b"pack_lanes=7 < n=8"),
    (dict(elem_bytes=8), b"elem_bytes=8"),
    (dict(elem_bytes=0), b"elem_bytes=0"),
])
def test_pack_entries_refuse_bad_arguments(name, bad, match):
    lib = _lib.load_library()
    rc = getattr(lib, name)(*_entry_args(name, **bad))
    assert rc == 1  # SRL_ERR_INVALID_ARG
    msg = lib.srl_last_error()
    assert name.encode() in msg and match in msg, msg


@pytest.mark.gpu
def test_without_a_pack_the_existing_entries_are_called(monkeypatch):
    called = []
    monkeypatch.setattr(ops._lib, "call", lambda fn, *a: called.append(fn))
    T, n = 2, 8
    f = lambda *s: torch.zeros(s, device="cuda")
    leaves = dict(old_logp=f(T, n), old_value=f(T, n), ret=f(T, n), adv=f(T, n),
                  on_reset_next=torch.zeros(T, n, dtype=torch.uint8, device="cuda"))
    stats = dict(norm_stats=torch.ones(3, dtype=torch.float64, device="cuda"), hyper=ops.LossHyper())
    act = torch.zeros(T, n, 1, dtype=torch.int32, device="cuda")
    pack = ops.new_pack(T + 1, n, "cuda")
    for dt, sfx in ((torch.float32, ""), (torch.bfloat16, "_bf16")):
        ops.ppo_loss_from_logits(f(T, n, 5).to(dt), act, [5], f(T, n).to(dt), **leaves, **stats)
        ops.ppo_loss_from_logits(f(T, n, 5).to(dt), act, [5], f(T, n).to(dt), available=f(T, n, 5) + 1, **leaves, **stats)
        ops.ppo_loss_from_gaussian(f(T, n, 3).to(dt), f(3), f(T, n, 3), f(T, n).to(dt), **leaves, **stats)
        assert called[-3:] == ["srl_ppo_loss_from_logits" + sfx, "srl_ppo_loss_from_logits_masked" + sfx,
                               "srl_ppo_loss_from_gaussian" + sfx]
    none = dict(old_logp=None, old_value=None, ret=None, adv=None, on_reset_next=None)
    ops.ppo_loss_from_logits(f(T, n, 5), act, [5], f(T, n), **none, pack=pack, **stats)
    ops.ppo_loss_from_gaussian(f(T, n, 3), f(3), f(T, n, 3), f(T, n), **none, pack=pack, pack_row_lo=1, **stats)
    assert called[-2:] == ["srl_ppo_loss_from_logits_pack", "srl_ppo_loss_from_gaussian_pack"]
