"""K4d (srl_ppo_loss_from_beta(_bf16, _pack), ops.ppo_loss_from_beta, ops.PPOBetaLossFunction, MultiAgentPPOB200 with a
Beta head): the PPO loss starting from a Beta actor head, against torch.distributions.Beta in float64 feeding the
oracle's loss, with autograd to both concentrations.  Bars as in test_gpu_parity.py: 1e-5 * max(1, |ref|), gradients on
the g * sum(mask) scale.  The head-result contract and the host-side argument checks run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import ref_math as M
from srl_b200 import _lib, api, build, synth
from srl_b200.api import PPOHeadAnalyzedResult
from srl_b200.namedarray import NamedArray
from tests.beta_ref import logp_entropy_from_beta_ref
from tests.doubles import SampleAnalyzedResult, TinyActorCriticPolicy
from tests.test_gpu_bf16_logits import assert_bf16_grad_close
from tests.test_gpu_gaussian import CONFIGS as GAUSSIAN_CONFIGS
from tests.test_gpu_gaussian import OUT_KEYS, STAT_KEYS, _popart, away_from_clip_edges
from tests.test_gpu_trainer_head import HYPER, SHAPES, _same, _scan, _zero_rows
from tests.util import assert_close_ref, assert_grad_close

CONFIGS = dict(GAUSSIAN_CONFIGS, smoothl1=dict(dual_clip=True, value_loss="smoothl1", entropy_bonus_weight=0.05))
NAMES = ("g_concentration1", "g_concentration0", "g_value", "out", "out_f32", "logp", "entropy")
X_LO, X_HI = np.float32(1e-6), np.float32(1 - 1e-6)


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()  # must load the in-tree .so, loudly
    return _ops


def bf16_exact(x):
    """float32 array -> the float32 array of its values rounded to bfloat16 (nearest even)."""
    return torch.from_numpy(np.ascontiguousarray(x)).bfloat16().float().numpy()


def make_case(T, n, D, seed, N=None, bf16=False):
    """Seeded inputs of one minibatch.  Concentrations log-uniform over [0.2, 100]; actions drawn from the Beta itself,
    clamped to [1e-6, 1 - 1e-6], and about 3 % of them at each end exactly.  Sample side [T + 1, N] (N >= n lanes),
    old_logp the head's log-prob perturbed so that ratios straddle the clip range.  bf16: concentrations and v_pred are
    bfloat16 numbers."""
    N = n if N is None else N
    rng = np.random.default_rng(seed)
    f32 = lambda x: np.asarray(x, dtype=np.float32)
    c1 = f32(np.exp(rng.uniform(np.log(0.2), np.log(100.0), (T, n, D))))
    c0 = f32(np.exp(rng.uniform(np.log(0.2), np.log(100.0), (T, n, D))))
    if bf16:
        c1, c0 = bf16_exact(c1), bf16_exact(c0)
    x = f32(np.clip(rng.beta(c1.astype(np.float64), c0.astype(np.float64)), X_LO, X_HI))
    u = rng.random((T, n, D))
    x = np.where(u < 0.03, X_LO, np.where(u > 0.97, X_HI, x)).astype(np.float32)
    on_reset = (rng.random((T + 1, N)) < 0.1).astype(np.uint8)
    value = f32(rng.standard_normal((T + 1, N)))
    ret = f32(rng.standard_normal((T + 1, N)) * 2.0)
    adv = f32(rng.standard_normal((T + 1, N)))
    lane_idx = np.arange(n, dtype=np.int32) if N == n else rng.permutation(N)[:n].astype(np.int32)
    with torch.no_grad():
        lp, _ = logp_entropy_from_beta_ref(*(torch.from_numpy(a).double() for a in (c1, c0, x)))
    old_logp = np.zeros((T + 1, N), np.float32)
    old_logp[:T, lane_idx] = away_from_clip_edges(lp.numpy(), lp.numpy() + 0.15 * rng.standard_normal((T, n)))
    v_pred = f32(value[:T, lane_idx] + 0.1 * rng.standard_normal((T, n)))
    if bf16:
        v_pred = bf16_exact(v_pred)
    return dict(c1=c1, c0=c0, action=x, on_reset=on_reset, value=value, ret=ret, adv=adv, old_logp=old_logp,
                v_pred=v_pred, lane_idx=lane_idx, T=T, n=n, N=N, D=D)


def oracle(c, hp_kw, popart=None, loss_dtype=torch.float32):
    """Beta log-prob / entropy in float64 -> the oracle's loss, autograd back to both concentrations, on the CPU."""
    T = c["T"]
    take = lambda x: torch.from_numpy(np.ascontiguousarray(x[:T][:, c["lane_idx"]])).to(loss_dtype)
    c1 = torch.from_numpy(c["c1"]).double().requires_grad_(True)
    c0 = torch.from_numpy(c["c0"]).double().requires_grad_(True)
    lp, en = logp_entropy_from_beta_ref(c1, c0, torch.from_numpy(c["action"]).double())
    mask = 1 - torch.from_numpy(np.ascontiguousarray(c["on_reset"][1:T + 1][:, c["lane_idx"]])).to(loss_dtype)
    adv = take(c["adv"])
    res = M.ppo_loss_ref(lp.detach().to(loss_dtype), take(c["old_logp"]), torch.from_numpy(c["v_pred"]).to(loss_dtype),
                         take(c["value"]), take(c["ret"]), adv, en.detach().to(loss_dtype), mask, M.LossHyper(**hp_kw),
                         popart=popart)
    (lp * res["g_logp"].double()).sum().add((en * res["g_entropy"].double()).sum()).backward()
    res.update(lp=lp.detach(), en=en.detach(), g_c1=c1.grad, g_c0=c0.grad, mask_sum=float(mask.sum()),
               norm_stats=[float(x) for x in M.masked_sums_ref(adv, mask)] + [0.0] * 5)
    return res


def run(ops, c, hp_kw, norm_stats, dtype=torch.float32, popart_ms=None, use_lane_idx=False, inputs=None, **kw):
    """One launch with the policy side in `dtype`; `inputs` overrides (c1, c0, action) with device tensors."""
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    c1, c0, act = inputs if inputs is not None else (d(c["c1"]).to(dtype), d(c["c0"]).to(dtype), d(c["action"]))
    r = ops.ppo_loss_from_beta(
        c1, c0, act, d(c["v_pred"]).to(dtype), d(c["old_logp"])[:T], d(c["value"])[:T], d(c["ret"])[:T],
        d(c["adv"])[:T], d(c["on_reset"])[1:T + 1], d(np.asarray(norm_stats, dtype=np.float64)), ops.LossHyper(**hp_kw),
        popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=d(c["lane_idx"]) if use_lane_idx else None, **kw)
    torch.cuda.synchronize()
    return r


def _grid(config, D, seed_base, bf16=False):
    """T = 20, n = 37: two full tiles of 256 transitions (bulk copies) and a partial one (element-wise staging)."""
    use_idx = config == "lane_idx"
    c = make_case(20, 37, D, seed=seed_base + 100 * D, N=53 if use_idx else None, bf16=bf16)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    return c, pa, ms, use_idx


def _check_outputs(ref, out, out32, logp, ent):
    msum = ref["mask_sum"]
    assert_close_ref(logp.cpu(), ref["lp"], what="logp")
    assert_close_ref(ent.cpu(), ref["en"], what="entropy")
    out = out.cpu().numpy()
    for k, name in OUT_KEYS:
        assert_close_ref(out[k], ref[name], what=name)
    for k, name in STAT_KEYS:
        if name in ref["stats"]:
            assert_close_ref(out[k], ref["stats"][name], what=name)
    assert out[9] == msum
    assert_close_ref(out32.cpu().numpy(), out[:4].astype(np.float32), what="out_f32")


# ---- 1. parity with torch.distributions.Beta + the oracle's loss -----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_beta_loss_matches_oracle(ops, D, config):
    hp_kw = CONFIGS[config]
    c, pa, ms, use_idx = _grid(config, D, 0)
    ref = oracle(c, hp_kw, popart=pa)
    g1, g0, g_v, out, out32, logp, ent = run(ops, c, hp_kw, ref["norm_stats"], popart_ms=ms, use_lane_idx=use_idx,
                                             want_logp_entropy=True)
    _check_outputs(ref, out, out32, logp, ent)
    msum = ref["mask_sum"]
    assert_grad_close(g_v.cpu(), ref["g_value"], msum, what="g_value")
    assert_grad_close(g1.cpu(), ref["g_c1"], msum, what="g_concentration1")
    assert_grad_close(g0.cpu(), ref["g_c0"], msum, what="g_concentration0")


@pytest.mark.gpu
def test_beta_masked_transitions_get_zero_gradients(ops):
    c, _, _, _ = _grid("mse_dual_clip", 6, 3)
    ref = oracle(c, CONFIGS["mse_dual_clip"])
    g1, g0, g_v, _, _, _, _ = run(ops, c, CONFIGS["mse_dual_clip"], ref["norm_stats"])
    masked = torch.from_numpy(c["on_reset"][1:c["T"] + 1] != 0).cuda()
    assert bool(masked.any())
    assert not g1[masked].any() and not g0[masked].any() and not g_v[masked].any()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_beta_non_positive_concentrations_give_nan_and_the_launch_ends(ops, dtype):
    """Out of the contract: a concentration of -inf or -1e30 (where x + 1 == x in float64, so a digamma recurrence
    towards x >= 6 would never end).  The launch completes; those transitions' logp and entropy and the gradients of
    those elements are NaN, every other transition's gradients are finite."""
    T, n, D = 4, 64, 3
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_case(T, n, D, seed=31, bf16=dtype == torch.bfloat16)
    ns = oracle(c, hp_kw)["norm_stats"]  # depends on adv and the mask only
    bad = [(1, 5, 0, "c1", -np.inf), (2, 9, 2, "c0", np.float32(-1e30))]
    rows = np.zeros((T, n), bool)
    for t, j, dd, k, v in bad:
        c[k][t, j, dd] = v
        c["on_reset"][t + 1, j] = 0  # a valid transition
        rows[t, j] = True
    g1, g0, g_v, _, _, logp, ent = run(ops, c, hp_kw, ns, dtype, want_logp_entropy=True)
    for t, j, dd, _, _ in bad:
        for name, x in (("logp", logp[t, j]), ("entropy", ent[t, j]), ("g_concentration1", g1[t, j, dd]),
                        ("g_concentration0", g0[t, j, dd])):
            assert bool(torch.isnan(x.float())), f"{name} at {(t, j)}: {x}"
    good = torch.from_numpy(~rows).cuda()
    for name, x in (("g_concentration1", g1), ("g_concentration0", g0), ("g_value", g_v)):
        assert bool(torch.isfinite(x[good].float()).all()), f"{name} of an in-contract transition is not finite"


# ---- 2. bfloat16 -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_bf16_beta_equals_the_float32_entry_bit_for_bit(ops, D, config):
    """The bfloat16 entry on x and the float32 entry on x.float(): logp, entropy, out and out_f32 are identical; the
    gradients are the float32 entry's rounded to bfloat16."""
    hp_kw = CONFIGS[config]
    c, pa, ms, use_idx = _grid(config, D, 1, bf16=True)
    ns = oracle(c, hp_kw, popart=pa)["norm_stats"]
    kw = dict(popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
    a = run(ops, c, hp_kw, ns, torch.bfloat16, **kw)
    b = run(ops, c, hp_kw, ns, torch.float32, **kw)
    assert a[0].dtype == a[1].dtype == a[2].dtype == torch.bfloat16
    assert a[5].dtype == a[6].dtype == torch.float32
    for k in (3, 4, 5, 6):
        assert torch.equal(a[k], b[k]), f"{NAMES[k]} differs from the float32 entry's"
    for k in (0, 1, 2):
        assert torch.equal(a[k], b[k].to(torch.bfloat16)), f"{NAMES[k]} is not the float32 entry's rounded to bfloat16"


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["huber_clip_value", "popart_normalize_old_value"])
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_bf16_beta_matches_oracle(ops, D, config):
    """On the widened bfloat16 values: logp, entropy and out within 1e-5 * max(1, |ref|), the bfloat16 gradients within
    half a bfloat16 ulp of the oracle's plus that bar."""
    hp_kw = CONFIGS[config]
    c, pa, ms, use_idx = _grid(config, D, 2, bf16=True)
    ref = oracle(c, hp_kw, popart=pa)
    g1, g0, g_v, out, out32, logp, ent = run(ops, c, hp_kw, ref["norm_stats"], torch.bfloat16, popart_ms=ms,
                                             use_lane_idx=use_idx, want_logp_entropy=True)
    _check_outputs(ref, out, out32, logp, ent)
    msum = ref["mask_sum"]
    assert_bf16_grad_close(g_v, ref["g_value"], msum, "g_value")
    assert_bf16_grad_close(g1, ref["g_c1"], msum, "g_concentration1")
    assert_bf16_grad_close(g0, ref["g_c0"], msum, "g_concentration0")


# ---- 3. unaligned pointers -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("D", [3, 17])
def test_beta_unaligned_pointers_give_the_aligned_bytes(ops, D, dtype):
    """Concentrations and actions one element off a 16-byte boundary take the element-wise staging path on every tile;
    every output is the bulk-copy path's, bit for bit."""
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_case(12, 50, D, seed=40 + D, bf16=dtype == torch.bfloat16)
    ns = oracle(c, hp_kw)["norm_stats"]

    def shifted(x, dt):
        t = torch.from_numpy(np.ascontiguousarray(x)).to(dt).cuda().reshape(-1)
        buf = torch.empty(t.numel() + 8, dtype=dt, device="cuda")
        v = buf[1:1 + t.numel()]
        v.copy_(t)
        assert v.data_ptr() % 16 != 0
        return v.view(x.shape)

    a = run(ops, c, hp_kw, ns, dtype, want_logp_entropy=True)
    b = run(ops, c, hp_kw, ns, dtype, want_logp_entropy=True,
            inputs=(shifted(c["c1"], dtype), shifted(c["c0"], dtype), shifted(c["action"], torch.float32)))
    for name, x, y in zip(NAMES, a, b):
        _same(x, y, name)


# ---- 4. the pack form ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_beta_pack_form_is_bit_identical_to_leaves(ops, shape, dtype):
    T, n, lo, idx, pack, leaves, stats = _scan(shape, seed=4)
    g = torch.Generator(device="cuda").manual_seed(5)
    Db = 6
    c1 = torch.exp(torch.rand(T, n, Db, device="cuda", generator=g) * 5 - 1.6).to(dtype)
    c0 = torch.exp(torch.rand(T, n, Db, device="cuda", generator=g) * 5 - 1.6).to(dtype)
    action = torch.rand(T, n, Db, device="cuda", generator=g).clamp(1e-6, 1 - 1e-6)
    v_pred = torch.randn(T, n, device="cuda", generator=g).to(dtype)
    common = dict(hyper=HYPER, lane_idx=idx, want_logp_entropy=True, **stats)
    ws = [ops.new_loss_workspace("cuda")[0] for _ in range(3)]
    ref = ops.ppo_loss_from_beta(c1, c0, action, v_pred, workspace=ws[0], **leaves, **common)
    got = ops.ppo_loss_from_beta(c1, c0, action, v_pred, None, None, None, None, None, workspace=ws[1], pack=pack,
                                 pack_row_lo=lo, **common)
    for name, a, b in zip(NAMES, ref, got):
        _same(a, b, name)
    deferred = ops.ppo_loss_from_beta(c1, c0, action, v_pred, None, None, None, None, None, workspace=ws[2], defer=True,
                                      pack=pack, pack_row_lo=lo, **common)
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    ops.loss_finalize(ws[2].view(1, -1), out)
    _same(deferred[0], ref[0], "g_concentration1 (deferred)")
    _same(deferred[1], ref[1], "g_concentration0 (deferred)")
    _same(out[0], ref[3], "out (deferred)")
    torch.cuda.synchronize()
    assert int(ws[0].count_nonzero()) == 0 and int(ws[1].count_nonzero()) == 0 and _zero_rows(ws[2])


# ---- 5. determinism and finalisation ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T,n,D", [(128, 1000, 17), (128, 512, 6)], ids=["T128_n1000_D17", "cfg2_minibatch_D6"])
def test_beta_deterministic_and_workspace_left_zero(ops, T, n, D):
    """Two launches: bit-identical gradients and outputs.  Deferred mode (out = NULL, then srl_ppo_loss_finalize on the
    slot) gives the immediate mode's bits.  The workspace is zero after every launch, except the bytes a deferred launch
    hands to the finaliser (slot bytes 4-31).  The second shape is cfg2's 512-lane minibatch."""
    hp_kw = CONFIGS["mse_dual_clip"]
    c = make_case(T, n, D, seed=11 + D)
    ref = oracle(c, hp_kw)
    ws = ops.new_loss_workspace("cuda")[0]
    a = run(ops, c, hp_kw, ref["norm_stats"], workspace=ws)
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = run(ops, c, hp_kw, ref["norm_stats"], workspace=ws)
    assert not ws.any()
    for x, y, name in zip(a[:5], b[:5], NAMES):
        assert torch.equal(x, y), f"{name} differs between two launches"
    msum = ref["mask_sum"]
    assert_grad_close(a[0].cpu(), ref["g_c1"], msum, what="g_concentration1")
    assert_grad_close(a[1].cpu(), ref["g_c0"], msum, what="g_concentration0")
    g1, g0, g_v, out_d, out32_d, _, _ = run(ops, c, hp_kw, ref["norm_stats"], workspace=ws, defer=True)
    assert out_d is None and out32_d is None
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    out32 = torch.zeros((1, 4), dtype=torch.float32, device="cuda")
    ops.loss_finalize(ws.view(1, -1), out, out32)
    torch.cuda.synchronize()
    assert torch.equal(out[0], a[3]) and torch.equal(out32[0], a[4])
    assert torch.equal(g1, a[0]) and torch.equal(g0, a[1]) and torch.equal(g_v, a[2])
    rest = torch.cat([ws[:4], ws[32:]])
    assert not rest.any(), "deferred mode + finalize left the workspace dirty"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_beta_autograd_function_hands_the_launch_gradients(ops, dtype):
    """PPOBetaLossFunction: the loss is out_f32[0] and backward hands the launch's gradients, in the inputs' dtype, to
    concentration1, concentration0 and v_pred."""
    T, n, D = 16, 100, 4
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_case(T, n, D, seed=21, bf16=dtype == torch.bfloat16)
    ns = oracle(c, hp_kw)["norm_stats"]
    want = run(ops, c, hp_kw, ns, dtype)
    d = lambda k: torch.from_numpy(np.ascontiguousarray(c[k])).cuda()
    c1 = d("c1").to(dtype).requires_grad_(True)
    c0 = d("c0").to(dtype).requires_grad_(True)
    vp = d("v_pred").to(dtype).requires_grad_(True)
    loss, out = ops.PPOBetaLossFunction.apply(c1, c0, d("action"), vp, d("old_logp")[:T], d("value")[:T], d("ret")[:T],
                                              d("adv")[:T], d("on_reset")[1:T + 1],
                                              torch.tensor(ns, dtype=torch.float64, device="cuda"), None, None, None,
                                              ops.LossHyper(**hp_kw))
    loss.backward()
    torch.cuda.synchronize()
    assert torch.equal(loss, want[4][0]) and torch.equal(out, want[3])
    for x, g in ((c1, want[0]), (c0, want[1]), (vp, want[2])):
        assert x.grad.dtype == dtype and torch.equal(x.grad, g)


# ---- 6. the trainer against the CPU restatement ----------------------------------------------------------------------
OBS_DIM, DB = 6, 3


class BetaDouble(TinyActorCriticPolicy):
    """A Beta policy over D = 3 bounded actions: the actor layer's 2 D outputs -> softplus(.) + 1 = (concentration1,
    concentration0).  target="ppo" is torch.distributions.Beta, target="ppo_head" returns the concentrations."""
    ppo_head = True

    def __init__(self, device, seed=3):
        super().__init__(OBS_DIM, 2 * DB, device=device, seed=seed)

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        net = self._net
        h = net.body(sample.obs.vec[burn_in_steps:])
        raw, value = net.actor(h), net.critic(h)
        # softplus runs in float32 under autocast; the head is handed over in the network's own dtype, as the value is
        conc = (F.softplus(raw) + 1.0).to(raw.dtype)
        c1, c0 = conc[..., :DB], conc[..., DB:]
        action = sample.action.x[burn_in_steps:]
        if target == "ppo_head":
            return PPOHeadAnalyzedResult(state_values=value, action=action, concentration1=c1, concentration0=c0)
        d = torch.distributions.Beta(c1, c0)
        return SampleAnalyzedResult(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                                    new_action_log_probs=d.log_prob(action).sum(-1, keepdim=True), state_values=value,
                                    entropy=d.entropy().sum(-1, keepdim=True))


def make_beta_sample(cfg, seed):
    s = synth.make_sample_scalars(cfg, seed)
    rng = np.random.default_rng(seed + 99)
    lead = s["value"].shape[:-1]
    obs = dict(vec=rng.standard_normal(lead + (OBS_DIM,)).astype(np.float32))
    x = rng.uniform(0.02, 0.98, lead + (DB,)).astype(np.float32)
    s["old_logp"] = rng.normal(0.3, 0.5, s["old_logp"].shape).astype(np.float32)
    info = NamedArray(episode_return=rng.standard_normal(lead + (1,)).astype(np.float32))
    info_mask = (rng.random(lead + (1,)) < 0.1).astype(np.float32)
    return api.SampleBatch(obs=NamedArray(**obs), on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"],
                           action=NamedArray(x=x), reward=s["reward"], info=info, info_mask=info_mask,
                           analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))


CASES = {
    "atari": (synth.PathConfig("t_atari", T=12, B=16, p_end=0.08),
              dict(clip_value=True, dual_clip=False, value_loss="huber", value_loss_config=dict(delta=10.0),
                   value_loss_weight=1.0, ppo_epochs=2)),
    "minibatch": (synth.PathConfig("t_mb", T=8, B=16, p_end=0.1),
                  dict(clip_value=True, value_loss="mse", ppo_epochs=2, num_minibatches=4, shuffle_seed=5)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_beta_head_path_matches_reference_restatement(case, monkeypatch):
    from oracle.ref_trainer import RefPPOTrainer
    from srl_b200.hotpath import HotPath
    from srl_b200.trainer import MultiAgentPPOB200
    calls = []
    orig = HotPath.loss_from_beta
    monkeypatch.setattr(HotPath, "loss_from_beta", lambda self, *a, **k: calls.append(1) or orig(self, *a, **k))
    cfg, kw = CASES[case]
    kw = dict(kw, discount_rate=cfg.gamma, optimizer="sgd", optimizer_config=dict(lr=0.05))
    pol_gpu, pol_cpu = BetaDouble("cuda:0"), BetaDouble("cpu")
    mine, ref = MultiAgentPPOB200(pol_gpu, prefetch=False, **kw), RefPPOTrainer(pol_cpu, **kw)
    assert mine.ppo_head
    for it in range(3):
        s_gpu, s_cpu = make_beta_sample(cfg, 10 + it), make_beta_sample(cfg, 10 + it)
        got = mine.step(s_gpu)
        want_stats, want_version = ref.step(s_cpu)
        assert got.step == want_version == it
        np.testing.assert_array_equal(s_gpu.analyzed_result.adv, s_cpu.analyzed_result.adv)
        for k, v in want_stats.items():
            assert_close_ref(got.stats[k], v, tol=2e-5, what=f"stat {k} at step {it}")
    assert calls, "the Beta head never reached loss_from_beta"
    for (n1, p1), (n2, p2) in zip(pol_gpu.net.state_dict().items(), pol_cpu.net.state_dict().items()):
        assert n1 == n2
        assert_close_ref(p1.cpu(), p2, tol=2e-5, what=f"parameter {n1}")


# ---- 7. autocast bfloat16 training -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_autocast_beta_policy_trains_through_the_head_path_without_casts(monkeypatch):
    """As test_gpu_trainer_head.py's autocast test: the bfloat16 concentrations and value reach loss_from_beta as the
    policy returned them, every parameter gets a gradient of its own dtype, and the stats are within 1e-2 of the float32
    run's."""
    from srl_b200.hotpath import HotPath
    from srl_b200.trainer import MultiAgentPPOB200
    cfg = synth.PathConfig("t_bf16", T=16, B=64, p_end=0.1)
    kw = dict(clip_value=True, value_loss="mse", ppo_epochs=2, num_minibatches=4, shuffle_seed=5, discount_rate=cfg.gamma,
              optimizer="sgd", optimizer_config=dict(lr=1e-3))
    seen = []
    orig = HotPath.loss_from_beta

    def spy(self, e, j, c1, c0, action, v_pred):
        seen.append((c1.dtype, c0.dtype, v_pred.dtype))
        return orig(self, e, j, c1, c0, action, v_pred)
    monkeypatch.setattr(HotPath, "loss_from_beta", spy)
    stats = {}
    for mode in ("f32", "bf16"):
        pol = BetaDouble("cuda:0")
        tr = MultiAgentPPOB200(pol, prefetch=False, **kw)
        seen.clear()
        for it in range(2):
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16")):
                stats[mode, it] = tr.step(make_beta_sample(cfg, 20 + it)).stats
        want = torch.bfloat16 if mode == "bf16" else torch.float32
        assert seen and all(d == want for t in seen for d in t), seen
        for p in pol.parameters():
            assert p.grad is not None and p.grad.dtype == p.dtype
    for it in range(2):
        for k, v in stats["f32", it].items():
            assert_close_ref(stats["bf16", it][k], v, tol=1e-2, what=f"bf16 stat {k} at step {it}")


# ---- 8. contract errors ----------------------------------------------------------------------------------------------
def _head(**over):
    T, B = 4, 3
    z = lambda *s: torch.zeros(s)
    f = dict(state_values=z(T, B, 1), action=z(T, B, 2), concentration1=z(T, B, 2) + 1, concentration0=z(T, B, 2) + 1)
    f.update(over)
    return PPOHeadAnalyzedResult(**f)


@pytest.mark.parametrize("res,match", [
    (_head(concentration0=None), "concentration0 is required"),
    (_head(concentration1=None), "concentration1 is required"),
    (_head(concentration0=torch.ones(4, 3, 3)), "concentration0"),
    (_head(concentration1=torch.ones(4, 3, 2, dtype=torch.bfloat16)), "concentration1"),
    (_head(concentration0=torch.ones(4, 3, 2, dtype=torch.bfloat16)), "concentration0"),
    (_head(concentration1=torch.ones(4, 3, 1, 2), concentration0=torch.ones(4, 3, 1, 2)), "concentration1"),
    (_head(concentration1=torch.ones(4, 3, 65), concentration0=torch.ones(4, 3, 65), action=torch.zeros(4, 3, 65)),
     "concentration1: D = 65"),
    (_head(action=torch.zeros(4, 3, 2, dtype=torch.float64)), "action"),
    (_head(action=torch.zeros(4, 3, 3)), "action"),
    (_head(logits=torch.zeros(4, 3, 7), head_sizes=[4, 3]), "exactly one"),
    (_head(mean=torch.zeros(4, 3, 2), log_std=torch.zeros(2)), "exactly one"),
    (_head(concentration1=None, mean=torch.zeros(4, 3, 2), log_std=torch.zeros(2)), "exactly one"),
], ids=lambda x: None)
def test_malformed_beta_head_results_are_refused(res, match):
    from srl_b200.trainer import _head_fields
    with pytest.raises(ValueError, match=match):
        _head_fields(res, 4, 3)


def test_well_formed_beta_head_results_pass():
    from srl_b200.trainer import _head_fields
    _head_fields(_head(), 4, 3)
    _head_fields(_head(concentration1=torch.ones(4, 3, 64), concentration0=torch.ones(4, 3, 64),
                       action=torch.zeros(4, 3, 64)), 3, 3)


def test_ppo_loss_from_beta_refuses_mixed_dtypes():
    """The dtype checks come before any device access: no GPU needed."""
    from srl_b200 import ops
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt)
    args = lambda c1, c0, a, v: (c1, c0, a, v) + (None,) * 6 + (ops.LossHyper(),)
    with pytest.raises(ValueError, match="concentration1: expected dtype"):
        ops.ppo_loss_from_beta(*args(z(2, 3, 2, dt=torch.float16), z(2, 3, 2), z(2, 3, 2), z(2, 3)))
    with pytest.raises(ValueError, match="v_pred has dtype"):
        ops.ppo_loss_from_beta(*args(z(2, 3, 2, dt=torch.bfloat16), z(2, 3, 2, dt=torch.bfloat16), z(2, 3, 2), z(2, 3)))
    with pytest.raises(ValueError, match="concentration0 has dtype"):
        ops.ppo_loss_from_beta(*args(z(2, 3, 2), z(2, 3, 2, dt=torch.bfloat16), z(2, 3, 2), z(2, 3)))
    with pytest.raises(ValueError, match="action: expected dtype torch.float32"):
        ops.ppo_loss_from_beta(*args(z(2, 3, 2), z(2, 3, 2), z(2, 3, 2, dt=torch.bfloat16), z(2, 3)))


ENTRIES = ["srl_ppo_loss_from_beta", "srl_ppo_loss_from_beta_bf16", "srl_ppo_loss_from_beta_pack"]
FAKE = 4096  # a non-null, 16-byte aligned device address that no refused call dereferences


def _beta_args(name, D=3, c1=FAKE, c0=FAKE, ws_bytes=None, elem_bytes=4, pack=FAKE, T=2, n=8):
    """The arguments of one of the three entries: every call below is refused on the host before any CUDA call."""
    lib = _lib.load_library()
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)
    ws_bytes = lib.srl_ppo_loss_workspace_bytes(T, n) if ws_bytes is None else ws_bytes
    stats = (FAKE, FAKE, None, ctypes.byref(hc))
    outs = (FAKE, FAKE, FAKE, None, None, FAKE, None, FAKE, ws_bytes, None)
    if name == "srl_ppo_loss_from_beta_pack":
        return (c1, c0, FAKE, D, elem_bytes, FAKE, pack, n, 0, None, T, n) + stats + outs
    return (c1, c0, FAKE, D, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, n, None, T, n) + stats + outs


def _refused(name, **kw):
    build.build()
    lib = _lib.load_library()
    rc = getattr(lib, name)(*_beta_args(name, **kw))
    msg = lib.srl_last_error().decode()
    assert rc == 1, (rc, msg)  # SRL_ERR_INVALID_ARG
    assert name in msg, msg
    return msg


@pytest.mark.parametrize("name", ENTRIES)
def test_beta_entries_refuse_bad_arguments(name):
    assert "D=0" in _refused(name, D=0)
    assert "D=65" in _refused(name, D=65)
    assert "null pointer concentration1" in _refused(name, c1=None)
    assert "null pointer concentration0" in _refused(name, c0=None)
    lib = _lib.load_library()
    need = lib.srl_ppo_loss_workspace_bytes(2, 8)
    assert "workspace too small" in _refused(name, ws_bytes=need - 8)
    if name.endswith("_pack"):
        assert "16-byte aligned" in _refused(name, pack=FAKE + 8)
        assert "pack is null" in _refused(name, pack=None)
        assert "elem_bytes=8" in _refused(name, elem_bytes=8)
        assert "elem_bytes=0" in _refused(name, elem_bytes=0)
