"""K4b-wide (srl_ppo_loss_from_logits_wide / _wide_pack): the fused categorical PPO loss for rows wider than K4b's staged tile
takes, up to 262144 logits per transition, and ops.ppo_loss_from_logits routing such rows to it.

  oracle   : logp, entropy, the ten outputs, g_logits and g_value against masked_fill + Categorical per head
             (oracle/ref_math.py) -> the oracle's loss -> autograd; float64 for unmasked rows, float32 (torch's rounding of
             a fully unavailable head) with a mask.  Bars of test_gpu_parity.py: 1e-5 * max(1, |ref|), gradients on the
             g * sum(mask) scale.  The narrow head sets of K4b run through the wide entry too.
  edges    : fully unavailable heads, chosen-but-unavailable actions, -inf logits without a mask
  identity : bfloat16 against float32, pack against leaves, two launches, deferred against immediate, unaligned logits
  routing  : which C entry ops.ppo_loss_from_logits calls
  training : PPOCategoricalLossFunction and MultiAgentPPOB200 with wide heads against the CPU restatement
The host-side argument checks run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from srl_b200 import _lib, api, build, synth
from srl_b200.namedarray import NamedArray
from tests.doubles import SampleAnalyzedResult, TinyActorCriticPolicy
from tests.test_gpu_bf16_logits import assert_bf16_grad_close, bf16_exact
from tests.test_gpu_gaussian import away_from_clip_edges
from tests.test_gpu_masked_logits import OUT_KEYS, STAT_KEYS, _popart
from tests.test_gpu_trainer_head import HYPER, OBS_DIM, HeadTiny, _same, _scan, _zero_rows
from tests.util import assert_close_ref, assert_grad_close

ids = lambda h: "x".join(map(str, h))
WIDE = "srl_ppo_loss_from_logits_wide"

CONFIGS = {
    "huber_clip_value": dict(dual_clip=False, clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0),
                             entropy_bonus_weight=0.05),
    "lane_idx": dict(clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0), entropy_bonus_weight=0.05),
    "popart_dual_clip": dict(dual_clip=True, c_clip=3.0, value_loss="huber", value_loss_config=dict(delta=10.0),
                             value_loss_weight=1.0, entropy_bonus_weight=0.05),
    "mse": dict(clip_value=False, value_loss="mse", entropy_bonus_weight=0.01),
}

# (heads, masked, p_available, T, n).  T * n = 740 rows: 92 CTAs of eight rows and a last one of four.
CASES = [
    ((200,), False, 1.0, 20, 37),
    ((160,), True, 0.5, 20, 37),
    ((1, 250), False, 1.0, 20, 37),
    ((4, 33, 300, 7), False, 1.0, 20, 37),
    ((4, 33, 300, 7), True, 0.3, 20, 37),
    ((64, 32, 16, 8, 4, 2, 40, 50), False, 1.0, 20, 37),  # eight heads, sum K = 216
    ((362,), False, 1.0, 20, 37),  # Go, 19 x 19 + pass
    ((4672,), True, 0.01, 4, 37),  # chess (AlphaZero's encoding), about 1 % of the actions legal
    ((32000,), False, 1.0, 3, 7),
    ((131072,), False, 1.0, 2, 3),
]
# K4b's own widths, through the wide entry (routing thresholds lowered)
NARROW = [((18,), False, 1.0, 20, 37), ((11, 11, 11, 2, 2), False, 1.0, 20, 37), ((199,), False, 1.0, 20, 37),
          ((36,), True, 0.3, 20, 37)]
case_id = lambda c: ids(c[0]) + ("-masked" if c[1] else "")


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()  # must load the in-tree .so, loudly
    return _ops


@pytest.fixture
def calls(ops, monkeypatch):
    """The C entries ops calls, in order (the calls still run)."""
    seen = []
    orig = ops._lib.call

    def spy(fn, *a):
        seen.append(fn)
        return orig(fn, *a)
    monkeypatch.setattr(ops._lib, "call", spy)
    return seen


def make_wide(heads, T, n, seed, masked=False, p_available=0.5, N=None, bf16=False, odd_rows=True):
    """Seeded inputs of one minibatch.  Logits N(0, 2^2), float32 (or bfloat16 numbers); with a mask every chosen action is
    available, except, with odd_rows, every 11th transition's head-0 action, and every 7th transition has one head with no
    available action.  Sample side [T + 1, N] as in test_gpu_masked_logits.make_case."""
    N = n if N is None else N
    rng = np.random.default_rng(seed)
    SK = sum(heads)
    offs = np.concatenate([[0], np.cumsum(heads)[:-1]]).astype(np.int64)
    logits = (rng.standard_normal((T, n, SK), dtype=np.float32) * 2).astype(np.float32)
    if bf16:
        logits = bf16_exact(logits)
    actions = np.stack([rng.integers(0, K, (T, n)) for K in heads], -1).astype(np.int32)
    avail = np.ones((T, n, SK), np.uint8)
    chosen_masked = np.zeros(T * n, bool)
    if masked:
        avail = (rng.random((T, n, SK)) < p_available).astype(np.uint8)
        np.put_along_axis(avail, (actions + offs).astype(np.int64), 1, -1)
        fa, fact = avail.reshape(T * n, SK), actions.reshape(T * n, -1)
        if odd_rows:
            for i in range(0, T * n, 7):
                h = (i // 7) % len(heads)
                fa[i, offs[h]:offs[h] + heads[h]] = 0
            chosen_masked[3::11] = True
            fa[chosen_masked, fact[chosen_masked, 0]] = 0
    on_reset = (rng.random((T + 1, N)) < 0.1).astype(np.uint8)
    f32 = lambda x: np.asarray(x, dtype=np.float32)
    value = f32(rng.standard_normal((T + 1, N)))
    ret = f32(rng.standard_normal((T + 1, N)) * 2.0)
    adv = f32(rng.standard_normal((T + 1, N)))
    lane_idx = np.arange(n, dtype=np.int32) if N == n else rng.permutation(N)[:n].astype(np.int32)
    with torch.no_grad():
        lp, _ = M.logp_entropy_from_logits_ref(torch.from_numpy(logits), torch.from_numpy(actions).long(), heads,
                                               available=torch.from_numpy(avail) if masked else None)
    lp = lp[..., 0].numpy().astype(np.float64)
    behaviour = np.where(chosen_masked.reshape(T, n), -1.5, lp)
    old_logp = np.zeros((T + 1, N), np.float32)
    old_logp[:T, lane_idx] = away_from_clip_edges(lp, behaviour + 0.15 * rng.standard_normal((T, n)))
    v_pred = f32(value[:T, lane_idx] + 0.1 * rng.standard_normal((T, n)))
    if bf16:
        v_pred = bf16_exact(v_pred)
    return dict(logits=logits, actions=actions, available=avail if masked else None, heads=tuple(heads), on_reset=on_reset,
                value=value, ret=ret, adv=adv, old_logp=old_logp, v_pred=v_pred, lane_idx=lane_idx, T=T, n=n, N=N)


def oracle(c, hp_kw, popart=None, dtype=torch.float64):
    """masked_fill + Categorical per head in `dtype` -> the oracle's loss (float32) -> autograd back to the logits."""
    T = c["T"]
    take = lambda x: torch.from_numpy(np.ascontiguousarray(x[:T][:, c["lane_idx"]]))
    zl = torch.from_numpy(c["logits"]).to(dtype).requires_grad_(True)
    avail = None if c["available"] is None else torch.from_numpy(c["available"])
    lp, en = M.logp_entropy_from_logits_ref(zl, torch.from_numpy(c["actions"]).long(), c["heads"], available=avail)
    mask = 1 - take(c["on_reset"][1:]).float()
    adv = take(c["adv"])
    res = M.ppo_loss_ref(lp[..., 0].detach().float(), take(c["old_logp"]), torch.from_numpy(c["v_pred"]), take(c["value"]),
                         take(c["ret"]), adv, en[..., 0].detach().float(), mask, M.LossHyper(**hp_kw), popart=popart)
    (lp[..., 0] * res["g_logp"].to(dtype)).sum().add((en[..., 0] * res["g_entropy"].to(dtype)).sum()).backward()
    res.update(lp=lp.detach()[..., 0], en=en.detach()[..., 0], g_logits=zl.grad, mask_sum=float(mask.sum()),
               norm_stats=[float(x) for x in M.masked_sums_ref(adv, mask)] + [0.0] * 5)
    return res


def run(ops, c, hp_kw, norm_stats, dtype=torch.float32, popart_ms=None, use_lane_idx=False, logits=None, **kw):
    """One launch through ops.ppo_loss_from_logits with the policy side in `dtype`."""
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    r = ops.ppo_loss_from_logits(
        d(c["logits"]).to(dtype) if logits is None else logits, d(c["actions"]), c["heads"], d(c["v_pred"]).to(dtype),
        d(c["old_logp"])[:T], d(c["value"])[:T], d(c["ret"])[:T], d(c["adv"])[:T], d(c["on_reset"])[1:T + 1],
        d(np.asarray(norm_stats, dtype=np.float64)), ops.LossHyper(**hp_kw),
        popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=d(c["lane_idx"]) if use_lane_idx else None,
        available=None if c["available"] is None else d(c["available"]), **kw)
    torch.cuda.synchronize()
    return r


def check_against_oracle(ref, r, c, bf16):
    g_logits, g_v, out, out32, logp, ent = r
    msum = ref["mask_sum"]
    for x, name in ((g_logits, "g_logits"), (g_v, "g_value"), (out, "out"), (logp, "logp"), (ent, "entropy")):
        assert bool(torch.isfinite(x).all()), f"{name} has non-finite values"
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
    if bf16:
        assert_bf16_grad_close(g_v, ref["g_value"].float(), msum, what="g_value")
        assert_bf16_grad_close(g_logits, ref["g_logits"], msum, what="g_logits")
    else:
        assert_grad_close(g_v.cpu(), ref["g_value"], msum, what="g_value")
        assert_grad_close(g_logits.cpu(), ref["g_logits"], msum, what="g_logits")
    if c["available"] is not None:
        unavailable = torch.from_numpy(c["available"]).cuda() == 0
        assert bool((g_logits[unavailable] == 0).all()), "non-zero gradient at an unavailable logit"


def _oracle_case(ops, case, config, dtype, seed):
    heads, masked, p_av, T, n = case
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    bf16 = dtype == torch.bfloat16
    c = make_wide(heads, T, n, seed, masked=masked, p_available=p_av, N=n + 16 if use_idx else None, bf16=bf16)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    ref = oracle(c, hp_kw, popart=pa, dtype=torch.float32 if masked else torch.float64)
    r = run(ops, c, hp_kw, ref["norm_stats"], dtype=dtype, popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
    assert r[0].dtype == r[1].dtype == dtype
    check_against_oracle(ref, r, c, bf16)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_wide_logits_match_oracle(ops, calls, case, config, dtype):
    _oracle_case(ops, case, config, dtype, seed=sum(case[0]) % 1000 + len(config))
    assert calls == [WIDE]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("config", ["huber_clip_value", "lane_idx", "popart_dual_clip"])
@pytest.mark.parametrize("case", NARROW, ids=case_id)
def test_wide_entry_at_k4b_widths_matches_oracle(ops, calls, monkeypatch, case, config, dtype):
    monkeypatch.setattr(ops, "SRL_K4B_MAX_SUM_K", 0)
    monkeypatch.setattr(ops, "SRL_K4B_MAX_SUM_K_MASKED", 0)
    _oracle_case(ops, case, config, dtype, seed=sum(case[0]) + 5)
    assert calls == [WIDE]


@pytest.mark.gpu
@pytest.mark.parametrize("heads", [(160,), (4, 33, 300, 7)], ids=ids)
def test_fully_unavailable_heads_and_unavailable_chosen_actions(ops, heads):
    """A head with no available action adds exactly 0 to logp and to the entropy (torch: its log-sum-exp rounds to -1e10,
    every lp_k is 0), and a chosen unavailable action gives a finite row with ratio 0; no NaN anywhere, and exactly 0
    gradient at every unavailable logit."""
    T, n = 20, 37
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_wide(heads, T, n, seed=4, masked=True, p_available=0.4)
    ref = oracle(c, hp_kw, dtype=torch.float32)
    r = run(ops, c, hp_kw, ref["norm_stats"], want_logp_entropy=True)
    check_against_oracle(ref, r, c, bf16=False)
    logp, ent = r[4].cpu(), r[5].cpu()
    # the same rows with the fully unavailable head left out of the row (its logits dropped): identical logp and entropy
    av = c["available"].reshape(T * n, -1)
    offs = np.concatenate([[0], np.cumsum(heads)[:-1]])
    for i in range(0, T * n, 7):
        h = (i // 7) % len(heads)
        assert not av[i, offs[h]:offs[h] + heads[h]].any()
        if len(heads) == 1:
            assert logp.view(-1)[i] == 0 and ent.view(-1)[i] == 0, f"row {i}: {logp.view(-1)[i]}, {ent.view(-1)[i]}"
        else:
            keep = [k for k in range(len(heads)) if k != h]
            z = torch.from_numpy(c["logits"].reshape(T * n, -1)[i])
            a = torch.from_numpy(c["actions"].reshape(T * n, -1)[i]).long()
            m = torch.from_numpy(av[i])
            parts = [M.logp_entropy_from_logits_ref(z[offs[k]:offs[k] + heads[k]], a[k:k + 1], (heads[k],),
                                                     available=m[offs[k]:offs[k] + heads[k]]) for k in keep]
            assert_close_ref(logp.view(-1)[i], sum(p[0] for p in parts)[0], what=f"logp of row {i}")
            assert_close_ref(ent.view(-1)[i], sum(p[1] for p in parts)[0], what=f"entropy of row {i}")
    # the rows whose chosen head-0 action is unavailable: logp about -1e10, finite (unless head 0 has no available action
    # at all in that row: then it adds 0)
    rows = [i for i in range(3, T * n, 11) if av[i, :heads[0]].any()]
    assert len(rows) > 20
    assert bool((logp.view(-1)[rows] < -1e9).all())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_unmasked_minus_inf_logits(ops, dtype):
    """Dead agents of an unmasked policy carry -inf logits: the entropy and every gradient stay finite (lp clamped at
    -FLT_MAX as Categorical.entropy clamps it), and a chosen -inf action gives logp -inf and ratio 0."""
    T, n, heads = 20, 37, (362,)
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_wide(heads, T, n, seed=8, bf16=dtype == torch.bfloat16)
    lg = c["logits"].reshape(T * n, -1)
    act = c["actions"].reshape(T * n)
    rng = np.random.default_rng(3)
    dead = rng.random(lg.shape) < 0.5
    dead[np.arange(T * n), act] = False
    lg[dead] = -np.inf
    chosen_inf = np.zeros(T * n, bool)
    chosen_inf[5::13] = True
    lg[chosen_inf, act[chosen_inf]] = -np.inf
    ref = oracle(c, hp_kw, dtype=torch.float64)
    g_logits, g_v, out, out32, logp, ent = run(ops, c, hp_kw, ref["norm_stats"], dtype=dtype, want_logp_entropy=True)
    for x, name in ((g_logits, "g_logits"), (g_v, "g_value"), (out, "out"), (ent, "entropy")):
        assert bool(torch.isfinite(x).all()), f"{name} has non-finite values"
    lp = logp.cpu().view(-1)
    assert bool(torch.isneginf(lp[torch.from_numpy(chosen_inf)]).all())
    assert bool(torch.isfinite(lp[torch.from_numpy(~chosen_inf)]).all())
    assert bool(torch.isneginf(ref["lp"].view(-1)[torch.from_numpy(chosen_inf)]).all())
    assert_close_ref(lp[torch.from_numpy(~chosen_inf)], ref["lp"].view(-1)[torch.from_numpy(~chosen_inf)], what="logp")
    assert_close_ref(ent.cpu(), ref["en"], what="entropy")
    out = out.cpu().numpy()
    for k, name in OUT_KEYS:
        assert_close_ref(out[k], ref[name], what=name)
    for k, name in STAT_KEYS:
        if name in ref["stats"]:
            assert_close_ref(out[k], ref["stats"][name], what=f"{name} (rows of ratio 0 included)")
    # dead logits get exactly 0 gradient; a chosen -inf action's row has ratio 0, so g_lp = 0 and its own logit gets 0 too
    dead_t = torch.from_numpy(dead).view(T, n, -1).cuda()
    assert bool((g_logits[dead_t] == 0).all())
    rows = np.nonzero(chosen_inf)[0]
    assert bool((g_logits.view(T * n, -1)[torch.from_numpy(rows).cuda(), torch.from_numpy(act[rows]).cuda()] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["lane_idx", "popart_dual_clip"])
@pytest.mark.parametrize("case", [CASES[i] for i in (0, 1, 4, 6, 7, 8)], ids=case_id)
def test_bf16_equals_float32_bit_for_bit(ops, case, config):
    """The bfloat16 launch on x and the float32 launch on x.float(): logp, entropy, out and out_f32 identical, g_logits and
    g_value the float32 launch's rounded to bfloat16 (the same element-to-lane assignment and grid for both types)."""
    heads, masked, p_av, T, n = case
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    c = make_wide(heads, T, n, seed=17, masked=masked, p_available=p_av, N=n + 5 if use_idx else None, bf16=True)
    _, ms = _popart() if config.startswith("popart") else (None, None)
    ns = oracle(c, hp_kw, dtype=torch.float32)["norm_stats"] if sum(heads) < 32000 else [T * n * 0.9, 3.0, T * n * 1.1]
    kw = dict(popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
    g16, gv16, o16, o3216, lp16, en16 = run(ops, c, hp_kw, ns, dtype=torch.bfloat16, **kw)
    g32, gv32, o32, o3232, lp32, en32 = run(ops, c, hp_kw, ns, dtype=torch.float32, **kw)
    assert torch.equal(lp16, lp32), "logp differs from the float32 launch's"
    assert torch.equal(en16, en32), "entropy differs from the float32 launch's"
    assert torch.equal(g16, g32.to(torch.bfloat16)), "g_logits is not the float32 launch's rounded to bfloat16"
    assert torch.equal(gv16, gv32.to(torch.bfloat16)), "g_value is not the float32 launch's rounded to bfloat16"
    assert torch.equal(o16, o32) and torch.equal(o3216, o3232), "out / out_f32 differ"


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["odd", "tiles", "agents"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("masked", [False, True], ids=["plain", "masked"])
@pytest.mark.parametrize("heads", [(362,), (100, 100, 60)], ids=ids)
def test_wide_pack_form_is_bit_identical_to_leaves(calls, shape, dtype, masked, heads):
    """The sample side from K2's pack (srl_ppo_loss_from_logits_wide_pack) against the five leaves it was written from, with
    the same lane_idx: every output bit for bit, deferred mode included, and the workspace slots clean afterwards."""
    from srl_b200 import ops
    T, n, lo, idx, pack, leaves, stats = _scan(shape)
    calls.clear()
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
    assert calls[:2] == [WIDE, WIDE + "_pack"] and calls[2] == WIDE + "_pack"


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True], ids=["plain", "masked"])
def test_wide_deterministic_deferred_and_unaligned(ops, masked):
    """Two launches are bit-identical and leave the workspace zero; a deferred launch + loss_finalize gives the immediate
    launch's bits; logits one element off a 16-byte boundary give the same bits."""
    T, n, heads = 16, 300, (362,)
    hp_kw = CONFIGS["popart_dual_clip"]
    c = make_wide(heads, T, n, seed=11, masked=masked, p_available=0.3)
    _, ms = _popart()
    ns = oracle(c, hp_kw, dtype=torch.float32)["norm_stats"]
    ws = ops.new_loss_workspace("cuda")
    a = run(ops, c, hp_kw, ns, popart_ms=ms, workspace=ws[0], want_logp_entropy=True)
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = run(ops, c, hp_kw, ns, popart_ms=ms, workspace=ws[0], want_logp_entropy=True)
    assert not ws.any()
    for x, y, name in zip(a, b, ("g_logits", "g_value", "out", "out_f32", "logp", "entropy")):
        assert torch.equal(x, y), f"{name} differs between two launches"
    g_logits, g_v, out_d, out32_d, _, _ = run(ops, c, hp_kw, ns, popart_ms=ms, workspace=ws[0], defer=True)
    assert out_d is None and out32_d is None
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    out32 = torch.zeros((1, 4), dtype=torch.float32, device="cuda")
    ops.loss_finalize(ws, out, out32)
    torch.cuda.synchronize()
    assert torch.equal(out[0], a[2]) and torch.equal(out32[0], a[3])
    assert torch.equal(g_logits, a[0]) and torch.equal(g_v, a[1])
    assert not torch.cat([ws[0, :4], ws[0, 32:]]).any(), "deferred mode + finalize left the workspace dirty"
    buf = torch.empty(c["logits"].size + 1, dtype=torch.float32, device="cuda")
    lg = buf[1:].view(c["logits"].shape)
    lg.copy_(torch.from_numpy(c["logits"]))
    assert lg.data_ptr() % 16 == 4
    u = run(ops, c, hp_kw, ns, popart_ms=ms, logits=lg, want_logp_entropy=True)
    for x, y, name in zip(u, a, ("g_logits", "g_value", "out", "out_f32", "logp", "entropy")):
        assert torch.equal(x, y), f"{name} differs with the logits unaligned"


@pytest.mark.gpu
def test_routing_by_row_width(monkeypatch):
    """Rows K4b takes (sum K <= 199, <= 159 with a mask) still go to the entries they went to; wider rows go to the _wide
    entries, the pack form to _wide_pack."""
    from srl_b200 import ops
    called = []
    monkeypatch.setattr(ops._lib, "call", lambda fn, *a: called.append((fn, a[1] if "wide" in fn or "pack" in fn else None)))
    T, n = 2, 8
    f = lambda *s: torch.zeros(s, device="cuda")
    leaves = dict(old_logp=f(T, n), old_value=f(T, n), ret=f(T, n), adv=f(T, n),
                  on_reset_next=torch.zeros(T, n, dtype=torch.uint8, device="cuda"))
    none = dict(old_logp=None, old_value=None, ret=None, adv=None, on_reset_next=None)
    stats = dict(norm_stats=torch.ones(3, dtype=torch.float64, device="cuda"), hyper=ops.LossHyper())
    pack = ops.new_pack(T + 1, n, "cuda")
    for dt, sfx, eb in ((torch.float32, "", 4), (torch.bfloat16, "_bf16", 2)):
        for K, masked, want in ((199, False, "srl_ppo_loss_from_logits" + sfx),
                                (159, True, "srl_ppo_loss_from_logits_masked" + sfx), (200, False, WIDE), (160, True, WIDE),
                                (262144, False, WIDE)):
            act = torch.zeros(T, n, 1, dtype=torch.int32, device="cuda")
            av = dict(available=f(T, n, K) + 1) if masked else {}
            called.clear()
            ops.ppo_loss_from_logits(f(T, n, K).to(dt), act, [K], f(T, n).to(dt), **leaves, **stats, **av)
            assert called == [(want, eb if want == WIDE else None)], (K, masked, dt, called)
            called.clear()
            ops.ppo_loss_from_logits(f(T, n, K).to(dt), act, [K], f(T, n).to(dt), **none, pack=pack, **stats, **av)
            wide = K > (159 if masked else 199)
            assert called == [(WIDE + "_pack" if wide else "srl_ppo_loss_from_logits_pack", eb)], (K, masked, dt, called)


@pytest.mark.gpu
def test_categorical_autograd_function_at_362_actions(ops):
    """PPOCategoricalLossFunction on (362,) logits: logits.grad and v_pred.grad match the float64 oracle's."""
    T, n, heads = 20, 37, (362,)
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_wide(heads, T, n, seed=23)
    ref = oracle(c, hp_kw)
    d = lambda k: torch.from_numpy(np.ascontiguousarray(c[k])).cuda()
    z = d("logits").requires_grad_(True)
    v = d("v_pred").requires_grad_(True)
    ns = torch.tensor(ref["norm_stats"], dtype=torch.float64, device="cuda")
    T_ = c["T"]
    loss, out = ops.PPOCategoricalLossFunction.apply(z, None, d("actions"), heads, v, d("old_logp")[:T_], d("value")[:T_],
                                                     d("ret")[:T_], d("adv")[:T_], d("on_reset")[1:T_ + 1], ns, None, None,
                                                     None, ops.LossHyper(**hp_kw))
    (2.0 * loss).backward()
    assert_close_ref(loss.item(), ref["loss"], what="loss")
    assert_grad_close(z.grad.cpu(), 2.0 * ref["g_logits"], ref["mask_sum"], what="logits.grad")
    assert_grad_close(v.grad.cpu(), 2.0 * ref["g_value"], ref["mask_sum"], what="v_pred.grad")


# ---- the trainer -------------------------------------------------------------------------------------------------------
class MaskedWide(TinyActorCriticPolicy):
    """Categorical heads of the given widths with SMAC's availability mask in obs.avail: target="ppo" builds the masked
    Categoricals in torch, target="ppo_head" returns logits + mask."""
    ppo_head = True

    def __init__(self, device, heads, seed=3):
        super().__init__(OBS_DIM, sum(heads), device=device, seed=seed)
        self.heads = tuple(heads)

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kwargs):
        logits, value = self._net(sample.obs.vec[burn_in_steps:])
        avail = sample.obs.avail[burn_in_steps:]
        action = sample.action.x[burn_in_steps:]
        if target == "ppo_head":
            return api.PPOHeadAnalyzedResult(state_values=value, action=action, logits=logits, head_sizes=self.heads,
                                             available=avail)
        lp, en = M.logp_entropy_from_logits_ref(logits, action.long(), self.heads, available=avail)
        return SampleAnalyzedResult(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                                    new_action_log_probs=lp, state_values=value, entropy=en)


def wide_sample(cfg, seed, heads, masked):
    s = synth.make_sample_scalars(cfg, seed)
    rng = np.random.default_rng(seed + 99)
    lead = s["value"].shape[:-1]
    obs = dict(vec=rng.standard_normal(lead + (OBS_DIM,)).astype(np.float32))
    x = np.stack([rng.integers(0, K, lead) for K in heads], -1).astype(np.float32)
    if masked:
        avail = rng.random(lead + (sum(heads),)) < 0.3
        off = 0
        for k, K in enumerate(heads):  # the actors only took available actions
            np.put_along_axis(avail[..., off:off + K], x[..., k:k + 1].astype(np.int64), True, -1)
            off += K
        obs["avail"] = avail.astype(np.float32)
    # near the uniform policy's log-prob, so that the ratios straddle the clip range
    p_av = 0.3 if masked else 1.0
    s["old_logp"] = rng.normal(-float(np.sum(np.log(p_av * np.asarray(heads) + (1 - p_av)))), 0.3,
                               s["old_logp"].shape).astype(np.float32)
    info = NamedArray(episode_return=rng.standard_normal(lead + (1,)).astype(np.float32))
    info_mask = (rng.random(lead + (1,)) < 0.1).astype(np.float32)
    return api.SampleBatch(obs=NamedArray(**obs), on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"],
                           action=NamedArray(x=x), reward=s["reward"], info=info, info_mask=info_mask,
                           analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))


TRAIN_KW = dict(clip_value=True, value_loss="mse", ppo_epochs=2, num_minibatches=4, shuffle_seed=5, optimizer="sgd",
                optimizer_config=dict(lr=0.05))
POLICIES = {"k362": ((362,), False), "masked_300x64": ((300, 64), True)}


def _policy(kind, device):
    heads, masked = POLICIES[kind]
    return MaskedWide(device, heads) if masked else HeadTiny(OBS_DIM, heads[0], device=device, seed=3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(POLICIES))
def test_wide_head_policy_matches_reference_restatement(kind, calls):
    """MultiAgentPPOB200 trains a ppo_head policy with wide heads through K4b-wide reading K2's pack (4 minibatches); the CPU
    restatement drives the same policy through target="ppo".  Statistics and parameters agree to 2e-5."""
    from oracle.ref_trainer import RefPPOTrainer
    from srl_b200.trainer import MultiAgentPPOB200
    heads, masked = POLICIES[kind]
    cfg = synth.PathConfig("t_wide", T=8, B=16, p_end=0.1)
    kw = dict(TRAIN_KW, discount_rate=cfg.gamma)
    pol_gpu, pol_cpu = _policy(kind, "cuda:0"), _policy(kind, "cpu")
    mine, ref = MultiAgentPPOB200(pol_gpu, prefetch=False, **kw), RefPPOTrainer(pol_cpu, **kw)
    assert mine.ppo_head
    for it in range(3):
        got = mine.step(wide_sample(cfg, 10 + it, heads, masked))
        want_stats, want_version = ref.step(wide_sample(cfg, 10 + it, heads, masked))
        assert got.step == want_version == it
        for k, v in want_stats.items():
            assert_close_ref(got.stats[k], v, tol=2e-5, what=f"stat {k} at step {it}")
    for (n1, p1), (n2, p2) in zip(pol_gpu.net.state_dict().items(), pol_cpu.net.state_dict().items()):
        assert n1 == n2
        assert_close_ref(p1.cpu(), p2, tol=2e-5, what=f"parameter {n1}")
    assert WIDE + "_pack" in calls and "srl_ppo_loss_from_logits_pack" not in calls


@pytest.mark.gpu
def test_autocast_wide_head_reaches_the_wide_pack_entry_as_bfloat16(ops, monkeypatch):
    """Under torch.autocast(bfloat16) the 362-action head's bfloat16 logits and value reach srl_ppo_loss_from_logits_wide_pack
    as they are (elem_bytes 2, no cast), and the step's statistics stay near the float32 step's."""
    from srl_b200.trainer import MultiAgentPPOB200
    seen = []
    orig = ops._lib.call

    def spy(fn, *a):
        if fn.startswith(WIDE):
            seen.append((fn, a[1]))
        return orig(fn, *a)
    monkeypatch.setattr(ops._lib, "call", spy)
    cfg = synth.PathConfig("t_wide_bf16", T=16, B=64, p_end=0.1)
    kw = dict(TRAIN_KW, discount_rate=cfg.gamma, optimizer_config=dict(lr=1e-3))
    stats = {}
    for mode in ("f32", "bf16"):
        tr = MultiAgentPPOB200(_policy("k362", "cuda:0"), prefetch=False, **kw)
        seen.clear()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16")):
            stats[mode] = tr.step(wide_sample(cfg, 20, (362,), False)).stats
            stats[mode] = tr.step(wide_sample(cfg, 21, (362,), False)).stats
        want = 2 if mode == "bf16" else 4
        assert seen and all(s == (WIDE + "_pack", want) for s in seen), seen
    for k, v in stats["f32"].items():
        assert_close_ref(stats["bf16"][k], v, tol=1e-2, what=f"bf16 stat {k}")


# ---- host-side argument checks (no GPU) ----------------------------------------------------------------------------------
def _wide_args(heads=(5,), elem_bytes=4, null=None, ws=None, pack=False, pack_ptr=4096, pack_lanes=8, pack_row_lo=0):
    """Arguments of the two wide entries with fake, non-null device pointers: every call below is refused before any is
    used.  `null` names a pointer argument to pass as NULL."""
    P = 4096
    T, n = 2, 8
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)
    hs = (ctypes.c_int32 * max(1, len(heads)))(*heads)
    ptr = lambda name: None if null == name else P
    ws_bytes = _lib.load_library().srl_ppo_loss_workspace_bytes(T, n) if ws is None else ws
    head = (ptr("logits"), elem_bytes, None, ptr("action"), hs, len(heads), ptr("v_pred"))
    tail = (None, T, n, ptr("norm_stats"), ptr("local_stats"), None, ctypes.byref(hc), ptr("g_logits"), ptr("g_value"), None,
            None, P, None, ptr("workspace"), ws_bytes, None)
    if pack:
        return head + (pack_ptr, pack_lanes, pack_row_lo) + tail
    return head + (ptr("old_logp"), None, ptr("ret"), ptr("adv"), ptr("on_reset_next"), n) + tail


@pytest.mark.parametrize("pack", [False, True], ids=["leaves", "pack"])
@pytest.mark.parametrize("bad,rc,match", [
    (dict(null="logits"), 1, "null pointer"),
    (dict(null="g_logits"), 1, "null pointer"),
    (dict(null="workspace"), 1, "null pointer"),
    (dict(heads=()), 1, "heads=0 outside [1, 8]"),
    (dict(heads=(1,) * 9), 1, "heads=9 outside [1, 8]"),
    (dict(heads=(300, 0, 4)), 1, "head 1 has no actions"),
    (dict(elem_bytes=8), 1, "elem_bytes=8, need 4 (float32) or 2 (bfloat16)"),
    (dict(ws=64), 1, "workspace too small"),
    (dict(heads=(262144, 1)), 2, "sum K = 262145 too wide (max 262144)"),
])
def test_wide_entries_refuse_bad_arguments(pack, bad, rc, match):
    build.build()
    lib = _lib.load_library()
    name = WIDE + ("_pack" if pack else "")
    got = getattr(lib, name)(*_wide_args(pack=pack, **bad))
    msg = lib.srl_last_error().decode()
    assert got == rc and msg.startswith(name + ":") and match in msg, (got, msg)


@pytest.mark.parametrize("bad,match", [
    (dict(pack_ptr=None), "pack is null"),
    (dict(pack_ptr=4096 + 8), "16-byte aligned"),
    (dict(pack_row_lo=-1), "pack_row_lo=-1"),
    (dict(pack_lanes=7), "pack_lanes=7 < n=8"),
    (dict(elem_bytes=0), "elem_bytes=0"),
])
def test_wide_pack_entry_refuses_bad_packs(bad, match):
    build.build()
    lib = _lib.load_library()
    assert lib.srl_ppo_loss_from_logits_wide_pack(*_wide_args(pack=True, **bad)) == 1
    msg = lib.srl_last_error().decode()
    assert msg.startswith(WIDE + "_pack:") and match in msg, msg


def test_wide_limit_and_abi():
    build.build()
    lib = _lib.load_library()
    assert lib.srl_abi_version() == _lib.ABI_VERSION == 12
    assert _lib.SRL_K4B_WIDE_MAX_SUM_K == 262144
    # the largest row is accepted by the host checks (refused later only for the fake workspace size)
    assert lib.srl_ppo_loss_from_logits_wide(*_wide_args(heads=(131072, 131072), ws=64)) == 1
    assert "workspace too small" in lib.srl_last_error().decode()
