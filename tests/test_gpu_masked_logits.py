"""K4b with an availability mask (srl_ppo_loss_from_logits_masked, ops.ppo_loss_from_logits(available=...),
ops.PPOCategoricalLossFunction): the reference's masked categorical policy (actor_critic_policy.py:135-136,
logits.masked_fill(available == 0, -1e10) before the per-head Categorical) feeding the oracle's loss, with autograd to the
logits.  Bars as in test_gpu_parity.py: 1e-5 * max(1, |ref|), gradients on the g * sum(mask) scale.  The host-side
argument checks run without a GPU."""
import ctypes
import dataclasses

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from srl_b200 import _lib, build, synth
from tests.test_gpu_gaussian import away_from_clip_edges
from tests.util import assert_close_ref, assert_grad_close

OUT_KEYS = ((0, "loss"), (1, "policy_loss"), (2, "value_loss"), (3, "entropy_loss"))
STAT_KEYS = ((4, "advantage"), (5, "importance_weight"), (6, "clip_ratio"), (7, "value_targets"), (8, "denorm_value"))

# (18,): one head in registers; (36,): SMAC 27m, the row walk; (11, 11, 11, 2, 2): hide-and-seek; (4, 33, 7, 32): both
# paths in one row; (27, 100, 32): sum K = 159, the largest a mask allows, where e_k is not cached (CACHE_E off)
HEAD_SETS = [(18,), (36,), (11, 11, 11, 2, 2), (4, 33, 7, 32), (27, 100, 32)]

CONFIGS = {
    "huber_clip_value": dict(dual_clip=False, clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0),
                             entropy_bonus_weight=0.05),
    "lane_idx": dict(clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0), entropy_bonus_weight=0.05),
    # cfg3 (SMAC 27m): PopArt targets, dual clip
    "popart_dual_clip": dict(dual_clip=True, c_clip=3.0, value_loss="huber", value_loss_config=dict(delta=10.0),
                             value_loss_weight=1.0, entropy_bonus_weight=0.05),
}


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()  # must load the in-tree .so, loudly
    return _ops


def make_case(heads, T, n, p_unavailable, seed, N=None, odd_rows=True):
    """Seeded inputs of one minibatch: logits, availability and actions [T, n, .] from synth; with odd_rows every 7th
    transition gets a head with no available action, every 11th its chosen action of head 0 made unavailable (padded rows
    can hold one).  Sample side [T + 1, N]; old_logp is the masked head's log-prob perturbed so that ratios straddle the clip range (a
    transition whose chosen action is unavailable keeps an ordinary old_logp: its ratio is 0)."""
    N = n if N is None else N
    cfg = dataclasses.replace(synth.CONFIGS["cfg3_smac_27m"], num_actions=tuple(heads))
    logits, actions, avail = synth.make_masked_logits_actions(cfg, (T, n), seed=seed, p_unavailable=p_unavailable)
    rng = np.random.default_rng(seed)
    flat_avail = avail.reshape(T * n, -1)
    flat_act = actions.reshape(T * n, -1)
    offs = np.concatenate([[0], np.cumsum(heads)[:-1]])
    for i in range(0, T * n if odd_rows else 0, 7):
        h = (i // 7) % len(heads)
        flat_avail[i, offs[h]:offs[h] + heads[h]] = 0
    chosen_masked = np.zeros(T * n, bool)
    chosen_masked[3::11] = odd_rows
    flat_avail[chosen_masked, flat_act[chosen_masked, 0]] = 0
    on_reset = (rng.random((T + 1, N)) < 0.1).astype(np.uint8)
    f32 = lambda x: np.asarray(x, dtype=np.float32)
    value = f32(rng.standard_normal((T + 1, N)))
    ret = f32(rng.standard_normal((T + 1, N)) * 2.0)
    adv = f32(rng.standard_normal((T + 1, N)))
    lane_idx = np.arange(n, dtype=np.int32) if N == n else rng.permutation(N)[:n].astype(np.int32)
    with torch.no_grad():
        lp, _ = M.logp_entropy_from_logits_ref(torch.from_numpy(logits), torch.from_numpy(actions).long(), heads,
                                               available=torch.from_numpy(avail))
    lp = lp[..., 0].numpy().astype(np.float64)
    behaviour = np.where(chosen_masked.reshape(T, n), -1.5, lp)
    old_logp = np.zeros((T + 1, N), np.float32)
    old_logp[:T, lane_idx] = away_from_clip_edges(lp, behaviour + 0.15 * rng.standard_normal((T, n)))
    v_pred = f32(value[:T, lane_idx] + 0.1 * rng.standard_normal((T, n)))
    return dict(logits=logits, actions=actions, available=avail, heads=tuple(heads), on_reset=on_reset, value=value,
                ret=ret, adv=adv, old_logp=old_logp, v_pred=v_pred, lane_idx=lane_idx, T=T, n=n, N=N)


def _popart():
    pa = M.RunningMeanStdRef((1,), beta=0.999)
    pa.update(torch.randn(64, 1, generator=torch.Generator().manual_seed(1)) * 2 + 1)
    m_, s_ = pa.mean_std()
    return pa, [m_.item(), s_.item()]


def oracle(c, hp_kw, popart=None):
    """masked_fill + Categorical per head (the oracle's logp_entropy_from_logits_ref) -> the oracle's loss, autograd back
    to the logits, in float32 on the CPU as the reference trains."""
    T = c["T"]
    take = lambda x: torch.from_numpy(np.ascontiguousarray(x[:T][:, c["lane_idx"]]))
    zl = torch.from_numpy(c["logits"]).requires_grad_(True)
    lp, en = M.logp_entropy_from_logits_ref(zl, torch.from_numpy(c["actions"]).long(), c["heads"],
                                            available=torch.from_numpy(c["available"]))
    mask = 1 - take(c["on_reset"][1:]).float()
    adv = take(c["adv"])
    res = M.ppo_loss_ref(lp[..., 0].detach(), take(c["old_logp"]), torch.from_numpy(c["v_pred"]), take(c["value"]),
                         take(c["ret"]), adv, en[..., 0].detach(), mask, M.LossHyper(**hp_kw), popart=popart)
    (lp[..., 0] * res["g_logp"]).sum().add((en[..., 0] * res["g_entropy"]).sum()).backward()
    res.update(lp=lp.detach()[..., 0], en=en.detach()[..., 0], g_logits=zl.grad, mask_sum=float(mask.sum()),
               norm_stats=[float(x) for x in M.masked_sums_ref(adv, mask)] + [0.0] * 5)
    return res


def run(ops, c, hp_kw, norm_stats, popart_ms=None, use_lane_idx=False, available="dense", logits=None, **kw):
    """One launch; `available` = "dense" (c's uint8 mask), None (the unmasked entry) or a CUDA tensor."""
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    if isinstance(available, str):
        available = d(c["available"])
    r = ops.ppo_loss_from_logits(
        d(c["logits"]) if logits is None else logits, d(c["actions"]), c["heads"], d(c["v_pred"]), d(c["old_logp"])[:T],
        d(c["value"])[:T], d(c["ret"])[:T], d(c["adv"])[:T], d(c["on_reset"])[1:T + 1],
        d(np.asarray(norm_stats, dtype=np.float64)), ops.LossHyper(**hp_kw),
        popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=d(c["lane_idx"]) if use_lane_idx else None, available=available, **kw)
    torch.cuda.synchronize()
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("p_unavailable", [0.3, 0.9])
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("heads", HEAD_SETS, ids=lambda h: "x".join(map(str, h)))
def test_masked_logits_match_oracle(ops, heads, config, p_unavailable):
    """T = 20, n = 37: two full tiles of 256 transitions (mask brought in with the logits' bulk copy) and a partial one
    (element-wise staging).  Rows with a head of no available action and rows whose chosen action is unavailable are in
    every case; g_logits is exactly 0 wherever the mask is 0."""
    T, n = 20, 37
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    c = make_case(heads, T, n, p_unavailable, seed=sum(heads) + int(10 * p_unavailable), N=53 if use_idx else None)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    ref = oracle(c, hp_kw, popart=pa)
    g_logits, g_v, out, out32, logp, ent = run(ops, c, hp_kw, ref["norm_stats"], popart_ms=ms, use_lane_idx=use_idx,
                                               want_logp_entropy=True)
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
    assert_grad_close(g_v.cpu(), ref["g_value"], msum, what="g_value")
    assert_grad_close(g_logits.cpu(), ref["g_logits"], msum, what="g_logits")
    unavailable = torch.from_numpy(c["available"]) == 0
    assert bool((g_logits.cpu()[unavailable] == 0).all()), "non-zero gradient at an unavailable logit"


@pytest.mark.gpu
@pytest.mark.parametrize("heads", [(36,), (4, 33, 7, 32)], ids=["36", "4x33x7x32"])
def test_masked_logits_unaligned_pointers_take_the_staging_path(ops, heads):
    """Logits one float off a 16-byte boundary, or the mask one byte off, are staged element by element in every tile:
    the results equal the aligned launch's bit for bit."""
    T, n = 20, 37
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_case(heads, T, n, 0.3, seed=3)
    ns = oracle(c, hp_kw)["norm_stats"]
    base = run(ops, c, hp_kw, ns, want_logp_entropy=True)
    buf = torch.empty(c["logits"].size + 1, dtype=torch.float32, device="cuda")
    lg = buf[1:].view(c["logits"].shape)
    lg.copy_(torch.from_numpy(c["logits"]))
    mb = torch.empty(c["available"].size + 1, dtype=torch.uint8, device="cuda")
    mk = mb[1:].view(c["available"].shape)
    mk.copy_(torch.from_numpy(c["available"]))
    assert lg.data_ptr() % 16 == 4 and mk.data_ptr() % 16 == 1
    for kw in (dict(logits=lg), dict(available=mk)):
        r = run(ops, c, hp_kw, ns, want_logp_entropy=True, **kw)
        for x, y, name in zip(r, base, ("g_logits", "g_value", "out", "out_f32", "logp", "entropy")):
            assert torch.equal(x, y), f"{name} differs with {list(kw)[0]} unaligned"


@pytest.mark.gpu
@pytest.mark.parametrize("heads", [(18,), (36,), (11, 11, 11, 2, 2), (4, 33, 7, 32)], ids=lambda h: "x".join(map(str, h)))
def test_all_ones_mask_equals_the_unmasked_entry(ops, heads):
    """Every action available (as uint8, bool and float32): g_logits, g_value, logp and entropy equal the unmasked
    launch's bit for bit.  `out` agrees to 1e-12: its partial rows are folded in grid order, and the grid follows the
    resident CTAs, which the mask's shared memory may change."""
    T, n = 64, 300
    hp_kw = CONFIGS["popart_dual_clip"]
    c = make_case(heads, T, n, 0.3, seed=21)
    _, ms = _popart()
    ns = oracle(c, hp_kw)["norm_stats"]
    plain = run(ops, c, hp_kw, ns, popart_ms=ms, available=None, want_logp_entropy=True)
    ones = torch.ones(c["logits"].shape, dtype=torch.uint8, device="cuda")
    for mask in (ones, ones.bool(), ones.float()):
        r = run(ops, c, hp_kw, ns, popart_ms=ms, available=mask, want_logp_entropy=True)
        for k, name in ((0, "g_logits"), (1, "g_value"), (4, "logp"), (5, "entropy")):
            assert torch.equal(r[k], plain[k]), f"{name} differs from the unmasked entry ({mask.dtype} mask)"
        assert_close_ref(r[2].cpu(), plain[2].cpu(), tol=1e-12, what=f"out ({mask.dtype} mask)")
        assert_close_ref(r[3].cpu(), plain[3].cpu(), tol=1e-6, what=f"out_f32 ({mask.dtype} mask)")


@pytest.mark.gpu
def test_masked_logits_deterministic_and_deferred(ops):
    """Two launches are bit-identical and leave the workspace zero; a deferred launch followed by loss_finalize gives the
    immediate launch's bits (the slot keeps only the bytes 4-31 a deferred launch hands to the finaliser)."""
    T, n = 128, 1000
    hp_kw = CONFIGS["popart_dual_clip"]
    c = make_case((36,), T, n, 0.3, seed=11)
    _, ms = _popart()
    ns = oracle(c, hp_kw)["norm_stats"]
    ws = ops.new_loss_workspace("cuda")
    a = run(ops, c, hp_kw, ns, popart_ms=ms, workspace=ws[0])
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = run(ops, c, hp_kw, ns, popart_ms=ms, workspace=ws[0])
    assert not ws.any()
    for x, y, name in zip(a[:4], b[:4], ("g_logits", "g_value", "out", "out_f32")):
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


@pytest.mark.gpu
def test_categorical_autograd_function_trains_a_masked_policy(ops):
    """A SMAC-shaped policy: nn.Linear logits (36 actions) and value heads, actions sampled from the masked distribution,
    the loss through PPOCategoricalLossFunction, then loss.backward().  Every parameter gradient matches the same network's
    in float64 through masked_fill + Categorical and the oracle's loss."""
    import copy
    T, n, F, heads = 24, 300, 11, (36,)
    torch.manual_seed(0)

    class Policy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.pi = torch.nn.Linear(F, sum(heads))
            self.v = torch.nn.Linear(F, 1)

    pol = Policy()
    ref_pol = copy.deepcopy(pol)
    pol = pol.cuda()
    # no head without an available action here: in float64 its log-sum-exp, -1e10 + log K, does not round to -1e10 as
    # it does in float32, so the float64 oracle would see a uniform head where float32 torch (and the kernel) see none
    c = make_case(heads, T, n, 0.3, seed=5, odd_rows=False)
    avail = torch.from_numpy(c["available"])
    obs = torch.randn(T, n, F)
    with torch.no_grad():
        z0 = ref_pol.pi(obs).masked_fill(avail == 0, -1e10)
        act = torch.distributions.Categorical(logits=z0).sample().unsqueeze(-1)
        c["actions"] = act.int().numpy()
        lp0, _ = M.logp_entropy_from_logits_ref(ref_pol.pi(obs).double(), act, heads, available=avail)
        lp0 = lp0[..., 0].numpy()
        c["old_logp"][:T] = away_from_clip_edges(lp0, lp0 + 0.15 * np.random.default_rng(1).standard_normal((T, n)))
    hp_kw = CONFIGS["huber_clip_value"]
    # oracle: the same network on the CPU, in float64 (its parameter gradients are sums over T * n transitions)
    ref_pol = ref_pol.double()
    z_r, v_r = ref_pol.pi(obs.double()), ref_pol.v(obs.double())[..., 0]
    lp, en = M.logp_entropy_from_logits_ref(z_r, act, heads, available=avail)
    lp, en = lp[..., 0], en[..., 0]
    mask = 1 - torch.from_numpy(c["on_reset"][1:T + 1]).float()
    t = lambda k: torch.from_numpy(c[k][:T])
    res = M.ppo_loss_ref(lp.detach().float(), t("old_logp"), v_r.detach().float(), t("value"), t("ret"), t("adv"),
                         en.detach().float(), mask, M.LossHyper(**hp_kw))
    (lp * res["g_logp"].double()).sum().add((en * res["g_entropy"].double()).sum()).add(
        (v_r * res["g_value"].double()).sum()).backward()
    ns = torch.tensor([float(x) for x in M.masked_sums_ref(t("adv"), mask)] + [0.0] * 5, dtype=torch.float64).cuda()
    # the fused path
    d = lambda k: torch.from_numpy(np.ascontiguousarray(c[k])).cuda()
    obs_d = obs.cuda()
    loss, out = ops.PPOCategoricalLossFunction.apply(pol.pi(obs_d), d("available"), d("actions"), heads, pol.v(obs_d)[..., 0],
                                                     d("old_logp")[:T], d("value")[:T], d("ret")[:T], d("adv")[:T],
                                                     d("on_reset")[1:T + 1], ns, None, None, None, ops.LossHyper(**hp_kw))
    loss.backward()
    torch.cuda.synchronize()
    msum = float(mask.sum())
    assert_close_ref(loss.item(), res["loss"], what="loss")
    for (name, p), (_, q) in zip(pol.named_parameters(), ref_pol.named_parameters()):
        assert p.grad is not None, f"{name} received no gradient"
        # a weight's gradient is a sum over the 7200 transitions of terms of either sign, compared on the scale of its
        # tensor's largest element (as in test_gpu_gaussian.py); the head's gradients are pinned element by element above
        scale = msum / max(1.0, float(q.grad.abs().max()) * msum)
        assert_close_ref(p.grad.cpu().double() * scale, q.grad * scale, what=f"d loss / d {name}")


def test_masked_logits_host_side_argument_checks():
    """Rejected on the host before any CUDA call, with a status and a message -- no GPU needed.  The non-null device
    pointers are never dereferenced."""
    build.build()
    lib = _lib.load_library()
    T, n = 4, 8
    fake = 256
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)

    def call(heads, available=fake):
        hs = (ctypes.c_int32 * len(heads))(*heads)
        rc = lib.srl_ppo_loss_from_logits_masked(fake, available, fake, hs, len(heads), fake, fake, fake, fake, fake, fake,
                                                 n, None, T, n, fake, fake, None, ctypes.byref(hc), fake, fake, None, None,
                                                 fake, None, fake, lib.srl_ppo_loss_workspace_bytes(T, n), None)
        return rc, lib.srl_last_error().decode()

    rc, msg = call((36,), available=None)
    assert rc == 1 and "null pointer available" in msg, msg
    too_wide = (100, _lib.SRL_K4B_MAX_SUM_K_MASKED + 1 - 100)
    rc, msg = call(too_wide)
    assert rc == 2 and f"sum K = {sum(too_wide)} too wide (max {_lib.SRL_K4B_MAX_SUM_K_MASKED})" in msg, msg
    rc, msg = call((0, 5))
    assert rc == 1 and "srl_ppo_loss_from_logits_masked: head 0 has no actions" in msg, msg


def test_masked_logits_ops_argument_checks():
    """ops.ppo_loss_from_logits refuses a mask of another dtype, another shape, a stride-0 expand or a non-contiguous
    view with a ValueError naming `available` (checked before anything touches the device)."""
    from srl_b200 import ops
    T, n, K = 3, 5, 36
    logits = torch.zeros(T, n, K)
    rest = dict(action=torch.zeros(T, n, 1, dtype=torch.int32), head_sizes=(K,), v_pred=torch.zeros(T, n),
                old_logp=None, old_value=None, ret=None, adv=None, on_reset_next=None, norm_stats=None,
                hyper=ops.LossHyper())
    bad = [torch.ones(T, n, K, dtype=torch.int32), torch.ones(T, n, K - 1, dtype=torch.uint8),
           torch.ones(1, 1, K, dtype=torch.uint8).expand(T, n, K), torch.ones(T, K, n, dtype=torch.uint8).transpose(1, 2),
           torch.ones(T, n, K)]  # the last is valid but on the CPU
    for mask, what in zip(bad, ("dtype", "shape", "stride-0", "contiguous", "CUDA")):
        with pytest.raises(ValueError, match="available") as e:
            ops.ppo_loss_from_logits(logits, available=mask, **rest)
        assert what in str(e.value), str(e.value)
