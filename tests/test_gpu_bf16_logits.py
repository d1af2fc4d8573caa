"""K4b with a bfloat16 policy side (srl_ppo_loss_from_logits_bf16, srl_ppo_loss_from_logits_masked_bf16,
ops.ppo_loss_from_logits on bfloat16 logits and value, ops.PPOCategoricalLossFunction under torch.autocast).  The logits and
values of every case are bfloat16 numbers; the float32 entry and the oracle see them widened, which is exact.  The bfloat16
entries compute in float32 and round each gradient once, so where both entries cache the exponentials alike their results
are the float32 entry's bit for bit, with the gradients rounded.  The host-side argument checks run without a GPU."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from srl_b200 import _lib, build
from tests.test_gpu_gaussian import away_from_clip_edges
from tests.test_gpu_masked_logits import CONFIGS, HEAD_SETS, OUT_KEYS, STAT_KEYS, _popart, make_case, oracle
from tests.util import assert_close_ref

# (60, 60): sum K = 120, unmasked, where the bfloat16 entry keeps e_k in shared memory (up to 133) and the float32 entry
# does not (up to 99); the two entries take different paths there, so it is compared with the oracle only
PARITY_HEAD_SETS = HEAD_SETS + [(60, 60)]
ids = lambda h: "x".join(map(str, h))


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


def bf16_case(heads, T, n, p_unavailable, seed, masked=True, N=None):
    """make_case with bfloat16 logits and v_pred; old_logp kept away from the clip edges for the rounded logits' log-prob.
    Unmasked: every action available and no row with an unavailable chosen action."""
    c = make_case(heads, T, n, p_unavailable, seed, N=N, odd_rows=masked)
    if not masked:
        c["available"] = np.ones_like(c["available"])
    c["logits"], c["v_pred"] = bf16_exact(c["logits"]), bf16_exact(c["v_pred"])
    with torch.no_grad():
        lp, _ = M.logp_entropy_from_logits_ref(torch.from_numpy(c["logits"]), torch.from_numpy(c["actions"]).long(), heads,
                                               available=torch.from_numpy(c["available"]))
    idx = c["lane_idx"]
    c["old_logp"][:T, idx] = away_from_clip_edges(lp[..., 0].numpy().astype(np.float64), c["old_logp"][:T, idx])
    return c


def launch(ops, c, hp_kw, norm_stats, dtype, masked=True, popart_ms=None, use_lane_idx=False, logits=None,
           available=None, **kw):
    """One launch with the policy side in `dtype` (c's values are bfloat16 numbers, so either dtype holds them exactly)."""
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    if available is None and masked:
        available = d(c["available"])
    r = ops.ppo_loss_from_logits(
        d(c["logits"]).to(dtype) if logits is None else logits, d(c["actions"]), c["heads"], d(c["v_pred"]).to(dtype),
        d(c["old_logp"])[:T], d(c["value"])[:T], d(c["ret"])[:T], d(c["adv"])[:T], d(c["on_reset"])[1:T + 1],
        d(np.asarray(norm_stats, dtype=np.float64)), ops.LossHyper(**hp_kw),
        popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=d(c["lane_idx"]) if use_lane_idx else None, available=available, **kw)
    torch.cuda.synchronize()
    return r


def assert_bf16_grad_close(g, ref, mask_sum, what):
    """A bfloat16 gradient against the oracle's float32 one, on the g * sum(mask) scale: within half a bfloat16 ulp (of the
    larger magnitude: the rounding of a value near a power of two) plus the usual 1e-5 * max(1, |ref|)."""
    x = g.float().cpu().numpy().astype(np.float64)
    r = ref.numpy().astype(np.float64)
    mag = np.maximum(np.abs(x), np.abs(r))  # the ulp of the unscaled gradient, the number that was rounded
    half_ulp = np.where(mag > 0, np.exp2(np.floor(np.log2(np.where(mag > 0, mag, 1.0))) - 8), 0.0) * mask_sum
    x, r = x * mask_sum, r * mask_sum
    err = np.abs(x - r)
    bad = ~(err <= half_ulp + 1e-5 * np.maximum(1.0, np.abs(r)))
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err - half_ulp, 0)), err.shape)
        raise AssertionError(f"{what}: {bad.sum()} of {bad.size} elements outside half a bfloat16 ulp + 1e-5; worst at {i}: "
                             f"got {x[i]!r}, reference {r[i]!r}")


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [True, False], ids=["masked", "unmasked"])
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("heads", HEAD_SETS, ids=ids)
def test_bf16_entry_equals_the_float32_entry_bit_for_bit(ops, heads, config, masked):
    """The bfloat16 entry on x and the float32 entry on x.float() (T = 20, n = 37: two bulk-copied tiles and a staged one):
    logp and entropy are identical, g_logits and g_value are the float32 entry's rounded to bfloat16."""
    T, n = 20, 37
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    c = bf16_case(heads, T, n, 0.3, seed=sum(heads) + 7, masked=masked, N=53 if use_idx else None)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    ns = oracle(c, hp_kw, popart=pa)["norm_stats"]
    kw = dict(masked=masked, popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
    g16, gv16, _, _, lp16, en16 = launch(ops, c, hp_kw, ns, torch.bfloat16, **kw)
    g32, gv32, _, _, lp32, en32 = launch(ops, c, hp_kw, ns, torch.float32, **kw)
    assert g16.dtype == gv16.dtype == torch.bfloat16 and lp16.dtype == en16.dtype == torch.float32
    assert torch.equal(lp16, lp32), "logp differs from the float32 entry's"
    assert torch.equal(en16, en32), "entropy differs from the float32 entry's"
    assert torch.equal(g16, g32.to(torch.bfloat16)), "g_logits is not the float32 entry's rounded to bfloat16"
    assert torch.equal(gv16, gv32.to(torch.bfloat16)), "g_value is not the float32 entry's rounded to bfloat16"
    if masked:
        assert bool((g16[torch.from_numpy(c["available"]).cuda() == 0] == 0).all()), "non-zero gradient at an unavailable logit"


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [True, False], ids=["masked", "unmasked"])
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("heads", PARITY_HEAD_SETS, ids=ids)
def test_bf16_logits_match_oracle(ops, heads, config, masked):
    """Against masked_fill + Categorical per head feeding the oracle's loss, on the widened bfloat16 values: `out`, logp and
    entropy within 1e-5 * max(1, |ref|), the bfloat16 gradients within half a bfloat16 ulp of the oracle's plus that bar."""
    T, n = 20, 37
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    c = bf16_case(heads, T, n, 0.3, seed=sum(heads) + 3, masked=masked, N=53 if use_idx else None)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    ref = oracle(c, hp_kw, popart=pa)
    g_logits, g_v, out, out32, logp, ent = launch(ops, c, hp_kw, ref["norm_stats"], torch.bfloat16, masked=masked,
                                                  popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
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
    assert_bf16_grad_close(g_v, ref["g_value"], msum, what="g_value")
    assert_bf16_grad_close(g_logits, ref["g_logits"], msum, what="g_logits")
    if masked:
        unavailable = torch.from_numpy(c["available"]) == 0
        assert bool((g_logits.cpu()[unavailable] == 0).all()), "non-zero gradient at an unavailable logit"


@pytest.mark.gpu
@pytest.mark.parametrize("heads", [(36,), (4, 33, 7, 32)], ids=ids)
def test_bf16_unaligned_pointers_take_the_staging_path(ops, heads):
    """bfloat16 logits one element (2 bytes) off a 16-byte boundary, or the mask one byte off, are staged element by element
    in every tile: the results equal the aligned launch's bit for bit."""
    T, n = 20, 37
    hp_kw = CONFIGS["huber_clip_value"]
    c = bf16_case(heads, T, n, 0.3, seed=3)
    ns = oracle(c, hp_kw)["norm_stats"]
    base = launch(ops, c, hp_kw, ns, torch.bfloat16, want_logp_entropy=True)
    buf = torch.empty(c["logits"].size + 1, dtype=torch.bfloat16, device="cuda")
    lg = buf[1:].view(c["logits"].shape)
    lg.copy_(torch.from_numpy(c["logits"]))
    mb = torch.empty(c["available"].size + 1, dtype=torch.uint8, device="cuda")
    mk = mb[1:].view(c["available"].shape)
    mk.copy_(torch.from_numpy(c["available"]))
    assert lg.data_ptr() % 16 == 2 and mk.data_ptr() % 16 == 1
    for kw in (dict(logits=lg), dict(available=mk)):
        r = launch(ops, c, hp_kw, ns, torch.bfloat16, want_logp_entropy=True, **kw)
        for x, y, name in zip(r, base, ("g_logits", "g_value", "out", "out_f32", "logp", "entropy")):
            assert torch.equal(x, y), f"{name} differs with {list(kw)[0]} unaligned"


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [True, False], ids=["masked", "unmasked"])
def test_bf16_logits_deterministic_and_deferred(ops, masked):
    """Two launches are bit-identical and leave the workspace zero; a deferred launch followed by loss_finalize gives the
    immediate launch's bits."""
    T, n = 128, 1000
    hp_kw = CONFIGS["popart_dual_clip"]
    c = bf16_case((36,), T, n, 0.3, seed=11, masked=masked)
    _, ms = _popart()
    ns = oracle(c, hp_kw)["norm_stats"]
    ws = ops.new_loss_workspace("cuda")
    a = launch(ops, c, hp_kw, ns, torch.bfloat16, masked=masked, popart_ms=ms, workspace=ws[0])
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = launch(ops, c, hp_kw, ns, torch.bfloat16, masked=masked, popart_ms=ms, workspace=ws[0])
    assert not ws.any()
    for x, y, name in zip(a[:4], b[:4], ("g_logits", "g_value", "out", "out_f32")):
        assert torch.equal(x, y), f"{name} differs between two launches"
    g_logits, g_v, out_d, out32_d, _, _ = launch(ops, c, hp_kw, ns, torch.bfloat16, masked=masked, popart_ms=ms,
                                                 workspace=ws[0], defer=True)
    assert out_d is None and out32_d is None
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    out32 = torch.zeros((1, 4), dtype=torch.float32, device="cuda")
    ops.loss_finalize(ws, out, out32)
    torch.cuda.synchronize()
    assert torch.equal(out[0], a[2]) and torch.equal(out32[0], a[3])
    assert torch.equal(g_logits, a[0]) and torch.equal(g_v, a[1])
    assert not torch.cat([ws[0, :4], ws[0, 32:]]).any(), "deferred mode + finalize left the workspace dirty"


@pytest.mark.gpu
def test_autocast_policy_trains_through_the_bf16_entry_without_casts(ops):
    """A SMAC-shaped policy (nn.Linear logits over 36 actions and value) under torch.autocast(bfloat16), loss through
    PPOCategoricalLossFunction with the mask: once on its bfloat16 outputs as they are, once through the cast path
    (.float() on both outputs, the float32 entry, autograd casting the gradients back).  The gradients reaching the
    bfloat16 outputs are the same bfloat16 bits, so every parameter gradient is bit-identical."""
    T, n, F, heads = 24, 300, 11, (36,)
    torch.manual_seed(0)

    class Policy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.pi = torch.nn.Linear(F, sum(heads))
            self.v = torch.nn.Linear(F, 1)

    pol = Policy().cuda()
    pol_cast = copy.deepcopy(pol)
    c = make_case(heads, T, n, 0.3, seed=5, odd_rows=False)
    d = lambda k: torch.from_numpy(np.ascontiguousarray(c[k])).cuda()
    avail = d("available")
    obs = torch.randn(T, n, F, device="cuda")
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        z0 = pol.pi(obs).float().masked_fill(avail == 0, -1e10)
    act = torch.distributions.Categorical(logits=z0).sample().unsqueeze(-1)
    with torch.no_grad():
        lp0, _ = M.logp_entropy_from_logits_ref(z0.cpu(), act.cpu(), heads, available=avail.cpu())
    lp0 = lp0[..., 0].numpy().astype(np.float64)
    c["old_logp"][:T] = away_from_clip_edges(lp0, lp0 + 0.15 * np.random.default_rng(1).standard_normal((T, n)))
    mask = 1 - torch.from_numpy(c["on_reset"][1:T + 1]).float()
    ns = torch.tensor([float(x) for x in M.masked_sums_ref(torch.from_numpy(c["adv"][:T]), mask)] + [0.0] * 5,
                      dtype=torch.float64).cuda()
    hp = ops.LossHyper(**CONFIGS["huber_clip_value"])
    smp = (d("old_logp")[:T], d("value")[:T], d("ret")[:T], d("adv")[:T], d("on_reset")[1:T + 1], ns, None, None, None, hp)
    action = act.int()

    with torch.autocast("cuda", dtype=torch.bfloat16):
        z, v = pol.pi(obs), pol.v(obs)[..., 0]
        z_c, v_c = pol_cast.pi(obs), pol_cast.v(obs)[..., 0]
    assert z.dtype == v.dtype == torch.bfloat16
    for t in (z, v, z_c, v_c):
        t.retain_grad()
    loss, _ = ops.PPOCategoricalLossFunction.apply(z, avail, action, heads, v, *smp)
    loss_c, _ = ops.PPOCategoricalLossFunction.apply(z_c.float(), avail, action, heads, v_c.float(), *smp)
    loss.backward()
    loss_c.backward()
    torch.cuda.synchronize()
    assert_close_ref(loss.item(), loss_c.item(), tol=1e-6, what="loss")
    assert z.grad.dtype == v.grad.dtype == torch.bfloat16
    assert torch.equal(z.grad, z_c.grad), "d loss / d logits differs from the cast path's"
    assert torch.equal(v.grad, v_c.grad), "d loss / d value differs from the cast path's"
    for (name, p), (_, q) in zip(pol.named_parameters(), pol_cast.named_parameters()):
        assert p.grad is not None, f"{name} received no gradient"
        assert torch.equal(p.grad, q.grad), f"d loss / d {name} differs from the cast path's"


def test_bf16_logits_host_side_argument_checks():
    """Rejected on the host before any CUDA call, with a status and a message -- no GPU needed.  The non-null device
    pointers are never dereferenced."""
    build.build()
    lib = _lib.load_library()
    assert lib.srl_abi_version() == _lib.ABI_VERSION == 12
    T, n = 4, 8
    fake = 256
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)

    def call(heads, masked, available=fake):
        hs = (ctypes.c_int32 * len(heads))(*heads)
        tail = (fake, hs, len(heads), fake, fake, fake, fake, fake, fake, n, None, T, n, fake, fake, None, ctypes.byref(hc),
                fake, fake, None, None, fake, None, fake, lib.srl_ppo_loss_workspace_bytes(T, n), None)
        if masked:
            rc = lib.srl_ppo_loss_from_logits_masked_bf16(fake, available, *tail)
        else:
            rc = lib.srl_ppo_loss_from_logits_bf16(fake, *tail)
        return rc, lib.srl_last_error().decode()

    rc, msg = call((36,), True, available=None)
    assert rc == 1 and "srl_ppo_loss_from_logits_masked_bf16: null pointer available" in msg, msg
    # the widest rows are the float32 entries' for both dtypes
    for masked, limit in ((False, _lib.SRL_K4B_MAX_SUM_K), (True, _lib.SRL_K4B_MAX_SUM_K_MASKED)):
        too_wide = (100, limit + 1 - 100)
        rc, msg = call(too_wide, masked)
        assert rc == 2 and f"sum K = {limit + 1} too wide (max {limit})" in msg, msg
    rc, msg = call((0, 5), False)
    assert rc == 1 and "srl_ppo_loss_from_logits_bf16: head 0 has no actions" in msg, msg


def test_bf16_logits_ops_argument_checks():
    """ops.ppo_loss_from_logits takes float32 or bfloat16 logits with a v_pred of the same dtype; anything else is a
    ValueError before anything touches the device."""
    from srl_b200 import ops
    T, n, K = 3, 5, 36
    rest = dict(action=torch.zeros(T, n, 1, dtype=torch.int32), head_sizes=(K,), old_logp=None, old_value=None, ret=None,
                adv=None, on_reset_next=None, norm_stats=None, hyper=ops.LossHyper())
    for lg, vp in ((torch.bfloat16, torch.float32), (torch.float32, torch.bfloat16)):
        with pytest.raises(ValueError, match="cast one of them") as e:
            ops.ppo_loss_from_logits(torch.zeros(T, n, K, dtype=lg), v_pred=torch.zeros(T, n, dtype=vp), **rest)
        assert str(lg) in str(e.value) and str(vp) in str(e.value), str(e.value)
    for dt in (torch.float16, torch.float64):
        with pytest.raises(ValueError, match=r"torch\.float32 or torch\.bfloat16, got " + str(dt).replace(".", r"\.")):
            ops.ppo_loss_from_logits(torch.zeros(T, n, K, dtype=dt), v_pred=torch.zeros(T, n, dtype=dt), **rest)
