"""K4c with a bfloat16 policy side (srl_ppo_loss_from_gaussian_bf16, ops.ppo_loss_from_gaussian on bfloat16 mean, value and
per-transition log_std, ops.PPOGaussianLossFunction under torch.autocast).  The mean, value and per-transition log_std of
every case are bfloat16 numbers; the float32 entry and the oracle see them widened, which is exact.  The action stays
float32.  The bfloat16 entry computes what the float32 entry computes and rounds each bfloat16 gradient once, so on the
same launch grid its results are the float32 entry's bit for bit, with the gradients rounded.  The host-side argument
checks run without a GPU."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from srl_b200 import _lib, build
from tests.gaussian_ref import logp_entropy_from_gaussian_ref
from tests.test_gpu_bf16_logits import assert_bf16_grad_close
from tests.test_gpu_gaussian import CONFIGS, OUT_KEYS, STAT_KEYS, _popart, away_from_clip_edges, make_case, oracle
from tests.util import assert_close_ref, assert_grad_close

NAMES = ("g_mean", "g_log_std", "g_value", "out", "out_f32", "logp", "entropy")


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


def bf16_case(T, n, D, shared, seed, N=None):
    """make_case with bfloat16 mean, v_pred and per-transition log_std (a shared [D] log_std stays float32, as autocast
    leaves an nn.Parameter); old_logp kept away from the clip edges for the rounded values' log-prob."""
    c = make_case(T, n, D, shared, seed, N=N)
    c["mean"], c["v_pred"] = bf16_exact(c["mean"]), bf16_exact(c["v_pred"])
    if not shared:
        c["log_std"] = bf16_exact(c["log_std"])
    with torch.no_grad():
        lp, _ = logp_entropy_from_gaussian_ref(*(torch.from_numpy(c[k]).double() for k in ("mean", "log_std", "action")))
    idx = c["lane_idx"]
    c["old_logp"][:T, idx] = away_from_clip_edges(lp.numpy(), c["old_logp"][:T, idx])
    return c


def launch(ops, c, hp_kw, norm_stats, dtype, popart_ms=None, use_lane_idx=False, mean=None, log_std=None, action=None,
           **kw):
    """One launch with the policy side in `dtype` (c's values are bfloat16 numbers, so either dtype holds them exactly);
    a shared log_std is passed as float32."""
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    if log_std is None:
        log_std = d(c["log_std"])
        log_std = log_std.to(dtype) if log_std.dim() > 1 else log_std
    r = ops.ppo_loss_from_gaussian(
        d(c["mean"]).to(dtype) if mean is None else mean, log_std, d(c["action"]) if action is None else action,
        d(c["v_pred"]).to(dtype), d(c["old_logp"])[:T], d(c["value"])[:T], d(c["ret"])[:T], d(c["adv"])[:T],
        d(c["on_reset"])[1:T + 1], d(np.asarray(norm_stats, dtype=np.float64)), ops.LossHyper(**hp_kw),
        popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=d(c["lane_idx"]) if use_lane_idx else None, **kw)
    torch.cuda.synchronize()
    return r


def _grid(config, D, shared, seed_base):
    use_idx = config == "lane_idx"
    c = bf16_case(20, 37, D, shared, seed=seed_base + 100 * D + int(shared), N=53 if use_idx else None)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    return c, pa, ms, use_idx


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("shared", [False, True], ids=["per_row", "shared"])
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_bf16_gaussian_equals_the_float32_entry_bit_for_bit(ops, D, shared, config):
    """The bfloat16 entry on x and the float32 entry on x.float() (T = 20, n = 37: two bulk-copied tiles and a staged one):
    logp, entropy, out, out_f32 and a shared (float32) g_log_std are identical; g_mean, g_value and a per-row g_log_std
    are the float32 entry's rounded to bfloat16."""
    hp_kw = CONFIGS[config]
    c, pa, ms, use_idx = _grid(config, D, shared, 1)
    ns = oracle(c, hp_kw, popart=pa)["norm_stats"]
    kw = dict(popart_ms=ms, use_lane_idx=use_idx, want_logp_entropy=True)
    a = launch(ops, c, hp_kw, ns, torch.bfloat16, **kw)
    b = launch(ops, c, hp_kw, ns, torch.float32, **kw)
    assert a[0].dtype == a[2].dtype == torch.bfloat16
    assert a[1].dtype == (torch.float32 if shared else torch.bfloat16)
    assert a[5].dtype == a[6].dtype == torch.float32
    for k in (3, 4, 5, 6):
        assert torch.equal(a[k], b[k]), f"{NAMES[k]} differs from the float32 entry's"
    for k in (0, 2):
        assert torch.equal(a[k], b[k].to(torch.bfloat16)), f"{NAMES[k]} is not the float32 entry's rounded to bfloat16"
    if shared:
        assert torch.equal(a[1], b[1]), "the shared g_log_std differs from the float32 entry's"
    else:
        assert torch.equal(a[1], b[1].to(torch.bfloat16)), "g_log_std is not the float32 entry's rounded to bfloat16"


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("shared", [False, True], ids=["per_row", "shared"])
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_bf16_gaussian_matches_oracle(ops, D, shared, config):
    """Against Normal in float64 feeding the oracle's loss, on the widened bfloat16 values: `out`, logp and entropy within
    1e-5 * max(1, |ref|), the bfloat16 gradients within half a bfloat16 ulp of the oracle's plus that bar, a shared
    (float32) g_log_std within the float32 entry's bar."""
    hp_kw = CONFIGS[config]
    c, pa, ms, use_idx = _grid(config, D, shared, 2)
    ref = oracle(c, hp_kw, popart=pa)
    g_mean, g_ls, g_v, out, out32, logp, ent = launch(ops, c, hp_kw, ref["norm_stats"], torch.bfloat16, popart_ms=ms,
                                                      use_lane_idx=use_idx, want_logp_entropy=True)
    msum = ref["mask_sum"]
    for x, name in zip((g_mean, g_ls, g_v, out, logp, ent), ("g_mean", "g_log_std", "g_value", "out", "logp", "entropy")):
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
    assert_bf16_grad_close(g_mean, ref["g_mean"], msum, what="g_mean")
    if shared:
        assert g_ls.dtype == torch.float32 and tuple(g_ls.shape) == (D,)
        assert_grad_close(g_ls.cpu(), ref["g_log_std"], msum, what="g_log_std")
    else:
        assert_bf16_grad_close(g_ls, ref["g_log_std"], msum, what="g_log_std")


@pytest.mark.gpu
@pytest.mark.parametrize("D", [6, 17])
def test_bf16_gaussian_unaligned_pointers_take_the_staging_path(ops, D):
    """bfloat16 mean or per-row log_std one element (2 bytes) off a 16-byte boundary, or the float32 action one element
    (4 bytes) off, are staged element by element in every tile: the results equal the aligned launch's bit for bit."""
    T, n = 20, 37
    hp_kw = CONFIGS["huber_clip_value"]
    c = bf16_case(T, n, D, False, seed=3)
    ns = oracle(c, hp_kw)["norm_stats"]
    base = launch(ops, c, hp_kw, ns, torch.bfloat16, want_logp_entropy=True)

    def unaligned(key, dtype):
        buf = torch.empty(c[key].size + 1, dtype=dtype, device="cuda")
        x = buf[1:].view(c[key].shape)
        x.copy_(torch.from_numpy(c[key]))
        assert x.data_ptr() % 16 == x.element_size()
        return x

    for key, dtype in (("mean", torch.bfloat16), ("log_std", torch.bfloat16), ("action", torch.float32)):
        r = launch(ops, c, hp_kw, ns, torch.bfloat16, want_logp_entropy=True, **{key: unaligned(key, dtype)})
        for x, y, name in zip(r, base, NAMES):
            assert torch.equal(x, y), f"{name} differs with {key} unaligned"


@pytest.mark.gpu
@pytest.mark.parametrize("D,shared", [(6, True), (17, False)], ids=["D6_shared", "D17_per_row"])
def test_bf16_gaussian_full_size(ops, D, shared):
    """cfg2's shape (T = 128, N = 4096): the grid is a full resident wave (a shared [D] gradient folded from one partial row
    per CTA); compared with the oracle evaluated in float64 on the widened values."""
    T, n = 128, 4096
    hp_kw = CONFIGS["huber_clip_value"]
    c = bf16_case(T, n, D, shared, seed=7)
    ref = oracle(c, hp_kw, loss_dtype=torch.float64)
    g_mean, g_ls, g_v, out, _, _, _ = launch(ops, c, hp_kw, ref["norm_stats"], torch.bfloat16)
    msum = ref["mask_sum"]
    out = out.cpu().numpy()
    for k, name in OUT_KEYS:
        assert_close_ref(out[k], ref[name], what=name)
    if shared:
        assert_grad_close(g_ls.cpu(), ref["g_log_std"], msum, what="g_log_std")
    else:
        assert_bf16_grad_close(g_ls, ref["g_log_std"], msum, what="g_log_std")
    assert_bf16_grad_close(g_mean, ref["g_mean"], msum, what="g_mean")
    assert_bf16_grad_close(g_v, ref["g_value"], msum, what="g_value")


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True], ids=["per_row", "shared"])
def test_bf16_gaussian_deterministic_and_workspace_left_zero(ops, shared):
    """Two launches: bit-identical gradients and outputs.  Deferred mode (out = NULL, then srl_ppo_loss_finalize on the
    workspace's slot) gives the immediate mode's bits and the same gradients.  The workspace is zero after every launch,
    except the bytes a deferred launch hands to the finaliser (slot bytes 4-31: n_rows, sum(mask), weights)."""
    T, n, D = 128, 1000, 17
    hp_kw = CONFIGS["mse_dual_clip"]
    c = bf16_case(T, n, D, shared, seed=11)
    ns = oracle(c, hp_kw)["norm_stats"]
    ws = ops.new_gaussian_loss_workspace("cuda", T, n, D, shared)
    a = launch(ops, c, hp_kw, ns, torch.bfloat16, workspace=ws)
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = launch(ops, c, hp_kw, ns, torch.bfloat16, workspace=ws)
    assert not ws.any()
    for x, y, name in zip(a[:5], b[:5], NAMES):
        assert torch.equal(x, y), f"{name} differs between two launches"
    g_mean, g_ls, g_v, out_d, out32_d, _, _ = launch(ops, c, hp_kw, ns, torch.bfloat16, workspace=ws, defer=True)
    assert out_d is None and out32_d is None
    out = torch.zeros((1, 16), dtype=torch.float64, device="cuda")
    out32 = torch.zeros((1, 4), dtype=torch.float32, device="cuda")
    ops.loss_finalize(ws.view(1, -1), out, out32)
    torch.cuda.synchronize()
    assert torch.equal(out[0], a[3]) and torch.equal(out32[0], a[4])
    assert torch.equal(g_mean, a[0]) and torch.equal(g_ls, a[1]) and torch.equal(g_v, a[2])
    rest = torch.cat([ws[:4], ws[32:]])
    assert not rest.any(), "deferred mode + finalize left the workspace dirty"


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["param_log_std", "per_row_log_std", "module_bf16"])
def test_autocast_gaussian_policy_trains_through_the_bf16_entry_without_casts(ops, variant):
    """A continuous-action policy (nn.Linear mean and value heads) under torch.autocast(bfloat16), loss through
    PPOGaussianLossFunction: once on its outputs as they are, once through the cast path (.float() on mean, log_std and
    value, the float32 entry, autograd casting the gradients back).  log_std is (a) a float32 nn.Parameter, (b) a third
    nn.Linear head, or (c) a bfloat16 [D] parameter of a module cast with .bfloat16().  The gradients reaching the policy's
    outputs are the same bits either way, so every parameter gradient is bit-identical."""
    T, n, D, F = 24, 300, 6, 11
    torch.manual_seed(0)
    per_row = variant == "per_row_log_std"

    class Policy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.mu = torch.nn.Linear(F, D)
            self.v = torch.nn.Linear(F, 1)
            if per_row:
                self.ls = torch.nn.Linear(F, D)
            else:
                self.log_std = torch.nn.Parameter(torch.linspace(-0.8, 0.3, D))

        def forward(self, obs):
            return self.mu(obs), self.ls(obs) if per_row else self.log_std, self.v(obs)[..., 0]

    pol = Policy().cuda()
    if variant == "module_bf16":
        pol = pol.bfloat16()
    pol_cast = copy.deepcopy(pol)
    c = make_case(T, n, D, True, seed=5)
    d = lambda k: torch.from_numpy(np.ascontiguousarray(c[k])).cuda()
    obs = torch.randn(T, n, F, device="cuda")
    # the actors' sample: float32 and without a graph (with a [D] parameter the forward hands back the parameter itself,
    # so exp() of it outside no_grad would tie both losses below to one shared node)
    with torch.no_grad():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            mean0, ls0, _ = pol(obs)
        mean0, ls0 = mean0.float(), ls0.float()
        action = (mean0 + ls0.exp() * torch.randn(T, n, D, device="cuda")).contiguous()
        lp0, _ = logp_entropy_from_gaussian_ref(mean0.double().cpu(), ls0.double().cpu(), action.double().cpu())
    assert not action.requires_grad
    lp0 = lp0.numpy()
    c["old_logp"][:T] = away_from_clip_edges(lp0, lp0 + 0.15 * np.random.default_rng(1).standard_normal((T, n)))
    mask = 1 - torch.from_numpy(c["on_reset"][1:T + 1]).float()
    ns = torch.tensor([float(x) for x in M.masked_sums_ref(torch.from_numpy(c["adv"][:T]), mask)] + [0.0] * 5,
                      dtype=torch.float64).cuda()
    hp = ops.LossHyper(**CONFIGS["huber_clip_value"])
    smp = (d("old_logp")[:T], d("value")[:T], d("ret")[:T], d("adv")[:T], d("on_reset")[1:T + 1], ns, None, None, None, hp)

    with torch.autocast("cuda", dtype=torch.bfloat16):
        mean, log_std, v = pol(obs)
        mean_c, log_std_c, v_c = pol_cast(obs)
    assert mean.dtype == v.dtype == torch.bfloat16
    assert log_std.dtype == (torch.float32 if variant == "param_log_std" else torch.bfloat16)
    outs = (mean, log_std, v, mean_c, log_std_c, v_c)
    for t in outs:
        if not t.is_leaf:
            t.retain_grad()
    loss, _ = ops.PPOGaussianLossFunction.apply(mean, log_std, action, v, *smp)
    loss_c, _ = ops.PPOGaussianLossFunction.apply(mean_c.float(), log_std_c.float(), action, v_c.float(), *smp)
    loss.backward()
    loss_c.backward()
    torch.cuda.synchronize()
    assert torch.equal(loss, loss_c), "the loss differs from the cast path's"
    for x, y, name in zip(outs[:3], outs[3:], ("mean", "log_std", "value")):
        assert x.grad.dtype == x.dtype, f"d loss / d {name} is {x.grad.dtype}, its input {x.dtype}"
        assert torch.equal(x.grad, y.grad), f"d loss / d {name} differs from the cast path's"
    for (name, p), (_, q) in zip(pol.named_parameters(), pol_cast.named_parameters()):
        assert p.grad is not None, f"{name} received no gradient"
        assert torch.equal(p.grad, q.grad), f"d loss / d {name} differs from the cast path's"


def test_bf16_gaussian_host_side_argument_checks():
    """The bfloat16 entry returns the float32 entry's statuses and messages, under its own name, before any CUDA call -- no
    GPU needed.  The non-null device pointers are never dereferenced."""
    build.build()
    lib = _lib.load_library()
    T, n, D = 4, 8, 6
    fake = 256
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)
    need = lib.srl_ppo_loss_gaussian_workspace_bytes(T, n, D, 1)

    def call(entry, D=D, mean=fake, old_value=fake, ws_bytes=need, hyper=hc):
        args = dict(mean=mean, log_std=fake, shared=1, action=fake, D=D, v_pred=fake, old_logp=fake, old_value=old_value,
                    ret=fake, adv=fake, rs=fake, ld_smp=n, lane_idx=None, T=T, n=n, ns=fake, ls=fake, pm=None,
                    hyper=ctypes.byref(hyper), g_mean=fake, g_ls=fake, g_v=fake, logp=None, ent=None, out=fake,
                    out32=None, ws=fake, ws_bytes=ws_bytes, stream=None)
        rc = getattr(lib, entry)(*args.values())
        return rc, lib.srl_last_error().decode()

    clip = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 1, 1, 0)
    for kw in (dict(D=0), dict(D=65), dict(mean=None), dict(ws_bytes=need - 8), dict(old_value=None, hyper=clip)):
        rc32, msg32 = call("srl_ppo_loss_from_gaussian", **kw)
        rc16, msg16 = call("srl_ppo_loss_from_gaussian_bf16", **kw)
        assert rc32 == 1 and msg32.startswith("srl_ppo_loss_from_gaussian: "), msg32
        assert rc16 == rc32, (kw, rc16, rc32)
        assert msg16 == msg32.replace("srl_ppo_loss_from_gaussian:", "srl_ppo_loss_from_gaussian_bf16:", 1), msg16
    assert "D=65" in call("srl_ppo_loss_from_gaussian_bf16", D=65)[1]
    assert "null pointer mean" in call("srl_ppo_loss_from_gaussian_bf16", mean=None)[1]


def test_bf16_gaussian_ops_argument_checks():
    """ops.ppo_loss_from_gaussian takes float32 or bfloat16 mean with a v_pred and a per-transition log_std of the same
    dtype, and a float32 action; anything else is a ValueError before anything touches the device."""
    from srl_b200 import ops
    T, n, D = 3, 5, 6
    z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt)
    rest = dict(old_logp=None, old_value=None, ret=None, adv=None, on_reset_next=None, norm_stats=None,
                hyper=ops.LossHyper())
    for m, vp in ((torch.bfloat16, torch.float32), (torch.float32, torch.bfloat16)):
        with pytest.raises(ValueError, match="cast one of them") as e:
            ops.ppo_loss_from_gaussian(z(T, n, D, dt=m), z(D), z(T, n, D), z(T, n, dt=vp), **rest)
        assert str(m) in str(e.value) and str(vp) in str(e.value), str(e.value)
    for m, ls in ((torch.bfloat16, torch.float32), (torch.float32, torch.bfloat16)):
        with pytest.raises(ValueError, match="cast one of them") as e:
            ops.ppo_loss_from_gaussian(z(T, n, D, dt=m), z(T, n, D, dt=ls), z(T, n, D), z(T, n, dt=m), **rest)
        assert "log_std" in str(e.value) and str(m) in str(e.value) and str(ls) in str(e.value), str(e.value)
    with pytest.raises(ValueError, match="float32 actions the actors sampled"):
        ops.ppo_loss_from_gaussian(z(T, n, D, dt=torch.bfloat16), z(D), z(T, n, D, dt=torch.bfloat16),
                                   z(T, n, dt=torch.bfloat16), **rest)
    for dt in (torch.float16, torch.float64):
        with pytest.raises(ValueError, match=r"torch\.float32 or torch\.bfloat16, got " + str(dt).replace(".", r"\.")):
            ops.ppo_loss_from_gaussian(z(T, n, D, dt=dt), z(D), z(T, n, D), z(T, n, dt=dt), **rest)
