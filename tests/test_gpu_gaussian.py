"""K4c (srl_ppo_loss_from_gaussian, ops.ppo_loss_from_gaussian, ops.PPOGaussianLossFunction): the PPO loss starting
from a diagonal-Gaussian actor head, against torch.distributions.Normal feeding the oracle's loss, with autograd to the
head's mean and log_std.  Bars as in test_gpu_parity.py: 1e-5 * max(1, |ref|), gradients on the g * sum(mask) scale.
The host-side argument checks run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from srl_b200 import _lib, build
from tests.gaussian_ref import logp_entropy_from_gaussian_ref
from tests.util import assert_close_ref, assert_grad_close

OUT_KEYS = ((0, "loss"), (1, "policy_loss"), (2, "value_loss"), (3, "entropy_loss"))
STAT_KEYS = ((4, "advantage"), (5, "importance_weight"), (6, "clip_ratio"), (7, "value_targets"), (8, "denorm_value"))


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()  # must load the in-tree .so, loudly
    return _ops


def away_from_clip_edges(logp, old_logp, eps_clip=0.2, margin=1e-4):
    """float32 old_logp whose ratios exp(logp - old_logp) stay `margin` away from 1 -/+ eps_clip: two float32 evaluations of
    the head's log-prob differ in the last bits, and a ratio that close to an edge of the clipped surrogate may land on
    either side of it (a zero or a full gradient for that transition) -- not a property of either evaluation."""
    old = np.asarray(old_logp, dtype=np.float64)
    for _ in range(4):
        r = np.exp(logp - old.astype(np.float32).astype(np.float64))
        near = (np.abs(r - (1 - eps_clip)) < margin) | (np.abs(r - (1 + eps_clip)) < margin)
        if not near.any():
            break
        old = np.where(near, old + 10 * margin, old)
    return old.astype(np.float32)


def make_case(T, n, D, shared, seed, N=None):
    """Seeded inputs of one minibatch.  Sample side [T + 1, N] (N >= n lanes; on_reset one row longer), policy side
    [T, n, D]; old_logp is the head's log-prob perturbed so that ratios straddle the clip range."""
    N = n if N is None else N
    rng = np.random.default_rng(seed)
    f32 = lambda x: np.asarray(x, dtype=np.float32)
    mean = f32(rng.standard_normal((T, n, D)))
    log_std = f32(rng.uniform(-1.0, 0.5, D if shared else (T, n, D)))
    sig = np.exp(log_std.astype(np.float64))
    action = f32(mean + sig * rng.standard_normal((T, n, D)) * 1.3)
    on_reset = (rng.random((T + 1, N)) < 0.1).astype(np.uint8)
    value = f32(rng.standard_normal((T + 1, N)))
    ret = f32(rng.standard_normal((T + 1, N)) * 2.0)
    adv = f32(rng.standard_normal((T + 1, N)))
    lane_idx = np.arange(n, dtype=np.int32) if N == n else rng.permutation(N)[:n].astype(np.int32)
    with torch.no_grad():
        lp, _ = logp_entropy_from_gaussian_ref(*(torch.from_numpy(x).double() for x in (mean, log_std, action)))
    old_logp = np.zeros((T + 1, N), np.float32)
    old_logp[:T, lane_idx] = away_from_clip_edges(lp.numpy(), lp.numpy() + 0.15 * rng.standard_normal((T, n)))
    v_pred = f32(value[:T, lane_idx] + 0.1 * rng.standard_normal((T, n)))
    return dict(mean=mean, log_std=log_std, action=action, on_reset=on_reset, value=value, ret=ret, adv=adv,
                old_logp=old_logp, v_pred=v_pred, lane_idx=lane_idx, T=T, n=n, N=N, D=D)


def oracle(c, hp_kw, popart=None, loss_dtype=torch.float32):
    """Normal log-prob / entropy -> the oracle's loss, autograd back to mean, log_std (a [D] leaf when shared) and
    v_pred, on the CPU.  The head and its backward run in float64: a shared log_std's gradient is a sum of T * n
    cancelling terms, which float32 autograd does not get to 1e-5.  The loss runs in `loss_dtype`."""
    T = c["T"]
    take = lambda x: torch.from_numpy(np.ascontiguousarray(x[:T][:, c["lane_idx"]])).to(loss_dtype)
    mean = torch.from_numpy(c["mean"]).double().requires_grad_(True)
    log_std = torch.from_numpy(c["log_std"]).double().requires_grad_(True)
    lp, en = logp_entropy_from_gaussian_ref(mean, log_std, torch.from_numpy(c["action"]).double())
    mask = 1 - torch.from_numpy(np.ascontiguousarray(c["on_reset"][1:T + 1][:, c["lane_idx"]])).to(loss_dtype)
    adv = take(c["adv"])
    res = M.ppo_loss_ref(lp.detach().to(loss_dtype), take(c["old_logp"]), torch.from_numpy(c["v_pred"]).to(loss_dtype),
                         take(c["value"]), take(c["ret"]), adv, en.detach().to(loss_dtype), mask, M.LossHyper(**hp_kw),
                         popart=popart)
    (lp * res["g_logp"].double()).sum().add((en * res["g_entropy"].double()).sum()).backward()
    res.update(lp=lp.detach(), en=en.detach(), g_mean=mean.grad, g_log_std=log_std.grad, mask_sum=float(mask.sum()),
               norm_stats=[float(x) for x in M.masked_sums_ref(adv, mask)] + [0.0] * 5)
    return res


def run(ops, c, hp_kw, popart_ms=None, use_lane_idx=False, **kw):
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    T = c["T"]
    li = d(c["lane_idx"]) if use_lane_idx else None
    ns = kw.pop("norm_stats")
    r = ops.ppo_loss_from_gaussian(
        d(c["mean"]), d(c["log_std"]), d(c["action"]), d(c["v_pred"]), d(c["old_logp"])[:T], d(c["value"])[:T],
        d(c["ret"])[:T], d(c["adv"])[:T], d(c["on_reset"])[1:T + 1], d(np.asarray(ns, dtype=np.float64)),
        ops.LossHyper(**hp_kw), popart_mean_std=None if popart_ms is None else d(np.asarray(popart_ms, np.float64)),
        lane_idx=li, **kw)
    torch.cuda.synchronize()
    return r


def _popart():
    pa = M.RunningMeanStdRef((1,), beta=0.999)
    pa.update(torch.randn(64, 1, generator=torch.Generator().manual_seed(1)) * 2 + 1)
    m_, s_ = pa.mean_std()
    return pa, [m_.item(), s_.item()]


CONFIGS = {
    "mse_dual_clip": dict(dual_clip=True, entropy_bonus_weight=0.05),
    "huber_clip_value": dict(dual_clip=False, clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0),
                             entropy_bonus_weight=0.05),
    "popart_normalize_old_value": dict(clip_value=True, normalize_old_value=True, entropy_bonus_weight=0.05),
    "lane_idx": dict(clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0), entropy_bonus_weight=0.05),
}


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("shared", [False, True], ids=["per_row", "shared"])
@pytest.mark.parametrize("D", [1, 6, 17, 64])
def test_gaussian_loss_matches_oracle(ops, D, shared, config):
    """T = 20, n = 37: two full tiles of 256 transitions (bulk copies) and a partial one (element-wise staging)."""
    T, n = 20, 37
    hp_kw = CONFIGS[config]
    use_idx = config == "lane_idx"
    c = make_case(T, n, D, shared, seed=100 * D + int(shared), N=53 if use_idx else None)
    pa, ms = _popart() if config.startswith("popart") else (None, None)
    ref = oracle(c, hp_kw, popart=pa)
    g_mean, g_ls, g_v, out, out32, logp, ent = run(ops, c, hp_kw, popart_ms=ms, use_lane_idx=use_idx,
                                                   norm_stats=ref["norm_stats"], want_logp_entropy=True)
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
    assert tuple(g_ls.shape) == ((D,) if shared else (T, n, D))
    assert_grad_close(g_v.cpu(), ref["g_value"], msum, what="g_value")
    assert_grad_close(g_mean.cpu(), ref["g_mean"], msum, what="g_mean")
    assert_grad_close(g_ls.cpu(), ref["g_log_std"], msum, what="g_log_std")


@pytest.mark.gpu
def test_gaussian_full_size_shared_log_std(ops):
    """cfg2's shape (T = 128, N = 4096) with D = 6 and a shared log_std: the [D] gradient is folded from one partial row
    per CTA of a full grid; compared with the oracle evaluated in float64."""
    T, n, D = 128, 4096, 6
    hp_kw = CONFIGS["huber_clip_value"]
    c = make_case(T, n, D, True, seed=7)
    ref = oracle(c, hp_kw, loss_dtype=torch.float64)
    g_mean, g_ls, g_v, out, _, _, _ = run(ops, c, hp_kw, norm_stats=ref["norm_stats"])
    msum = ref["mask_sum"]
    out = out.cpu().numpy()
    for k, name in OUT_KEYS:
        assert_close_ref(out[k], ref[name], what=name)
    assert_grad_close(g_ls.cpu(), ref["g_log_std"], msum, what="g_log_std")
    assert_grad_close(g_mean.cpu(), ref["g_mean"], msum, what="g_mean")
    assert_grad_close(g_v.cpu(), ref["g_value"], msum, what="g_value")


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True], ids=["per_row", "shared"])
def test_gaussian_deterministic_and_workspace_left_zero(ops, shared):
    """Two launches: bit-identical gradients and outputs.  Deferred mode (out = NULL, then srl_ppo_loss_finalize on the
    workspace's slot) gives the immediate mode's bits and the same [D] gradient.  The workspace is zero after every
    launch, except the bytes a deferred launch hands to the finaliser (slot bytes 4-31: n_rows, sum(mask), weights)."""
    T, n, D = 128, 1000, 17
    hp_kw = CONFIGS["mse_dual_clip"]
    c = make_case(T, n, D, shared, seed=11)
    ref = oracle(c, hp_kw)
    ws = ops.new_gaussian_loss_workspace("cuda", T, n, D, shared)
    a = run(ops, c, hp_kw, norm_stats=ref["norm_stats"], workspace=ws)
    assert not ws.any(), "immediate mode left the workspace dirty"
    b = run(ops, c, hp_kw, norm_stats=ref["norm_stats"], workspace=ws)
    assert not ws.any()
    for x, y, name in zip(a[:5], b[:5], ("g_mean", "g_log_std", "g_value", "out", "out_f32")):
        assert torch.equal(x, y), f"{name} differs between two launches"
    g_mean, g_ls, g_v, out_d, out32_d, _, _ = run(ops, c, hp_kw, norm_stats=ref["norm_stats"], workspace=ws, defer=True)
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
def test_gaussian_autograd_function_trains_a_policy(ops):
    """A continuous-action policy: nn.Linear mean and value heads plus a state-independent nn.Parameter log_std, the loss
    through PPOGaussianLossFunction, then loss.backward().  Every parameter gradient matches the same network's through
    torch.distributions.Normal and the oracle's loss."""
    import copy
    T, n, D, F = 24, 300, 6, 11
    torch.manual_seed(0)

    class Policy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.mu = torch.nn.Linear(F, D)
            self.v = torch.nn.Linear(F, 1)
            self.log_std = torch.nn.Parameter(torch.linspace(-0.8, 0.3, D))

    pol = Policy()
    ref_pol = copy.deepcopy(pol)
    pol = pol.cuda()
    c = make_case(T, n, D, True, seed=5)
    obs = torch.randn(T, n, F)
    with torch.no_grad():
        mean0 = ref_pol.mu(obs)
        c["action"] = (mean0 + ref_pol.log_std.exp() * torch.randn(T, n, D)).numpy()
        lp0, _ = logp_entropy_from_gaussian_ref(mean0.double(), ref_pol.log_std.double(), torch.from_numpy(c["action"]).double())
        c["old_logp"][:T] = away_from_clip_edges(lp0.numpy(), (lp0 + 0.15 * torch.randn(T, n, dtype=torch.float64)).numpy())
    hp_kw = CONFIGS["huber_clip_value"]
    # oracle: the same network on the CPU, in float64 (its parameter gradients are sums over T * n transitions)
    ref_pol = ref_pol.double()
    mean_r, v_r = ref_pol.mu(obs.double()), ref_pol.v(obs.double())[..., 0]
    lp, en = logp_entropy_from_gaussian_ref(mean_r, ref_pol.log_std, torch.from_numpy(c["action"]).double())
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
    loss, out = ops.PPOGaussianLossFunction.apply(pol.mu(obs_d), pol.log_std, d("action"), pol.v(obs_d)[..., 0],
                                                  d("old_logp")[:T], d("value")[:T], d("ret")[:T], d("adv")[:T],
                                                  d("on_reset")[1:T + 1], ns, None, None, None, ops.LossHyper(**hp_kw))
    loss.backward()
    torch.cuda.synchronize()
    msum = float(mask.sum())
    assert_close_ref(loss.item(), res["loss"], what="loss")
    for (name, p), (_, q) in zip(pol.named_parameters(), ref_pol.named_parameters()):
        assert p.grad is not None, f"{name} received no gradient"
        # a weight's gradient is a sum over the 7200 transitions of terms of either sign: float32 rounding of the head's
        # gradients (1e-7 each) adds up to ~1e-4 of a typical term there, so an element is compared on the scale of its
        # tensor's largest one -- the head's gradients themselves are pinned element by element above
        scale = msum / max(1.0, float(q.grad.abs().max()) * msum)
        assert_close_ref(p.grad.cpu().double() * scale, q.grad * scale, what=f"d loss / d {name}")


def test_gaussian_host_side_argument_checks():
    """Rejected on the host before any CUDA call, with status 1 (SRL_ERR_INVALID_ARG) and a message naming the argument
    -- no GPU needed.  The non-null device pointers are never dereferenced."""
    build.build()
    lib = _lib.load_library()
    T, n, D = 4, 8, 6
    fake = 256
    hc = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 0, 1, 0)
    need = lib.srl_ppo_loss_gaussian_workspace_bytes(T, n, D, 1)
    assert need == lib.srl_ppo_loss_workspace_bytes(T, n) + 2048 * D * 8
    assert lib.srl_ppo_loss_gaussian_workspace_bytes(T, n, D, 0) == lib.srl_ppo_loss_workspace_bytes(T, n)

    def call(D=D, mean=fake, old_value=fake, ws_bytes=need, hyper=hc):
        args = dict(mean=mean, log_std=fake, shared=1, action=fake, D=D, v_pred=fake, old_logp=fake, old_value=old_value,
                    ret=fake, adv=fake, rs=fake, ld_smp=n, lane_idx=None, T=T, n=n, ns=fake, ls=fake, pm=None,
                    hyper=ctypes.byref(hyper), g_mean=fake, g_ls=fake, g_v=fake, logp=None, ent=None, out=fake,
                    out32=None, ws=fake, ws_bytes=ws_bytes, stream=None)
        rc = lib.srl_ppo_loss_from_gaussian(*args.values())
        return rc, lib.srl_last_error().decode()

    rc, msg = call(D=0)
    assert rc == 1 and "D=0" in msg, msg
    rc, msg = call(D=65)
    assert rc == 1 and "D=65" in msg, msg
    rc, msg = call(mean=None)
    assert rc == 1 and "null pointer mean" in msg, msg
    rc, msg = call(ws_bytes=need - 8)
    assert rc == 1 and "workspace too small" in msg, msg
    clip = _lib.PpoHyper(0.2, 0.2, 3.0, 0.5, 0.01, 0.0, 1e-5, 0, 1, 1, 0)
    rc, msg = call(old_value=None, hyper=clip)
    assert rc == 1 and "clip_value needs old_value" in msg, msg
