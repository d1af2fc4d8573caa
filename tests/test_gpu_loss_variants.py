"""K4, the scalar PPO loss (srl_ppo_loss_fwd_bwd_batched), on every kernel instantiation the library contains, against the
float64 oracle.

The host code picks one of five routes by sample-side form, shape, row strides and alignment (ppo_loss.cu
srl_ppo_loss_fwd_bwd_batched, ppo_loss_pair.cu loss_pair_eligible, ppo_loss.cuh launch_loss_mode / launch_loss_static), and
one hyper-parameter configuration per route: 53 instantiations in all.  CASES names, for every row, the instantiation its
inputs route to; `expected_kernel` restates the routing rules, the profiler shows which kernel actually ran, and a CPU test
checks that the table names every instantiation in the built library.

The sample side (leaves, K2's loss pack, lane_aos, minibatch_part) is built on the host from the oracle's adv / ret, so the
matrix does not depend on which scan kernel would have written it.  Per case: loss scalars, statistics and gradients against
oracle/ref_math.ppo_loss_ref, the exact parts of the contract (mask count, zero tail, float32 copies, clip count, masked and
entropy gradients), no byte written outside the gradients' [T, n] views (gap columns of strided rows included), the
workspace slot left as include/srl_b200.h documents, a second launch bit-identical, every problem of a batch bit-identical
to its own launch, and a deferred launch against its immediate twin.
"""
import ctypes
import dataclasses
import re
import zlib
from typing import Optional

import numpy as np
import pytest
import torch

from oracle import ref_math as M
from tests.kernel_variants import F32_SENTINEL, Guarded, launched, library_kernels
from tests.util import assert_close_ref

GAMMA, LMBDA = 0.995, 0.9
EPS_CLIP, C_CLIP, WV, WE = 0.2, 3.0, 0.5, 0.01
PACK_MASKED_ADV = 0x7FC00000  # gae_common.cuh kPackMaskedAdv
MAX_BATCH = 32  # SRL_MAX_LOSS_BATCH
EDGE = 4e-7  # |ratio - (1 +- eps)| of a clipped-surrogate decision boundary (test_gpu_parity.test_loss_full_size_lane_subset)
VL_CODE = {"mse": 0, "huber": 1, "smoothl1": 2}
STAT_SLOTS = dict(advantage=4, importance_weight=5, clip_ratio=6, value_targets=7, denorm_value=8)


# ---------------------------------------------------------------------------------------------------------------------
# Routing: ppo_loss.cu srl_ppo_loss_fwd_bwd_batched, ppo_loss_pair.cu loss_pair_eligible / launch_loss_pair,
# ppo_loss.cuh launch_loss_mode / launch_loss_static, ppo_loss_pack.cu launch_loss_pack.  No rule depends on the SM count.
# ---------------------------------------------------------------------------------------------------------------------
def _b(x: bool) -> str:
    return "true" if x else "false"


def cfg_name(vl: str, clip: bool, dual: bool, popart: bool) -> str:
    """The element-math configuration of the four-lane and pair kernels: StaticCfg for {mse, huber}, else RuntimeCfg."""
    if vl == "smoothl1":
        return "RuntimeCfg"
    return f"StaticCfg<{VL_CODE[vl]}, {_b(clip)}, {_b(dual)}, {_b(popart)}>"


def expected_kernel(n: int, ld_pol: int, ld_grad: int, pol16: bool, pol8: bool, smp_vec: bool, pack: bool, has_idx: bool,
                    lane_aos: bool, vl: str, clip: bool, dual: bool, popart: bool) -> Optional[str]:
    """The instantiation srl_ppo_loss_fwd_bwd_batched launches, or None when the call is refused (SRL_ERR_UNSUPPORTED).
    pol16 / pol8: every policy-side tensor, gradient and lane_idx of every problem 16- / 8-byte aligned; smp_vec: the sample
    leaves allow 128-bit loads (ld_smp % 4 == 0, 16-byte aligned float leaves, 4-byte aligned flags; never with a pack)."""
    dense_ok = n % 4 == 0 and ld_pol % 4 == 0 and ld_grad % 4 == 0 and pol16
    pair = pack and pol8 and n % 2 == 0 and ld_pol % 2 == 0 and ld_grad % 2 == 0 and (not lane_aos or n <= 1024)
    if lane_aos and not pair:
        return None
    cfg = cfg_name(vl, clip, dual, popart)
    if pack:
        return f"ppo_loss_pair_kernel<{cfg}>" if pair else "ppo_loss_kernel<1, 2, RuntimeCfg>"
    if not has_idx and dense_ok and smp_vec:
        return f"ppo_loss_kernel<4, 0, {cfg}>"
    return f"ppo_loss_kernel<4, 1, {cfg}>" if dense_ok else "ppo_loss_kernel<1, 1, RuntimeCfg>"


_K4_RE = re.compile(r"\b(ppo_loss_kernel|ppo_loss_pair_kernel)<")


def _split_top(s: str):
    """Template arguments split at the commas outside nested <...>."""
    parts, depth, cur = [], 0, []
    for ch in s:
        depth += (ch == "<") - (ch == ">")
        if ch == "," and depth == 0:
            parts.append("".join(cur))
            cur = []
        else:
            cur.append(ch)
    parts.append("".join(cur))
    return parts


def _norm_arg(a: str) -> str:
    a = re.sub(r"\b\w+::", "", a.strip())  # srl::loss::StaticCfg -> StaticCfg
    m = re.fullmatch(r"(\w+)\s*<(.*)>", a, re.S)
    if m:
        return f"{m.group(1)}<{', '.join(_norm_arg(x) for x in _split_top(m.group(2)))}>"
    m = re.fullmatch(r"\(bool\)([01])", a)
    if m:
        return _b(m.group(1) == "1")
    m = re.fullmatch(r"(?:\((?:unsigned )?\w+\))?(-?\d+)[uUlL]*", a)
    if m:
        return str(int(m.group(1)))  # (int)4 -> 4
    return a


def kernel_id(name: str) -> Optional[str]:
    """A demangled K4 kernel name (profiler or cu++filt spelling, nested StaticCfg<...> included) -> "name<args>" with
    namespaces dropped and `true`/`false`/`(bool)1`, `4`/`(int)4` written one way; None for any other kernel."""
    m = _K4_RE.search(name)
    if m is None:
        return None
    depth, j = 1, m.end()
    while depth and j < len(name):
        depth += (name[j] == "<") - (name[j] == ">")
        j += 1
    return f"{m.group(1)}<{', '.join(_norm_arg(a) for a in _split_top(name[m.end():j - 1]))}>"


# ---------------------------------------------------------------------------------------------------------------------
# The case table
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class Case:
    kernel: str  # the instantiation these inputs route to
    T: int
    n: int
    vl: str = "mse"
    clip: bool = False
    dual: bool = False
    popart: bool = False
    pack: bool = False  # sample side: K2's pack (else the five leaves)
    N: Optional[int] = None  # sample lanes (the pack's N); None = n
    row_lo: int = 0  # sample row of loss row 0 (pack_row_lo)
    # None; "perm" (random lanes of N); "arange"; "env4" / "env2mix" (environments of 4 / 2 agents: every thread of the
    # four-lane gather takes the run of four / half of them do); "env4+2" (environments of 4 shifted by 2 lanes: consecutive
    # runs that are not 4-aligned)
    idx: Optional[str] = None
    pol_off: int = 0  # policy-side tensors, gradients and lane_idx: elements past a 256-byte boundary
    smp_off: int = 0  # sample leaves: elements past a 256-byte boundary
    ld_pol: Optional[int] = None  # row strides (elements); None = n
    ld_grad: Optional[int] = None
    problems: int = 1
    defer: bool = False
    stats: str = "norm"  # "norm" (norm_stats / local_stats), "aos" (lane_aos), "part" (lane_aos + minibatch_part)
    veps: Optional[float] = None  # value_eps_clip; None = eps_clip
    norm_old: bool = False  # normalize_old_value
    descending: bool = False  # new_logp / v_pred / entropy (and the gradients) carved from one buffer, high to low

    @property
    def lanes(self) -> int:
        return self.N if self.N is not None else self.n

    @property
    def lp(self) -> int:
        return self.ld_pol if self.ld_pol is not None else self.n

    @property
    def lg(self) -> int:
        return self.ld_grad if self.ld_grad is not None else self.n


STATIC = [(vl, c, d, p) for vl in ("mse", "huber") for c in (False, True) for d in (False, True) for p in (False, True)]


def _hname(vl, clip, dual, popart) -> str:
    return vl + ("-clip" if clip else "") + ("-dual" if dual else "") + ("-pa" if popart else "")


def _hk(vl, clip, dual, popart) -> dict:
    return dict(vl=vl, clip=clip, dual=dual, popart=popart)


def _dense(h, T, n, **kw):
    return Case(f"ppo_loss_kernel<4, 0, {cfg_name(*h)}>", T, n, **_hk(*h), **kw)


def _gather4(h, T, n, **kw):
    return Case(f"ppo_loss_kernel<4, 1, {cfg_name(*h)}>", T, n, **_hk(*h), **kw)


def _pair(h, T, n, **kw):
    return Case(f"ppo_loss_pair_kernel<{cfg_name(*h)}>", T, n, pack=True, **_hk(*h), **kw)


G1 = "ppo_loss_kernel<1, 1, RuntimeCfg>"
PK1 = "ppo_loss_kernel<1, 2, RuntimeCfg>"
SL1 = ("smoothl1", True, True, False)
SL1_PA = ("smoothl1", False, False, True)

# one edge per static configuration and route, in STATIC's order
_DENSE_EDGES = [dict(T=1, n=64), dict(T=9, n=4), dict(T=9, n=516), dict(T=5, n=2052), dict(T=1001, n=64),
                dict(T=33, n=256, problems=3), dict(T=16, n=128, defer=True), dict(T=12, n=96, row_lo=3),
                dict(T=1, n=4), dict(T=9, n=516, defer=True), dict(T=7, n=2052), dict(T=1001, n=64, problems=2),
                dict(T=64, n=512, ld_pol=516, ld_grad=520), dict(T=8, n=1024), dict(T=13, n=36, row_lo=1),
                dict(T=40, n=200, problems=5, defer=True)]
_GATHER4_EDGES = [dict(T=9, n=256, N=1024, idx="perm"), dict(T=16, n=512, N=1024, idx="env4"),
                  dict(T=16, n=512, N=1026, idx="env4+2"), dict(T=33, n=512, N=2048, idx="env2mix"),
                  dict(T=12, n=256, N=1024, idx="perm", smp_off=1), dict(T=12, n=256, smp_off=1),
                  dict(T=1, n=4, N=64, idx="perm"), dict(T=9, n=1024, N=4096, idx="env4", problems=4, defer=True),
                  dict(T=20, n=2052, N=4096, idx="perm"), dict(T=17, n=256, N=1026, idx="env4+2", defer=True),
                  dict(T=8, n=512, N=2048, idx="env2mix", problems=3), dict(T=30, n=128, smp_off=1, row_lo=2),
                  dict(T=24, n=256, N=512, idx="perm", ld_pol=260, ld_grad=268), dict(T=9, n=516, N=600, idx="env4"),
                  dict(T=9, n=64, N=300, idx="perm", smp_off=1), dict(T=50, n=1024, N=1024, idx="arange")]
_PAIR_EDGES = [dict(T=1, n=128, N=1024, idx="perm", row_lo=1), dict(T=2, n=128, N=1024, idx="perm", row_lo=1),
               dict(T=7, n=130, N=512, idx="env4", row_lo=3), dict(T=10, n=130, N=512, idx="perm", row_lo=5),
               dict(T=1, n=2, N=64, idx="perm", row_lo=0), dict(T=2, n=128, row_lo=2),  # T = 2 at an even row: cpp = 1
               dict(T=9, n=1024, N=4096, idx="perm", row_lo=4), dict(T=12, n=256, row_lo=0, problems=2),
               dict(T=257, n=1000, N=2048, idx="perm", row_lo=1, problems=32),
               dict(T=5, n=64, N=256, idx="perm", row_lo=1, problems=33, defer=True),
               dict(T=16, n=256, N=1024, idx="perm", row_lo=2, defer=True), dict(T=33, n=130, N=256, idx="env2mix", row_lo=1),
               dict(T=24, n=256, N=512, idx="perm", ld_pol=260, ld_grad=258), dict(T=11, n=512, N=512, idx="perm", row_lo=6),
               dict(T=20, n=128, N=256, idx="perm", row_lo=3, descending=True), dict(T=3, n=1024, row_lo=1, defer=True)]

CASES = {}
for (h, e) in zip(STATIC, _DENSE_EDGES):
    CASES[f"dense-{_hname(*h)}"] = _dense(h, **e)
for (h, e) in zip(STATIC, _GATHER4_EDGES):
    CASES[f"gather4-{_hname(*h)}"] = _gather4(h, **e)
for (h, e) in zip(STATIC, _PAIR_EDGES):
    CASES[f"pair-{_hname(*h)}"] = _pair(h, **e)
CASES.update({
    # ---- smoothl1 (RuntimeCfg) on the three routes that also have static configurations --------------------------------
    "dense-smoothl1": _dense(SL1, 9, 132),
    "dense-smoothl1-pa-defer": _dense(SL1_PA, 17, 64, defer=True, problems=2),
    "gather4-smoothl1": _gather4(SL1, 10, 256, N=1024, idx="env4"),
    "gather4-smoothl1-pa": _gather4(SL1_PA, 10, 128, smp_off=1),
    "pair-smoothl1": _pair(SL1, 10, 256, N=1024, idx="perm", row_lo=1),
    "pair-smoothl1-pa-veps": _pair(SL1_PA, 9, 130, N=512, idx="perm", row_lo=2, veps=0.5),
    # ---- gather, one lane per thread (odd widths, or 4-byte aligned policy tensors) --------------------------------------
    "gather1-n1": Case(G1, 9, 1, **_hk(*SL1)),
    "gather1-n1-idx": Case(G1, 8, 1, N=7, idx="perm", **_hk("huber", True, False, True)),
    "gather1-n5": Case(G1, 13, 5, **_hk("mse", False, True, False)),
    "gather1-n5-idx": Case(G1, 4, 5, N=40, idx="perm", **_hk("mse", True, False, True), norm_old=True),
    "gather1-n1029": Case(G1, 9, 1029, **_hk("huber", True, True, False), defer=True),
    "gather1-n1029-idx": Case(G1, 10, 1029, N=2048, idx="perm", **_hk(*SL1), problems=3),
    "gather1-pol-offset": Case(G1, 12, 256, pol_off=1, **_hk("huber", False, True, True)),
    "gather1-stride-odd": Case(G1, 12, 256, ld_pol=257, ld_grad=259, **_hk("mse", True, True, False)),
    # ---- pack, row tile: one lane per thread (odd widths, 4-byte aligned policy tensors, odd strides) --------------------
    "pack-n1": Case(PK1, 9, 1, pack=True, N=16, idx="perm", row_lo=1, **_hk("mse", True, True, True)),
    "pack-n37": Case(PK1, 12, 37, pack=True, row_lo=2, **_hk(*SL1)),
    "pack-n1023": Case(PK1, 11, 1023, pack=True, N=2048, idx="perm", row_lo=3, **_hk("huber", True, False, False),
                       defer=True),
    "pack-pol-offset-odd-row": Case(PK1, 10, 256, pack=True, N=1024, idx="perm", row_lo=1, pol_off=1,
                                    **_hk("huber", False, False, True)),
    "pack-pol-offset-even-row": Case(PK1, 7, 256, pack=True, row_lo=4, pol_off=1, problems=2, **_hk(*SL1_PA)),
    "pack-stride-odd": Case(PK1, 12, 256, pack=True, N=1024, idx="perm", row_lo=1, ld_pol=259, ld_grad=262,
                            **_hk("mse", True, True, False)),
    # ---- pair kernel: statistics sources, hyper-parameters, the lane_aos width limit ------------------------------------
    "pair-aos": _pair(("mse", True, True, False), 16, 256, N=1024, idx="perm", row_lo=1, stats="aos"),
    "pair-aos-defer": _pair(("huber", False, True, False), 16, 256, N=1024, idx="perm", row_lo=1, stats="aos",
                            defer=True, problems=3),
    "pair-aos-n1024": _pair(("mse", False, False, False), 2, 1024, N=1024, idx="env4", row_lo=0, stats="aos"),
    "pair-aos-cta1": _pair(("huber", True, False, False), 2, 128, N=512, idx="perm", row_lo=0, stats="aos"),
    "pair-part": _pair(("huber", True, True, False), 12, 512, N=2048, idx="perm", row_lo=3, stats="part", problems=4),
    "pair-part-defer": _pair(("mse", True, False, False), 9, 256, N=1000, idx="env2mix", row_lo=1, stats="part",
                             defer=True, problems=2),
    "pair-popart-normold-clip": _pair(("huber", True, False, True), 14, 256, N=512, idx="perm", row_lo=1, norm_old=True),
    "pair-veps": _pair(("mse", True, True, False), 14, 256, N=512, idx="perm", row_lo=2, veps=0.05),
    "pair-aos-stride": _pair(("huber", True, False, False), 15, 256, N=1024, idx="perm", row_lo=1, stats="aos",
                             ld_pol=300, ld_grad=262),
})

# one set of inputs on every route its shape allows (test_routes_agree)
CROSS = {"mse-clip-dual-pa": ("mse", True, True, True), "huber-clip": ("huber", True, False, False),
         "smoothl1-clip-dual": SL1}


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table covers the library; the name normaliser; the refused width
# ---------------------------------------------------------------------------------------------------------------------
def test_case_table_names_every_loss_instantiation_in_the_library():
    """The set of ppo_loss_kernel / ppo_loss_pair_kernel instantiations in libsrl_b200.so (cuobjdump -symbols | cu++filt) is
    the set CASES names: 16 static configurations + RuntimeCfg on the dense, four-lane gather and pair routes, RuntimeCfg on
    the one-lane gather and pack routes."""
    built = library_kernels(kernel_id)
    assert len(built) == 53, sorted(built)
    named = {c.kernel for c in CASES.values()}
    assert built == named, f"in the library only: {sorted(built - named)}; in the table only: {sorted(named - built)}"


def test_kernel_names_normalise_both_spellings():
    cuobj = ("void srl::loss::ppo_loss_kernel<(int)4, (int)1, srl::loss::StaticCfg<(int)1, (bool)0, (bool)1, (bool)1>>"
             "(srl::loss::LossBatch)")
    prof = "void srl::loss::ppo_loss_kernel<4, 1, srl::loss::StaticCfg<1, false, true, true> >(srl::loss::LossBatch)"
    assert kernel_id(cuobj) == kernel_id(prof) == "ppo_loss_kernel<4, 1, StaticCfg<1, false, true, true>>"
    pc = ("void srl::loss::<unnamed>::ppo_loss_pair_kernel<srl::loss::RuntimeCfg>(srl::loss::LossBatch, "
          "srl::loss::<unnamed>::PairSched)")
    pp = ("void srl::loss::(anonymous namespace)::ppo_loss_pair_kernel<srl::loss::RuntimeCfg>(srl::loss::LossBatch, "
          "srl::loss::(anonymous namespace)::PairSched)")
    assert kernel_id(pc) == kernel_id(pp) == "ppo_loss_pair_kernel<RuntimeCfg>"
    assert kernel_id("void srl::loss::<unnamed>::ppo_loss_logits_kernel<(bool)1, (bool)0, float, (bool)0>(x)") is None
    assert kernel_id("void srl::loss::<unnamed>::loss_finalize_kernel(unsigned char *, unsigned long, double *, float *)") is None


def test_lane_aos_width_limit_is_refused():
    """lane_aos needs the pair kernel, which adds a minibatch's lane items for at most 1024 lanes: n = 1026 is refused;
    without lane_aos the same shape runs the pair kernel."""
    kw = dict(ld_pol=1026, ld_grad=1026, pol16=True, pol8=True, smp_vec=False, pack=True, has_idx=True, vl="mse",
              clip=False, dual=True, popart=False)
    assert expected_kernel(1026, lane_aos=True, **kw) is None
    assert expected_kernel(1026, lane_aos=False, **kw) == "ppo_loss_pair_kernel<StaticCfg<0, false, true, false>>"
    assert expected_kernel(1024, lane_aos=True, **kw) == "ppo_loss_pair_kernel<StaticCfg<0, false, true, false>>"
    # with a pack, the four-lane conditions imply the pair kernel's (ppo_loss_pack.cu)
    for n, lp, lg, a16, a8 in [(n, lp, lg, a16, a8) for n in (4, 6, 7) for lp in (n, n + 1, n + 2, n + 4)
                               for lg in (n, n + 2, n + 3) for a16 in (True, False) for a8 in (True, False) if a8 or not a16]:
        k = expected_kernel(n, lp, lg, a16, a8, False, True, True, False, "mse", False, False, False)
        dense_ok = n % 4 == 0 and lp % 4 == 0 and lg % 4 == 0 and a16
        assert not dense_ok or k.startswith("ppo_loss_pair_kernel<")


def test_case_table_covers_the_routes_asked_of_it():
    for route in ("ppo_loss_kernel<4, 0, ", "ppo_loss_kernel<4, 1, ", "ppo_loss_pair_kernel<"):
        cfgs = {c.kernel for c in CASES.values() if c.kernel.startswith(route)}
        assert len(cfgs) == 17, (route, sorted(cfgs))
    assert len(CASES) >= 53
    for name, c in CASES.items():
        assert c.stats == "norm" or (c.pack and c.idx is not None and not c.popart), name
        assert c.stats != "part" or c.problems <= MAX_BATCH, name


# ---------------------------------------------------------------------------------------------------------------------
# Inputs (host) and device placement
# ---------------------------------------------------------------------------------------------------------------------
def _lanes(case: Case, g: torch.Generator) -> torch.Tensor:
    n, N = case.n, case.lanes
    if case.idx in (None, "arange"):
        return torch.arange(n)
    if case.idx == "perm":
        return torch.randperm(N, generator=g)[:n]
    if case.idx in ("env4", "env4+2"):
        shift = 2 if case.idx == "env4+2" else 0
        env = torch.randperm((N - shift) // 4, generator=g)
        return ((env[:, None] * 4 + torch.arange(4)).reshape(-1) + shift)[:n]
    assert case.idx == "env2mix"  # blocks of two 2-agent environments; every other block has its two environments swapped
    blk = torch.randperm(N // 4, generator=g)
    order = torch.where((torch.arange(blk.numel()) % 2 == 0)[:, None], torch.arange(4), torch.tensor([2, 3, 0, 1]))
    return (blk[:, None] * 4 + order).reshape(-1)[:n]


def _popart(g: torch.Generator) -> M.RunningMeanStdRef:
    pa = M.RunningMeanStdRef((1,), beta=0.99)
    pa.update(torch.randn((64, 1), generator=g) * 2.5 + 0.7)
    return pa


def _inputs(seed: str, case: Case) -> dict:
    """Seeded host inputs: the [L, N] sample (GAE from the oracle), each problem's lanes and policy outputs.  They depend on
    the seed, the shape and the hyper-parameters only, not on the route."""
    g = torch.Generator().manual_seed(zlib.crc32(seed.encode()))
    T, n, N, lo = case.T, case.n, case.lanes, case.row_lo
    L = lo + T + 1
    flag = lambda p: (torch.rand((L, N), generator=g) < p).to(torch.uint8)
    reward, value = torch.randn((L, N), generator=g) * 4.0, torch.randn((L, N), generator=g) * 4.0
    done, truncated, on_reset = flag(0.05), flag(0.02), flag(0.12)
    old_logp = -torch.rand((L, N), generator=g) * 3.0
    pa = _popart(g) if case.popart else None
    adv, ret = M.adv_and_value_target_ref(reward, value, truncated, done, on_reset, GAMMA, LMBDA, popart=pa)
    adv, ret = M.pad_last_row(adv), M.pad_last_row(ret)
    veps = EPS_CLIP if case.veps is None else case.veps
    x = dict(L=L, old_logp=old_logp, value=value, ret=ret, adv=adv, on_reset=on_reset, popart=pa, lanes=[], pol=[])
    for _ in range(case.problems):
        li = _lanes(case, g)
        rows = slice(lo, lo + T)
        ol, ov, rt = old_logp[rows][:, li], value[rows][:, li], ret[rows][:, li]
        mask = on_reset[lo + 1:lo + T + 1][:, li] == 0
        nl = ol + torch.randn((T, n), generator=g) * 0.25  # ratios on both sides of 1 +- eps
        nl[(~mask) & (torch.rand((T, n), generator=g) < 0.5)] = -float("inf")  # dead agents
        tgt = pa.normalize(rt) if pa is not None else rt  # PopArt clips some of these returns to +-5
        ovn = pa.normalize(ov) if (pa is not None and case.norm_old) else ov
        vp = tgt + torch.randn((T, n), generator=g) * 1.5  # Huber / smoothl1 differences on both sides of 1
        if case.clip:  # half the predictions inside the value-clip window: |da| == |db| ties
            near = ovn + (torch.rand((T, n), generator=g) * 2 - 1) * veps
            vp = torch.where(torch.rand((T, n), generator=g) < 0.5, near, vp)
        en = torch.rand((T, n), generator=g) * 2.0
        x["lanes"].append(li)
        x["pol"].append((nl.contiguous(), vp.contiguous(), en.contiguous()))
    return x


def _masked_sums(x: dict, case: Case, li: torch.Tensor):
    """float64 {sum mask, sum adv * mask, sum (adv * mask)^2} over the loss rows of the given lanes, per lane."""
    lo = case.row_lo
    m = (x["on_reset"][lo + 1:lo + case.T + 1][:, li] == 0).double()
    a = x["adv"][lo:lo + case.T][:, li].double() * m
    return torch.stack([m.sum(0), a.sum(0), a.square().sum(0)], 1)


def _pack(x: dict, N: int) -> torch.Tensor:
    """K2's pair-interleaved pack [ceil(L/2), N, 2, 4] of the sample: {old_logp, value, ret, mask ? adv : NaN}."""
    L = x["L"]
    P = (L + 1) // 2
    rows = torch.zeros((2 * P, N, 4))
    rows[:L, :, 0], rows[:L, :, 1], rows[:L, :, 2], rows[:L, :, 3] = x["old_logp"], x["value"], x["ret"], x["adv"]
    keep = torch.zeros((2 * P, N), dtype=torch.bool)
    keep[:L - 1] = x["on_reset"][1:] == 0
    bits = rows.view(torch.int32)
    bits[..., 3][~keep] = PACK_MASKED_ADV
    return rows.view(P, 2, N, 4).permute(0, 2, 1, 3).contiguous()


def _place(x: torch.Tensor, off: int) -> torch.Tensor:
    """x on the device, contiguous, its base `off` elements past a 256-byte boundary."""
    buf = torch.empty(x.numel() + off, dtype=x.dtype, device="cuda")
    out = buf[off:].view(x.shape)
    out.copy_(x)
    return out


def _slot(rows: int, ld: int) -> int:
    return -(-rows * ld // 64) * 64  # arrays of a carved buffer start 256 bytes apart (alignment shared with the base)


class Device:
    """A case's inputs on the device: sample side, per problem the policy tensors (carved from one buffer, rows of stride
    ld_pol, gap columns NaN), lane_idx and statistics."""

    def __init__(self, case: Case, x: dict):
        T, n, N, lo = case.T, case.n, case.lanes, case.row_lo
        self.case, self.x = case, x
        self.ptr_leaf = {}
        if case.pack:
            self.pack = _pack(x, N).cuda()
        else:
            self.leaf = {k: _place(x[k], case.smp_off) for k in ("old_logp", "value", "ret", "adv", "on_reset")}
            fs = 4
            self.ptr_leaf = dict(old_logp=self.leaf["old_logp"].data_ptr() + lo * N * fs,
                                 old_value=self.leaf["value"].data_ptr() + lo * N * fs if case.clip else None,
                                 ret=self.leaf["ret"].data_ptr() + lo * N * fs, adv=self.leaf["adv"].data_ptr() + lo * N * fs,
                                 on_reset_next=self.leaf["on_reset"].data_ptr() + (lo + 1) * N)
        S = _slot(T, case.lp)
        order = (2, 1, 0) if case.descending else (0, 1, 2)
        self.pol, self.pol_ptr, self.idx, self.sums = [], [], [], []
        for k in range(case.problems):
            buf = torch.full((3 * S + case.pol_off,), float("nan"))
            for a, t in zip(order, x["pol"][k]):
                v = buf[case.pol_off + a * S:case.pol_off + a * S + T * case.lp].view(T, case.lp)
                v[:, :n] = t
            buf = buf.cuda()
            self.pol.append(buf)
            self.pol_ptr.append([buf.data_ptr() + 4 * (case.pol_off + a * S) for a in order])
            li = x["lanes"][k].to(torch.int32)
            self.idx.append(_place(li, case.pol_off) if case.idx is not None else None)
            s = _masked_sums(x, case, x["lanes"][k]).sum(0)
            self.sums.append(s)
        self.norm = [torch.tensor([s[0], s[1], s[2]], dtype=torch.float64, device="cuda") for s in self.sums]
        self.local = [torch.tensor([s[0]], dtype=torch.float64, device="cuda") for s in self.sums]
        self.popart = None
        if x["popart"] is not None:
            m, sd = x["popart"].mean_std()
            self.popart = torch.tensor([m.item(), sd.item()], dtype=torch.float64, device="cuda")
        self.aos = self.part = None
        if case.stats in ("aos", "part"):
            aos = torch.zeros((N, 4), dtype=torch.float64)
            aos[:, :3] = _masked_sums(x, case, torch.arange(N))
            self.aos = aos.cuda()
            if case.stats == "part":
                ctas = (N + 31) // 32
                part = torch.zeros((MAX_BATCH, ctas, 4), dtype=torch.float64)
                for k, li in enumerate(x["lanes"]):
                    part[self.part_first + k].index_add_(0, li // 32, aos[li])
                self.part = part.cuda()

    @property
    def part_first(self) -> int:
        return MAX_BATCH - self.case.problems

    def flags(self) -> dict:
        """The alignment facts the host routing reads, from the actual pointers."""
        case = self.case
        pol = [p for ps in self.pol_ptr for p in ps] + [t.data_ptr() for t in self.idx if t is not None]
        # gradients share the policy side's offset inside a 256-byte aligned buffer (Out)
        ok = lambda a: all(p % a == 0 for p in pol) and (4 * case.pol_off) % a == 0
        smp_vec = False
        if not case.pack:
            lp = self.ptr_leaf
            fl = [lp["old_logp"], lp["ret"], lp["adv"]] + ([lp["old_value"]] if case.clip else [])
            smp_vec = case.lanes % 4 == 0 and all(p % 16 == 0 for p in fl) and lp["on_reset_next"] % 4 == 0
        return dict(pol16=ok(16), pol8=ok(8), smp_vec=smp_vec)


class Out:
    """The outputs of one launch: per problem the three gradients carved from one guarded buffer (rows of stride ld_grad),
    out [problems, 16] and out_f32 [problems, 4], guarded as well; a zeroed workspace slot per problem."""

    def __init__(self, case: Case, problems: int):
        T, n = case.T, case.n
        self.S = _slot(T, case.lg)
        self.order = (2, 1, 0) if case.descending else (0, 1, 2)
        self.grad = [Guarded((3 * self.S + case.pol_off,), torch.float32) for _ in range(problems)]
        self.out = Guarded((problems, 16), torch.float64)
        self.out32 = Guarded((problems, 4), torch.float32)
        from srl_b200 import ops
        self.ws = ops.new_loss_workspace("cuda", slots=problems)
        written = torch.zeros(3 * self.S + case.pol_off, dtype=torch.bool)
        for a in self.order:
            written[case.pol_off + a * self.S:case.pol_off + a * self.S + T * case.lg].view(T, case.lg)[:, :n] = True
        self.written = written
        self.case = case

    def grad_ptrs(self, k: int):
        return [self.grad[k].t.data_ptr() + 4 * (self.case.pol_off + a * self.S) for a in self.order]

    def grads(self, k: int):
        """g_logp, g_value, g_entropy of problem k as [T, n] host tensors."""
        c = self.case
        t = self.grad[k].t.cpu()
        return [t[c.pol_off + a * self.S:c.pol_off + a * self.S + c.T * c.lg].view(c.T, c.lg)[:, :c.n] for a in self.order]

    def bits(self) -> list:
        return [g.buf.view(torch.int32).clone() for g in self.grad] + [self.out.buf.view(torch.int64).clone(),
                                                                        self.out32.buf.view(torch.int32).clone()]


def _hyper(case: Case):
    from srl_b200 import ops
    vcfg = {"huber": {"delta": 1.0}, "smoothl1": {"beta": 1.0}}.get(case.vl)
    kw = dict(eps_clip=EPS_CLIP, clip_value=case.clip, value_eps_clip=case.veps, dual_clip=case.dual, c_clip=C_CLIP,
              value_loss=case.vl, value_loss_config=vcfg, value_loss_weight=WV, entropy_bonus_weight=WE,
              normalize_old_value=case.norm_old)
    return ops.LossHyper(**kw), M.LossHyper(**kw)


def _run(case: Case, dv: Device, which=None, defer: Optional[bool] = None, o: Optional[Out] = None) -> Out:
    """One srl_ppo_loss_fwd_bwd_batched call over the problems `which` (consecutive; default all), then, deferred,
    srl_ppo_loss_finalize over their slots.  `o`: fresh outputs allocated beforehand (so that a profiled call launches
    nothing but the loss)."""
    from srl_b200 import _lib, ops
    which = list(range(case.problems)) if which is None else which
    defer = case.defer if defer is None else defer
    o = Out(case, len(which)) if o is None else o
    arr = (_lib.LossProblem * len(which))()
    for i, k in enumerate(which):
        nl, vp, en = dv.pol_ptr[k]
        g = o.grad_ptrs(i)
        idx = dv.idx[k]
        arr[i] = _lib.LossProblem(nl, vp, en, idx.data_ptr() if idx is not None else None,
                                  None if dv.aos is not None else dv.norm[k].data_ptr(),
                                  None if dv.aos is not None else dv.local[k].data_ptr(), g[0], g[1], g[2],
                                  None if defer else o.out.t[i].data_ptr(), None if defer else o.out32.t[i].data_ptr(),
                                  o.ws[i].data_ptr())
    lp = dv.ptr_leaf
    hc = _hyper(case)[0].to_c()
    part_ctas = dv.part.shape[1] if dv.part is not None else 0
    _lib.call("srl_ppo_loss_fwd_bwd_batched", arr, len(which), case.lp, case.lg, lp.get("old_logp"), lp.get("old_value"),
              lp.get("ret"), lp.get("adv"), lp.get("on_reset_next"), case.lanes,
              dv.pack.data_ptr() if case.pack else None, case.row_lo, dv.aos.data_ptr() if dv.aos is not None else None,
              dv.part.data_ptr() if dv.part is not None else None, part_ctas, dv.part_first + which[0] if dv.part is not None else 0,
              case.T, case.n, dv.popart.data_ptr() if dv.popart is not None else None, ctypes.byref(hc), o.ws.shape[1], None,
              torch.cuda.current_stream().cuda_stream)
    if defer:
        ops.loss_finalize(o.ws, o.out.t, o.out32.t)
    return o


# ---------------------------------------------------------------------------------------------------------------------
# Checks
# ---------------------------------------------------------------------------------------------------------------------
def _check_problem(case: Case, x: dict, dv: Device, o: Out, k: int, i: int, what: str) -> int:
    """Problem k (row i of the launch's outputs) against the oracle and the contract; returns its excused elements."""
    T, n, lo = case.T, case.n, case.row_lo
    li = x["lanes"][k]
    rows = slice(lo, lo + T)
    ol, ov, rt, ad = (x[key][rows][:, li] for key in ("old_logp", "value", "ret", "adv"))
    valid = x["on_reset"][lo + 1:lo + T + 1][:, li] == 0
    mask = valid.float()
    nl, vp, en = x["pol"][k]
    s = dv.sums[k]
    hp = _hyper(case)[1]
    ref = M.ppo_loss_ref(nl, ol, vp, ov, rt, ad, en, mask, hp, popart=x["popart"], global_sums=(s[0], s[1], s[2]))
    out, out32 = o.out.t[i].cpu().numpy(), o.out32.t[i].cpu().numpy()
    Msum = float(mask.sum())
    # exact parts of the contract
    assert out[9] == Msum, f"{what}: out[9] = {out[9]}, sum(mask) = {Msum}"
    assert not out[10:].any(), f"{what}: out[10..15] not zero: {out[10:]}"
    assert np.array_equal(out32, out[:4].astype(np.float32)), f"{what}: out_f32 != float(out[0..3])"
    for slot, key in ((0, "loss"), (1, "policy_loss"), (2, "value_loss"), (3, "entropy_loss")):
        assert_close_ref(out[slot], ref[key], what=f"{what} {key}")
        assert_close_ref(out32[slot], ref[key], what=f"{what} {key} (float32)")
    for key, slot in STAT_SLOTS.items():
        if key in ref["stats"]:
            assert_close_ref(out[slot], ref["stats"][key], what=f"{what} {key}")
    if not case.popart:
        assert out[8] == 0.0, f"{what}: denorm_value without PopArt"
    ratio = (nl.double() - ol.double()).exp()
    edge = valid & (((ratio - (1 - EPS_CLIP)).abs() <= EDGE) | ((ratio - (1 + EPS_CLIP)).abs() <= EDGE))
    n_edge = int(edge.sum())
    clips = round(ref["stats"]["clip_ratio"] * Msum)
    assert abs(round(out[6] * Msum) - clips) <= n_edge, f"{what}: clip count {round(out[6] * Msum)}, oracle {clips}"
    # gradients: the O(1) scale on valid transitions; exact zeros on masked ones, dead agents included
    g = o.grads(i)
    excused = 0
    for name, got in zip(("g_logp", "g_value", "g_entropy"), g):
        assert bool(torch.isfinite(got).all()), f"{what}: {name} not finite"
        assert bool((got[~valid] == 0).all()), f"{what}: {name} of masked transitions not zero"
        a, b = got.double() * Msum, ref[name].double() * Msum
        bad = valid & ((a - b).abs() > 1e-5 * b.abs().clamp(min=1.0))
        if name == "g_logp":
            excused += int((bad & edge).sum())
            bad = bad & ~edge
        assert not bool(bad.any()), f"{what}: {name}: {int(bad.sum())} of {int(valid.sum())} outside 1e-5 at the O(1) scale"
    ge = np.float32(-np.float32(WE)) * (np.float32(1.0) / np.float32(Msum))
    assert bool((g[2][valid] == torch.tensor(ge)).all()), f"{what}: g_entropy != -we * (1/M as float32)"
    return excused


def _check_guards(o: Out, what: str):
    for k, gb in enumerate(o.grad):
        assert gb.guards_intact(), f"{what}: problem {k}: written before / after its gradient buffer"
        b = gb.t.view(torch.int32).cpu()
        assert bool((b[~o.written] == F32_SENTINEL).all()), f"{what}: problem {k}: written outside the [T, n] views"
        assert bool((b[o.written] != F32_SENTINEL).all()), f"{what}: problem {k}: a gradient element was not written"
    for name, gb in (("out", o.out), ("out_f32", o.out32)):
        assert gb.guards_intact(), f"{what}: {name} written outside its rows"


def _check_workspace(o: Out, deferred: bool, what: str):
    ws = o.ws.cpu()
    if deferred:  # bytes 4-31 keep n_rows / sum(mask) / the weights for the finaliser
        assert not ws[:, :4].any() and not ws[:, 32:].any(), f"{what}: workspace not zero outside bytes 4-31"
    else:
        assert not ws.any(), f"{what}: workspace not zero after an immediate launch"


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()
    return _ops


def _route(dv: Device) -> Optional[str]:
    c = dv.case
    return expected_kernel(c.n, c.lp, c.lg, has_idx=c.idx is not None, pack=c.pack, lane_aos=c.stats != "norm", vl=c.vl,
                           clip=c.clip, dual=c.dual, popart=c.popart, **dv.flags())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every case
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_loss_variant_matches_oracle(ops, name):
    case = CASES[name]
    x = _inputs(name, case)
    dv = Device(case, x)
    want = _route(dv)
    assert want == case.kernel, f"{name}: these inputs route to {want}, not {case.kernel}"
    o = Out(case, case.problems)
    _, names = launched(lambda: _run(case, dv, o=o), lambda s: s)
    k4 = [kernel_id(s) for s in names if kernel_id(s) is not None]
    fin = [s for s in names if "loss_finalize_kernel" in s]
    assert set(k4) == {case.kernel} and len(k4) == -(-case.problems // MAX_BATCH), f"{name}: launched {names}"
    ours = [s for s in names if "srl::" in s and not s.startswith("cuda")]  # the library's kernels (no runtime API events)
    assert len(fin) == int(case.defer) and len(k4) + len(fin) == len(ours), f"{name}: launched {ours}"
    excused = max(_check_problem(case, x, dv, o, k, k, f"{name} problem {k}") for k in range(case.problems))
    assert excused <= 2, f"{name}: {excused} boundary elements in one problem: more than rounding can explain"
    _check_guards(o, name)
    _check_workspace(o, case.defer, name)
    again = _run(case, dv)
    torch.cuda.synchronize()
    for a, b in zip(o.bits(), again.bits()):
        assert torch.equal(a, b), f"{name}: a second launch changed an output"
    if case.problems > 1:
        for k in range(case.problems):
            one = _run(case, dv, which=[k])
            assert torch.equal(o.grad[k].buf.view(torch.int32), one.grad[0].buf.view(torch.int32)), \
                f"{name}: problem {k} in the batch differs from its own launch"
    if case.defer:
        now = _run(case, dv, defer=False)
        torch.cuda.synchronize()
        for k in range(case.problems):
            assert torch.equal(o.grad[k].buf.view(torch.int32), now.grad[k].buf.view(torch.int32)), \
                f"{name}: problem {k}: deferred and immediate gradients differ"
        a, b = o.out.t.cpu().numpy(), now.out.t.cpu().numpy()
        if case.kernel.startswith("ppo_loss_pair_kernel<"):  # the in-kernel fold adds the rows in another order
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, err_msg=f"{name}: deferred vs immediate out")
        else:
            assert np.array_equal(a, b), f"{name}: deferred and immediate out differ"
        _check_workspace(now, False, f"{name} (immediate twin)")


@pytest.mark.gpu
def test_lane_aos_call_too_wide_is_refused(ops):
    """n = 1026 with lane_aos: SRL_ERR_UNSUPPORTED before any launch; the same call without lane_aos runs the pair kernel."""
    from srl_b200._lib import SrlCudaError
    base = Case("ppo_loss_pair_kernel<StaticCfg<0, false, true, false>>", 4, 1026, dual=True, pack=True, N=2048,
                idx="perm", row_lo=1)
    x = _inputs("aos-1026", base)
    aos = dataclasses.replace(base, stats="aos")
    with pytest.raises(SrlCudaError) as err:
        _run(aos, Device(aos, x))
    assert err.value.status == 2  # SRL_ERR_UNSUPPORTED
    dv = Device(base, x)
    assert _route(dv) == base.kernel
    o = Out(base, 1)
    _, ran = launched(lambda: _run(base, dv, o=o), kernel_id)
    assert ran == [base.kernel]
    _check_problem(base, x, dv, o, 0, 0, "n = 1026 without lane_aos")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: one set of inputs on every route
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("hname", sorted(CROSS))
def test_routes_agree(ops, hname):
    """The same inputs through the dense, four-lane gather (lane_idx = arange), one-lane gather and pack row-tile (policy
    tensors one element off) and pair routes: gradients bit-identical -- every route evaluates element<CFG> on the same float32
    values -- and the loss scalars within 2e-6 (the routes group the float32 partial sums differently)."""
    h = CROSS[hname]
    T, n, lo = 13, 256, 3
    routes = {
        f"ppo_loss_kernel<4, 0, {cfg_name(*h)}>": dict(),
        f"ppo_loss_kernel<4, 1, {cfg_name(*h)}>": dict(idx="arange"),
        G1: dict(pol_off=1),
        PK1: dict(pack=True, pol_off=1),
        f"ppo_loss_pair_kernel<{cfg_name(*h)}>": dict(pack=True),
    }
    x = None
    res = {}
    for kern, kw in routes.items():
        case = Case(kern, T, n, row_lo=lo, **_hk(*h), **kw)
        x = _inputs(f"cross-{hname}", case) if x is None else x
        dv = Device(case, x)
        assert _route(dv) == kern, (kern, _route(dv))
        o = Out(case, 1)
        _, ran = launched(lambda: _run(case, dv, o=o), kernel_id)
        assert ran == [kern]
        _check_problem(case, x, dv, o, 0, 0, f"{hname} on {kern}")
        res[kern] = (torch.stack([t.contiguous() for t in o.grads(0)]), o.out.t[0].cpu().numpy())
    (k0, (g0, out0)), rest = next(iter(res.items())), list(res.items())[1:]
    for kern, (g, out) in rest:
        diff = int((g.view(torch.int32) != g0.view(torch.int32)).sum())
        assert diff == 0, f"{hname}: {diff} gradient elements differ between {k0} and {kern}"
        assert_close_ref(out[:10], out0[:10], tol=2e-6, what=f"{hname}: loss scalars {kern} vs {k0}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the statistics from a real scan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pair_kernel_with_scan_minibatch_shares(ops):
    """End to end: srl_gae_scan_perm writes the pack, lane_aos, the step's permutation and every minibatch's per-CTA shares
    (part_valid); the pair kernel adds those shares itself (lane_aos + minibatch_part) and agrees with the same launch fed
    float64 norm_stats of the scan's own adv: loss scalars within 1e-12, gradients at the suite's bar (the two sums are
    added in different orders, so a normalised advantage may differ in its last bit)."""
    L, N, group, mbs = 13, 512, 4, 4  # the warp-specialised scan: 16 lane groups, aligned
    n = N // mbs
    g = torch.Generator().manual_seed(zlib.crc32(b"scan-part"))
    flag = lambda p: (torch.rand((L, N), generator=g) < p).to(torch.uint8)
    raw = dict(reward=torch.randn((L, N), generator=g), value=torch.randn((L, N), generator=g) * 2.0, done=flag(0.05),
               truncated=flag(0.02), on_reset=flag(0.1), old_logp=-torch.rand((L, N), generator=g) * 3.0)
    d = {k: v.cuda() for k, v in raw.items()}
    pack = ops.new_pack(L, N, "cuda")
    aos = torch.zeros((N, 4), dtype=torch.float64, device="cuda")
    perm = torch.empty((1, N), dtype=torch.int32, device="cuda")
    part = ops.new_minibatch_part(N, "cuda")
    job = dict(seed=77, epoch=0, n_epochs=1, n_env=N // group, group=group, out=perm, minibatches=mbs, part=part)
    adv, ret, _ = ops.gae_scan(d["reward"], d["value"], d["done"], d["truncated"], d["on_reset"], GAMMA, LMBDA, row_lo=0,
                               row_hi=L - 1, old_logp=d["old_logp"], pack=pack, lane_aos=aos, perm_job=job)
    torch.cuda.synchronize()
    assert job["part_valid"], "the scan did not leave the minibatch shares"
    hp = ops.LossHyper(clip_value=True, dual_clip=True, value_loss="huber", value_loss_config={"delta": 1.0})
    T = L - 1
    ws = ops.new_loss_workspace("cuda", slots=2 * mbs)
    mk = lambda k, w: dict(new_logp=(d["old_logp"][:T][:, perm[0, k * n:(k + 1) * n].long()] + 0.2).contiguous(),
                           v_pred=torch.zeros((T, n), device="cuda"), entropy=torch.ones((T, n), device="cuda"),
                           lane_idx=perm[0, k * n:(k + 1) * n].contiguous(),
                           grads=tuple(torch.empty((T, n), device="cuda") for _ in range(3)), workspace=ws[w],
                           out=torch.zeros(16, dtype=torch.float64, device="cuda"))
    a = [mk(k, k) for k in range(mbs)]
    b = [mk(k, mbs + k) for k in range(mbs)]
    for q in b:
        li = q["lane_idx"].long()
        m = (d["on_reset"][1:T + 1][:, li] == 0).double()
        x = adv[:T][:, li].double() * m
        q["norm_stats"] = torch.stack([m.sum(), x.sum(), x.square().sum()])
    ops.ppo_loss_batched(a, None, None, None, None, None, hp, pack=pack, pack_row_lo=0, lane_aos=aos, minibatch_part=part)
    ops.ppo_loss_batched(b, None, None, None, None, None, hp, pack=pack, pack_row_lo=0)
    torch.cuda.synchronize()
    for k in range(mbs):
        assert_close_ref(a[k]["out"].cpu(), b[k]["out"].cpu(), tol=1e-12, what=f"minibatch {k} out")
        Msum = float(b[k]["out"][9])
        for ga, gb in zip(a[k]["grads"], b[k]["grads"]):
            assert_close_ref(ga.cpu().double() * Msum, gb.cpu().double() * Msum, what=f"minibatch {k} gradients")
