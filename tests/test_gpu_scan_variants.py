"""K2 (srl_gae_scan / srl_gae_scan_perm) on every kernel instantiation the library contains, against the float64 oracle.

The host code picks one of three scan kernels by shape, alignment and flags (gae_scan.cu, gae_scan_tma.cu, gae_scan_ws.cu),
each templated further: 36 instantiations in all.  CASES names, for every row, the instantiation its inputs route to;
`expected_kernel` restates the routing rules, the profiler shows which kernel actually ran, and a CPU test checks that the
table names every instantiation in the built library -- a new one without a case, or a shape that silently lands on
another kernel, fails the suite.

Per case: adv / ret bit-exact against oracle/ref_math.py (padding row included), lane_part over the case's loss rows,
lane_aos, every column of the loss pack against its definition, no byte written outside the outputs, and a second launch
that reproduces the first bit for bit.
"""
import ctypes
import dataclasses
import re
import shutil
import subprocess
import zlib
from typing import Callable, Optional, Tuple, Union

import numpy as np
import pytest
import torch

from oracle import ref_math as M

GAMMA, LMBDA = 0.995, 0.9
RHO, C = 1.0, 0.9  # V-trace clips: rho != c, and the ratios below straddle both
SMEM_BUDGET = 200 * 1024  # gae_scan.cu kSmemBudget
F32_SENTINEL = 0x7FA5A5A5  # signalling-NaN bit patterns no kernel writes
F64_SENTINEL = 0x7FF4A5A5A5A5A5A5
PACK_MASKED_ADV = 0x7FC00000  # gae_common.cuh kPackMaskedAdv


# ---------------------------------------------------------------------------------------------------------------------
# Routing: gae_scan.cu (gae_scan_impl, launch), gae_scan_tma.cu (gae_tma_eligible, launch_gae_tma_lpw), gae_scan_ws.cu
# (gae_ws_eligible, launch_gae_ws)
# ---------------------------------------------------------------------------------------------------------------------
def _b(x: bool) -> str:
    return "true" if x else "false"


def tile_smem_bytes(L: int, lw: int, pack: bool) -> int:
    """gae_scan.cu gae_smem_bytes: the [L][LW] tile, or the reduction scratch if that is larger."""
    return max(L * lw * (16 + 4 + 4 + 1 + (8 if pack else 0)), 256 * 7 * 8)


def tile_max_L(pack: bool) -> int:
    """The longest trajectory the tile kernel takes (at its narrowest tile, LW = 8)."""
    return SMEM_BUDGET // (8 * (25 + (8 if pack else 0)))


def expected_kernel(L: int, N: int, aligned: bool, vtrace: bool, popart: bool, pack: bool, sms: int) -> Optional[str]:
    """The instantiation srl_gae_scan launches for these inputs on a device with `sms` SMs, as
    "name<template arguments>"; None when the call is refused (L too long for the tile kernel)."""
    groups = (N + 31) // 32
    eligible = aligned and N % 16 == 0  # TMA: 16-byte aligned bases and row pitches
    if groups >= 2 * sms and eligible:
        spec = N % 32 == 0 and not vtrace
        return f"gae_scan_tma_kernel<{_b(vtrace)}, {_b(pack)}, {_b(spec)}, {_b(spec and popart)}, 32>"
    if groups >= 8 and eligible and not vtrace:
        return f"gae_scan_ws_kernel<{_b(pack)}, 16, {9 if groups <= sms else 3}>"
    lw = 32
    while lw > 8 and (tile_smem_bytes(L, lw, pack) > SMEM_BUDGET or -(-N // lw) < 2 * sms):
        lw //= 2
    if tile_smem_bytes(L, lw, pack) > SMEM_BUDGET:
        return None
    rows_per_thread = -(-L // (256 // lw))
    un = rows_per_thread if not vtrace and rows_per_thread in (5, 6) else 4
    return f"gae_scan_kernel<{lw}, {_b(vtrace)}, {_b(pack)}, {un}>"


_KERNEL_RE = re.compile(r"\b(gae_scan(?:_tma|_ws)?_kernel)<([^<>]*)>")


def _template_arg(s: str) -> str:
    s = s.strip()
    m = re.fullmatch(r"\(bool\)([01])", s)
    if m:
        return _b(m.group(1) == "1")
    if s in ("true", "false"):
        return s
    return str(int(re.sub(r"^\((?:unsigned )?\w+\)", "", s)))  # (int)16 -> 16


def kernel_id(name: str) -> Optional[str]:
    """A demangled kernel name (profiler, cu++filt) -> "name<args>" with `true`/`false`/`(bool)1`/`(bool)0` and `(int)16`/`16`
    written one way; None for any other kernel."""
    m = _KERNEL_RE.search(name)
    if m is None:
        return None
    return f"{m.group(1)}<{', '.join(_template_arg(a) for a in m.group(2).split(','))}>"


# ---------------------------------------------------------------------------------------------------------------------
# The case table
# ---------------------------------------------------------------------------------------------------------------------
def per_sm(groups_per_sm: int, extra: int) -> Callable[[int], int]:
    """N = groups_per_sm 32-lane groups per SM + extra lanes: the routing thresholds scale with the SM count
    (at 148 SMs: per_sm(2, 0) = 9472, per_sm(1, 16) = 4752)."""
    return lambda sms: groups_per_sm * 32 * sms + extra


@dataclasses.dataclass(frozen=True)
class Case:
    kernel: str  # the instantiation these inputs route to
    L: int
    N: Union[int, Callable[[int], int]]  # lanes, or lanes as a function of the SM count
    aligned: bool = True  # False: every input one element (flags: one byte) past a 16-byte boundary
    vtrace: bool = False
    popart: bool = False
    pack: bool = False
    rows: Optional[Tuple[int, int]] = None  # [row_lo, row_hi); None = [0, L-1)
    perm: Optional[Tuple[int, int, int]] = None  # srl_gae_scan_perm: (group, epochs, minibatches), n_env = N / group

    def lanes(self, sms: int) -> int:
        return self.N(sms) if callable(self.N) else self.N

    def window(self) -> Tuple[int, int]:
        return self.rows if self.rows is not None else (0, self.L - 1)


def _tile(lw, vt, pk, un):
    return f"gae_scan_kernel<{lw}, {_b(vt)}, {_b(pk)}, {un}>"


def _tma(vt, pk, spec, pa):
    return f"gae_scan_tma_kernel<{_b(vt)}, {_b(pk)}, {_b(spec)}, {_b(pa)}, 32>"


def _ws(pk, slots):
    return f"gae_scan_ws_kernel<{_b(pk)}, 16, {slots}>"


LW16_N = per_sm(1, 264)  # 5000 at 148 SMs: ragged, too few lanes for 2 x SMs tiles of 32
LW32_N = per_sm(2, 28)  # 9500: ragged, enough for 32-lane tiles
TMA_SPEC_N = per_sm(2, 0)  # 9472: whole warps
TMA_GEN_N = per_sm(2, 16)  # 9488: the last warp half filled
WS3_N = per_sm(1, 16)  # 4752: more lane groups than SMs, the last warp half filled

CASES = {
    # ---- tile kernel, LW = 8 (fewer than 2 x SMs tiles of 16 lanes, or a long trajectory) -----------------------------
    "tile8-L2": Case(_tile(8, 0, 0, 4), 2, 37),
    "tile8-pack-popart-rows": Case(_tile(8, 0, 1, 4), 37, 4001, pack=True, popart=True, rows=(3, 29)),
    "tile8-un5-popart": Case(_tile(8, 0, 0, 5), 131, 37, popart=True),
    "tile8-un5-pack-rows": Case(_tile(8, 0, 1, 5), 160, 4001, pack=True, rows=(7, 150)),
    "tile8-un6": Case(_tile(8, 0, 0, 6), 161, 1000),
    "tile8-un6-pack": Case(_tile(8, 0, 1, 6), 192, 37, pack=True),
    "tile8-vtrace-perm": Case(_tile(8, 1, 0, 4), 131, 40, vtrace=True, perm=(4, 3, 2)),
    "tile8-vtrace-pack-popart": Case(_tile(8, 1, 1, 4), 33, 4001, vtrace=True, pack=True, popart=True, rows=(1, 30)),
    "tile8-L5-pack": Case(_tile(8, 0, 1, 4), 5, 37, pack=True),
    "tile8-maxL": Case(_tile(8, 0, 0, 4), tile_max_L(False), 37, rows=(100, 1000)),
    "tile8-maxL-pack": Case(_tile(8, 0, 1, 4), tile_max_L(True), 37, pack=True),
    # ---- tile kernel, LW = 16 ------------------------------------------------------------------------------------------
    "tile16-L2-perm": Case(_tile(16, 0, 0, 4), 2, LW16_N, perm=(8, 2, 5)),
    "tile16-pack-smem-bound": Case(_tile(16, 0, 1, 4), 300, LW32_N, pack=True, rows=(9, 290)),  # LW lowered by smem
    "tile16-un5-popart-rows": Case(_tile(16, 0, 0, 5), 65, LW16_N, popart=True, rows=(1, 60)),
    "tile16-un5-pack-offset": Case(_tile(16, 0, 1, 5), 80, WS3_N, aligned=False, pack=True),
    "tile16-un6": Case(_tile(16, 0, 0, 6), 81, LW16_N),
    "tile16-un6-pack-popart": Case(_tile(16, 0, 1, 6), 96, LW16_N, pack=True, popart=True, rows=(5, 90)),
    "tile16-vtrace": Case(_tile(16, 1, 0, 4), 65, LW16_N, vtrace=True),
    "tile16-vtrace-pack-offset": Case(_tile(16, 1, 1, 4), 41, WS3_N, aligned=False, vtrace=True, pack=True, rows=(2, 33)),
    # ---- tile kernel, LW = 32 ------------------------------------------------------------------------------------------
    "tile32-L2": Case(_tile(32, 0, 0, 4), 2, LW32_N),
    "tile32-pack-offset": Case(_tile(32, 0, 1, 4), 12, TMA_SPEC_N, aligned=False, pack=True, rows=(1, 10)),
    "tile32-un5-popart": Case(_tile(32, 0, 0, 5), 33, LW32_N, popart=True),
    "tile32-un5-pack": Case(_tile(32, 0, 1, 5), 40, LW32_N, pack=True, rows=(2, 37)),
    "tile32-un6-offset": Case(_tile(32, 0, 0, 6), 41, TMA_SPEC_N, aligned=False),
    "tile32-un6-pack-popart": Case(_tile(32, 0, 1, 6), 48, LW32_N, pack=True, popart=True),
    "tile32-vtrace-popart": Case(_tile(32, 1, 0, 4), 33, LW32_N, vtrace=True, popart=True),
    "tile32-vtrace-pack-offset": Case(_tile(32, 1, 1, 4), 100, TMA_SPEC_N, aligned=False, vtrace=True, pack=True,
                                      rows=(3, 97)),
    "tile32-maxL": Case(_tile(32, 0, 0, 4), 256, LW32_N, rows=(8, 250)),
    # ---- TMA kernel (>= 2 lane groups per SM, 16-byte aligned) ----------------------------------------------------------
    "tma-general-L2": Case(_tma(0, 0, 0, 0), 2, TMA_GEN_N),
    "tma-general-popart": Case(_tma(0, 0, 0, 0), 29, TMA_GEN_N, popart=True, rows=(4, 20)),
    # a window on stage boundaries: stages 1..3 take the interior body, stages 0 and 4 the EDGE body, in one launch
    "tma-spec-stage-window-perm": Case(_tma(0, 0, 1, 0), 37, TMA_SPEC_N, rows=(8, 32), perm=(4, 2, 8)),
    "tma-spec-popart-L5": Case(_tma(0, 0, 1, 1), 5, TMA_SPEC_N, popart=True),
    "tma-spec-popart-rows": Case(_tma(0, 0, 1, 1), 150, TMA_SPEC_N, popart=True, rows=(11, 141)),
    "tma-general-pack-popart": Case(_tma(0, 1, 0, 0), 41, TMA_GEN_N, pack=True, popart=True, rows=(3, 29)),
    "tma-spec-pack-L12": Case(_tma(0, 1, 1, 0), 12, TMA_SPEC_N, pack=True, rows=(0, 11)),
    "tma-spec-pack-popart": Case(_tma(0, 1, 1, 1), 161, TMA_SPEC_N, pack=True, popart=True, rows=(16, 144)),
    "tma-spec-pack-popart-mid": Case(_tma(0, 1, 1, 1), 33, per_sm(2, 512), pack=True, popart=True, rows=(3, 29)),
    "tma-spec-pack-popart-L2": Case(_tma(0, 1, 1, 1), 2, TMA_SPEC_N, pack=True, popart=True),
    "tma-vtrace-popart": Case(_tma(1, 0, 0, 0), 37, TMA_SPEC_N, vtrace=True, popart=True, rows=(5, 35)),
    "tma-vtrace-general": Case(_tma(1, 0, 0, 0), 9, TMA_GEN_N, vtrace=True),
    "tma-vtrace-pack": Case(_tma(1, 1, 0, 0), 40, TMA_GEN_N, vtrace=True, pack=True, rows=(8, 32)),
    "tma-vtrace-pack-L2": Case(_tma(1, 1, 0, 0), 2, TMA_SPEC_N, vtrace=True, pack=True),
    # ---- warp-specialised kernel (8 .. 2 x SMs lane groups, aligned, no V-trace) ----------------------------------------
    "ws-deep-L2": Case(_ws(0, 9), 2, 256),
    "ws-deep-wrap-popart": Case(_ws(0, 9), 161, 4096, popart=True, rows=(16, 150)),  # 11 chunks: the 9-slot ring wraps
    "ws-deep-pack-perm": Case(_ws(1, 9), 12, 272, pack=True, rows=(1, 10), perm=(8, 8, 2)),
    "ws-deep-pack-popart-wrap": Case(_ws(1, 9), 145, 4080, pack=True, popart=True, rows=(5, 133)),
    "ws3-L5": Case(_ws(0, 3), 5, WS3_N),
    "ws3-wrap-popart-perm": Case(_ws(0, 3), 50, per_sm(1, 1664), popart=True, rows=(16, 48), perm=(1, 2, 4)),
    "ws3-pack-perm": Case(_ws(1, 3), 37, per_sm(1, 1408), pack=True, rows=(3, 35), perm=(8, 4, 4)),  # N = 6144 at 148
    "ws3-pack-L2": Case(_ws(1, 3), 2, WS3_N, pack=True),
    "ws3-pack-popart-wrap": Case(_ws(1, 3), 67, WS3_N, pack=True, popart=True, rows=(17, 63)),
}

# the same seeded inputs aligned (the TMA / warp-specialised kernel) and offset (the tile kernel)
CROSS = ["tma-spec-pack-popart", "tma-general-pack-popart", "tma-vtrace-pack", "ws-deep-pack-popart-wrap", "ws3-pack-perm",
         "tma-spec-stage-window-perm"]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table covers the library
# ---------------------------------------------------------------------------------------------------------------------
def test_case_table_names_every_scan_instantiation_in_the_library():
    """The set of gae_scan*_kernel instantiations in libsrl_b200.so (cuobjdump -symbols | cu++filt) is the set CASES names:
    an instantiation with no case, or a case naming one that does not exist, fails here."""
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not available")
    from srl_b200 import _lib, build
    build.build()
    sym = subprocess.run(["cuobjdump", "-symbols", _lib.lib_path()], capture_output=True, text=True)
    if sym.returncode != 0:
        pytest.skip("cuobjdump not available")
    names = subprocess.run(["cu++filt"], input=sym.stdout, capture_output=True, text=True, check=True).stdout
    built = {k for k in (kernel_id(line) for line in names.splitlines()) if k is not None}
    assert len(built) == 36, sorted(built)
    named = {c.kernel for c in CASES.values()}
    assert built == named, f"in the library only: {sorted(built - named)}; in the table only: {sorted(named - built)}"


def test_kernel_names_normalise_both_spellings():
    cuobj = "void srl::<unnamed>::gae_scan_tma_kernel<(bool)0, (bool)1, (bool)1, (bool)0, (int)32>(srl::<unnamed>::GaeTmaParams)"
    prof = "void srl::(anonymous namespace)::gae_scan_tma_kernel<false, true, true, false, 32>(srl::(anonymous namespace)::GaeTmaParams)"
    assert kernel_id(cuobj) == kernel_id(prof) == _tma(0, 1, 1, 0)
    assert kernel_id("void srl::philox_perm_kernel<(int)8>(int)") is None
    assert expected_kernel(130, 4096, True, False, False, True, 148) == _ws(1, 9)
    assert expected_kernel(tile_max_L(True) + 1, 37, True, False, False, True, 148) is None


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test instead")
    from srl_b200 import ops as _ops
    _ops._lib.load_library()
    return _ops


@pytest.fixture(scope="module")
def sms(ops):
    n, major, minor = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
    ops._lib.call("srl_device_info", ctypes.byref(n), ctypes.byref(major), ctypes.byref(minor))
    return n.value


def _place(x: torch.Tensor, aligned: bool) -> torch.Tensor:
    """x on the device as a contiguous [L, N] tensor; aligned = False: its base one element past a 256-byte boundary."""
    if aligned:
        return x.cuda()
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device="cuda")
    out = buf[1:].view(x.shape)
    out.copy_(x)
    return out


class Guarded:
    """An output as a view into a larger buffer: 256 bytes of sentinel on both sides (the view stays 256-byte aligned, so
    routing does not change) and the view itself pre-filled with the sentinel."""

    def __init__(self, shape, dtype):
        self.n = int(np.prod(shape))
        self.g = 256 // torch.empty((), dtype=dtype).element_size()
        self.ity = torch.int32 if dtype == torch.float32 else torch.int64
        self.sentinel = F32_SENTINEL if dtype == torch.float32 else F64_SENTINEL
        self.buf = torch.empty(self.n + 2 * self.g, dtype=dtype, device="cuda")
        self.buf.view(self.ity).fill_(self.sentinel)
        self.t = self.buf[self.g:self.g + self.n].view(shape)

    def guards_intact(self) -> bool:
        b = self.buf.view(self.ity)
        return bool((b[:self.g] == self.sentinel).all()) and bool((b[self.g + self.n:] == self.sentinel).all())


def _inputs(name: str, case: Case, N: int) -> dict:
    """Seeded CPU inputs of a case; they depend on the name and shape only, not on the alignment."""
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    L = case.L
    flag = lambda p: (torch.rand((L, N), generator=g) < p).to(torch.uint8)
    x = dict(reward=torch.randn((L, N), generator=g), value=torch.randn((L, N), generator=g) * 2.0,
             done=flag(0.06), truncated=flag(0.03), on_reset=flag(0.08),
             old_logp=-torch.rand((L, N), generator=g) * 3.0)
    if case.vtrace:
        # a different tensor from old_logp, so that the pack shows which of the two it carries
        x["vt_old"] = -torch.rand((L - 1, N), generator=g) * 2.0
        x["vt_new"] = x["vt_old"] + (torch.rand((L - 1, N), generator=g) * 0.8 - 0.4)  # ratios in [0.67, 1.49]
    if case.popart:
        pa = M.RunningMeanStdRef((1,), beta=0.99)
        pa.update(torch.randn((64, 1), generator=g) * 2.5 + 0.7)
        x["popart"] = pa
    return x


def _run(ops, case: Case, x: dict, N: int, aligned: bool, perm_job: Optional[dict] = None) -> dict:
    """One srl_gae_scan(_perm) launch with every output in a guarded buffer."""
    L = case.L
    d = {k: _place(x[k], aligned) for k in ("reward", "value", "done", "truncated", "on_reset", "old_logp")}
    kw = {}
    if case.vtrace:
        kw.update(vtrace_new_logp=_place(x["vt_new"], aligned), vtrace_old_logp=_place(x["vt_old"], aligned), rho=RHO, c=C)
    if case.popart:
        m, s = x["popart"].mean_std()
        kw["popart_mean_std"] = torch.tensor([m.item(), s.item()], dtype=torch.float64, device="cuda")
    out = dict(adv=Guarded((L, N), torch.float32), ret=Guarded((L, N), torch.float32),
               lane_part=Guarded((8, N), torch.float64), lane_aos=Guarded((N, 4), torch.float64))
    if case.pack:
        out["pack"] = Guarded((ops.pack_rows(L) // 2, N, 2, 4), torch.float32)
        kw.update(old_logp=d["old_logp"], pack=out["pack"].t)
    lo, hi = case.window()
    ops.gae_scan(d["reward"], d["value"], d["done"], d["truncated"], d["on_reset"], GAMMA, LMBDA, row_lo=lo, row_hi=hi,
                 adv=out["adv"].t, ret=out["ret"].t, lane_part=out["lane_part"].t, lane_aos=out["lane_aos"].t,
                 perm_job=perm_job, **kw)
    if case.vtrace:  # the importance ratio as torch computes it on the device from the same float32 leaves
        out["ratio"] = (kw["vtrace_new_logp"] - kw["vtrace_old_logp"]).exp().cpu()
    return out


def _launched(fn):
    """fn()'s result and the gae_scan*_kernel instantiations it launched (kernel_id strings, from the CUDA profiler)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, [k for k in (kernel_id(e.name) for e in prof.events()) if k is not None]


def _oracle(case: Case, x: dict, ratio: Optional[torch.Tensor]):
    """adv, ret [L, N] (padding row included) and lane_part [8, N] from oracle/ref_math.py."""
    f = {k: x[k].float() for k in ("reward", "value", "done", "truncated", "on_reset")}
    pa = x.get("popart")
    if case.vtrace:
        base = pa.denormalize(f["value"]) if pa is not None else f["value"]
        boot = base * (1 - f["done"])  # mappo.py:120-124
        adv = M.gae_trace_ref(f["reward"][:-1], boot, f["truncated"], f["done"], f["on_reset"], GAMMA, LMBDA, vtrace=True,
                              imp_ratio=ratio, rho=RHO, c=C)
        ret = adv + boot[:-1]
    else:
        adv, ret = M.adv_and_value_target_ref(f["reward"], f["value"], f["truncated"], f["done"], f["on_reset"], GAMMA,
                                              LMBDA, popart=pa)
    adv, ret = M.pad_last_row(adv), M.pad_last_row(ret)
    lo, hi = case.window()
    mask = 1 - f["on_reset"][lo + 1:hi + 1].double()
    xs, ys = adv[lo:hi].double() * mask, ret[lo:hi].double() * mask
    part = torch.stack([mask.sum(0), xs.sum(0), xs.square().sum(0), ys.sum(0), ys.square().sum(0),
                        f["done"][lo:hi].double().sum(0), f["truncated"][lo:hi].double().sum(0),
                        torch.zeros(adv.shape[1], dtype=torch.float64)])
    return adv, ret, part


def _check_lane_part(got: torch.Tensor, want: torch.Tensor, what: str):
    got = got.cpu()
    for k in (0, 5, 6):  # counts
        assert torch.equal(got[k], want[k]), f"{what}: lane_part row {k} (a count) differs"
    np.testing.assert_allclose(got[1:5].numpy(), want[1:5].numpy(), rtol=1e-12, atol=1e-12, err_msg=f"{what}: lane_part sums")
    assert torch.equal(got[7], torch.zeros_like(got[7])), f"{what}: lane_part row 7 is not zero"


def _check_case(ops, case: Case, x: dict, out: dict, what: str):
    L = case.L
    adv, ret = out["adv"].t.cpu(), out["ret"].t.cpu()
    ra, rr, rpart = _oracle(case, x, out.get("ratio"))
    assert torch.equal(adv, ra), f"{what}: adv not bit-exact ({int((adv != ra).sum())} elements differ)"
    assert torch.equal(ret, rr), f"{what}: ret not bit-exact ({int((ret != rr).sum())} elements differ)"
    _check_lane_part(out["lane_part"].t, rpart, what)
    aos = out["lane_aos"].t.cpu()
    assert torch.equal(aos[:, :3], out["lane_part"].t[:3].t().cpu()), f"{what}: lane_aos != lane_part[:3].T"
    assert not aos[:, 3].any(), f"{what}: lane_aos column 3 is not zero"
    if case.pack:
        pk = ops.unpack_rows(out["pack"].t)[:L].cpu()  # row L of an odd L is not part of the contract
        if case.vtrace:  # the V-trace leaf, rows 0..L-2; 0 in the padding row; old_logp is not read
            want_ol = torch.cat([x["vt_old"], torch.zeros_like(x["vt_old"][:1])])
        else:
            want_ol = x["old_logp"]
        assert torch.equal(pk[..., 0], want_ol), f"{what}: pack old_logp column"
        assert torch.equal(pk[..., 1], x["value"]), f"{what}: pack value column is not the value as stored"
        assert torch.equal(pk[..., 2], rr), f"{what}: pack ret column"
        keep = torch.zeros((L, adv.shape[1]), dtype=torch.bool)
        keep[:-1] = x["on_reset"][1:] == 0
        assert torch.equal(pk[..., 3][keep], ra[keep]), f"{what}: pack adv column (kept transitions)"
        masked_bits = pk[..., 3].contiguous().view(torch.int32)[~keep]
        assert bool((masked_bits == PACK_MASKED_ADV).all()), f"{what}: pack adv column of masked transitions is not NaN"
    for k, gb in out.items():
        if isinstance(gb, Guarded):
            assert gb.guards_intact(), f"{what}: {k} written outside its [{gb.n}] elements"


def _bits(out: dict) -> dict:
    return {k: v.buf.view(v.ity).clone() for k, v in out.items() if isinstance(v, Guarded)}


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every case
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_scan_variant_matches_oracle(ops, sms, name):
    """The case's inputs route to its instantiation (by the rules and by the profiler), and every output matches the
    oracle and the stated contract.  V-trace is compared with gae_trace_ref fed the importance ratio torch computes on the
    device from the same float32 leaves (both sides reach expf through libdevice): bit-exact as well."""
    case = CASES[name]
    N = case.lanes(sms)
    want = expected_kernel(case.L, N, case.aligned, case.vtrace, case.popart, case.pack, sms)
    assert want == case.kernel, f"{name}: at {sms} SMs these inputs route to {want}, not {case.kernel}"
    x = _inputs(name, case, N)
    out, launched = _launched(lambda: _run(ops, case, x, N, case.aligned))
    assert launched and set(launched) == {case.kernel}, f"{name}: launched {launched}, expected {case.kernel}"
    _check_case(ops, case, x, out, name)
    again = _run(ops, case, x, N, case.aligned)
    torch.cuda.synchronize()
    first, second = _bits(out), _bits(again)
    for k in first:
        assert torch.equal(first[k], second[k]), f"{name}: a second launch changed {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("pack", [False, True])
def test_tile_kernel_refuses_one_row_too_many(ops, pack):
    """One row past the longest trajectory the tile kernel takes is refused on the host (SRL_ERR_UNSUPPORTED), with the
    limit that applies to the call in the message."""
    from srl_b200._lib import SrlCudaError
    L, N = tile_max_L(pack) + 1, 37
    z = torch.zeros((L, N), device="cuda")
    f = torch.zeros((L, N), dtype=torch.uint8, device="cuda")
    kw = dict(old_logp=z, pack=ops.new_pack(L, N, "cuda")) if pack else {}
    with pytest.raises(SrlCudaError) as err:
        ops.gae_scan(z, z, f, f, f, GAMMA, LMBDA, **kw)
    assert err.value.status == 2  # SRL_ERR_UNSUPPORTED
    assert f"max L = {tile_max_L(pack)}" in err.value.message, err.value.message
    adv, _, _ = ops.gae_scan(z[:-1], z[:-1], f[:-1], f[:-1], f[:-1], GAMMA, LMBDA)  # the device is fine
    torch.cuda.synchronize()
    assert not adv.any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", CROSS)
def test_aligned_and_offset_inputs_agree(ops, sms, name):
    """The same seeded inputs aligned (TMA or warp-specialised kernel) and one element off (tile kernel): adv, ret and the
    pack bit-identical, lane_part counts equal and its sums within 1e-12 (the kernels add in different orders)."""
    case = CASES[name]
    N = case.lanes(sms)
    off = dataclasses.replace(case, aligned=False)
    k_off = expected_kernel(off.L, N, False, off.vtrace, off.popart, off.pack, sms)
    assert k_off.startswith("gae_scan_kernel<") and not case.kernel.startswith("gae_scan_kernel<")
    x = _inputs(name, case, N)
    a = _run(ops, case, x, N, True)
    b = _run(ops, off, x, N, False)
    torch.cuda.synchronize()
    for k in ("adv", "ret"):
        assert torch.equal(a[k].buf.view(a[k].ity), b[k].buf.view(b[k].ity)), f"{name}: {k} differs between {case.kernel} and {k_off}"
    if case.pack:  # rows < L: row L of an odd L is not part of the contract (the warp-specialised kernel writes it)
        pka, pkb = (ops.unpack_rows(o["pack"].t)[:case.L].contiguous().view(torch.int32) for o in (a, b))
        assert torch.equal(pka, pkb), f"{name}: pack differs between {case.kernel} and {k_off}"
    pa, pb = a["lane_part"].t.cpu(), b["lane_part"].t.cpu()
    for k in (0, 5, 6, 7):
        assert torch.equal(pa[k], pb[k])
    np.testing.assert_allclose(pa[1:5].numpy(), pb[1:5].numpy(), rtol=1e-12, atol=1e-12)
    _check_case(ops, off, x, b, f"{name} (offset)")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(n for n, c in CASES.items() if c.perm is not None))
def test_perm_job_on_every_kernel(ops, sms, name):
    """srl_gae_scan_perm: the permutations are the oracle's Philox permutation on every kernel, the scan's outputs do not
    change, only the warp-specialised kernel computes them itself (fused / part_valid), and there every scan CTA's share of
    every minibatch's {count, sum, sum of squares} matches the oracle's lane sums."""
    case = CASES[name]
    N = case.lanes(sms)
    group, epochs, mbs = case.perm
    assert N % group == 0 and N % mbs == 0
    n_env = N // group
    x = _inputs(name, case, N)
    plain = _run(ops, case, x, N, case.aligned)
    perm = torch.full((epochs, N), -7, dtype=torch.int32, device="cuda")
    part = ops.new_minibatch_part(N, "cuda").view(torch.int64).fill_(F64_SENTINEL).view(torch.float64)
    job = dict(seed=0x5EED1234ABCD, epoch=3, n_epochs=epochs, n_env=n_env, group=group, out=perm, minibatches=mbs, part=part)
    fused = _run(ops, case, x, N, case.aligned, perm_job=job)
    torch.cuda.synchronize()
    a, b = _bits(plain), _bits(fused)
    for k in a:
        assert torch.equal(a[k], b[k]), f"{name}: the permutation job changed {k}"
    lanes = np.stack([(M.philox_perm_ref(0x5EED1234ABCD, 3 + e, n_env).astype(np.int64)[:, None] * group +
                       np.arange(group)[None]).reshape(-1) for e in range(epochs)])
    assert np.array_equal(perm.cpu().numpy(), lanes), f"{name}: permutations differ from the oracle"
    is_ws = case.kernel.startswith("gae_scan_ws_kernel<")
    assert job["fused"] == is_ws and job["part_valid"] == is_ws
    tb = part.cpu()
    if not is_ws:
        assert bool((tb.view(torch.int64) == F64_SENTINEL).all()), f"{name}: minibatch table written by {case.kernel}"
        return
    _, _, lp = _oracle(case, x, plain.get("ratio"))
    ctas, per = (N + 31) // 32, N // mbs
    for e in range(epochs):
        for j in range(mbs):
            mb = lanes[e, j * per:(j + 1) * per]
            want = np.zeros((ctas, 3))
            for k in range(3):
                np.add.at(want[:, k], mb // 32, lp[k].numpy()[mb])
            got = tb[e * mbs + j].numpy()
            assert np.array_equal(got[:, 0], want[:, 0]), f"{name}: minibatch {e},{j} counts"
            np.testing.assert_allclose(got[:, 1:3], want[:, 1:3], rtol=1e-12, atol=1e-12)
            assert not got[:, 3].any()
    assert bool((tb[epochs * mbs:].view(torch.int64) == F64_SENTINEL).all()), f"{name}: table slots past the step written"
