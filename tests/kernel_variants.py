"""Helpers shared by the kernel-variant matrices (test_gpu_scan_variants.py, test_gpu_loss_variants.py): outputs in
sentinel-guarded buffers, the kernels a call launched (CUDA profiler), and the kernels the built library contains
(cuobjdump -symbols | cu++filt)."""
import shutil
import subprocess
from typing import Callable, Optional, Set

import numpy as np
import pytest
import torch

F32_SENTINEL = 0x7FA5A5A5  # signalling-NaN bit patterns no kernel writes
F64_SENTINEL = 0x7FF4A5A5A5A5A5A5


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


def launched(fn: Callable, kernel_id: Callable[[str], Optional[str]]):
    """fn()'s result and the demangled names of every kernel it launched, mapped through kernel_id (None: dropped), in
    launch order, from the CUDA profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, [k for k in (kernel_id(e.name) for e in prof.events()) if k is not None]


def library_kernels(kernel_id: Callable[[str], Optional[str]]) -> Set[str]:
    """kernel_id of every symbol in the built libsrl_b200.so (cuobjdump -symbols | cu++filt), building it first; skips
    where the CUDA binary utilities are missing."""
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not available")
    from srl_b200 import _lib, build
    build.build()
    sym = subprocess.run(["cuobjdump", "-symbols", _lib.lib_path()], capture_output=True, text=True)
    if sym.returncode != 0:
        pytest.skip("cuobjdump not available")
    names = subprocess.run(["cu++filt"], input=sym.stdout, capture_output=True, text=True, check=True).stdout
    return {k for k in (kernel_id(line) for line in names.splitlines()) if k is not None}

