"""Host build of csrc/decode.cu with its Zstd decoder (csrc/decode_zstd.cuh, XRS_HOST_ZSTD): the shim and exports of
:mod:`tests.hostmath.zarr_decode`, plus what k_zstd_decode needs -- one static instance as every block's shared
memory (a launch runs its blocks one after another), ``__clz``, and the repeat-offset counter hook XRS_ZSTD_COUNT,
read back through ``xrsh_zstd_events_take``."""

from __future__ import annotations

import os
import re
import shutil
import subprocess

from . import CSRC, ROOT, RSK_SHIM, _without_include
from .zarr_decode import DECODE_EXPORT, DECODE_SHIM

ZSTD_SHIM = r"""
#define XRS_HOST_ZSTD 1
#define __shared__ static
static inline int __clz(int v) { return v ? __builtin_clz(static_cast<unsigned>(v)) : 32; }
// repeat-offset events of k_zstd_decode: 0-2 repeat offset 1-3 after literals, 4-6 after none
static long xrsh_zstd_events[8];
#define XRS_ZSTD_COUNT(event) __atomic_fetch_add(&xrsh_zstd_events[(event)], 1, __ATOMIC_RELAXED)
"""

ZSTD_EXPORT = r"""
// repeat-offset events since the last call (8 counts, see XRS_ZSTD_COUNT); resets them
extern "C" void xrsh_zstd_events_take(long *out) {
    for (int k = 0; k < 8; ++k) out[k] = __atomic_exchange_n(&xrsh_zstd_events[k], 0, __ATOMIC_RELAXED);
}
"""


def build_zstd_decode(out_dir: str) -> str:
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = _without_include(open(os.path.join(CSRC, "common.cuh")).read(), '"xrs.h"', "common.cuh")
    m = re.search(r"#define XRS_DISPATCH_DTYPE\(.*?\n    }\n", common, re.S)
    assert m, "XRS_DISPATCH_DTYPE moved"
    text = _without_include(open(os.path.join(CSRC, "decode.cu")).read(), '"common.cuh"', "decode.cu")
    zstd = open(os.path.join(CSRC, "decode_zstd.cuh")).read()
    text, n = re.subn(r'#include "decode_zstd.cuh"\n', lambda _: zstd, text)
    assert n == 1, "decode.cu no longer includes decode_zstd.cuh exactly once"
    text, n = re.subn(r"([A-Za-z_]\w*(?:<[^<>;()]*>)?)<<<([^<>;]*?)>>>\(\s*", r"xrshd_launch(\2, &\1, ", text)
    assert n == 4 and "<<<" not in text, "launch syntax of decode.cu / decode_zstd.cuh changed"
    src = os.path.join(out_dir, "decode_zstd_host.cpp")
    with open(src, "w") as fh:
        fh.write(RSK_SHIM + DECODE_SHIM + ZSTD_SHIM + m.group(0) + "\n" + text + DECODE_EXPORT + ZSTD_EXPORT)
    so = os.path.join(out_dir, "libxrs_zstddecodehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-Wl,-Bsymbolic",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of decode.cu with its Zstd decoder failed:\n" + res.stderr[-6000:])
    return so
