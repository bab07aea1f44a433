"""Host build of csrc/decode.cu with its Deflate decoder (csrc/decode_deflate.cuh, XRS_HOST_DEFLATE): the shim and
exports of :mod:`tests.hostmath.zarr_decode`, plus what k_inflate needs -- one static instance as every block's shared
memory (a launch runs its blocks one after another) -- and the coverage counter hook XRS_DEFLATE_COUNT, read back
through ``xrsh_deflate_events_take``."""

from __future__ import annotations

import os
import re
import shutil
import subprocess

from . import CSRC, ROOT, RSK_SHIM, _without_include
from .zarr_decode import DECODE_EXPORT, DECODE_SHIM

N_EVENTS = 128

DEFLATE_SHIM = r"""
#define XRS_HOST_DEFLATE 1
#define __shared__ static
#define __noinline__ __attribute__((noinline))
// what k_inflate decodes (the event numbers of decode_deflate.cuh)
static long xrsh_deflate_events[128];
#define XRS_DEFLATE_COUNT(event) __atomic_fetch_add(&xrsh_deflate_events[(event)], 1, __ATOMIC_RELAXED)
"""

DEFLATE_EXPORT = r"""
// events since the last call (128 counts, see XRS_DEFLATE_COUNT); resets them
extern "C" void xrsh_deflate_events_take(long *out) {
    for (int k = 0; k < 128; ++k) out[k] = __atomic_exchange_n(&xrsh_deflate_events[k], 0, __ATOMIC_RELAXED);
}
"""


def build_deflate_decode(out_dir: str) -> str:
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = _without_include(open(os.path.join(CSRC, "common.cuh")).read(), '"xrs.h"', "common.cuh")
    m = re.search(r"#define XRS_DISPATCH_DTYPE\(.*?\n    }\n", common, re.S)
    assert m, "XRS_DISPATCH_DTYPE moved"
    text = _without_include(open(os.path.join(CSRC, "decode.cu")).read(), '"common.cuh"', "decode.cu")
    deflate = open(os.path.join(CSRC, "decode_deflate.cuh")).read()
    text, n = re.subn(r'#include "decode_deflate.cuh"\n', lambda _: deflate, text)
    assert n == 1, "decode.cu no longer includes decode_deflate.cuh exactly once"
    text, n = re.subn(r"([A-Za-z_]\w*(?:<[^<>;()]*>)?)<<<([^<>;]*?)>>>\(\s*", r"xrshd_launch(\2, &\1, ", text)
    assert n == 4 and "<<<" not in text, "launch syntax of decode.cu / decode_deflate.cuh changed"
    src = os.path.join(out_dir, "decode_deflate_host.cpp")
    with open(src, "w") as fh:
        fh.write(RSK_SHIM + DECODE_SHIM + DEFLATE_SHIM + m.group(0) + "\n" + text + DECODE_EXPORT + DEFLATE_EXPORT)
    so = os.path.join(out_dir, "libxrs_deflatedecodehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-Wl,-Bsymbolic",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of decode.cu with its Deflate decoder failed:\n" + res.stderr[-6000:])
    return so
