"""Host build of csrc/decode.cu with its CRC-32C check (csrc/decode_crc32c.cuh, XRS_HOST_CRC32C) and, so that every
Zarr v3 compressor runs, its Zstd and Deflate decoders: the shims and exports of :mod:`tests.hostmath.zarr_decode`,
:mod:`tests.hostmath.zstd_decode` and :mod:`tests.hostmath.deflate_decode`, each kernel's shared memory one static
instance (a launch runs its blocks one after another).  ``xrsh_crc32c`` runs k_crc32c alone over any table."""

from __future__ import annotations

import os
import re
import shutil
import subprocess

from . import CSRC, ROOT, RSK_SHIM, _without_include
from .deflate_decode import DEFLATE_EXPORT, DEFLATE_SHIM
from .zarr_decode import DECODE_EXPORT, DECODE_SHIM
from .zstd_decode import ZSTD_EXPORT, ZSTD_SHIM

CRC32C_SHIM = r"""
#define XRS_HOST_CRC32C 1
"""

CRC32C_EXPORT = r"""
// k_crc32c alone over a caller's table, without xrs_zarr_decode's header checks, so that any bytes can be a payload:
// a flagged entry's last 4 bytes are checked against the CRC-32C of the rest, then flag and trailer are dropped
extern "C" int xrsh_crc32c(const uint8_t *data, xrs_zarr_chunk *chunks, long n_chunks, uint32_t *err) {
    return xrs::launch_crc32c(data, chunks, n_chunks, err, cudaStream_t{});
}
"""


def build_crc32c_decode(out_dir: str) -> str:
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = _without_include(open(os.path.join(CSRC, "common.cuh")).read(), '"xrs.h"', "common.cuh")
    m = re.search(r"#define XRS_DISPATCH_DTYPE\(.*?\n    }\n", common, re.S)
    assert m, "XRS_DISPATCH_DTYPE moved"
    text = _without_include(open(os.path.join(CSRC, "decode.cu")).read(), '"common.cuh"', "decode.cu")
    for header in ("decode_crc32c.cuh", "decode_zstd.cuh", "decode_deflate.cuh"):
        body = open(os.path.join(CSRC, header)).read()
        text, n = re.subn(r'#include "' + re.escape(header) + r'"\n', lambda _: body, text)
        assert n == 1, f"decode.cu no longer includes {header} exactly once"
    text, n = re.subn(r"([A-Za-z_]\w*(?:<[^<>;()]*>)?)<<<([^<>;]*?)>>>\(\s*", r"xrshd_launch(\2, &\1, ", text)
    assert n == 6 and "<<<" not in text, "launch syntax of decode.cu or its decoders changed"
    src = os.path.join(out_dir, "decode_crc32c_host.cpp")
    with open(src, "w") as fh:
        fh.write(RSK_SHIM + DECODE_SHIM + ZSTD_SHIM + DEFLATE_SHIM + CRC32C_SHIM + m.group(0) + "\n" + text
                 + DECODE_EXPORT + ZSTD_EXPORT + DEFLATE_EXPORT + CRC32C_EXPORT)
    so = os.path.join(out_dir, "libxrs_crc32cdecodehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-Wl,-Bsymbolic",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of decode.cu with its CRC-32C check failed:\n" + res.stderr[-6000:])
    return so
