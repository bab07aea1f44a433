"""Streaming of data variables host -> device -> host around the gather kernels.

The reference hands every dask chunk of every variable to a tile task (``rectify.py:263-309``,
``reproject.py:189-265``).  Here the source-index information of a call (rectify: the ij image,
reproject: the tile tables) is computed once and stays resident; the data variables then stream
through the device in band chunks on three streams -- upload of chunk k+1 (H2D copy engine), kernels
of chunk k, download of chunk k-1 (D2H copy engine) -- so that a PCIe-bound call costs
max(H2D, D2H) instead of their sum.

* A host array that several output variables are computed from (the same bands rectified with two
  interpolation methods) is uploaded ONCE per chunk and feeds every target.
* Only the part of the source a call needs is uploaded: ``segments`` lists sub-rectangles of the
  source image (the ragged footprint of a target row band, ``bands.py``); they land in a
  full-pitch device slot at their true position, so the kernels address the source as usual.
* Results are written straight into rows ``rows`` of the caller's (page-locked) output arrays --
  with several GPUs, every GPU fills its own row band of ONE array.

All copies are strided 2-D copies on the copy engines (``xrs_copy2d_slices``); torch supplies
streams, events and device buffers.
"""

from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _dev
from ._lib import XrsError, check, load


@dataclass
class Target:
    """One output variable computed from a source group."""

    name: str
    method: str
    fill: float
    out_host: np.ndarray          # (bands, H_out, W_out), rows `rows` are filled
    out_dtype: np.dtype = None
    row0: int = 0                 # target row held by out_host[:, 0] (a band-only array of a torchrun rank)

    def __post_init__(self):
        self.out_dtype = np.dtype(self.out_host.dtype)


@dataclass
class SourceGroup:
    """One host array ``values`` (bands, h, w) and the targets computed from it."""

    values: np.ndarray
    targets: list = field(default_factory=list)


def as_bands(values):
    """(h, w) or (bands, h, w) -> (bands, h, w) view with unit stride along x; lazy sources
    (``io.LazySource``: bands still in a chunked store) pass through."""
    if hasattr(values, "read_bands"):
        return values
    v = values if values.ndim == 3 else values[None]
    if v.strides[-1] != v.itemsize or v.strides[-2] < v.shape[-1] * v.itemsize or not v.flags.aligned:
        v = np.ascontiguousarray(v)
    return v


def group_by_buffer(items) -> list[SourceGroup]:
    """``items``: iterable of (values, Target).  Variables that are views of the same host memory
    (same address, shape, strides, dtype) form one group -- uploaded once."""
    groups: dict = {}
    for values, target in items:
        v = as_bands(values)
        key = ("lazy", id(v)) if hasattr(v, "read_bands") else \
            (v.__array_interface__["data"][0], v.shape, v.strides, v.dtype.str)
        if key not in groups:
            groups[key] = SourceGroup(v)
        groups[key].targets.append(target)
    return list(groups.values())


def pair_targets(targets: list, src_dtype) -> list[tuple]:
    """Jobs of one source group: ``(interp_target, nearest_target)`` pairs where a bilinear / triangular
    target and a nearest target share the group's bands and dtype (one launch gives both,
    ``xrs_gather_ij2``), single-target jobs ``(target,)`` for the rest; the order of first appearance is kept."""
    src_dtype = np.dtype(src_dtype)
    same = [t for t in targets if t.out_dtype == src_dtype]
    near = [t for t in same if t.method == "nearest"]
    interp = [t for t in same if t.method in ("bilinear", "triangular")]
    partner = {id(a): b for a, b in zip(interp, near)}
    partner.update({id(b): a for a, b in zip(interp, near)})
    jobs, seen = [], set()
    for t in targets:
        if id(t) in seen:
            continue
        other = partner.get(id(t))
        if other is None:
            jobs.append((t,))
            seen.add(id(t))
        else:
            a, b = (t, other) if t.method != "nearest" else (other, t)
            jobs.append((a, b))
            seen.update((id(a), id(b)))
    return jobs


def chunk_schedule(bands: int, chunk: int) -> list[tuple[int, int]]:
    """Band chunks 1, 2, 4, ..., chunk, chunk, ...: a short first chunk starts the download early."""
    out, b0, size = [], 0, 1
    while b0 < bands:
        nb = min(size, chunk, bands - b0)
        out.append((b0, nb))
        b0 += nb
        size *= 2
    return out


def copy2d(dst_addr: int, dst_pitch: int, dst_slice: int, src_addr: int, src_pitch: int, src_slice: int,
           width: int, rows: int, slices: int, device) -> None:
    """``xrs_copy2d_slices`` on the current stream of ``device`` (all quantities in bytes)."""
    check(load().xrs_copy2d_slices(ctypes.c_void_p(dst_addr), dst_pitch, dst_slice, ctypes.c_void_p(src_addr),
                                   src_pitch, src_slice, width, rows, slices, _dev.stream_ptr(device)),
          "xrs_copy2d_slices")


def _zarr_geometry(source):
    """(stored ZarrV2Source, chunk (bands, h, w), dtype code, big-endian flag, CF struct or None) of a source with a
    device read (``io.ZarrV2Source`` or ``io.DecodedSource`` over one)."""
    from .constants import DTYPE_CODES
    from ._lib import XrsZarrCF

    stored = getattr(source, "source", source)
    raw = np.dtype(stored.dtype)
    chunk = tuple(stored.chunks) if len(stored.chunks) == 3 else (1,) + tuple(stored.chunks)
    cf = None
    if stored is not source:
        p = source.device_cf()
        cf = XrsZarrCF.from_params(DTYPE_CODES[np.dtype(p["out_dtype"])], p["fills"], p["scale"], p["offset"])
    return stored, chunk, DTYPE_CODES[raw.newbyteorder("=")], int(raw.byteorder == ">"), cf


def zarr_workspace_bytes(lib, source, table) -> int:
    """``xrs_zarr_decode_workspace_bytes`` for the chunk table of a device read of ``source``."""
    _, (cb, ch, cw), code, _, _ = _zarr_geometry(source)
    n = lib.xrs_zarr_decode_workspace_bytes(ctypes.c_void_p(table.ctypes.data), len(table), cb, ch, cw, code)
    if n < 0:
        check(1, "xrs_zarr_decode_workspace_bytes")
    return int(n)


def zarr_decode(lib, source, data_addr: int, n_bytes: int, table, dst_addr: int, pitch: int, band_stride: int,
                window, b0: int, nb: int, ws_addr: int, ws_bytes: int, err_addr: int, stream) -> int:
    """``xrs_zarr_decode`` of a device read of ``source`` (``lib``: libxrs or a host build with the same ABI);
    returns the status."""
    stored, (cb, ch, cw), code, big, cf = _zarr_geometry(source)
    h, w = stored.shape[-2:]
    return lib.xrs_zarr_decode(ctypes.c_void_p(data_addr), n_bytes, ctypes.c_void_p(table.ctypes.data), len(table),
                               cb, ch, cw, code, big, stored.device_fill_bits(),
                               None if cf is None else ctypes.byref(cf), h, w, ctypes.c_void_p(dst_addr), pitch,
                               band_stride, int(window[0]), int(window[1]), b0, nb, ctypes.c_void_p(ws_addr), ws_bytes,
                               ctypes.c_void_p(err_addr), stream)


DECODE_ERRORS = {1: "a block offset or stream size points outside the file", 2: "a match offset of 0",
                 3: "a match reaching before the stream's start", 4: "literals past the decoded size",
                 5: "a match past the decoded size", 6: "the stream ends inside a sequence, header or block",
                 7: "the stream ends short of its decoded size", 8: "a bad zstd frame, zlib or gzip header",
                 9: "a reserved zstd block type or a block above the block size limit",
                 10: "a bad zstd literals section", 11: "a bad zstd Huffman tree description",
                 12: "a bad zstd FSE table description", 13: "a bad zstd sequences section",
                 14: "bytes after the zstd frame or gzip member",
                 15: "a checksum mismatch (zstd content checksum, zlib Adler-32, gzip CRC-32 or size)",
                 16: "a bad Deflate block type or stored block length",
                 17: "a bad Deflate code description", 18: "an invalid Deflate litlen or distance code",
                 19: "a CRC-32C trailer that does not match the chunk's bytes"}


def decode_error(word: int, paths) -> str | None:
    """The message for an ``xrs_zarr_decode`` error word (``paths``: the chunk files of that call)."""
    if word == 0:
        return None
    chunk = (word & 0xFFFFFF) - 1
    where = paths[chunk] if 0 <= chunk < len(paths) else f"chunk {chunk}"
    return f"{where}: malformed chunk file: {DECODE_ERRORS.get(word >> 24, f'error {word >> 24}')}"


class GatherPipeline:
    """Three-stream pipeline over the band chunks of a list of :class:`SourceGroup`.

    ``src_window = (j0, j1)``: source rows resident on the device (slot height); ``segments``:
    (j0, j1, i0, i1) sub-rectangles of the source image to upload per band (default: the whole
    window); ``rows``: target rows computed; ``process(src_view, target, out_view, b0)`` enqueues the
    kernel for one chunk and one target on the current stream -- ``src_view`` is the
    (nb, j1 - j0, w) view of the slot, ``out_view`` the (nb, rows, W) output slot.
    """

    def __init__(self, device, src_hw, out_w: int, rows, src_window=None, segments=None, chunk_bands: int = 4,
                 pitch_bytes: int = 128):
        self.dev = _dev.require_cuda(device)
        self.h, self.w = int(src_hw[0]), int(src_hw[1])
        self.rows = (int(rows[0]), int(rows[1]))
        self.out_w = int(out_w)
        self.win = (0, self.h) if src_window is None else (int(src_window[0]), int(src_window[1]))
        self.segments = [(self.win[0], self.win[1], 0, self.w)] if segments is None else list(segments)
        self.chunk = int(chunk_bands)
        self.pitch_bytes = int(pitch_bytes)
        self._in_slots: dict = {}
        self._out_slots: dict = {}
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._pending = None
        self._keep = None
        self._decode_checks = []  # (error words, chunk file paths per band chunk) of device-decoded sources

    def _slots(self, cache, key, shape, dtype, n=2):
        if key not in cache or len(cache[key]) < n:
            cache[key] = [torch.empty(shape, dtype=_dev.torch_dtype(dtype), device=self.dev) for _ in range(n)]
        return cache[key]

    def wait(self) -> None:
        """Block until everything enqueued by :meth:`run` has landed in host memory."""
        if self._pending is not None:
            s_out, main = self._pending
            s_out.synchronize()
            main.synchronize()  # main waited for every decode on s_in
            self._pending = None
        checks, self._decode_checks = self._decode_checks, []
        for errs, paths_of in checks:
            for word, paths in zip(errs.cpu().tolist(), paths_of):
                msg = decode_error(word & 0xFFFFFFFF, paths)
                if msg:
                    raise XrsError(msg)

    def run(self, groups: list[SourceGroup], process, wait: bool = True, process_pair=None) -> None:
        """Enqueue uploads, kernels and downloads of every band chunk; ``wait=False`` returns as soon as
        everything is enqueued (call :meth:`wait` before touching the outputs or dropping the inputs).

        ``process_pair(src_view, target_interp, target_nearest, out_interp, out_nearest, b0)``, when given,
        computes a bilinear / triangular target and a nearest target of the same group in one launch
        (:func:`pair_targets` decides which); everything else goes through ``process``."""
        dev = self.dev
        main = torch.cuda.current_stream(dev)
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        n_rows = self.rows[1] - self.rows[0]
        win_h = self.win[1] - self.win[0]
        k_in = k_out = 0
        in_free = [torch.cuda.Event() for _ in range(2)]
        # output slots: double-buffered per target of a job, so that the kernels of chunk k+1 never wait for
        # the downloads of chunk k (a pair job fills two slots at once)
        # (XRS_PIPE_OUT_SLOTS overrides the count for measurements: with two slots a pair's kernel waits for
        # both downloads of the previous chunk, 147 vs 141 ms per C2 call, profiles/r02c_e2e_ab_same_box.json)
        n_out = int(os.environ.get("XRS_PIPE_OUT_SLOTS", 4 if process_pair is not None else 2))
        out_free = [torch.cuda.Event() for _ in range(n_out)]
        for e in in_free + out_free:
            e.record(main)
        keep = []
        for grp in groups:
            v = grp.values
            lazy = hasattr(v, "read_bands")
            on_device = lazy and getattr(v, "device_decodable", False)  # compressed chunks decode on the device
            dtype = np.dtype(v.dtype).newbyteorder("=") if on_device else np.dtype(v.dtype)
            bands = (1 if v.ndim == 2 else v.shape[0]) if lazy else v.shape[0]
            h, w = v.shape[-2:]
            if (h, w) != (self.h, self.w):
                raise ValueError(f"variable of shape {(h, w)} does not match the source image {(self.h, self.w)}")
            isz = dtype.itemsize
            per = max(1, self.pitch_bytes // isz)
            wp = -(-w // per) * per
            chunk = max(1, min(self.chunk, bands))
            in_slots = self._slots(self._in_slots, (dtype.str, chunk), (chunk, win_h, wp), dtype)
            schedule = chunk_schedule(bands, chunk)
            if on_device:
                # the chunk files of band chunk k+1 are read into one of two page-locked byte buffers on a reader
                # thread while chunk k's files are uploaded and decoded into its slot (xrs_zarr_decode)
                from concurrent.futures import ThreadPoolExecutor

                lib = load()
                files = [None, None]
                stage_done = [None, None]
                reader = ThreadPoolExecutor(max_workers=1)
                pending = reader.submit(v.device_read, schedule[0][0], schedule[0][1], self.segments, self.win)
                with torch.cuda.stream(s_in):
                    errs = torch.zeros(len(schedule), dtype=torch.int32, device=dev)
                dev_bytes = ws = None
                paths_of = []
                self._decode_checks.append((errs, paths_of))
                keep.append(files)
            elif lazy:
                # the I/O edge: band chunk k+1 is read from the store into one of two page-locked staging
                # buffers on a reader thread while chunk k is copied to the device
                from concurrent.futures import ThreadPoolExecutor

                stage = [_dev.pinned_empty((chunk, h, w), dtype) for _ in range(2)]
                stage_done = [None, None]
                reader = ThreadPoolExecutor(max_workers=1)
                pending = reader.submit(v.read_bands, schedule[0][0], schedule[0][1], stage[0])
                keep.append(stage)
            else:
                base = v.__array_interface__["data"][0]
                sb, sr = v.strides[0], v.strides[1]
            for ci, (b0, nb) in enumerate(schedule):
                if on_device:
                    files[ci % 2] = pending.result()
                    buf, n_bytes, table, paths = files[ci % 2]
                    paths_of.append(paths)
                    if ci + 1 < len(schedule):
                        if stage_done[(ci + 1) % 2] is not None:
                            stage_done[(ci + 1) % 2].synchronize()  # its previous decode has left the buffer
                        prev = files[(ci + 1) % 2]
                        pending = reader.submit(v.device_read, schedule[ci + 1][0], schedule[ci + 1][1], self.segments,
                                                self.win, None if prev is None else prev[0])
                elif lazy:
                    pending.result()
                    base, sb, sr = stage[ci % 2].__array_interface__["data"][0], h * w * isz, w * isz
                    if ci + 1 < len(schedule):
                        if stage_done[(ci + 1) % 2] is not None:
                            stage_done[(ci + 1) % 2].synchronize()  # its previous upload has left the buffer
                        pending = reader.submit(v.read_bands, schedule[ci + 1][0], schedule[ci + 1][1],
                                                stage[(ci + 1) % 2])
                b_off = 0 if lazy else b0
                slot = k_in % 2
                k_in += 1
                src_slot = in_slots[slot]
                with torch.cuda.stream(s_in):
                    s_in.wait_event(in_free[slot])
                    if on_device:
                        ws_bytes = zarr_workspace_bytes(lib, v, table)
                        if dev_bytes is None or dev_bytes.numel() < n_bytes:
                            dev_bytes = torch.empty(max(n_bytes + (n_bytes >> 3), 1 << 20), dtype=torch.uint8, device=dev)
                        if ws is None or ws.numel() < ws_bytes:
                            ws = torch.empty(max(ws_bytes + (ws_bytes >> 3), 1 << 20), dtype=torch.uint8, device=dev)
                        if n_bytes:
                            copy2d(dev_bytes.data_ptr(), n_bytes, n_bytes, buf.ctypes.data, n_bytes, n_bytes, n_bytes, 1,
                                   1, dev)
                        check(zarr_decode(lib, v, dev_bytes.data_ptr(), n_bytes, table, src_slot.data_ptr(), wp,
                                          win_h * wp, self.win, b0, nb, ws.data_ptr(), ws.numel(),
                                          errs.data_ptr() + 4 * ci, _dev.stream_ptr(dev)), "xrs_zarr_decode")
                        self.h2d_bytes += n_bytes
                        keep.append((dev_bytes, ws))
                    else:
                        for (j0, j1, i0, i1) in self.segments:
                            copy2d(src_slot.data_ptr() + ((j0 - self.win[0]) * wp + i0) * isz, wp * isz,
                                   win_h * wp * isz, base + b_off * sb + j0 * sr + i0 * isz, sr, sb, (i1 - i0) * isz,
                                   j1 - j0, nb, dev)
                            self.h2d_bytes += (i1 - i0) * isz * (j1 - j0) * nb
                    ready = torch.cuda.Event()
                    ready.record(s_in)
                if lazy:
                    stage_done[ci % 2] = ready
                main.wait_event(ready)
                src_view = src_slot[:nb, :, :w]
                for job in (pair_targets(grp.targets, dtype) if process_pair is not None
                            else [(t,) for t in grp.targets]):
                    # one output slot per target of the job (a pair takes both slots of its dtype)
                    views, oslots = [], []
                    for tgt in job:
                        oslot = k_out % n_out
                        k_out += 1
                        out_slots = self._slots(self._out_slots, (tgt.out_dtype.str, chunk),
                                                (chunk, n_rows, self.out_w), tgt.out_dtype, n_out)
                        main.wait_event(out_free[oslot])
                        views.append(out_slots[oslot][:nb])
                        oslots.append(oslot)
                    if len(job) == 2:
                        process_pair(src_view, job[0], job[1], views[0], views[1], b0)
                    else:
                        process(src_view, job[0], views[0], b0)
                    done = torch.cuda.Event()
                    done.record(main)
                    for tgt, out_view, oslot in zip(job, views, oslots):
                        oh = tgt.out_host
                        osz = oh.itemsize
                        if oh.ndim != 3 or oh.shape[2] != self.out_w or oh.strides[2] != osz:
                            raise ValueError("output arrays must be (bands, rows, width) with unit x stride")
                        with torch.cuda.stream(s_out):
                            s_out.wait_event(done)
                            copy2d(oh.__array_interface__["data"][0] + b0 * oh.strides[0]
                                   + (self.rows[0] - tgt.row0) * oh.strides[1],
                                   oh.strides[1], oh.strides[0], out_view.data_ptr(), self.out_w * osz,
                                   n_rows * self.out_w * osz, self.out_w * osz, n_rows, nb, dev)
                            self.d2h_bytes += self.out_w * osz * n_rows * nb
                            out_free[oslot].record(s_out)
                in_free[slot].record(main)
            if lazy:
                reader.shutdown(wait=True)
            keep.append(v)
        self._keep = keep
        self._pending = (s_out, main)
        if wait:
            self.wait()
