#!/usr/bin/env python
"""bench.py -- throughput of the rectify hot path on B200 (BASELINE.json configs[1], "C2").

Workload: Sentinel-3 OLCI-shaped swath (4865 x 4091 lon/lat float64, 21 float32 bands) rectified to
a regular 0.0027 deg (~300 m) EPSG:4326 grid with nearest AND bilinear interpolation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *scene pass* is ONE ``rectify_dataset`` call that produces the 21 bands with both methods (the
band stack enters the dataset under two variable names with ``interp_methods`` per variable): as in
the reference (rectify.py:146), the source-index image is computed once per call and shared by all
variables -- K0 (tile windows) + K1 (ij image) + K2 gather x 2.  One *step* on N GPUs rectifies N
scenes; every scene is cut into N target row bands and rank r computes band r of every scene (weak
scaling: one scene-equivalent per GPU and step).  The only exchange step is the MIN all-reduce
(NCCL) of the partial tile / footprint tables that the ranks get from scanning 1/N of the swath
coordinates each.  ``value`` is output Mpix*band/s with the inputs resident in HBM; ``e2e`` is the
same metric through the public API with host (pinned) inputs and outputs, copies inside the timed
region.  Rank 0 prints ONE JSON line.

The device-resident part is timed twice over K steps each: eagerly, launch after launch, with a
CUDA event pair around every kernel (the per-kernel durations of ``roofline``), then as K replays
of a CUDA graph of the same step (``value``; ``--no-graph`` takes it from the eager region).
At N=1 the line also carries ``configs``: kernel times of the other BASELINE.json configurations
(C1 affine, C3 reproject, C4 coarsen, C5 reproject row band) with a CPU figure beside each.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "output Mpix*band/s"
UNIT = "Mpix*band/s"
TILE = 512
METHODS = ("nearest", "bilinear")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the scene (debugging only; 1.0 = BASELINE config)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (debugging only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (debugging only)")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1/C3/C4/C5 kernel timings (debugging only)")
    ap.add_argument("--fused", action="store_true",
                    help="device-resident leg: one fused xrs_rectify_gather per method (ij in registers, claims "
                         "computed per method) instead of the shared ij image + xrs_gather_ij")
    ap.add_argument("--dual", dest="dual", action="store_true", default=None,
                    help="device-resident leg: nearest + bilinear of the scene in ONE gather launch (xrs_gather_ij2); "
                         "default: what rectify_dataset does (rectify.DUAL_GATHER)")
    ap.add_argument("--no-dual", dest="dual", action="store_false",
                    help="one xrs_gather_ij launch per method (the round-1/early round-2 form)")
    ap.add_argument("--chains", type=int, default=4, help="N > 1: concurrent chains of scenes inside the step's CUDA graph")
    ap.add_argument("--split-k2", action="store_true",
                    help="N = 1: run the nearest and the bilinear gather of the scene as two concurrent chains "
                         "(measured slower than back to back: 3.53 vs 3.46 ms)")
    ap.add_argument("--no-graph", action="store_true", help="take `value` from the eager, sequential region")
    ap.add_argument("--cpu-kind", default="auto", choices=["auto", "reference", "port"],
                    help="CPU baseline: the reference's own numba kernels (oracle/_ref) or the C restatement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's outputs as DIR/<name>.npy "
                         "(float32, every band at the same seeded target pixels; with N > 1 GPUs rank 0's row band) "
                         "to compare two builds; --impl reference writes nothing and says so in its result line")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------
def make_scene(scale=1.0, seed=0, n_bands=None):
    from xcube_resampling_b200 import synthetic as syn

    w = max(64, int(round(syn.OLCI_WIDTH * scale)))
    h = max(64, int(round(syn.OLCI_HEIGHT * scale)))
    nb = syn.OLCI_BANDS if n_bands is None else n_bands
    lon, lat = syn.swath(w, h, res=syn.OLCI_RES_DEG, theta=12.0, seed=seed)
    size, xy_min = syn.covering_grid_args(lon, lat, syn.OLCI_RES_DEG)
    bands = syn.band_stack(nb, h, w, seed=seed)
    return lon, lat, bands, size, xy_min, syn.OLCI_RES_DEG


def workload_config(w, h, nb, size, n_gpus):
    return {
        "workload": "rectify_dataset: OLCI-shaped swath -> regular 300 m EPSG:4326 grid, nearest + bilinear",
        "source": f"{w}x{h} lon/lat float64, {nb} float32 bands",
        "target": f"{size[0]}x{size[1]} @0.0027deg, reference tile_size {TILE}",
        "scene_pass": "ONE rectify_dataset call giving the 21 bands with nearest and with bilinear interpolation: "
                      "K0 tile windows + K1 ij image once (shared by both, as in the reference), K2 gather of both methods",
        "scenes_per_step": n_gpus,
        "partition": "target row bands, rank r = band r of every scene; exchange step: one NCCL all-reduce(MIN) of "
                     "the partial tile/footprint tables (each rank scans 1/N of the swath coordinates)",
        "l2": "inputs (2.0 GB) and outputs (3.3 GB per method) exceed the 126 MB L2; no explicit flush",
    }


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled while the timed region runs.

    In-process NVML (the counters behind nvidia-smi's clocks.sm / clocks_event_reasons.* columns)
    every 10 ms from a thread that is joined when the timed region ends -- the device-resident
    region lasts tens of milliseconds, too short for ``nvidia-smi -lms``.  Falls back to an
    ``nvidia-smi -lms 100`` child (killed and reaped in stop()) when the NVML binding is missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASON_BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.thread = None
        self.stop_flag = threading.Event()
        self.sm, self.smax, self.reasons = [], [], set()
        self.source = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            handle = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.smax.append(float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM)))

            def loop():
                while not self.stop_flag.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)))
                        mask = int(reasons_fn(handle))
                        self.reasons.update(name for name, bit in self.REASON_BITS.items() if mask & bit)
                    except pynvml.NVMLError:
                        pass
                    self.stop_flag.wait(0.01)

            self.source = "nvml"
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:  # no NVML binding: the nvidia-smi child below
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _nvml_index(self):
        # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a list of indices
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join()
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.kill()
            self.proc.wait()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for ln in self.lines:
                f = [t.strip() for t in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    self.sm.append(float(f[1]))
                    self.smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(names, f[5:9]):
                    if val.lower().startswith("active"):
                        self.reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.smax) if self.smax else None, "samples": len(self.sm),
                "source": self.source, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------
# CPU arm: the reference's own numba kernels (oracle/_ref), or the C restatement (oracle port)
# ---------------------------------------------------------------------------
def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1)."""
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def run_cpu_port(steps, warmup, scale):
    """C/OpenMP restatement of the reference kernels (oracle/xrs_oracle.c), whole scenes."""
    import oracle
    from oracle import grid as ogrid
    from oracle import rectify as orect

    oracle.build()
    lon, lat, bands, size, xy_min, res = make_scene(scale=scale)
    oracle.lib().xrso_set_num_threads(host_threads())
    cores = oracle.lib().xrso_num_threads()
    g = ogrid.regular_grid(size, xy_min, res, tile_size=TILE)

    def scene_pass():
        windows = orect.source_windows(lon, lat, g)
        ij = orect.rectify_ij(lon, lat, g, windows=windows)
        return sum(orect.gather(bands, ij, m, np.nan).size for m in METHODS)

    for _ in range(warmup):
        scene_pass()
    t0 = time.perf_counter()
    units = sum(scene_pass() for _ in range(steps))
    dt = time.perf_counter() - t0
    h, w = lon.shape
    sample = (f"{steps} scene pass(es) of the {w}x{h} swath, {bands.shape[0]} bands -> {size[0]}x{size[1]}, "
              f"nearest+bilinear with one shared ij image, {dt:.1f} s")
    return {"value": units / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
            "ms_per_step": dt / steps * 1e3,
            "what": "oracle/xrs_oracle.c: C/OpenMP restatement of the reference's numba kernels"}


def run_cpu_reference(steps, warmup, scale, budget_s=25.0):
    """The reference's own numba kernels (unmodified package in oracle/_ref), tile by tile on a
    thread pool = dask's threaded scheduler with nogil kernels.  A step processes a bounded sample of
    the scene's target tiles (every k-th tile, so that empty corner tiles and full centre tiles are
    represented in proportion); throughput = output pixels*bands of those tiles / time."""
    from oracle import grid as ogrid
    from oracle import refkernels as rk

    rk.load()
    lon, lat, bands, size, xy_min, res = make_scene(scale=scale)
    g = ogrid.regular_grid(size, xy_min, res, tile_size=TILE)
    nty, ntx = g.n_tiles
    n_tiles = nty * ntx
    cores = host_threads()
    # JIT warm-up on a tiny scene (excluded), then one probe tile set to size the sample
    l2, a2, b2, s2, m2, _ = make_scene(scale=0.03, n_bands=2)
    rk.rectify_pass(l2, a2, b2, ogrid.regular_grid(s2, m2, res, tile_size=64), METHODS, cores)
    stride = max(1, n_tiles // max(cores, 8))
    ids = np.arange(0, n_tiles, stride)
    t0 = time.perf_counter()
    units = rk.rectify_pass(lon, lat, bands, g, METHODS, cores, tile_ids=ids)[0]
    probe = time.perf_counter() - t0
    per_tile = probe / len(ids)
    n_steps = max(1, steps)
    want = max(len(ids), min(n_tiles, int(budget_s / n_steps / max(per_tile, 1e-6))))
    stride = max(1, n_tiles // want)
    ids = np.arange(0, n_tiles, stride)
    for _ in range(max(0, warmup - 1)):
        rk.rectify_pass(lon, lat, bands, g, METHODS, cores, tile_ids=ids)
    t0 = time.perf_counter()
    units = 0
    for _ in range(n_steps):
        units += rk.rectify_pass(lon, lat, bands, g, METHODS, cores, tile_ids=ids)[0]
    dt = time.perf_counter() - t0
    h, w = lon.shape
    sample = (f"{n_steps} step(s) over {len(ids)} of the {n_tiles} {TILE}x{TILE} target tiles (every {stride}-th) of the "
              f"{w}x{h} swath -> {size[0]}x{size[1]}, {bands.shape[0]} bands, nearest+bilinear with one shared ij "
              f"image, {dt:.1f} s; numba JIT warm-up excluded")
    return {"value": units / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample,
            "ms_per_step": dt / n_steps * 1e3,
            "what": "xcube_resampling's own numba kernels (compute_ij_bboxes, _compute_target_source_ij_sequential, "
                    "_compute_var_image_sequential) from oracle/_ref, per target tile on a ThreadPoolExecutor"}


def run_cpu(steps, warmup, scale, kind="auto"):
    notes = None
    if kind in ("auto", "reference"):
        try:
            return run_cpu_reference(steps, warmup, scale)
        except Exception as e:  # reference package or numba missing on this box: say so, use the port
            notes = f"reference kernels unavailable ({type(e).__name__}: {e}); fell back to the C restatement"
            if kind == "reference":
                raise
    out = run_cpu_port(steps, warmup, scale)
    if notes:
        out["note"] = notes
    return out


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpu = run_cpu(args.steps, args.warmup, args.scale, args.cpu_kind)
    from xcube_resampling_b200 import synthetic as syn

    w, h = max(64, int(round(syn.OLCI_WIDTH * args.scale))), max(64, int(round(syn.OLCI_HEIGHT * args.scale)))
    lon, lat = syn.swath(w, h, res=syn.OLCI_RES_DEG, theta=12.0, seed=0)
    size, _ = syn.covering_grid_args(lon, lat, syn.OLCI_RES_DEG)
    value = cpu["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cpu.pop("ms_per_step"), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(w, h, syn.OLCI_BANDS, size, args.gpus),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:  # the CPU arm times a sample of target tiles; it has no whole outputs to write
        line["notes"] = ["--dump-outputs: nothing written; it writes the outputs of the GPU path (--impl ours)"]
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def pin_to_gpu_numa_node(gpu_index):
    """Restrict this process to the CPUs NVML reports as local to the GPU, so that page-locked host
    buffers (first touched here) sit on the NUMA node of the GPU's PCIe root.  Returns the original
    CPU set (restored before the CPU baseline runs); a no-op when NVML is unavailable."""
    try:
        original = os.sched_getaffinity(0)
    except (AttributeError, OSError):
        return None
    from xcube_resampling_b200._affinity import bind_to_device

    bind_to_device(gpu_index)  # best effort: no NVML / nothing local in the cpuset leave the affinity as inherited
    return original


def load_traffic_table():
    """ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, keyed by kernel name, from the
    committed capture summary profiles/kernel_traffic.json (written by tools/ncu_traffic.py from a
    `ncu --set full` run of this workload at N=1)."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as fh:
            return json.load(fh)
    except (OSError, ValueError):
        return {}


def ours(args):
    import torch
    import torch.distributed as dist

    import xcube_resampling_b200 as xrs
    from xcube_resampling_b200 import _dev, _lib, _pipeline, bands as xbands, multigpu, rectify as xrect

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    all_cpus = pin_to_gpu_numa_node(local_rank)  # pinned host buffers land next to the GPU's PCIe root
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    notes = []
    dual = (xrect.DUAL_GATHER if args.dual is None else args.dual) and not args.fused
    xrect.DUAL_GATHER = dual  # the end-to-end leg (rectify_dataset / rectify_band_stream) takes the same form

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        return xbands.max_over_ranks(ms, dev)

    def sum_over_ranks(v):
        return xbands.sum_over_ranks(v, dev)

    # ---- scene + geometry (every rank builds the same synthetic scene) ----------------
    lon, lat, bands, size, xy_min, res = make_scene(scale=args.scale)
    nb, h, w = bands.shape
    target_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=TILE)
    W_t, H_t = target_gm.size
    group = int(lib.xrs_quad_row_group())
    n_groups = -(-(h - 1) // group)
    x_dev = _dev.to_device(lon)
    y_dev = _dev.to_device(lat)

    # ---- end to end through the public API with host buffers --------------------------
    # (This leg runs before the device-resident one, so that neither the clock sampler nor the
    # device-resident buffers' allocation is in flight while it is timed.)
    e2e = None
    if not args.no_e2e:
        lon_p, lat_p = _dev.pinned_empty(lon.shape, np.float64), _dev.pinned_empty(lat.shape, np.float64)
        lon_p[...] = lon
        lat_p[...] = lat
        bands_p = _dev.pinned_empty(bands.shape, np.float32)
        bands_p[...] = bands
        e2e_steps = args.steps
        interp = {"bands_nearest": "nearest", "bands_bilinear": "bilinear"}
        if world == 1:
            ds = xrs.Dataset(data_vars=dict(bands_nearest=(("band", "y", "x"), bands_p),
                                            bands_bilinear=(("band", "y", "x"), bands_p)),
                             coords=dict(lon=(("y", "x"), lon_p), lat=(("y", "x"), lat_p)))
            source_gm = xrs.GridMapping.from_coords(lon_p, lat_p, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
            h2d_scene = lon_p.nbytes + lat_p.nbytes + bands_p.nbytes
            d2h_scene = len(METHODS) * nb * H_t * W_t * 4

            def e2e_step():
                out = xrs.rectify_dataset(ds, target_gm=target_gm, source_gm=source_gm, interp_methods=interp)
                return sum(out[name].values.size for name in interp), h2d_scene, d2h_scene

            api = "rectify_dataset(ds, target_gm, source_gm, interp_methods={var: method})"
        else:
            edges_e2e = multigpu.default_band_edges(H_t, world)
            r0, r1 = edges_e2e[rank], edges_e2e[rank + 1]
            outs_p = {m: _dev.pinned_empty((nb, max(r1 - r0, 1), W_t), np.float32) for m in METHODS}
            groups = _pipeline.group_by_buffer(
                [(bands_p, _pipeline.Target(f"bands_{m}", m, np.nan, outs_p[m], row0=r0)) for m in METHODS])
            exchange = multigpu.DistExchange()
            plans_e2e = [xrect.RectifyPlan(target_gm, dev, rows=(r0, r1)) for _ in range(2)]

            def e2e_step():
                # the step's N scenes as one stream of band jobs: the prologue of scene s+1 (slab scan, NCCL
                # all-reduce of the tables, footprint, K1) overlaps the data streaming of scene s
                stats = multigpu.rectify_band_stream(((lon_p, lat_p, groups) for _ in range(world)), target_gm,
                                                     edges_e2e, rank, exchange, device=dev, plans=plans_e2e)
                n = world * len(METHODS) * nb * (r1 - r0) * W_t
                return n, sum(st.h2d_bytes for st in stats), sum(st.d2h_bytes for st in stats)

            api = ("multigpu.rectify_band_stream per rank (the per-device worker of rectify_dataset(..., devices=range(N)), "
                   "over the step's N scenes): slab scan + NCCL all-reduce(MIN) of the tables + footprint-only uploads "
                   "+ band download")

        # Warm-up to steady state.  The first step page-locks the output buffers (seconds); for two to
        # three seconds after that, single steps were measured to take 1.5-4x longer at random on
        # this pool (host-side).  Warm-up therefore runs for at least 4 s after the first step AND until
        # three consecutive steps agree within 3 % on every rank (at most 60 steps or 25 s).
        warm_ms = []
        t_first = None
        while len(warm_ms) < 60:
            ts = time.perf_counter()
            e2e_step()
            warm_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
            if t_first is None:
                t_first = time.perf_counter()
            last = warm_ms[-3:]
            waited = time.perf_counter() - t_first
            steady = (len(warm_ms) >= 4 and max(last) <= 1.03 * min(last) and waited >= 4.0) or waited >= 25.0
            if max_over_ranks(0.0 if steady else 1.0) == 0.0:
                break
        barrier()
        t0 = time.perf_counter()
        n_units = h2d = d2h = 0
        step_ms = []
        for _ in range(e2e_steps):
            ts = time.perf_counter()
            n, a, b = e2e_step()
            n_units += n
            h2d += a
            d2h += b
            step_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
        torch.cuda.synchronize()
        dt_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        n_units = sum_over_ranks(float(n_units))
        h2d = sum_over_ranks(float(h2d)) / e2e_steps
        d2h = sum_over_ranks(float(d2h)) / e2e_steps
        e2e = {"value": n_units / (dt_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": dt_ms / e2e_steps,
               "rank0_step_ms": step_ms, "rank0_warmup_step_ms": warm_ms,
               "api": api + ": pinned host arrays in, pinned host arrays out, host clock around synchronised calls"}
        if world > 1:
            del outs_p, groups
        del bands_p

    # ---- device-resident leg ----------------------------------------------------------
    if world == 1:
        edges = [0, H_t]
    else:
        # Row bands of equal WORK, not equal height: a rotated swath leaves the top and bottom rows of
        # the target mostly empty.  The weights come from one full ij image (valid pixels per row plus
        # a constant for the fill writes: measured at N=1, a valid pixel costs ~103 ps across K1 + both
        # gathers, a fill pixel ~31 ps, i.e. row cost ~ valid + 0.43 * width); every rank derives the
        # same partition.
        ij_full = xrect.RectifyPlan(target_gm, dev).ij(x_dev, y_dev)
        valid_per_row = (~torch.isnan(ij_full[0])).sum(dim=1).cpu().numpy().astype(np.float64)
        del ij_full
        bands_w = xbands.weighted_row_bands(valid_per_row + 0.43 * W_t, world, align=8)
        edges = [b[0] for b in bands_w] + [H_t]
    rows = (edges[rank], edges[rank + 1])
    band_px = (rows[1] - rows[0]) * W_t
    src_dev = _dev.to_device_pitched(bands, dev)  # 128-byte row pitch -> TMA-staged gather
    n_chains = max(1, args.chains)
    n_plans = 1 if world == 1 else min(n_chains, world)
    # one set of output buffers per concurrent chain of scenes
    outs_c = [{m: torch.empty((nb, rows[1] - rows[0], W_t), dtype=torch.float32, device=dev) for m in METHODS}
              for _ in range(n_plans)]
    outs = outs_c[0]
    plans = [xrect.RectifyPlan(target_gm, dev, rows=rows) for _ in range(max(n_plans, 2 if args.fused else 1))]
    n_tiles = plans[0].ntx * plans[0].nty
    table_len = 4 * n_tiles + 2 * world * n_groups
    s0, s1 = multigpu.source_slabs(h, world, group)[rank]
    s1v = min(h, s1 + 1)
    tables = _dev.empty((world, table_len), np.int32, dev)  # one min-form table per scene of the step
    torch.cuda.synchronize()
    pending = []  # (name, start event, end event) of the eager region's phases

    def mark(record):
        if not record:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def scan_scene(scene, plan):
        if s1 > s0:
            plan.scan_slab(x_dev[s0:s1v], y_dev[s0:s1v], s0, s1 - s0, h, w, edges, tables[scene])

    def check_rc(rc):
        _lib.check(rc, "libxrs")

    def gather_scene(plan, scene, record, outs=outs, split=False):
        """K1 on this rank's band (restricted to the band's footprint when N > 1) + K2 per method."""
        e0 = mark(record)
        if world == 1:
            boxes = plan.windows(x_dev, y_dev)
            e1 = mark(record)
            if args.fused:
                e2 = e1
            else:
                ij = plan.ij(x_dev, y_dev, boxes)
                e2 = mark(record)
        else:
            boxes = plan.finalize_windows(tables[scene], w, h)
            e1 = mark(record)
            col_ranges = tables[scene][4 * n_tiles:].view(world, n_groups, 2)[rank]
            ij = plan.ij_window(x_dev, y_dev, 0, h, w, boxes, col_ranges)
            e2 = mark(record)
        ends = []
        if split:  # the two gathers of the scene side by side: bilinear is fp64-issue bound, nearest HBM bound
            main = torch.cuda.current_stream(dev)
            fork = torch.cuda.Event()
            fork.record(main)
            chains[0].wait_event(fork)
            with torch.cuda.stream(chains[0]):
                xrect.gather_ij(src_dev, ij, METHODS[0], np.nan, out=outs[METHODS[0]])
                joined = torch.cuda.Event()
                joined.record(chains[0])
            xrect.gather_ij(src_dev, ij, METHODS[1], np.nan, out=outs[METHODS[1]])
            main.wait_event(joined)
            return
        if dual:  # both methods of the scene from ONE pass over ij and the source
            xrect.gather_ij_pair(src_dev, ij, METHODS[1], np.nan, np.nan, outs[METHODS[1]], outs[METHODS[0]])
            if record:
                pending.append(("k0", e0, e1))
                pending.append(("k1", e1, e2))
                pending.append(("k2_nearest+bilinear", e2, mark(record)))
            return
        for k, m in enumerate(METHODS):
            if world == 1 and args.fused:
                plans[k].rectify_gather(x_dev, y_dev, src_dev, m, np.nan, out=outs[m], tile_boxes=boxes)
            else:
                xrect.gather_ij(src_dev, ij, m, np.nan, out=outs[m])
            ends.append(mark(record))
        if record:
            pending.append(("k0", e0, e1))
            pending.append(("k1", e1, e2))
            pending.append(("k2_nearest", e2, ends[0]))
            pending.append(("k2_bilinear", ends[0], ends[1]))

    chains = [torch.cuda.Stream(dev) for _ in range(n_chains)]

    def step(record=False, concurrent=False):
        if world == 1:
            gather_scene(plans[0], 0, record, split=concurrent and args.split_k2 and not args.fused and not dual)
            return
        # N > 1: scan 1/N of the coordinates of every scene of the step, ONE all-reduce(MIN) for all
        # their tables, then the band kernels scene after scene (two chains: a rank's band kernels are
        # 10-250 us, K0 finalize / K1 scatter latency-bound)
        e0 = mark(record)
        check_rc(lib.xrs_minform_init(_dev.ptr(tables), world * table_len, _dev.stream_ptr(dev)))  # all scenes at once
        main = torch.cuda.current_stream(dev)
        multi = concurrent and n_plans > 1

        def on_chains(work):
            """work(c) on chain c, forked from and joined to the main stream."""
            fork = torch.cuda.Event()
            fork.record(main)
            for c in range(n_plans):
                chains[c].wait_event(fork)
                with torch.cuda.stream(chains[c]):
                    work(c)
                    joined = torch.cuda.Event()
                    joined.record(chains[c])
                main.wait_event(joined)

        if multi:  # the slab scans of the scenes are latency-bound kernels of 40-70 us: side by side
            on_chains(lambda c: [scan_scene(scene, plans[c]) for scene in range(c, world, n_plans)])
        else:
            for scene in range(world):
                scan_scene(scene, plans[0])
        dist.all_reduce(tables, op=dist.ReduceOp.MIN)
        e1 = mark(record)
        if record:
            pending.append(("scan+allreduce", e0, e1))
        if multi:
            on_chains(lambda c: [gather_scene(plans[c], scene, False, outs=outs_c[c]) for scene in range(c, world, n_plans)])
        else:
            for scene in range(world):
                gather_scene(plans[0], scene, record)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.profile_collect()
    use_graph = not args.no_graph
    # Region A (every N): K eager steps, one launch after the other on one stream, with libxrs's
    # per-launch CUDA events -- the per-kernel durations behind `roofline`.
    launches0 = lib.xrs_launch_count()
    _lib.profile_enable(True)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(args.steps):
        step(record=True)
    a1.record()
    torch.cuda.synchronize()
    _lib.profile_enable(False)
    kernel_times = _lib.profile_collect()
    launches = lib.xrs_launch_count() - launches0
    eager_ms = max_over_ranks(a0.elapsed_time(a1))
    e0, e1 = a0, a1
    graph_used = False
    graph = None
    if use_graph:
        # Region B, the one `value` is computed from: the same step captured once in a CUDA graph and
        # replayed K times (at N > 1 the all-reduce is captured with it).
        try:
            step(concurrent=True)  # eagerly once: every chain's plan allocates its workspaces / uploads its tables
            barrier()
            launches0 = lib.xrs_launch_count()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step(concurrent=True)
            per_step = lib.xrs_launch_count() - launches0
            graph.replay()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(args.steps):
                graph.replay()
            g1.record()
            torch.cuda.synchronize()
            e0, e1 = g0, g1
            launches = per_step * args.steps
            graph_used = True
        except Exception as e:  # capture not possible on this box (e.g. NCCL refuses): keep the eager region
            notes.append(f"CUDA-graph capture failed ({type(e).__name__}: {e}); value is from the eager region")
            torch.cuda.synchronize()
    graph_ok = max_over_ranks(0.0 if graph_used else 1.0) == 0.0
    if use_graph and not graph_ok:
        e0, e1 = a0, a1
    my_ms = e0.elapsed_time(e1)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = max_over_ranks(my_ms)
    units_rank = args.steps * world * len(METHODS) * nb * band_px
    units = sum_over_ranks(float(units_rank))
    value = units / (total_ms * 1e-3) / 1e6
    phase_ms = {}
    for name, ea, eb in pending:
        phase_ms[name] = phase_ms.get(name, 0.0) + ea.elapsed_time(eb)
    n_pass = args.steps * world
    phase_ms = {k: v / (args.steps if k == "scan+allreduce" else n_pass) for k, v in phase_ms.items()}

    # ---- parity spot-check of the timed outputs against the oracle (rank 0) ----------------
    parity = None
    if rank == 0:
        ij_ref = None
        try:
            ij_ref = oracle_ij(lon, lat, size, xy_min, res)
            parity = spot_check(bands, ij_ref, outs, rows, plans[0] if not args.fused else None)
        except Exception as e:
            parity = {"error": f"{type(e).__name__}: {e}"}
        if args.dump_outputs:
            try:
                if ij_ref is None:
                    ij_ref = oracle_ij(lon, lat, size, xy_min, res)
                dump_outputs(outs, args.dump_outputs, np.isfinite(ij_ref[0, rows[0]:rows[1]]))
            except Exception as e:  # the result line below still goes out, saying so
                notes.append(f"--dump-outputs failed ({type(e).__name__}: {e})")

    # ---- roofline of the dominant kernel (largest share of the timed region) ------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    S = float(h * w)
    if world == 1:
        s_used = S
    else:
        # source pixels a band's kernels address: its ragged quad footprint (+1 vertex, +2 taps)
        fp = _dev.to_host(tables[0][4 * n_tiles:].view(world, n_groups, 2)[rank]).astype(np.int64)
        ok = fp[:, 0] != np.iinfo(np.int32).max
        s_used = float(np.sum((-fp[ok, 1] - fp[ok, 0] + 3) * group))
    T = float(band_px)
    fused = world == 1 and args.fused
    if fused:
        k2_index_bytes = 4.0 * T + 16.0 * S
        k2_model = "4*T (claims) + 16*S (winning quads' vertices) + 4*B*S_used (source once) + 4*B*T (output once)"
    else:
        k2_index_bytes, k2_model = 16.0 * T, "16*T (ij) + 4*B*S_used (source once) + 4*B*T (output once)"
    s_slab = float(max(s1v - s0, 0) * w)
    models = {
        "k0_tile_windows": (16.0 * (S if world == 1 else s_slab), "16*S_scanned (lon+lat fp64 read once)"),
        "kb_quad_footprints": (16.0 * s_slab, "16*S_slab (lon+lat fp64 of the slab read once)"),
        "k1_init_claims": (4.0 * T, "4*T (claim word per target pixel)"),
        "k1_scatter": (16.0 * s_used + 4.0 * T, "16*S_used (lon+lat fp64 read once) + 4*T (claim word per target pixel)"),
        "k1_scatter_slow": (0.0, "queue of border quads, no compulsory traffic of its own"),
        "k1_resolve": (4.0 * T + 16.0 * T + 16.0 * s_used, "4*T (claims) + 16*T (ij fp64 out) + 16*S_used (winning quads' vertices)"),
        "k2_gather_staged<nearest>": (k2_index_bytes + 4.0 * nb * s_used + 4.0 * nb * T, k2_model),
        "k2_gather_staged<bilinear>": (k2_index_bytes + 4.0 * nb * s_used + 4.0 * nb * T, k2_model),
        "k2_gather_dual<nearest+bilinear>": (16.0 * T + 4.0 * nb * s_used + 8.0 * nb * T,
                                             "16*T (ij) + 4*B*S_used (source once) + 8*B*T (nearest and bilinear output once each)"),
    }
    traffic_table = load_traffic_table() if (world == 1 and args.scale == 1.0) else {}
    traffic_key = "fused" if fused else "dual" if dual else "two_step"
    total_kernel_ms = sum(v[0] for v in kernel_times.values()) or 1.0
    kernels = []
    for name, (ms_total, n_launch) in sorted(kernel_times.items(), key=lambda kv: -kv[1][0]):
        ms_launch = ms_total / max(n_launch, 1)
        nbytes, model = models.get(name, (0.0, "n/a"))
        gbs = nbytes / (ms_launch * 1e-3) / 1e9 if ms_launch > 0 else 0.0
        traffic = (traffic_table.get(traffic_key, {}).get(name) or traffic_table.get("two_step", {}).get(name)
                   or {}).get("dram_bytes_per_launch")
        kernels.append({"kernel": name, "launches": int(n_launch), "ms_per_launch": ms_launch,
                        "share_of_kernel_time": ms_total / total_kernel_ms, "algorithmic_bytes_per_launch": nbytes,
                        "achieved_gbs": gbs, "frac": gbs / peak, "bytes_model": model, "traffic": traffic})
    top = kernels[0] if kernels else {"kernel": "none", "ms_per_launch": 0.0, "achieved_gbs": 0.0, "frac": 0.0,
                                      "algorithmic_bytes_per_launch": 0.0, "bytes_model": "n/a",
                                      "share_of_kernel_time": 0.0, "traffic": None}
    step_bytes = sum(k["algorithmic_bytes_per_launch"] * k["launches"] for k in kernels) / max(args.steps, 1)
    roofline = {
        "bound": "hbm", "kernel": top["kernel"], "achieved": top["achieved_gbs"], "peak": peak,
        "peak_kind": peak_kind, "unit": "GB/s", "frac": top["frac"],
        "traffic": top["traffic"],
        "traffic_source": ("profiles/kernel_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch from "
                           + str(traffic_table.get(traffic_key + "_source") if top["kernel"] in traffic_table.get(traffic_key, {})
                                 and traffic_table.get(traffic_key + "_source") else traffic_table.get("source")))
        if top["traffic"] else None,
        "algorithmic_bytes_per_launch": top["algorithmic_bytes_per_launch"], "bytes_model": top["bytes_model"],
        "ms_per_launch": top["ms_per_launch"], "share_of_kernel_time": top["share_of_kernel_time"],
        "timing": "CUDA events recorded by libxrs around every launch on the launching stream over K eager, "
                  "sequential steps (ms_per_step_eager)" +
                  ("; `value` is timed over K CUDA-graph replays of the same step" if graph_used and graph_ok
                   else "; `value` is that region"),
        "ms_per_step_eager": eager_ms / args.steps,
        "whole_step": {"algorithmic_bytes": step_bytes, "ms": total_ms / args.steps,
                       "frac": step_bytes / (total_ms / args.steps * 1e-3) / 1e9 / peak if total_ms > 0 else None},
        "kernels": kernels, "phase_ms_per_scene": phase_ms,
    }
    del src_dev, outs, outs_c, plans
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations (N=1 only) -------------------------------
    configs = None
    if rank == 0 and world == 1 and not args.no_configs and args.scale == 1.0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs

            configs = bench_configs.run_all(reps=3, cpu=not args.no_cpu, cpu_threads=len(all_cpus) if all_cpus else None,
                                            restore_affinity=all_cpus)
        except Exception as e:
            configs = [{"error": f"{type(e).__name__}: {e}"}]

    # ---- BASELINE.json configs[4] across the N GPUs by target row bands (N > 1) ----------------
    if world > 1 and not args.no_configs and args.scale == 1.0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs

            barrier()
            err5 = None
            try:
                c5 = bench_configs.c5_across(rank, world, reps=3, e2e=not args.no_e2e)
            except Exception as e:  # keep the ranks' collectives below in step whatever happened here
                err5 = f"{type(e).__name__}: {e}"
                c5 = {"kernel_ms": 1.0, "units": 0, "algorithmic_bytes": 0.0, "per_band_ms": [], "e2e_s": 1.0,
                      "h2d_bytes": 0, "d2h_bytes": 0}
                if args.no_e2e:
                    c5["e2e_s"] = None
            if max_over_ranks(1.0 if err5 else 0.0) != 0.0:
                raise RuntimeError(err5 or "C5 failed on another rank")
            kernel_ms = max_over_ranks(c5["kernel_ms"])
            units = sum_over_ranks(float(c5["units"]))
            alg = sum_over_ranks(c5["algorithmic_bytes"])
            barrier()
            line5 = {"config": f"C5 reproject global 0.01deg (36000x18000, 8 float32 variables) -> EPSG:3857 36000^2 across "
                               f"{world} GPUs by target row bands of 4500 rows, bilinear, float32 out",
                     "ms": kernel_ms, "Mpix_band_per_s": units / kernel_ms / 1e3, "algorithmic_bytes": alg,
                     "GB_per_s": alg / kernel_ms / 1e6, "frac": alg / kernel_ms / 1e6 / (peak * world),
                     "timing": "per rank: CUDA events around xrs_reproject of each of its bands (median of 3), summed; "
                               "max over ranks", "rank0_per_band_ms": c5["per_band_ms"]}
            if c5["e2e_s"] is not None:
                e2e_s = max_over_ranks(c5["e2e_s"])
                line5["e2e"] = {"Mpix_band_per_s": units / e2e_s / 1e6, "seconds": e2e_s,
                                "h2d_bytes": int(sum_over_ranks(float(c5["h2d_bytes"]))),
                                "d2h_bytes": int(sum_over_ranks(float(c5["d2h_bytes"]))),
                                "api": "reproject_groups per rank (the per-device worker of reproject_dataset(..., "
                                       "devices=range(N))): footprint-only upload from page-locked host arrays, band "
                                       "download into page-locked host arrays"}
            configs = [line5]
        except Exception as e:
            configs = [{"config": "C5 across GPUs", "error": f"{type(e).__name__}: {e}"}]

    # ---- CPU baseline beside it (rank 0, N=1 only) -------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if all_cpus:
            os.sched_setaffinity(0, all_cpus)  # the CPU arm uses every host core again
        try:
            cpu = run_cpu(steps=2, warmup=1, scale=args.scale, kind=args.cpu_kind)
            cpu.pop("ms_per_step", None)
        except Exception as e:
            cpu = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(w, h, nb, size, world), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "k2_form": "fused" if fused else "dual" if dual else "per-method",
            "roofline": roofline, "cpu_baseline": cpu, "parity_check": parity,
            "configs": configs, "notes": notes,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down: the CUDA graph holds captured NCCL kernels; it must be gone, and every rank idle,
        # before the communicator is destroyed (destroying it under a live graph was seen to hang the
        # last rank for the watchdog's 8 minutes).  A timer makes sure a stuck tear-down cannot keep
        # the GPUs -- the result line is already printed.
        graph = None  # noqa: F841
        import gc

        gc.collect()
        torch.cuda.synchronize()
        sys.stdout.flush()
        killer = threading.Timer(20.0, lambda: os._exit(0))
        killer.daemon = True
        killer.start()
        try:
            dist.barrier()
            dist.destroy_process_group()
        finally:
            killer.cancel()


def oracle_ij(lon, lat, size, xy_min, res):
    """The oracle's ij image of the whole target (C restatement on all host threads, ~1 s at full size)."""
    import oracle
    from oracle import grid as ogrid
    from oracle import rectify as orect

    oracle.build()
    oracle.lib().xrso_set_num_threads(host_threads())
    return orect.rectify_ij(lon, lat, ogrid.regular_grid(size, xy_min, res, tile_size=TILE))


def spot_check(bands, ij, outs, rows, plan, strip=48):
    """The timed region's own outputs against the oracle (its ij image ``ij``) on a strip of target rows in the
    middle of this rank's band: ij image (when the two-step path ran) and both gathers of all bands, bit for bit."""
    from oracle import rectify as orect

    mid = (rows[0] + rows[1]) // 2
    a = max(rows[0], mid - strip // 2)
    b = min(rows[1], a + strip)
    ij_strip = np.ascontiguousarray(ij[:, a:b])
    out = {"rows": [int(a), int(b)], "bands": int(bands.shape[0])}
    if plan is not None:
        got_ij = plan.ij_buf[:, a - rows[0]:b - rows[0]].cpu().numpy()
        out["ij_bit_exact"] = bool(np.array_equal(got_ij, ij_strip, equal_nan=True))
        out["valid_px"] = int(np.isfinite(ij_strip[0]).sum())
    for m in METHODS:
        want = orect.gather(bands, ij_strip, m, np.nan)
        got = outs[m][:, a - rows[0]:b - rows[0]].cpu().numpy()
        out[f"{m}_bit_exact"] = bool(np.array_equal(got, want, equal_nan=True))
        out[f"{m}_mismatch_fraction"] = float(np.mean(~((got == want) | (np.isnan(got) & np.isnan(want)))))
    return out


DUMP_PIXELS = 1 << 18  # covered pixels per method: 21 bands x 2^18 x 4 B = 22 MB
DUMP_FILL_PIXELS = 1 << 15  # uncovered pixels per method: 21 bands x 2^15 x 4 B = 2.8 MB


def _seeded_sample(mask, n, seed):
    """Flat indices of ``n`` pixels drawn with a seeded generator from those ``mask`` marks (all of them when
    there are fewer), in raster order."""
    idx = np.flatnonzero(mask)
    if idx.size > n:
        idx = np.sort(np.random.default_rng(seed).choice(idx, size=n, replace=False))
    return idx


def dump_outputs(outs, out_dir, covered, n_pixels=DUMP_PIXELS, n_fill=DUMP_FILL_PIXELS, seed=0):
    """What the timed step hands back -- one (bands, rows, cols) float32 image per method with the NaN fill
    where no source pixel lands -- as a fixed, finite sample.  ``covered`` is where the oracle finds a source
    pixel; it depends on the inputs alone, never on the build that computed ``outs``.

    * ``out_dir/bands_<method>.npy`` (bands, n): every band at ``n_pixels`` covered pixels, the values;
    * ``out_dir/fill_<method>.npy`` (bands, n): every band at ``n_fill`` uncovered pixels, 1.0 where the output
      holds the NaN fill and 0.0 where it holds anything else (a build that writes outside the swath).

    Both sets are drawn with seeded generators and kept in raster order."""
    import torch

    covered = np.asarray(covered, dtype=bool)
    idx = _seeded_sample(covered.ravel(), n_pixels, seed)
    idx_fill = _seeded_sample(~covered.ravel(), n_fill, seed + 1)
    os.makedirs(out_dir, exist_ok=True)
    for m, img in outs.items():
        nb, h, w = img.shape
        assert covered.shape == (h, w), f"coverage {covered.shape} does not match the output {(h, w)}"
        flat = img.reshape(nb, h * w)
        sample = flat[:, torch.from_numpy(idx).to(img.device)]
        np.save(os.path.join(out_dir, f"bands_{m}.npy"), sample.cpu().numpy())
        is_fill = torch.isnan(flat[:, torch.from_numpy(idx_fill).to(img.device)])
        np.save(os.path.join(out_dir, f"fill_{m}.npy"), is_fill.to(torch.float32).cpu().numpy())


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
