"""Host-side pieces of bench.py that run without a GPU: the reference arm (the reference's own numba
kernels from oracle/_ref, or the C port of them, on a bounded sample), its JSON contract, and the helpers' behaviour when NVML /
nvidia-smi are absent."""

import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          cwd=ROOT, env=env, timeout=300)


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--scale", "0.05", "--steps", "1", "--warmup", "0", "--gpus", "2"])
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "output Mpix*band/s" and line["unit"] == "Mpix*band/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 2 and line["gpu_launches"] == 0
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cpu = line["cpu_baseline"]
    # the reference's own numba kernels when oracle/_ref (or /root/reference) is there, else the C port
    assert cpu["kind"] in ("reference", "port") and cpu["cores"] >= 1 and cpu["value"] == line["value"]
    assert "swath" in cpu["sample"]
    # the config is the GPU arm's, key for key (the bounded sample is described in cpu_baseline)
    sys.path.insert(0, ROOT)
    import bench

    assert set(line["config"]) == set(bench.workload_config(1, 1, 1, (1, 1), 2))
    assert line["config"]["scenes_per_step"] == 2


def test_reference_arm_port_kind():
    r = _run(["--impl", "reference", "--scale", "0.05", "--steps", "1", "--warmup", "0", "--cpu-kind", "port"])
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["kind"] == "port" and line["value"] > 0


def test_reference_arm_only_rank_zero_works():
    r = _run(["--impl", "reference", "--scale", "0.05", "--steps", "1", "--warmup", "0"], {"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_argument_checks(tmp_path):
    r = _run(["--steps", "0"])
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    # the CPU arm has no whole outputs: nothing written, and its result line says so
    r = _run(["--impl", "reference", "--scale", "0.05", "--steps", "1", "--warmup", "0", "--cpu-kind", "port",
              "--dump-outputs", str(tmp_path / "dump")])
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert "--dump-outputs: nothing written" in line["notes"][0] and not (tmp_path / "dump").exists()


def test_dump_outputs_is_a_fixed_sample_of_every_band(tmp_path):
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    j, i = np.mgrid[:40, :50]
    covered = np.abs(i - 25 - 0.4 * (j - 20)) < 15  # a slanted swath; the NaN fill outside it
    imgs = {}
    for k, m in enumerate(bench.METHODS):
        img = torch.rand((3, 40, 50), generator=torch.Generator().manual_seed(k))
        img[:, torch.from_numpy(~covered)] = float("nan")
        imgs[m] = img
    bench.dump_outputs(imgs, str(tmp_path / "a"), covered, n_pixels=300, n_fill=100)
    bench.dump_outputs({m: img.clone() for m, img in imgs.items()}, str(tmp_path / "b"), covered, n_pixels=300,
                       n_fill=100)
    for m, img in imgs.items():
        a, b = np.load(tmp_path / "a" / f"bands_{m}.npy"), np.load(tmp_path / "b" / f"bands_{m}.npy")
        assert a.dtype == np.float32 and a.shape == (3, 300) and np.array_equal(a, b) and np.isfinite(a).all()
        flat = img.numpy().reshape(3, -1)
        cols = [int(np.flatnonzero(flat[0] == v)[0]) for v in a[0]]  # the sampled pixels, in raster order
        assert cols == sorted(set(cols)) and covered.ravel()[cols].all() and np.array_equal(a, flat[:, cols])
        fa, fb = np.load(tmp_path / "a" / f"fill_{m}.npy"), np.load(tmp_path / "b" / f"fill_{m}.npy")
        assert fa.dtype == np.float32 and fa.shape == (3, 100) and np.array_equal(fa, fb) and (fa == 1.0).all()
    # a build that writes values outside the swath, where the NaN fill belongs, shows in the fill sample
    wrong = {m: torch.nan_to_num(img, nan=0.5) for m, img in imgs.items()}
    bench.dump_outputs(wrong, str(tmp_path / "w"), covered, n_pixels=300, n_fill=100)
    assert np.array_equal(np.load(tmp_path / "w" / "bands_nearest.npy"), np.load(tmp_path / "a" / "bands_nearest.npy"))
    assert (np.load(tmp_path / "w" / "fill_nearest.npy") == 0.0).all()
    bench.dump_outputs(imgs, str(tmp_path / "c"), covered, n_pixels=10 ** 6)  # fewer covered pixels: all of them
    want = imgs["nearest"].numpy().reshape(3, -1)[:, covered.ravel()]
    assert np.array_equal(np.load(tmp_path / "c" / "bands_nearest.npy"), want)


def test_helpers_without_nvml():
    sys.path.insert(0, ROOT)
    import bench

    sampler = bench.ClockSampler(0)
    sampler.start()
    clocks = sampler.stop()
    assert set(clocks) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    before = os.sched_getaffinity(0)
    assert bench.pin_to_gpu_numa_node(0) == before
    assert os.sched_getaffinity(0) == before  # no NVML here: affinity untouched
    cfg = bench.workload_config(4865, 4091, 21, (7992, 5013), 8)
    assert cfg["scenes_per_step"] == 8 and "rectify_dataset" in cfg["workload"]


def test_traffic_source_expression_of_the_bench_line():
    """The `roofline.traffic_source` expression of bench.py, lifted from the source by its AST and evaluated
    with the committed profiles/kernel_traffic.json: names the capture a kernel's DRAM bytes come from, and is
    None when there is no traffic figure (N > 1, scaled scenes, kernels without a capture)."""
    import ast
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tree = ast.parse(open(os.path.join(root, "bench.py")).read())
    found = [v for node in ast.walk(tree) if isinstance(node, ast.Dict)
             for k, v in zip(node.keys, node.values) if isinstance(k, ast.Constant) and k.value == "traffic_source"]
    assert len(found) == 1
    expr = ast.Expression(found[0])
    ast.fix_missing_locations(expr)
    code = compile(expr, "bench.py", "eval")
    table = json.load(open(os.path.join(root, "profiles", "kernel_traffic.json")))
    assert "k2_gather_dual<nearest+bilinear>" in table["dual"] and "k1_scatter" in table["two_step"]

    def ev(key, kernel, traffic, tab=table):
        return eval(code, dict(traffic_table=tab, traffic_key=key, top={"kernel": kernel, "traffic": traffic}))

    assert "regex:k2_gather_dual" in ev("dual", "k2_gather_dual<nearest+bilinear>", 9.1e9)
    assert "regex:k2_gather_dual" not in ev("dual", "k1_scatter", 5e8) and "ncu --set full" in ev("dual", "k1_scatter", 5e8)
    assert "ncu --set full" in ev("two_step", "k2_gather_staged<bilinear>", 5.6e9)
    assert ev("dual", "k2_gather_dual<nearest+bilinear>", None) is None
    assert ev("dual", "k2_gather_dual<nearest+bilinear>", None, tab={}) is None
