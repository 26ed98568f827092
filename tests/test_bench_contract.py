"""The bench.py contract.  CPU: the reference arm prints exactly one JSON line on stdout with the agreed keys
(everything else goes to stderr), non-zero ranks stay silent; where oracle/_ref is not built the arm times the
oracle port.  GPU: --dump-outputs writes the same files on every run, and they hold the oracle's frame."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPU_KIND = "reference" if _ref.available() else "port"


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                           "cif8_n7", "--steps", "1", "--warmup", "1", *args],
                          capture_output=True, text=True, env=env, timeout=300)


def test_reference_arm_prints_one_json_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "arf_filtered_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "cif8_n7" and d["dtype"] == "u8" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == CPU_KIND and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["simd"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_generic_c_flavour_is_selectable():
    d = json.loads(_run(None, "--ref-simd", "c").stdout.strip())
    assert d["cpu_baseline"]["simd"].startswith("none")


def test_reference_arm_other_ranks_stay_silent():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_write_outputs_sample_the_same_positions_within_the_limit(tmp_path):
    """Above the limit every large array is cut to the same seeded sample of its elements; small ones (FRAME_DIFF)
    stay whole and exact; below the limit everything is written whole with its shape."""
    import bench
    rng = np.random.default_rng(3)
    arrays = {"y": rng.integers(0, 1024, (300, 400), dtype=np.uint16),
              "u": rng.integers(0, 1024, (150, 200), dtype=np.uint16),
              "frame_diff": np.array([123456789, (1 << 40) + 3], np.int64)}
    limit = 200_000
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays, limit)
    a, b = tmp_path / "a", tmp_path / "b"
    names = sorted(os.listdir(a))
    assert names == ["frame_diff.npy", "u.npy", "y.npy"]
    assert sum(os.path.getsize(a / n) for n in names) <= limit
    for n in names:
        assert np.array_equal(np.load(a / n), np.load(b / n)), n
    fd = np.load(a / "frame_diff.npy")
    assert fd.dtype == np.float64 and fd.tolist() == arrays["frame_diff"].tolist()
    for n in ("y", "u"):
        got = np.load(a / f"{n}.npy")
        assert got.dtype == np.float32 and 0 < got.size < arrays[n].size
        idx = np.sort(np.random.default_rng(0).choice(arrays[n].size, got.size, replace=False))
        assert np.array_equal(got, arrays[n].ravel()[idx])
    bench.write_outputs(str(tmp_path / "c"), arrays)
    assert np.array_equal(np.load(tmp_path / "c" / "y.npy"), arrays["y"])


@pytest.mark.gpu
def test_dump_outputs_repeat_and_hold_the_oracle_frame(tmp_path):
    """Two runs with the same arguments write identical float32 / float64 files, under 64 MB in all; a run with
    three timed steps launches three times the kernels of a run with one.  With one
    timed step the first context's last step filtered the first seeded window, so its files are the oracle's
    frame and FRAME_DIFF for that window."""
    import bench
    import _gpu
    import _oracle
    dirs = [tmp_path / "a", tmp_path / "b", tmp_path / "c"]
    lines = []
    for d, steps in zip(dirs, (1, 1, 3)):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cif8_n7", "--steps",
                            str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-400:]
        lines.append(json.loads(r.stdout.strip()))
        assert lines[-1]["steps"] == steps
    # --steps sets the timed work: the kernel launches counted over the timed steps scale with it
    assert lines[0]["gpu_launches"] > 0 and lines[2]["gpu_launches"] == 3 * lines[0]["gpu_launches"]
    dirs = dirs[:2]
    names = sorted(os.listdir(dirs[0]))
    assert names == sorted(os.listdir(dirs[1]))
    assert {"ctx0_y.npy", "ctx0_u.npy", "ctx0_v.npy", "ctx0_frame_diff.npy"} <= set(names)
    assert sum(os.path.getsize(dirs[0] / n) for n in names) <= 64_000_000
    for n in names:
        a, b = np.load(dirs[0] / n), np.load(dirs[1] / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    width, height, bd, n, _ = bench.WORKLOADS["cif8_n7"]
    frames = bench.make_window(width, height, bd, n, seed=1234)
    p = bench.window_params("cif8_n7")
    o = _oracle.OracleFilter(p, frames)
    p["noise_levels"] = tuple(o.estimate_noise())
    o.close()
    want = _gpu.oracle_run(p, frames)
    for pl, plane in enumerate("yuv"):
        assert np.array_equal(np.load(dirs[0] / f"ctx0_{plane}.npy"), want["out"][pl]), plane
    assert np.array_equal(np.load(dirs[0] / "ctx0_frame_diff.npy"), want["diff"])
