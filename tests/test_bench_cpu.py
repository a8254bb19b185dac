"""bench.py contract checks that need no GPU: stdout carries exactly ONE JSON line (native libraries
that print to fd 1 — NCCL's version banner under NCCL_DEBUG — are diverted to stderr), and the
reference arm (CPU restatement, the one arm that runs without a device) emits the agreed keys."""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_stdout_guard_diverts_native_writes():
    code = textwrap.dedent(f'''
        import os, sys
        sys.path.insert(0, {ROOT!r})
        import bench
        with bench._CleanStdout() as out:
            os.write(1, b"NCCL version 2.28.9+cuda12.9\\n")      # what a native library does
            print("a python print inside the run")
            out.emit('{{"ok": 1}}')
        print("after")
    ''')
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout == '{"ok": 1}\nafter\n'
    assert "NCCL version" in r.stderr and "a python print inside the run" in r.stderr


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["value"] > 0
    for key in ("metric", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_fixed_sample_within_64_mb(tmp_path):
    """--dump-outputs at the headline size (1 M splats, 1920x1080): float .npy files, at most 64 MB in all, the same
    seeded sample of pixels and splats on every run; small outputs are written whole."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(0)
    P, H, W = 1_000_000, 1080, 1920
    images = {"color": rng.random((3, H, W), np.float32), "allmap": rng.random((7, H, W), np.float32)}
    per_splat = {"radii": rng.integers(0, 50, P).astype(np.int32), "grad_shs": rng.random((P, 16, 3), np.float32)}
    names = bench.dump_outputs(str(tmp_path / "a"), images, per_splat)
    bench.dump_outputs(str(tmp_path / "b"), images, per_splat)
    assert names == ["allmap", "color", "grad_shs", "pixel_index", "radii", "splat_index"]
    files = sorted((tmp_path / "a").iterdir())
    assert [f.name for f in files] == [n + ".npy" for n in names]
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    for n in names:
        a, b = np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy"))
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    pix = np.load(tmp_path / "a" / "pixel_index.npy").astype(np.int64)
    spl = np.load(tmp_path / "a" / "splat_index.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "color.npy"), images["color"].reshape(3, -1)[:, pix])
    assert np.array_equal(np.load(tmp_path / "a" / "radii.npy"), per_splat["radii"][spl].astype(np.float32))
    assert np.load(tmp_path / "a" / "grad_shs.npy").shape == (len(spl), 16, 3)
    small = bench.dump_outputs(str(tmp_path / "c"), {"color": images["color"][:, :64, :64]}, {"radii": per_splat["radii"][:100]})
    assert small == ["color", "radii"]
    assert np.array_equal(np.load(tmp_path / "c" / "color.npy"), images["color"][:, :64, :64])


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
