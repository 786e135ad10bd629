"""CPU tests of the bench.py contract the driver relies on: the reference arm (the CPU port of
the reference's path, timed on the host cores) prints one JSON line with the agreed keys, and
the product arm fails loudly without a GPU instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "3", "--cpu-sample", "192")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "particle-steps/s" and d["unit"] == "particle-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["dtype"] == "f64"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3
    assert d["vs_baseline"] is None  # BASELINE.md holds no published number for this metric
    assert "4096x4096" in d["config"]["workload"] and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "192x192" in cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def test_product_arm_has_no_cpu_fallback():
    """Without an sm_100 device the b200 arm must stop with the library's error, not print a number."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the product arm runs")
    r = _run("--steps", "1", "--warmup", "3", "--no-cpu-baseline")
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert "no CPU fallback" in r.stderr


def test_dump_outputs_samples_a_large_strip(tmp_path):
    """--dump-outputs on a strip with more nodes than it dumps: the same seeded sample every time, every array float64,
    the values those of the model at the recorded nodes, and the default sample within 64 MB"""
    import numpy as np
    import bench
    from common import HostShim, cartesian_grid
    g = cartesian_grid(40, 30)
    e = HostShim(g, bench.params())
    e.seed(10.0, 10.0)
    e.step(0.0, 600.0, 10.0, 10.0, 10.0, 10.0)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), e, e.counters(), max_nodes=500)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and len(names) == 8
    A = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert A[n[:-4]].dtype == np.float64 and np.array_equal(A[n[:-4]], np.load(tmp_path / "b" / n))
    idx = A["node_index"].astype(np.int64)
    assert idx.shape == (500,) and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < 40 * 30
    assert np.array_equal(A["state"], e.state().reshape(3, -1)[:, idx])
    p = e.particles()
    assert np.array_equal(A["particles_u"], p["z"].reshape(5, -1)[:, idx])
    for k in ("t", "dt", "flags", "status"):
        assert np.array_equal(A["particles_" + k], p[k].reshape(-1)[idx]), k
    per_node = sum(a.nbytes for n, a in A.items() if n != "counters") / 500
    assert per_node * bench.DUMP_NODES + A["counters"].nbytes <= 64 * 2 ** 20


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(gpu_lib, tmp_path):
    """bench.py --dump-outputs writes State and the particles after exactly warmup + steps model steps (the oracle's,
    bit for bit, on the same box), and the same arguments dump the same arrays"""
    import numpy as np
    import bench
    from common import bits_equal, cartesian_grid, make_oracle
    warmup, steps = 3, 2
    for d in ("a", "b"):
        r = _run("--nx", "96", "--ny", "64", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
                 "--no-e2e", "--dump-outputs", str(tmp_path / d))
        assert r.returncode == 0, r.stderr
    names = sorted(os.listdir(tmp_path / "a"))
    for n in names:
        assert bits_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)), n
    A = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert np.array_equal(A["node_index"], np.arange(96 * 64))
    o = make_oracle(cartesian_grid(96, 64), bench.params())
    o.seed(10.0, 10.0)
    for k in range(warmup + steps):
        o.step(600.0 * k, 600.0, 10.0, 10.0, 10.0, 10.0)
    assert bits_equal(A["state"], o.state().reshape(3, -1))
    p = o.particles()
    act = (p["flags"].reshape(-1) & 8) != 0
    assert bits_equal(A["particles_u"][:, act], p["z"].reshape(5, -1)[:, act])
    assert bits_equal(A["particles_t"][act], p["t"].reshape(-1)[act])
    live = act & ((p["flags"].reshape(-1) & 4) == 0)  # dt means nothing while a step-size reset is pending
    assert bits_equal(A["particles_dt"][live], p["dt"].reshape(-1)[live])
    assert np.array_equal(A["particles_flags"][act], p["flags"].reshape(-1)[act])
    assert np.array_equal(A["particles_status"][act], p["status"].reshape(-1)[act])


def test_stale_library_is_rebuilt_outside_the_tree(tmp_path):
    """bench.py in a copy of the tree whose library is missing (as after a source edit, when it is older than its
    sources): the sources are compiled into a temporary directory and that library runs — on a GPU the bench line is
    printed, without one the library's own no-fallback error ends the run — and the tree is not written"""
    import shutil
    tree = tmp_path / "tree"
    shutil.copytree(ROOT, tree, ignore=shutil.ignore_patterns(".git", "_build", "__pycache__", "*.so"))
    listing = lambda: sorted(str(p.relative_to(tree)) for p in tree.rglob("*") if "__pycache__" not in p.parts)
    before = listing()
    r = subprocess.run([sys.executable, str(tree / "bench.py"), "--nx", "64", "--ny", "64", "--steps", "1", "--warmup", "3",
                        "--no-cpu-baseline", "--no-e2e"], capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert "building them into" in r.stderr, r.stderr
    assert listing() == before
    import torch
    if torch.cuda.is_available():
        assert r.returncode == 0, r.stderr
        assert len([l for l in r.stdout.splitlines() if l.startswith("{")]) == 1
    else:
        assert r.returncode != 0 and "no CPU fallback" in r.stderr, r.stderr


def test_bench_c5_grid_is_the_tests_grid():
    """bench.py builds the tripolar + land grid of its strong_c5 leg without touching tests/ or oracle/ (host mirror of
    make_boundaries); it must be the grid profiles/bench_configs.py and the GPU config tests build through the oracle"""
    import sys
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import bench
    from bench_configs import tripolar
    for nx, ny in ((432, 384), (270, 240)):
        a, b = bench.c5_grid(nx, ny), tripolar(nx, ny, True)
        assert a["bx"] == b["bx"] and a["by"] == b["by"]
        assert np.array_equal(a["mask"], b["mask"]) and a["mask"].dtype == np.uint8
        assert np.array_equal(a["M"], b["M"]) and np.array_equal(a["pc"], b["pc"])
