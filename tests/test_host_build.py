"""The host libraries the tests load are rebuilt exactly when a file the compiler read for them changes or their command
line does, and processes that load one at the same time build it once.  Works on a copy of the sources under tmp_path;
the last test guards the one hand-kept header list left, build_lib.HEADERS, against the compiler."""
import glob
import importlib.util
import os
import shlex
import shutil
import subprocess
import sys

import pytest

import build_lib
import host_build

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture
def tree(tmp_path):
    """the device headers, the public header, the oracle and the shim sources, copied; no build products"""
    shutil.copytree(os.path.join(ROOT, "picles_b200", "csrc"), tmp_path / "picles_b200" / "csrc")
    shutil.copytree(os.path.join(ROOT, "include"), tmp_path / "include")
    shutil.copytree(os.path.join(ROOT, "oracle"), tmp_path / "oracle",
                    ignore=shutil.ignore_patterns("_build", "__pycache__"))
    (tmp_path / "tests").mkdir()
    for f in ("host_shim.cpp", "host_shim_1d.cpp"):
        shutil.copy(os.path.join(HERE, f), tmp_path / "tests" / f)
    return tmp_path


def closure(cmd, src):
    """the files the compiler reads for src, headers outside the system directories included"""
    out = subprocess.run(cmd + ["-MM", src], capture_output=True, text=True, check=True).stdout
    return {os.path.realpath(p) for p in shlex.split(out.replace("\\\n", " "))[1:]}


def stamp(path):
    st = os.stat(path)
    return st.st_ino, st.st_mtime_ns


def bump(path, than):
    """make `path` newer than the file `than` by one nanosecond"""
    t = os.stat(than).st_mtime_ns + 1
    os.utime(path, ns=(t, t))


def check_rebuilds(tree, build, so, deps, must):
    """build() rebuilds `so` after each file of `deps` is bumped, and after no other header is"""
    deps = {os.path.realpath(p) for p in deps}
    assert {os.path.realpath(tree / p) for p in must} <= deps
    build()
    for p in sorted(deps):
        before = stamp(so)
        bump(p, so)
        build()
        assert stamp(so) != before, p
    others = set(glob.glob(str(tree / "picles_b200" / "csrc" / "*.h")) + glob.glob(str(tree / "include" / "*.h")))
    others = sorted({os.path.realpath(p) for p in others} - deps)
    assert others
    before = stamp(so)
    for p in others:
        bump(p, so)
    build()
    assert stamp(so) == before, others


@pytest.mark.parametrize("name, must", [
    ("host_shim", ["picles_b200/csrc/pmath_body.h", "picles_b200/csrc/pmath_exptab.h"]),
    ("host_shim_1d", ["include/picles_b200.h"]),
])
def test_shim_rebuilds_when_a_file_it_includes_changes(tree, name, must):
    src = str(tree / "tests" / (name + ".cpp"))
    out = tree / "tests" / "_build"
    deps = closure(["g++", "-std=c++17"], src)
    check_rebuilds(tree, lambda: host_build.load(name, src=src, build_dir=str(out)), out / ("lib%s.so" % name), deps,
                   must + ["tests/%s.cpp" % name])


def test_oracle_rebuilds_when_a_file_it_includes_changes(tree):
    spec = importlib.util.spec_from_file_location("oracle_copy", tree / "oracle" / "__init__.py")
    copy = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(copy)
    src = str(tree / "oracle" / "picles_oracle.c")
    deps = closure(["gcc", "-std=c11"], src)
    so = tree / "oracle" / "_build" / "libpicles_oracle.so"
    check_rebuilds(tree, lambda: copy.make("_build/libpicles_oracle.so"), so, deps,
                   ["picles_b200/csrc/pmath_exptab.h", "oracle/picles_oracle.c"])


def test_a_changed_flag_rebuilds(tree):
    src, out = str(tree / "tests" / "host_shim_1d.cpp"), str(tree / "tests" / "_build")
    so = os.path.join(out, "libhost_shim_1d.so")
    host_build.load("host_shim_1d", src=src, build_dir=out)
    stamps = [stamp(so)]
    for flags in (["-DPICLES_HOST_BUILD_TEST"], ["-DPICLES_HOST_BUILD_TEST"], []):
        host_build.load("host_shim_1d", src=src, flags=flags, build_dir=out)
        stamps.append(stamp(so))
    assert stamps[1] != stamps[0] and stamps[2] == stamps[1] and stamps[3] != stamps[2]


WORKER = r"""
import ctypes as C, subprocess, sys
sys.path.insert(0, sys.argv[1])
import host_build
builds, run = [], subprocess.run
def counted(cmd, **kw):
    builds.append(cmd)
    return run(cmd, **kw)
subprocess.run = counted
lib = host_build.load("host_shim", src=sys.argv[2], build_dir=sys.argv[3])
lib.shim_corner_target.restype = C.c_int64
lib.shim_corner_target.argtypes = [C.c_int] * 4 + [C.c_int64] * 2
print(len(builds), [lib.shim_corner_target(9, 7, 1, 2, i, j) for i in (-1, 0, 8, 9) for j in (-1, 0, 6, 7)])
"""


def test_processes_loading_at_once_build_once(tree):
    out = tree / "tests" / "_build"
    args = [sys.executable, "-c", WORKER, HERE, str(tree / "tests" / "host_shim.cpp"), str(out)]
    procs = [subprocess.Popen(args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for _ in range(4)]
    results = []
    for p in procs:
        stdout, stderr = p.communicate(timeout=600)
        assert p.returncode == 0, stderr
        results.append(stdout.split(" ", 1))
    assert sum(int(n) for n, _ in results) == 1
    assert len({r for _, r in results}) == 1
    assert sorted(os.listdir(out)) == ["libhost_shim.cmd", "libhost_shim.d", "libhost_shim.lock", "libhost_shim.so"]


def test_build_lib_headers_cover_the_include_closure_of_its_sources():
    """bench.py decides whether to rebuild the library from build_lib.HEADERS, so that list must name every header of
    the repository the CUDA sources include"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if os.path.exists(nvcc):
        cmd = [nvcc, "-std=c++17", "-M"]
    elif shutil.which("g++"):  # -MG: CUDA's headers may be missing too
        cuda = os.path.dirname(os.path.dirname(nvcc))
        cmd = ["g++", "-std=c++17", "-MM", "-MG", "-x", "c++", "-I", os.path.join(cuda, "include")]
    else:
        pytest.skip("neither nvcc nor g++ is installed")
    csrc, root = os.path.realpath(build_lib.CSRC), os.path.realpath(ROOT)
    listed = {os.path.realpath(os.path.join(csrc, h)) for h in build_lib.SOURCES + build_lib.HEADERS}
    ours = set()
    for s in build_lib.SOURCES:
        out = subprocess.run(cmd + [os.path.join(csrc, s)], capture_output=True, text=True, check=True).stdout
        read = {os.path.realpath(p) for p in shlex.split(out.replace("\\\n", " "))}
        ours |= {p for p in read if p.startswith(root + os.sep) and os.path.isfile(p)}  # not the target, nor CUDA's
    # the compiler reported headers that only other headers include
    assert {os.path.join(csrc, "pmath_body.h"), os.path.join(root, "include", "picles_b200.h")} <= ours
    assert ours <= listed, sorted(ours - listed)
