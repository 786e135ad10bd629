"""Host builds of the libraries the tests load: the host builds of the device headers (host_shim.cpp, host_shim_1d.cpp)
and sources the tests generate.  One flag set; a library is rebuilt when a file the compiler read for it is newer or its
command line changed, and processes that load it at the same time build it once and never see a partial file."""
from __future__ import annotations

import ctypes
import fcntl
import os
import shlex
import subprocess
from pathlib import Path

BUILD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_build")

# -ffp-contract=off, -fno-fast-math: every fused multiply-add in the headers is written out, so the host build gives
# the bits of the sm_100a kernels (built with --fmad=false) and of the oracle
FLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-shared"]
LANGS = {"c++17": ("g++", "-std=c++17", ".cpp"), "c99": ("gcc", "-std=c99", ".c")}


def _current(so, dep, cmd_file, cmd):
    """the library exists, was built by `cmd`, and no file its depfile names is newer"""
    try:
        if Path(cmd_file).read_text() != cmd:
            return False
        files = shlex.split(Path(dep).read_text().replace("\\\n", " "))[1:]  # "<target>: <source> <headers...>"
        t = os.stat(so).st_mtime_ns
        return all(os.stat(p).st_mtime_ns <= t for p in files)
    except FileNotFoundError:
        return False


def load(name, src=None, text=None, lang="c++17", flags=(), build_dir=BUILD):
    """lib<name>.so in build_dir, compiled from the file `src` or from the source `text` (written to build_dir), and
    loaded.  `flags` follow the common ones."""
    assert (src is None) != (text is None)
    cc, std, ext = LANGS[lang]
    cc = "/usr/bin/" + cc if os.path.exists("/usr/bin/" + cc) else cc
    os.makedirs(build_dir, exist_ok=True)
    base = os.path.join(build_dir, "lib" + name)
    so, dep = base + ".so", base + ".d"
    fd = os.open(base + ".lock", os.O_RDONLY | os.O_CREAT, 0o644)
    try:
        fcntl.flock(fd, fcntl.LOCK_EX)
        if text is not None:  # rewritten only when it changed, so that its mtime says when it last did
            src = Path(build_dir, name + ext)
            if not src.exists() or src.read_text() != text:
                src.write_text(text)
        argv = [cc, std, *FLAGS, *flags, os.path.abspath(src)]
        if not _current(so, dep, base + ".cmd", shlex.join(argv)):
            tmp = "%s.%d" % (base, os.getpid())
            r = subprocess.run(argv + ["-MMD", "-MF", tmp + ".d", "-o", tmp + ".so"], capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("host build of %s failed:\n%s" % (name, r.stderr))
            os.replace(tmp + ".d", dep)
            os.replace(tmp + ".so", so)
            Path(base + ".cmd").write_text(shlex.join(argv))
    finally:
        os.close(fd)
    return ctypes.CDLL(so)
