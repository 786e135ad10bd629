"""Shared pieces of the ensemble-scale tests (test_ensemble_scale_cpu.py, test_gpu_ensemble_scale.py).

- `graded_blocks`: the row blocks `advance_range` (picles_b200/csrc/picles_capi.cu) cuts one step's advance into, with
  the constants and the grading condition read out of that source, so the mirror cannot drift from it.
- `energy_sum_restated`: the deterministic two-stage energy reduction (`energy_partial` in picles_kernels.cu, then
  `energy_sums` in picles_capi.cu) restated in numpy, in the device's order.
- `member_winds`: E wind fields on one grid that vary in x, y and t and differ from member to member, so that a block
  advanced against the previous step's wind plane, or against another member's rows, changes bits.
"""
from __future__ import annotations

import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAPI = os.path.join(ROOT, "picles_b200", "csrc", "picles_capi.cu")

# the lines of advance_range that graded_blocks restates, as they stand in the source
LOOP_LINES = (
    "for (int c = 0; c < PIPE_CHUNKS && a < r1; c++) {",
    "const int b = (!graded || c == PIPE_CHUNKS - 1 || a + len >= r1) ? r1 : a + len;",
    "int rc = upload_rows(h, u_t, v_t, u_t1, v_t1, a, b, h->pev[c], h->stream);",
    "launch_advance(A, h->P, dt_model, h->d_counters, h->sms, h->stream, (int64_t)a * A.Nx, l_end, l_end, l_end, c);",
)


def _define(src, name):
    m = re.search(r"^#define %s\s+\(?\s*(\d+)\s*(?:<<\s*(\d+)\s*)?\)?" % name, src, re.M)
    if m is None:
        raise AssertionError(f"#define {name} not found in {CAPI}")
    v = int(m.group(1))
    return v << int(m.group(2)) if m.group(2) else v


def capi_constants(path=CAPI):
    """PIPE_CHUNKS, PIPE_MIN_NODES, ENERGY_BLOCKS and the grading rule of advance_range, read from the source"""
    with open(path) as f:
        src = f.read()
    body = re.search(r"static int advance_range\(.*?\n}\n", src, re.S)
    if body is None:
        raise AssertionError("advance_range not found")
    body = body.group(0)
    graded = re.search(r"const bool graded = \(u_t \|\| u_t1\) && \(int64_t\)\(r1 - r0\) \* A\.Nx (>=|>) PIPE_MIN_NODES;",
                       body)
    first = re.search(r"int a = r0, len = (\d+);", body)
    grow = re.search(r"a = b; len \*= (\d+);", body)
    if not (graded and first and grow):
        raise AssertionError("advance_range no longer has the shape graded_blocks restates: update the mirror")
    return dict(PIPE_CHUNKS=_define(src, "PIPE_CHUNKS"), PIPE_MIN_NODES=_define(src, "PIPE_MIN_NODES"),
                ENERGY_BLOCKS=_define(src, "ENERGY_BLOCKS"), graded_op=graded.group(1), first_rows=int(first.group(1)),
                growth=int(grow.group(1)), advance_range=body)


def graded_blocks(rows, Nx, uploads, consts=None):
    """[(a, b, slot)]: the row blocks [a, b) of one step's advance over `rows` rows of Nx nodes (an ensemble:
    rows = ny * members) and the work-queue slot of each, as advance_range cuts them.  uploads: host winds are given
    with the step (picles_step with a wind pointer), which is what grades the range."""
    k = capi_constants() if consts is None else consts
    nodes = rows * Nx
    big = nodes >= k["PIPE_MIN_NODES"] if k["graded_op"] == ">=" else nodes > k["PIPE_MIN_NODES"]
    graded = bool(uploads) and big
    out, a, ln = [], 0, k["first_rows"]
    for c in range(k["PIPE_CHUNKS"]):
        if a >= rows:
            break
        b = rows if (not graded or c == k["PIPE_CHUNKS"] - 1 or a + ln >= rows) else a + ln
        out.append((a, b, c))
        a, ln = b, ln * k["growth"]
    return out


def energy_sum_restated(plane, blocks=None, threads=256):
    """the energy sum of the last axis of `plane` (any leading axes: one sum each), in the device's order:
    thread t of block b sums e[b*threads + t + k*blocks*threads] for k = 0, 1, ... starting from 0.0; the block's
    shared-memory tree adds sh[t + o] into sh[t] for o = threads/2 ... 1; the host adds the blocks' partials in block
    order starting from 0.0.  Blocks past the last element hold +0.0 partials: only the blocks that own elements are
    formed, which leaves every sum of non-negative terms unchanged."""
    blocks = capi_constants()["ENERGY_BLOCKS"] if blocks is None else blocks
    e = np.asarray(plane, np.float64)
    lead, n = e.shape[:-1], e.shape[-1]
    e = e.reshape(-1, n)
    G = blocks * threads
    used = min(blocks, max(1, -(-n // threads)))  # blocks that own at least one element
    width = used * threads
    s = np.zeros((e.shape[0], width))
    for k0 in range(0, n, G):  # grid-stride loop, k = 0, 1, ...
        chunk = e[:, k0:k0 + width]
        s[:, :chunk.shape[1]] = s[:, :chunk.shape[1]] + chunk
    sh = s.reshape(-1, used, threads)
    o = threads // 2
    while o > 0:  # the tree
        sh[:, :, :o] = sh[:, :, :o] + sh[:, :, o:2 * o]
        o //= 2
    part = np.zeros((e.shape[0], blocks))
    part[:, :used] = sh[:, :, 0]
    total = np.zeros(e.shape[0])
    for b in range(blocks):  # the host, in block order
        total = total + part[:, b]
    return total.reshape(lead)


def energy_sum_scalar(values, blocks, threads):
    """energy_sum_restated of one plane written out element by element (the check of the vectorised form)"""
    e = [float(x) for x in values]
    n, G = len(e), blocks * threads
    partial = []
    for b in range(blocks):
        sh = []
        for t in range(threads):
            s, l = 0.0, b * threads + t
            while l < n:
                s += e[l]
                l += G
            sh.append(s)
        o = threads // 2
        while o > 0:
            for t in range(o):
                sh[t] += sh[t + o]
            o //= 2
        partial.append(sh[0])
    total = 0.0
    for p in partial:
        total += p
    return total


def unit_coords(g):
    """node coordinates scaled to [0, 1] (x, y of shape (Ny, Nx))"""
    x, y = np.asarray(g["x"], np.float64), np.asarray(g["y"], np.float64)
    sx = lambda a: (a - a.min()) / max(a.max() - a.min(), 1.0)
    return sx(x), sx(y)


def member_winds(g, speed, angle, phase):
    """winds(t) -> (U, V) of shape (E, Ny, Nx): member m blows at about speed[m] m/s towards angle[m] (radians), with
    a gradient in x and in y and a modulation in time that starts at phase[m]; members with different parameters have
    different winds at every node and every time"""
    xn, yn = unit_coords(g)
    s = np.asarray(speed, np.float64)[:, None, None]
    a = np.asarray(angle, np.float64)[:, None, None]
    ph = np.asarray(phase, np.float64)[:, None, None]
    cu, su = s * np.cos(a), s * np.sin(a)

    def winds(t):
        f = 1.0 + 0.15 * np.sin(2.0 * np.pi * t / 7200.0 + ph)
        u = (cu * (0.75 + 0.25 * xn) + 0.4 * yn) * f
        v = (su * (0.8 + 0.2 * yn) - 0.3 * xn) * f
        return u, v

    return winds
