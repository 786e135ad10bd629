"""CPU tests of the advance-kernel cases (tests/advance_cases.py): the selection mirror against the launcher of
picles_kernels.cu, proof that the cases launch all 22 advance kernels and reach every device-only path they claim,
the host build of the device header against the oracle on every case, and the oracle's right-hand side against
exact arithmetic at the premise edges the cases push the kernels to."""
import ctypes as C
import itertools
import math
import os
import re

import numpy as np
import pytest

import advance_cases as AC
import host_build
from common import HostShim, PiclesParams, ROOT, compare_models, default_params, make_oracle, shim_lib

KERNELS_CU = os.path.join(ROOT, "picles_b200", "csrc", "picles_kernels.cu")
LAUNCHERS = ("advance_kernels", "launch_advance_as", "launch_advance")


def _function_text(src, name):
    """the definition of `name` in src, from its template head or return type to its closing brace"""
    m = re.search(r"^(?:template\s*<[^>]*>\s*)?(?:static\s+)?void\s+" + name + r"\(", src, re.M)
    assert m, name
    i = src.index("{", m.end())
    depth = 0
    for j in range(i, len(src)):
        depth += {"{": 1, "}": -1}.get(src[j], 0)
        if depth == 0:
            return src[m.start():j + 1]
    raise AssertionError(name)


def _template_head(src, kernel):
    """the template parameter list of a kernel, default arguments included"""
    m = re.search(r"template\s*<([^>]*)>\s*__global__\s+void\s+(?:\w+(?:\([^)]*\))?\s+)?" + kernel + r"\(", src)
    assert m, kernel
    return m.group(1)


@pytest.fixture(scope="module")
def launch_selection():
    """launch_advance and the templates behind it as they stand in picles_kernels.cu, compiled for the host with
    physics.h (ph_advance_variant) and every kernel launch replaced by a call that records its template arguments
    (default arguments filled in by the compiler from the kernels' own template heads), with the launch counter kept
    as the library keeps it.  Each recorder instantiation registers itself when the library is loaded, so the
    registry lists every kernel the launcher can launch, whether or not some call reaches it."""
    src = open(KERNELS_CU).read()
    bodies = [_function_text(src, f) for f in LAUNCHERS]
    launch = re.compile(r"\b(k_advance(?:_resume)?)<([^<>]*)><<<[^>]*>>>\([^;]*\);")
    assert any(launch.search(b) for b in bodies)
    bodies = [launch.sub(r"\1_rec<\2>();", b) for b in bodies]
    body_text = "\n".join(bodies)
    code = f"""
#include <cstdint>
#include "physics.h"
using namespace picles;
typedef void* cudaStream_t;
struct DeviceCounters;
struct DeviceArrays {{ int members; const double* M[4]; }};
#define ADV_THREADS 128
#define ADV_MIN_BLOCKS 1
#define REG_MAX 64
static int n_reg = 0, reg[REG_MAX][5]; /* every recorder instantiation: kind, PER_NODE_M, AUTOSW, TSIT5, ENS */
static int rec_n = 0, rec[16], rec_launches = 0;
#define COUNT_LAUNCH(n) (rec_launches += (n))
static int grid_for(int64_t, int, int, int) {{ return 1; }}
static int add_reg(int kind, int pn, int autosw, int tsit5, int ens) {{
    if (n_reg < REG_MAX) {{ int* r = reg[n_reg]; r[0] = kind; r[1] = pn; r[2] = autosw; r[3] = tsit5; r[4] = ens; }}
    return n_reg++;
}}
template <bool PN, bool AUTOSW, int TSIT5, bool ENS> int k_advance_id = add_reg(0, PN, AUTOSW, TSIT5, ENS);
template <bool PN, bool ENS> int k_advance_resume_id = add_reg(1, PN, 0, 0, ENS);
template <{_template_head(src, "k_advance")}> void k_advance_rec() {{
    rec[rec_n++] = k_advance_id<PER_NODE_M, AUTOSW, TSIT5, ENS>; }}
template <{_template_head(src, "k_advance_resume")}> void k_advance_resume_rec() {{
    rec[rec_n++] = k_advance_resume_id<PER_NODE_M, ENS>; }}
{body_text}
extern "C" int registered(int* out) {{
    for (int i = 0; i < n_reg && i < REG_MAX; i++) for (int c = 0; c < 5; c++) out[5 * i + c] = reg[i][c];
    return n_reg;
}}
extern "C" int select_kernels(const picles_params_t* P, int per_node_M, int members, int* out, int* launches) {{
    static const double plane = 0.0;
    DeviceArrays A; A.members = members;
    for (int k = 0; k < 4; k++) A.M[k] = per_node_M ? &plane : nullptr;
    rec_n = 0; rec_launches = 0;
    launch_advance(A, *P, 600.0, nullptr, 148, nullptr, 0, 64, 64, 64, 0);
    for (int i = 0; i < rec_n; i++) for (int c = 0; c < 5; c++) out[5 * i + c] = reg[rec[i]][c];
    *launches = rec_launches;
    return rec_n;
}}
"""
    # -O0: the recorder runs no arithmetic, so optimising it would only slow the build; -I: the text includes
    # physics.h by name
    lib = host_build.load("launch_selection", text=code,
                          flags=["-O0", "-I", os.path.join(ROOT, "picles_b200", "csrc")])
    lib.select_kernels.restype = C.c_int
    lib.select_kernels.argtypes = [C.POINTER(PiclesParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.registered.restype = C.c_int
    lib.registered.argtypes = [C.c_void_p]

    def kernels(rows):
        ks = set()
        for row in rows:
            if row[0] == 0:
                ks.add(("k_advance", bool(row[1]), bool(row[2]), int(row[3]), bool(row[4])))
            else:
                ks.add(("k_advance_resume", bool(row[1]), bool(row[4])))
        assert len(ks) == len(rows)
        return ks

    def select(P, pn, members):
        out = np.zeros((16, 5), np.int32)
        nl = np.zeros(1, np.int32)
        n = lib.select_kernels(C.byref(P), int(pn), int(members), out.ctypes.data, nl.ctypes.data)
        return kernels(out[:n]), int(nl[0])

    out = np.zeros((64, 5), np.int32)
    n = lib.registered(out.ctypes.data)
    assert n <= len(out), n
    select.instantiated = kernels(out[:n])
    return select


def _combinations():
    for solver, prop, nan_eest, pn, E in itertools.product(("Tsit5", "DP5", "AutoTsit5"), (True, False), (False, True),
                                                          (False, True), (1, 2, 3)):
        yield default_params(solver=solver, propagation=prop, nan_eest_rejects=nan_eest), pn, E


def test_selection_mirror_equals_the_launcher(launch_selection):
    """for every solver x propagation x nan_eest_rejects x per-node kernel x (E = 1, E > 1), the kernels the source
    launches are the mirror's, and the library counts one launch per kernel; over all of them, the 22 kernels, and the
    launcher can launch no other"""
    assert launch_selection.instantiated == AC.ALL_KERNELS
    image = set()
    for P, pn, E in _combinations():
        got, launches = launch_selection(P, pn, E)
        want = AC.advance_kernels(P, pn, E)
        assert got == want, (int(P.solver), int(P.propagation), int(P.nan_eest_rejects), pn, E, got, want)
        assert launches == len(want)
        image |= got
    assert image == AC.ALL_KERNELS


def test_host_build_selects_as_the_device():
    """the specialised host build runs the copy of the instantiation launch_advance would launch"""
    lib = shim_lib()
    for P, pn, E in _combinations():
        if E == 1:
            (k,) = [k for k in AC.advance_kernels(P, pn, 1) if k[0] == "k_advance"]
            assert lib.shim_advance_template(C.byref(P), int(pn)) == k[3], (int(P.solver), pn)


def test_cases_cover_every_kernel_and_path():
    """each case's premises hold in its oracle run, and together the cases launch all 22 kernels and reach every path
    listed in advance_cases.REQUIRED; a path only one case reaches fails here when that case goes"""
    seen, launched = set(), set()
    for case in AC.CASES.values():
        held = AC.premises(case, AC.oracle_run(case))
        claims = AC.claims_of(case)
        assert claims <= held, (case.name, sorted(claims - held))
        seen |= claims
        launched |= case.kernels()
    assert launched == AC.ALL_KERNELS, sorted(AC.ALL_KERNELS - launched)
    assert AC.REQUIRED <= seen, sorted(AC.REQUIRED - seen)


def _compare_with_solver_state(ref, dut):
    compare_models(ref, dut)
    assert np.array_equal(ref.solver_state(), dut.solver_state())


@pytest.mark.parametrize("name", sorted(AC.CASES))
def test_host_build_bit_exact(name):
    """the host build of the device header with the copies the kernels pick (switch-free right-hand side, Tsit5, DP5
    and AutoTsit5 instantiations) against the oracle, bit for bit after every step"""
    case = AC.CASES[name]
    lib = shim_lib()
    lib.shim_set_specialised(1)
    try:
        AC.run_case(make_oracle(case.grid, case.params), HostShim(case.grid, case.params), case,
                    _compare_with_solver_state)
    finally:
        lib.shim_set_specialised(0)


# ---- the oracle at the edges -----------------------------------------------------------------------------------------

def _edge_inputs():
    """(case, P, z, u, v, M, pc) of the first right-hand side of one integrating particle of every case that pushes an
    operand of rhs3 to a premise edge"""
    wanted = ("std_rhs:", "general_rhs:", "f3", "tanh", "sech")
    for case in AC.CASES.values():
        if not any(c.startswith(wanted) for c in case.claims) or "std_rhs" in case.claims and len(case.claims) > 1:
            continue
        o = make_oracle(case.grid, case.params)
        u0, v0 = case.wind(0.0)
        o.seed(u0, v0)
        p = o.particles()
        j, i = np.argwhere((p["flags"] & AC.PF_ACTIVE) != 0)[0]
        g = case.grid
        M = g["M_const"] if g["M"] is None else g["M"][:, j, i]
        u = np.broadcast_to(u0, (g["Ny"], g["Nx"]))[j, i]
        v = np.broadcast_to(v0, (g["Ny"], g["Nx"]))[j, i]
        yield case.name, case.params, p["z"][:, j, i], float(u), float(v), M, 0.0 if g["pc"] is None else g["pc"][j, i]


def _direction_scale(mp, P, z, u, v):
    """the error scale of c̄ S_dir that mp_rhs leaves out: s2 is a difference of two products that cancel exactly when
    c̄ is parallel to the wind (every seeded particle), so its rounding error is an ulp of the larger product"""
    F = mp.mpf
    cx, cy, u, v, r_g = F(z[1]), F(z[2]), F(u), F(v), F(P.r_g)
    gx, gy = cx / r_g, cy / r_g
    us, sg = mp.sqrt(u ** 2 + v ** 2), mp.sqrt(gx ** 2 + gy ** 2)
    if us * sg == 0:
        return F(0), F(0)
    a2 = min(us / (2 * sg), F(500))
    s2 = (2 / (us * sg) ** 2) * (abs(u * v * (2 * gy ** 2 - sg ** 2)) + abs(gx * gy * (2 * v ** 2 - us ** 2)))
    w = a2 ** 2 * abs(F(P.C_varphi)) * s2 if P.direction else F(0)
    return abs(cy) * w, abs(cx) * w


# below this the float64 evaluation meets underflowed intermediates (|c̄|^2 of c̄ = 2^-486 is 2^-971); a value of
# that size is not resolved by either side
ABS_FLOOR = 2.0 ** -900


def test_oracle_rhs_at_the_premise_edges():
    """the oracle's right-hand side (the arithmetic every kernel is held to) against the 50-digit restatement of the
    Julia formulas, at every premise-edge input of the cases: within the conditioning-aware bound of
    test_independent_math where the exact value is a double; where it overflows or is undefined, the same class"""
    mp = pytest.importorskip("mpmath")
    import oracle
    from test_independent_math import mp_rhs
    F = mp.mpf
    big = F(np.finfo(np.float64).max)
    n = 0
    for name, P, z, u, v, M, pc in _edge_inputs():
        d = oracle.rhs(P, z, u, v, M=M, pc=pc)
        try:
            ref, scale = mp_rhs(P, z, u, v, M, pc)
            ds = _direction_scale(mp, P, z, u, v)
            scale = [scale[0], scale[1] + ds[0], scale[2] + ds[1], scale[3], scale[4]]
        except ZeroDivisionError:
            ref = None
        # an intermediate of the float64 lines that leaves the double range (|g|^2 for |c̄| = 2^450 over r_g = 2^-64)
        # makes the formula itself, the reference's too, give Inf or NaN where the exact value is finite
        g2 = (F(z[1]) ** 2 + F(z[2]) ** 2) / F(P.r_g) ** 2
        out_of_range = g2 > big
        for c in range(5):
            if out_of_range and not math.isfinite(d[c]):
                continue
            if ref is None or not mp.isfinite(ref[c]):
                assert not math.isfinite(d[c]), (name, c, d[c])
            elif abs(ref[c]) > big:
                assert math.isinf(d[c]) and (d[c] > 0) == (ref[c] > 0), (name, c, d[c], float(ref[c]))
            else:
                err = abs(F(float(d[c])) - ref[c])
                assert err <= F("1e-12") * scale[c] + F(ABS_FLOOR), (name, c, float(d[c]), float(ref[c]))
        n += 1
    assert n >= 30, n
