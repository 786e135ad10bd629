"""The compares of pmath.h that stand in for FP64 compares on the device fast paths (pm_ge_hw, pm_absge_hw, pm_iszero,
pm_maxc_i, pm_minc_i, pm_max_mag, pm_le_u, pm_lt_u), built for the host from the same header, against the FP64 compare
each replaces: at the edges of its stated premise (+-0, subnormals, +-inf, NaNs with payload only in the low word, the
constants and their neighbours) and on random operands inside it."""
import ctypes
import os

import numpy as np
import pytest

import host_build

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "picles_b200", "csrc")

SRC = r"""
#include "pmath.h"
#define LOOP(expr) for (long i = 0; i < n; i++) { double x = a[i], c = b[i]; out[i] = (expr); }
void ev(int op, const double* a, const double* b, long n, double* out) {
    switch (op) {
    case 0: LOOP(pm_ge_hw(x, c)) break;
    case 1: LOOP(pm_absge_hw(x, c)) break;
    case 2: LOOP(pm_iszero(x)) break;
    case 3: LOOP(pm_maxc_i(x, c)) break;
    case 4: LOOP(pm_minc_i(x, c)) break;
    case 5: LOOP(pm_max_mag(x, c)) break;
    case 6: LOOP(pm_le_u(x, c)) break;
    case 7: LOOP(pm_lt_u(x, c)) break;
    case 8: LOOP(pm_maxc(x, c)) break;
    case 9: LOOP(pm_min(c, x)) break;
    case 10: LOOP(pm_max(x, c)) break;
    }
}
"""
OPS = {"ge_hw": 0, "absge_hw": 1, "iszero": 2, "maxc_i": 3, "minc_i": 4, "max_mag": 5, "le_u": 6, "lt_u": 7,
       "maxc": 8, "min": 9, "max": 10}


@pytest.fixture(scope="module")
def lib():
    L = host_build.load("pmath_predicates", text=SRC, lang="c99", flags=["-I", CSRC])  # -I: SRC includes pmath.h by name
    dp = ctypes.POINTER(ctypes.c_double)
    L.ev.argtypes = [ctypes.c_int, dp, dp, ctypes.c_long, dp]

    def ev(op, x, c):
        x, c = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(c, np.float64))
        x, c = np.ascontiguousarray(x), np.ascontiguousarray(c)
        out = np.empty(x.shape)
        L.ev(OPS[op], x.ctypes.data_as(dp), c.ctypes.data_as(dp), x.size, out.ctypes.data_as(dp))
        return out
    return ev


def bits(a):
    return np.asarray(a, np.float64).view(np.uint64)


def f64(u):
    return np.array(u, np.uint64).view(np.float64)


def nb(c):
    """c and its neighbours at +-1 and +-2 ulp"""
    return [np.nextafter(np.nextafter(c, -np.inf), -np.inf), np.nextafter(c, -np.inf), c, np.nextafter(c, np.inf),
            np.nextafter(np.nextafter(c, np.inf), np.inf)]


TINY = 5e-324
SUB = [TINY, 2 * TINY, 2.2250738585072009e-308, 1e-310]      # subnormals
NAN_LO = f64([0x7FF0000000000001, 0x7FF00000FFFFFFFF, 0xFFF0000000000001, 0x7FF8000000000000, 0xFFF8000000000000])
RNG = np.random.default_rng(20261022)


def edges(cs):
    """+-0, subnormals, +-inf, huge, the constants and their neighbours, and the doubles where a high word reads as
    a float inf or NaN (2^1017)"""
    e = [0.0, -0.0, np.inf, -np.inf, 1.0, -1.0, 1.7976931348623157e308, -1.7976931348623157e308]
    e += SUB + [-s for s in SUB]
    for c in cs:
        e += nb(c) + [-v for v in nb(c)]
    e += nb(2.0 ** 1017) + nb(2.0 ** 1016)
    return np.array(e)


def randpos(n):
    """positive doubles over the whole exponent range, and near 1"""
    return np.concatenate([np.exp2(RNG.uniform(-1074, 1023.9, n)), RNG.uniform(0, 1000, n)])


HW_CONSTS = [22.0, 25.0, 350.0, 500.0, 700.0]


def test_hw_constants_have_zero_low_words():
    assert all(bits(c) & 0xFFFFFFFF == 0 for c in HW_CONSTS)


@pytest.mark.parametrize("c", HW_CONSTS)
def test_ge_hw(lib, c):
    """pm_ge_hw(x, c) == (x >= c) for every non-NaN x > -2^1017, and true for NaN"""
    x = np.concatenate([edges(HW_CONSTS), randpos(20000), -randpos(20000)])
    x = x[x > -(2.0 ** 1017)]
    assert np.array_equal(lib("ge_hw", x, c) != 0, x >= c)
    assert np.all(lib("ge_hw", NAN_LO, c) != 0)


@pytest.mark.parametrize("c", HW_CONSTS)
def test_absge_hw(lib, c):
    """pm_absge_hw(x, c) == (|x| >= c) for every non-NaN x, and true for NaN (the fast exp's flag)"""
    x = np.concatenate([edges(HW_CONSTS), randpos(20000), -randpos(20000)])
    assert np.array_equal(lib("absge_hw", x, c) != 0, np.abs(x) >= c)
    assert np.all(lib("absge_hw", NAN_LO, c) != 0)


def test_iszero(lib):
    x = np.concatenate([edges(HW_CONSTS), NAN_LO, randpos(2000), -randpos(2000)])
    with np.errstate(invalid="ignore"):
        assert np.array_equal(lib("iszero", x, 0.0) != 0, x == 0.0)


@pytest.mark.parametrize("c", [1e-2, 0.1, 1e-4, 5.0])
def test_maxc_minc(lib, c):
    """pm_maxc_i(a, c) is pm_maxc(a, c) bit for bit except for a negative NaN; pm_minc_i(a, c) is pm_min(c, a) except
    for a positive NaN"""
    x = np.concatenate([edges([c] + HW_CONSTS), randpos(20000), -randpos(2000)])
    assert np.array_equal(bits(lib("maxc_i", x, c)), bits(lib("maxc", x, c)))
    assert np.array_equal(bits(lib("minc_i", x, c)), bits(lib("min", x, c)))
    pos_nan, neg_nan = NAN_LO[bits(NAN_LO) >> 63 == 0], NAN_LO[bits(NAN_LO) >> 63 == 1]
    assert np.array_equal(bits(lib("maxc_i", pos_nan, c)), bits(pos_nan))
    assert np.array_equal(bits(lib("minc_i", neg_nan, c)), bits(neg_nan))


def test_max_mag(lib):
    """pm_max_mag(a, b) is pm_max(a, b) bit for bit on magnitudes (fabs of anything), except between two NaNs"""
    e = np.abs(np.concatenate([edges([1e-2, 0.1] + HW_CONSTS), randpos(300)]))
    a, b = np.meshgrid(e, e)
    a, b = a.ravel(), b.ravel()
    assert np.array_equal(bits(lib("max_mag", a, b)), bits(lib("max", a, b)))
    n = np.abs(NAN_LO)
    r = lib("max_mag", np.concatenate([n, e[:50]]), np.concatenate([e[:5], n[:5].repeat(10)]))
    assert np.all(np.isnan(r[:5])) and np.all(np.isnan(r[5:]))


@pytest.mark.parametrize("c", [1.0, 1e-4, 1e-12, 3.0e5, 0.0])
def test_le_u_lt_u(lib, c):
    """pm_le_u(x, c) == (x <= c) and pm_lt_u(x, c) == (x < c) for x >= +0 and every NaN (both false)"""
    x = np.concatenate([np.abs(edges([c, 1.0, 1e-4])), randpos(20000)])
    x = x[np.signbit(x) == 0]
    assert np.array_equal(lib("le_u", x, c) != 0, x <= c)
    assert np.array_equal(lib("lt_u", x, c) != 0, x < c)
    assert not np.any(lib("le_u", NAN_LO, c)) and not np.any(lib("lt_u", NAN_LO, c))
