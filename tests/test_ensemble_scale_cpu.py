"""CPU tests of the two statements the ensemble-scale GPU tests rest on: the mirror of advance_range's graded row
blocks (ensemble_scale_cases.graded_blocks), held to the source and to hand-worked cases, and the restatement of the
two-stage energy reduction (energy_sum_restated), held to an element-by-element form of the same order and to
math.fsum within the rounding-error bound of a sum of positive terms."""
import math

import numpy as np
import pytest

from ensemble_scale_cases import (LOOP_LINES, capi_constants, energy_sum_restated, energy_sum_scalar, graded_blocks)

K = capi_constants()


def sizes(blocks):
    return [b - a for a, b, _ in blocks]


def test_constants_read_from_the_source():
    assert (K["PIPE_CHUNKS"], K["PIPE_MIN_NODES"], K["ENERGY_BLOCKS"]) == (8, 1 << 20, 1024)
    assert (K["graded_op"], K["first_rows"], K["growth"]) == (">=", 64, 3)
    for line in LOOP_LINES:
        assert line in K["advance_range"], f"advance_range changed: {line!r} is gone, update graded_blocks"


def test_threshold_is_inclusive():
    # exactly 2^20 nodes: graded (32 x 32 x 1024 members, rows = 32768)
    b = graded_blocks(32 * 1024, 32, True)
    assert [(a, e) for a, e, _ in b] == [(0, 64), (64, 256), (256, 832), (832, 2560), (2560, 7744), (7744, 23296),
                                         (23296, 32768)]
    assert [c for _, _, c in b] == list(range(7))
    # one row less of 2^20 nodes (1023 members): one block
    assert graded_blocks(32 * 1023, 32, True) == [(0, 32 * 1023, 0)]
    # 2^20 - Nx nodes as one model
    assert graded_blocks(1023, 1024, True) == [(0, 1023, 0)]
    assert len(graded_blocks(1024, 1024, True)) == 4


def test_range_ending_inside_block_3():
    # 1024 rows of 1024: blocks of 64, 192, 576 rows, then the fourth block (slot 3) is cut short at row 1024
    b = graded_blocks(1024, 1024, True)
    assert b == [(0, 64, 0), (64, 256, 1), (256, 832, 2), (832, 1024, 3)]
    # 2000 rows of 600 nodes: slot 3 would run to 2560
    assert graded_blocks(2000, 600, True)[-1] == (832, 2000, 3)


def test_eighth_block_takes_the_rest():
    b = graded_blocks(72000, 16, True)  # 16 x 16 members x 4500
    assert len(b) == 8 and sizes(b) == [64, 192, 576, 1728, 5184, 15552, 46656, 2048]
    assert b[-1] == (69952, 72000, 7)
    # much larger ranges still stop at eight blocks
    b = graded_blocks(1_000_000, 8, True)
    assert len(b) == 8 and b[-1] == (69952, 1_000_000, 7)


def test_bench_shape_edges_fall_inside_members():
    b = graded_blocks(51 * 512, 51, True)
    assert len(b) == 7 and b[-1][1] == 51 * 512
    assert all(a % 51 != 0 for a, _, _ in b[1:])


def test_no_uploads_is_one_block():
    for rows, Nx in ((72000, 16), (32 * 1024, 32), (4096, 4096), (1, 1)):
        assert graded_blocks(rows, Nx, False) == [(0, rows, 0)]


def test_blocks_tile_the_range():
    for rows, Nx in ((1, 1 << 20), (65, 1 << 14), (257, 4096), (2561, 512), (70000, 16), (69953, 16), (69952, 16)):
        b = graded_blocks(rows, Nx, True)
        assert b[0][0] == 0 and b[-1][1] == rows
        assert all(b[k][1] == b[k + 1][0] for k in range(len(b) - 1))
        assert all(a < e for a, e, _ in b)


@pytest.mark.parametrize("blocks,threads,n", [(4, 8, 1), (4, 8, 31), (4, 8, 32), (4, 8, 33), (4, 8, 100),
                                              (3, 4, 50), (1024, 256, 1), (1024, 256, 300)])
def test_restatement_equals_the_element_by_element_order(blocks, threads, n):
    rng = np.random.default_rng(n + blocks)
    # values of one binade: nearly every addition rounds
    e = 1.0 + rng.random(n)
    assert energy_sum_restated(e, blocks, threads) == energy_sum_scalar(e, blocks, threads)


def test_restatement_order_at_the_device_shape():
    """two full strides and a partial third of the 1024 x 256 grid: every thread sums two or three values"""
    rng = np.random.default_rng(5)
    n = 2 * 262144 + 1000
    e = 1.0 + rng.random(n)
    s = energy_sum_restated(e)
    assert s == energy_sum_scalar(e, 1024, 256)
    # the same values in another order: other bits
    assert s != energy_sum_restated(e[::-1].copy())


def test_restatement_hand_worked_orders():
    """three planes whose sum depends on one stage's order: u = 2^-53, so 1 + u rounds to 1 (a tie, to even) and
    1 + 2u is exact"""
    u, G = 2.0 ** -53, 1024 * 256
    # the grid-stride loop runs before the tree: (e[0] + e[G]) + (e[1] + e[G+1]) = 1 + 2u; the tree first over each
    # stride would give (e[0] + e[1]) + (e[G] + e[G+1]) = 1
    e = np.zeros(G + 2)
    e[0], e[1], e[G + 1] = 1.0, u, u
    assert energy_sum_restated(e) == 1.0 + 2 * u == energy_sum_scalar(e, 1024, 256)
    # the tree pairs sh[t] with sh[t + o]: (e0 + e2) + (e1 + e3) = 1 + 2u; added in thread order it would be 1
    assert energy_sum_restated(np.array([1.0, u, 0.0, u])) == 1.0 + 2 * u
    # the host adds the partials in block order: (1 + u) + u = 1; a tree over the blocks would give 1 + 2u
    e = np.zeros(513)
    e[0], e[256], e[512] = 1.0, u, u
    assert energy_sum_restated(e) == 1.0 == energy_sum_scalar(e, 1024, 256)


def test_restatement_of_many_planes_is_each_plane():
    rng = np.random.default_rng(3)
    E, n = 37, 16
    e = rng.random((E, n)) * 2.0 ** rng.integers(-20, 20, (E, n))
    s = energy_sum_restated(e)
    assert s.shape == (E,)
    assert all(s[m] == energy_sum_scalar(e[m], 1024, 256) for m in range(E))
    assert energy_sum_restated(e.reshape(1, E, n))[0, 5] == s[5]


@pytest.mark.parametrize("n", [1, 255, 256, 257, 262144, 262145, 10 ** 6])
def test_restatement_within_the_rounding_bound(n):
    rng = np.random.default_rng(n)
    e = rng.random(n) * 2.0 ** rng.integers(-10, 10, n)
    s = energy_sum_restated(e)
    exact = math.fsum(e)
    # additions on the path of any one term: grid-stride loop, tree, host loop
    depth = -(-n // 262144) + 8 + 1023
    u = 2.0 ** -53
    assert abs(s - exact) <= depth * u / (1 - depth * u) * exact
    if n <= 256:  # all in thread 0..255 of block 0: an exact case for small integers
        assert energy_sum_restated(np.arange(n, dtype=np.float64)) == n * (n - 1) / 2


def test_restatement_of_ones_and_empty_blocks():
    for n in (1, 16, 255, 256, 257, 262144, 262145, 600000):
        assert energy_sum_restated(np.ones(n)) == float(n)
    # +0.0 partials of the blocks past the data leave the sum alone, whatever the block count
    e = np.random.default_rng(1).random(300)
    assert energy_sum_restated(e, blocks=1024) == energy_sum_restated(e, blocks=2)
