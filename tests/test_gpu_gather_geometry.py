"""GPU tests (-m gpu) of the projection gather k_project_remesh across its tile geometry and every reach regime: the cases
of tests/gather_cases.py on the CUDA path against the oracle's serial scatter, bit for bit after every step.

Besides State, particles and counters, the per-row reach the gather sizes its tiles with (B200Engine.row_reach) is
compared with the reach predicted from the particles' positions, and the regimes each case claims (tile guesses, tiles
narrowed by their rows' reach) are checked on the rows the device reports."""
import numpy as np
import pytest

import gather_cases as GC
from common import cartesian_grid, compare_models, make_oracle
from test_gpu_ensemble import run_ensemble
from test_gpu_parity import StripSet, engine_for

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", sorted(GC.CASES))
def test_gpu_gather_case_bit_exact(gpu_lib, name):
    case = GC.CASES[name]
    g, P = case.grid, case.params
    dut = StripSet(g, P, *case.strips) if case.strips else engine_for(g, P)
    reaches, rows = [], []

    def on_step(k, ref, dut, before):
        reaches.append(ref.counters()["reach"])
        if case.strips:
            rows.append(None)
            return
        rr = dut.row_reach()
        if case.propagation:
            assert np.array_equal(rr, GC.row_reach_prediction(g, before, case.dts[k])), f"step {k}: row reach"
        assert int(rr.max()) == reaches[-1]
        rows.append(rr)

    GC.run_case(make_oracle(g, P), dut, case, compare_models, on_step=on_step)
    obs = GC.observed(case, reaches, rows)
    assert case.claims <= obs, sorted(case.claims - obs)


def test_gpu_ensemble_members_of_different_reach(gpu_lib):
    """three members stepped together on 65 x 17 (partial last tiles in x and y): calm, reach 1, reach 11 — each member
    against its own oracle after every step, and each member's row reach its own"""
    case = GC.ensemble_case()
    eng, refs = run_ensemble(case.grid, case.params, case.winds, case.dts[0], len(case.dts))
    member_reaches = [r.counters()["reach"] for r in refs]
    assert member_reaches[0] == 0 and member_reaches[1] == 1 and member_reaches[2] >= 6, member_reaches
    rows = eng.row_reach()
    assert rows.shape == (3, case.grid["Ny"])
    assert [int(rows[m].max()) for m in range(3)] == member_reaches


def test_gpu_reach_beyond_supported_is_refused(gpu_lib):
    """a step whose deposits reach 16 cells raises PiclesError naming the supported reach (15); the step before it, at
    reach 2, matches the oracle.  What State holds after the refused step is not specified: only the error is."""
    from picles_b200 import PiclesError
    g = cartesian_grid(65, 17)
    P = GC.prop_params((2.0, 0.7))
    dts = GC.dts_for([2, 16], 2.0 / 2000.0)
    ref, dut = make_oracle(g, P), engine_for(g, P)
    ref.seed(5.0, 5.0)
    dut.seed(5.0, 5.0)
    ref.step(0.0, dts[0], 5.0, 5.0, 5.0, 5.0)
    dut.step(0.0, dts[0], 5.0, 5.0, 5.0, 5.0)
    compare_models(ref, dut)
    ref.step(dts[0], dts[1], 5.0, 5.0, 5.0, 5.0)
    assert ref.counters()["reach"] == 16
    with pytest.raises(PiclesError, match="ERR_HALO.*supported reach 15"):
        dut.step(dts[0], dts[1], 5.0, 5.0, 5.0, 5.0)


def test_gpu_strip_shorter_than_the_reach_is_refused(gpu_lib):
    """host-driven strips of 10, 4 and 10 rows with a halo of 4 rows, then a step of reach 6: the gather refuses
    (PICLES_ERR_HALO) and changes nothing; the 4-row strip cannot widen its exchange to 6 rows, so the error stands"""
    from picles_b200 import PiclesError
    g = cartesian_grid(65, 24)
    P = GC.prop_params((0.7, 2.0))
    s = StripSet(g, P, 3, 4, bounds=[(0, 10), (10, 14), (14, 24)])
    s.seed(5.0, 5.0)
    dt = GC.dts_for([6], 2.0 / 2000.0)[0]
    before = s.state()
    with pytest.raises(PiclesError, match="ERR_HALO"):
        s.step(0.0, dt, 5.0, 5.0, 5.0, 5.0)
    assert np.array_equal(s.state().view(np.uint64), before.view(np.uint64))
    assert max(e.reach() for e in s.e) == 6
    assert s.e[1].halo_rows() == (4, 4)
    with pytest.raises(PiclesError, match="ERR_HALO.*at most 4"):
        s.e[1].halo_widen(6)
