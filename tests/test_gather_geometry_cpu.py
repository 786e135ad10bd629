"""CPU tests of the gather cases (tests/gather_cases.py): the host build of the device header (gather_node and
axis_candidates at reach up to 15, the candidate lists across the tripolar fold, y-strips with a halo as deep as the
reach) against the oracle's serial scatter, bit for bit after every step — and proof that the generator reaches every
regime the GPU test relies on."""
import numpy as np
import pytest

import gather_cases as GC
from common import HostShim, compare_models, make_oracle


@pytest.mark.parametrize("name", sorted(GC.CASES))
def test_gather_case_bit_exact(name):
    case = GC.CASES[name]
    kw = dict(nstrips=case.strips[0], halo=case.strips[1]) if case.strips else {}
    GC.run_case(make_oracle(case.grid, case.params), HostShim(case.grid, case.params, **kw), case, compare_models)


@pytest.mark.parametrize("member", range(3))
def test_ensemble_case_members_bit_exact(member):
    """each member of the ensemble case, as a model of its own"""
    case = GC.ensemble_case()
    GC.run_case(make_oracle(case.grid, case.params), HostShim(case.grid, case.params), case, compare_models,
                wind=case.winds[member])


def oracle_run(case, wind):
    """the oracle's reach of every step and, for propagation-only cases, the predicted per-row reach (whose maximum must
    be the oracle's reach: the prediction is what the GPU test compares B200Engine.row_reach with)"""
    o = make_oracle(case.grid, case.params)
    o.seed(*wind(0.0))
    if case.accumulate:
        o.set_accumulate(True)
    reaches, rows, t = [], [], 0.0
    for dt in case.dts:
        pred = GC.row_reach_prediction(case.grid, o.particles(), dt) if case.propagation else None
        o.step(t, dt, *wind(t), *wind(t + dt))
        t += dt
        r = o.counters()["reach"]
        if pred is not None:
            assert int(pred.max()) == r, f"{case.name}: predicted row reach {int(pred.max())}, oracle reach {r}"
        reaches.append(r)
        rows.append(pred)
    return reaches, rows


def test_cases_reach_every_regime():
    """each case goes through the regimes it claims, and together they go through every regime of the gather that only
    a GPU runs: each reach class with both tile guesses, the three reach sequences, every boundary type (narrow periodic
    rings, the fold, two deposit classes), per-row reach narrowing tiles, accumulation on the untiled path, strips and
    an ensemble of calm / reach-1 / fast members, on every grid width and height of the matrix"""
    seen = set()
    for case in GC.CASES.values():
        reaches, rows = oracle_run(case, case.wind)
        assert max(reaches) <= GC.REACH_MAX, (case.name, reaches)
        obs = GC.observed(case, reaches, rows)
        assert case.claims <= obs, (case.name, sorted(case.claims - obs))
        seen |= obs
    ens = GC.ensemble_case()
    member_reaches = [max(oracle_run(ens, w)[0]) for w in ens.winds]
    obs = GC.observed(ens, [max(member_reaches)] * len(ens.dts), member_reaches=member_reaches)
    assert ens.claims <= obs, sorted(ens.claims - obs)
    seen |= obs
    assert GC.REQUIRED <= seen, sorted(GC.REQUIRED - seen)


def test_reach_classes_are_exact():
    """the reach of a propagation-only step is set by its length: (r - 1/2) cells per step gives reach r, for r = 1..16
    in both directions"""
    from common import cartesian_grid
    for c in ((2.0, 0.5), (-2.0, 0.5), (0.5, -2.0)):
        g = cartesian_grid(40, 40, dx=1000.0, dy=1000.0)
        P = GC.prop_params(c)
        reaches = list(range(1, 17))
        o = make_oracle(g, P)
        o.seed(5.0, 5.0)
        got, t = [], 0.0
        for dt in GC.dts_for(reaches, 2.0 / 1000.0):
            o.step(t, dt, 5.0, 5.0, 5.0, 5.0)
            t += dt
            got.append(o.counters()["reach"])
        assert got == reaches, (c, got)
    assert np.all(np.diff(GC.dts_for(reaches, 1.0)) > 0)
