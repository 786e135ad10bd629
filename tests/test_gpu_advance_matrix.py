"""GPU tests (-m gpu) of the advance kernels: the cases of tests/advance_cases.py on the CUDA path against the oracle,
bit for bit after every step — every k_advance and k_advance_resume instantiation, single model and ensemble, and the
device-only paths inside them (switch-free right-hand side at its premise edges, the steady / mixed warp vote, the
deferred-flag fallbacks f3_cold, step_control_cold, initdt_a_cold, initdt_b_cold and vertex_values_cold).

The CPU test (test_advance_matrix_cpu.py) proves that each case reaches what it claims; here the device has to agree
with the oracle there.  The library's launch counter is the one direct evidence of the selection the ABI exposes:
three launches per step under AutoTsit5 (advance, resume, gather), two otherwise."""
import numpy as np
import pytest

import advance_cases as AC
from common import TALLY_NAMES, compare_models, make_oracle
from test_gpu_ensemble import compare_member, ensemble_engine
from test_gpu_parity import StripSet, engine_for

pytestmark = pytest.mark.gpu


def launches_per_step(case):
    return 3 if case.params.solver == AC.SOLVER_AUTOTSIT5 else 2


class Counted:
    """an engine whose step() records how many kernels it launched"""

    def __init__(self, eng):
        self.eng = eng
        self.step_launches = []

    def __getattr__(self, name):
        return getattr(self.eng, name)

    def step(self, *a):
        k0 = self.eng.launch_count()
        self.eng.step(*a)
        self.step_launches.append(self.eng.launch_count() - k0)


def _compare(case):
    auto = case.params.solver == AC.SOLVER_AUTOTSIT5

    def cmp(ref, dut):
        compare_models(ref, dut)
        if auto:
            assert np.array_equal(ref.solver_state(), dut.solver_state()), "AutoSwitch state differs"
    return cmp


@pytest.mark.parametrize("name", sorted(AC.CASES))
def test_gpu_advance_case_bit_exact(gpu_lib, name):
    case = AC.CASES[name]
    dut = Counted(engine_for(case.grid, case.params))
    AC.run_case(make_oracle(case.grid, case.params), dut, case, _compare(case))
    assert dut.step_launches == [launches_per_step(case)] * len(case.dts)


def _members(case):
    """the case's winds, the same with v negated, and a calm member"""
    w = case.wind

    def flipped(t):
        u, v = w(t)
        return u, -np.asarray(v, np.float64)

    def calm(t):
        u, v = w(t)
        return np.zeros_like(np.asarray(u, np.float64)), np.zeros_like(np.asarray(v, np.float64))
    return [w, flipped, calm]


@pytest.mark.parametrize("name", sorted(AC.CASES))
def test_gpu_advance_case_as_ensemble(gpu_lib, name):
    """the case as an ensemble of three (the ensemble form of each instantiation), every member against its own
    oracle after every step; counters summed over the members"""
    case = AC.CASES[name]
    g, P = case.grid, case.params
    winds = _members(case)
    E = len(winds)
    eng = ensemble_engine(g, P, E)
    refs = [make_oracle(g, P) for _ in range(E)]
    full = lambda a: np.broadcast_to(np.asarray(a, np.float64), (g["Ny"], g["Nx"]))
    stack = lambda lv: (np.stack([full(a) for a, _ in lv]), np.stack([full(b) for _, b in lv]))
    u0, v0 = stack([w(0.0) for w in winds])
    eng.seed(u0, v0)
    for m, r in enumerate(refs):
        r.seed(u0[m], v0[m])
    if case.accumulate:
        eng.set_accumulate(True)
        for r in refs:
            r.set_accumulate(True)
    auto = P.solver == AC.SOLVER_AUTOTSIT5
    t = 0.0
    for k, dt in enumerate(case.dts):
        if case.inject is not None:
            S = case.inject(k)
            eng.set_state(np.stack([S] * E, axis=1))
            for r in refs:
                r.set_state(S)
        lv = [stack([w(t + dt * j / (case.n_mid + 1)) for w in winds]) for j in range(case.n_mid + 2)]
        if case.n_mid:
            eng.set_wind_midlevels([a for a, _ in lv[1:-1]], [b for _, b in lv[1:-1]])
            for m, r in enumerate(refs):
                r.set_wind_midlevels([a[m] for a, _ in lv[1:-1]], [b[m] for _, b in lv[1:-1]])
        k0 = eng.launch_count()
        eng.step(t, dt, *lv[0], *lv[-1])
        assert eng.launch_count() - k0 == launches_per_step(case)
        for m, r in enumerate(refs):
            r.step(t, dt, lv[0][0][m], lv[0][1][m], lv[-1][0][m], lv[-1][1][m])
        t += dt
        out = (eng.state(), eng.particles(), eng.solver_state() if auto else None)
        for m, r in enumerate(refs):
            compare_member(r, out, m, auto)
        c, cr = eng.counters(), [r.counters() for r in refs]
        for n in TALLY_NAMES:
            want = max(x[n] for x in cr) if n in ("reach", "max_attempts") else sum(x[n] for x in cr)
            assert c[n] == want, (k, n, c[n], want)


@pytest.mark.parametrize("name", sorted(n for n, c in AC.CASES.items() if c.strips))
def test_gpu_advance_case_in_strips(gpu_lib, name):
    """two strips with a host-driven exchange: particles parked for k_advance_resume are resumed strip by strip; the
    AutoSwitch state of the strips, put together, is the oracle's"""
    case = AC.CASES[name]
    auto = case.params.solver == AC.SOLVER_AUTOTSIT5

    def cmp(ref, dut):
        compare_models(ref, dut)
        if auto:
            sol = np.concatenate([e.solver_state() for e in dut.e], axis=0)
            assert np.array_equal(ref.solver_state(), sol), "AutoSwitch state differs"
    AC.run_case(make_oracle(case.grid, case.params), StripSet(case.grid, case.params, 2, 2), case, cmp)
