"""GPU (-m gpu): the randomized configurations of tests/test_independent_model.py through the CUDA path, bit for bit
against the oracle.

The host build of the same device header is bit-exact with the oracle on 150 seeds of this generator
(tests/test_device_path_cpu.py runs ten of them), but the CUDA path also has its fast arithmetic copies (unchecked
divisions and table-driven exp where the operand ranges are proven, with a checked fallback), which only a GPU
exercises."""
import numpy as np
import pytest

from common import compare_models, make_oracle
from scenarios import run_pair

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(10))
def test_gpu_random_configurations_bit_exact(gpu_lib, seed):
    from test_gpu_parity import engine_for
    from test_independent_model import fuzz_case
    g, P, winds, DT, _ = fuzz_case(seed)

    def wind(t):
        return tuple(np.array([[winds(g["x"][j, i], g["y"][j, i], t)[k] for i in range(g["Nx"])] for j in range(g["Ny"])])
                     for k in (0, 1))

    run_pair(make_oracle(g, P), engine_for(g, P), wind, DT, 4, compare_models)


@pytest.mark.parametrize("mode", ["one strip", "two strips"])
def test_gpu_nan_error_estimate_rejected(gpu_lib, mode):
    """picles_params_t::nan_eest_rejects = 1 on scenario dp5_blowup (the generic instantiation of the advance kernel
    carries the switch; the specialised ones are launched only with it off): nobody fails, bit for bit"""
    from test_device_path_cpu import _blowup_case
    from test_gpu_parity import StripSet, engine_for
    g, P, wind, DT, n = _blowup_case(True)
    dut = StripSet(g, P, 2, 2) if mode == "two strips" else engine_for(g, P)
    ref = make_oracle(g, P)
    run_pair(ref, dut, wind, DT, n, compare_models)
    assert ref.counters()["n_failed"] == 0
