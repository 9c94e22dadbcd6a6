"""The AMG V-cycle computes exactly the bits recorded in tests/golden/amg_cycle_bits.json
(tests/golden/make_amg_cycle_bits.py, written with the library from before the cycle's sweeps were
fused): the single-GPU cycle (csrc/amg.cu) and the one-rank row-partitioned solve (csrc/dist_amg.cu),
whose iterations must match as well."""
import importlib.util
import os

import pytest

from helpers import golden

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
BITS = golden("amg_cycle_bits.json")


def _maker():
    spec = importlib.util.spec_from_file_location("make_amg_cycle_bits",
                                                  os.path.join(HERE, "golden", "make_amg_cycle_bits.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


MAKER = _maker()


@pytest.mark.parametrize("name", MAKER.APPLY_CASES)
def test_amg_apply_bits(device, name):
    got = MAKER.digest(MAKER.apply_bits(device, name))
    assert got == BITS["apply"][name]


def test_dist_single_rank_solve_bits(device):
    x, info = MAKER.dist_bits(device)
    want = BITS["dist_single_rank"]
    assert int(info["distributed_levels"]) == want["distributed_levels"] >= 2
    assert int(info["iterations"]) == want["iterations"]
    assert MAKER.digest(x) == want["x"]
