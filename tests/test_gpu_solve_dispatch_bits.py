"""Circuit.solve takes the same path, computes the same bits and reports the same stats as recorded in
tests/golden/solve_dispatch_bits.json (tests/golden/make_solve_dispatch_bits.py, written with the library
from before the options were parsed once and the sparse paths run from one plan): SHA-256 of
Solution.result and Solution.stats without its timings, for every case of the maker."""
import importlib.util
import json
import os

import pytest

from helpers import golden

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
BITS = golden("solve_dispatch_bits.json")


def _maker():
    spec = importlib.util.spec_from_file_location("make_solve_dispatch_bits",
                                                  os.path.join(HERE, "golden", "make_solve_dispatch_bits.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


MAKER = _maker()


def same(got, want):
    """Equal as recorded (JSON text, so the NaN heads of a solve that ends in NaNs compare equal)."""
    return json.dumps(got, sort_keys=True) == json.dumps(want, sort_keys=True)


@pytest.mark.parametrize("name", list(MAKER.CASES))
def test_solve_bits(device, name):
    result, stats = MAKER.run_case(name)
    assert stats == BITS[name]["stats"]
    assert same(result, BITS[name]["result"]), (result, BITS[name]["result"])


@pytest.mark.parametrize("name,pairs", [("equivalent_resistances", MAKER.PORTS),
                                        ("equivalent_resistances_single", MAKER.PORTS[1:2])])
def test_port_bits(device, name, pairs):
    result, stats = MAKER.ports(pairs)
    assert stats == BITS[name]["stats"]
    assert same(result, BITS[name]["result"]), (result, BITS[name]["result"])
