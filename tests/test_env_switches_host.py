"""The environment variables the library reads (nodal_b200/csrc).  Each one is a second code path
that kernel changes must keep correct, so the set is pinned: a new switch is a deliberate decision
that updates this list."""
import glob
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "nodal_b200", "csrc")

KEPT = {
    "NODAL_SELL_WIDE",      # the wide SELL encoding: the reference the compact one is tested against
    "NODAL_DIST_NO_P2P",    # the NCCL back end of the row-partitioned solvers on a box with peer access
    "NODAL_DIST_DEBUG",     # timing report of the fused peer-memory iteration
}


def test_getenv_names_are_the_kept_switches():
    names = set()
    files = glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh"))
    assert files
    for path in files:
        with open(path) as f:
            src = f.read()
        names |= set(re.findall(r'getenv\(\s*"([^"]*)"\s*\)', src))
        # every getenv call names its variable literally, so the scan above sees all of them
        assert src.count("getenv(") == len(re.findall(r'getenv\(\s*"[^"]*"\s*\)', src)), path
    assert names == KEPT
