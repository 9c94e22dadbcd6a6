"""CPU tests of the SELL entry encodings (csrc/sell_core.cuh through tests/host_check/sell_host.cpp): which
matrices go compact, and that the compact entries decode to the wide ones bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sps

from sell_host import build


def csr_of(M):
    M = sps.csr_matrix(M)
    M.sort_indices()
    return M.shape[0], M.indptr, M.indices, M.data


def assert_lossless(s):
    assert s["compact"]
    assert np.array_equal(s["dcols"], s["cols"])
    assert np.array_equal(s["dvals"].view(np.uint64), s["vals"].view(np.uint64))
    assert np.all(np.diff(s["dict"].astype(np.uint64)) > 0) and s["dict"][0] == 0


def diagonal(values):
    v = np.asarray(values, dtype=np.float64)
    n = len(v)
    return n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32), v


@pytest.mark.parametrize("distinct,compact", [(255, True), (256, False)])
def test_table_holds_256_patterns_with_the_padding_zero(distinct, compact):
    # 255 nonzero values + the 0.0 of the padding fill the 256-entry table; one more does not fit
    s = build(*diagonal(np.arange(1, distinct + 1)))
    assert s["ndict"] == distinct + 1 and s["compact"] == compact
    if compact:
        assert_lossless(s)


def test_256_distinct_including_zero_fits():
    s = build(*diagonal(np.arange(0, 256)))
    assert s["ndict"] == 256
    assert_lossless(s)


def test_signed_zeros_are_two_values():
    s = build(*diagonal([0.0, -0.0, 1.0, -0.0]))
    assert s["ndict"] == 3
    assert_lossless(s)
    assert np.signbit(s["dvals"][1]) and not np.signbit(s["dvals"][0])


def test_nan_payloads_and_subnormals_by_bit_pattern():
    pats = np.array([0x7FF8000000000001, 0x7FF8000000000002, 0xFFF8000000000000, 0x0000000000000001,
                     0x8000000000000001, 0x000FFFFFFFFFFFFF], dtype=np.uint64)
    s = build(*diagonal(pats.view(np.float64)))
    assert s["ndict"] == len(pats) + 1
    assert_lossless(s)
    assert np.array_equal(s["dvals"][: len(pats)].view(np.uint64), pats)


@pytest.mark.parametrize("off,fits", [(32767, True), (32768, False), (-32768, True), (-32769, False)])
def test_offset_range(off, fits):
    n = 40000
    row = 32769 if off < 0 else 0
    M = sps.lil_matrix((n, n))
    M.setdiag(2.0)
    M[row, row + off] = -1.0
    s = build(*csr_of(M))
    assert s["fits"] == fits and s["compact"] == fits
    if fits:
        assert_lossless(s)


@pytest.mark.parametrize("n", [1, 31, 33, 70])
def test_tail_lanes_and_row_padding(n):
    rng = np.random.default_rng(n)
    M = sps.random(n, n, density=0.2, random_state=rng, format="csr")
    M.data = np.round(M.data * 4) - 2.0          # few values, some of them 0.0 stored explicitly
    M = M + sps.eye(n)
    n_, ip, ix, dv = csr_of(M)
    s = build(n_, ip, ix, dv)
    assert_lossless(s)
    ns = (n + 31) // 32
    sw = s["slice_w"]
    for lane in range(n - (ns - 1) * 32, 32):          # tail lanes: column n - 1, value +0.0
        for k in range(sw[ns - 1], sw[ns]):
            i = k * 32 + lane
            assert s["dcols"][i] == n - 1 and s["dvals"][i].view(np.uint64) == 0
    lens = np.diff(ip)
    for r in range(n):                                 # padding inside a row: the row itself
        s0, lane = divmod(r, 32)
        for k in range(sw[s0] + lens[r], sw[s0 + 1]):
            i = k * 32 + lane
            assert s["dcols"][i] == r and s["dvals"][i].view(np.uint64) == 0


def test_empty_matrix_is_wide():
    s = build(0, np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0))
    assert not s["compact"] and s["cols"].size == 0


def test_single_row():
    s = build(*diagonal([3.5]))
    assert_lossless(s)
    assert s["dcols"][0] == 0 and s["dvals"][0] == 3.5 and s["dcols"][1:].tolist() == [0] * 31
