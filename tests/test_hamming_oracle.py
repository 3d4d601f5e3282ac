"""The pigeonhole oracle of the k-mismatch search equals the window-scan oracle (no GPU needed): on every text of
test_gpu_hamming, for k = 0 .. 8, on the patterns that file generates.  The GPU tests at 2^20 symbols and 10^5
patterns rest on the pigeonhole oracle, so it is pinned here first."""
import numpy as np
import pytest

from _hamming_oracle import QgramTable, oracle_hits, part_bounds, pigeonhole_hits
from test_gpu_hamming import TEXTS, _concat, _offsets, patterns, text_of


def test_part_bounds_split_like_the_kernel():
    """k + 1 consecutive parts covering the pattern, the m mod (k + 1) longer ones first."""
    for k in range(9):
        for m in range(0, 40):
            st, ln = part_bounds(np.array([m]), k)
            st, ln = st[0].tolist(), ln[0].tolist()
            assert st[0] == 0 and st[-1] + ln[-1] == m
            assert all(a + b == c for a, b, c in zip(st, ln, st[1:]))
            assert ln == [m // (k + 1) + 1] * (m % (k + 1)) + [m // (k + 1)] * (k + 1 - m % (k + 1))


@pytest.mark.parametrize("name", TEXTS)
def test_pigeonhole_equals_window_scan(oracle, name):
    codes, sigma = text_of(oracle, name)
    isa = oracle.inverse(oracle.sa(codes))
    table = QgramTable(codes, sigma)
    rng = np.random.default_rng(len(codes) + sigma)
    npat = 40 if len(codes) > 20000 else 80
    pats = patterns(rng, codes, sigma, npat, 1, 60, 3)
    pats += [codes[s:s + 24].copy() for s in range(0, 600, 50)]
    pats += patterns(rng, codes, sigma, 30, 1, 12, 8)  # (m <= k comes up for the larger k)
    pat, off = _concat(pats), _offsets(pats)
    total = 0
    for k in range(9):
        want = [oracle_hits(codes, isa, p, k) for p in pats]
        got_off, L, R, d = pigeonhole_hits(table, isa, pat, off, k)
        assert got_off.tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), k
        assert list(zip(L.tolist(), R.tolist(), d.tolist())) == [h for w in want for h in w], k
        total += len(L)
    assert total > len(pats)  # (the comparison is not vacuous)
