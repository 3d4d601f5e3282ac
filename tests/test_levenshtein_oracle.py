"""The oracles of the edit-distance search agree (no GPU needed): the DP-from-every-start oracle equals a plain
dynamic program over every text window on small texts, and the pigeonhole oracle equals the DP oracle on every text
of test_gpu_hamming, for k = 0 .. 4, on the patterns test_gpu_levenshtein generates.  The GPU tests at 2^20 symbols
rest on the pigeonhole oracle, so it is pinned here first."""
import numpy as np
import pytest

from _hamming_oracle import QgramTable
from _levenshtein_oracle import oracle_hits, pigeonhole_hits
from test_gpu_hamming import TEXTS, _concat, _offsets, text_of
from test_gpu_levenshtein import ed, patterns


def test_dp_oracle_equals_every_window(oracle):
    rng = np.random.default_rng(1)
    checked = 0
    for case in range(60):
        nsym = int(rng.choice([1, 2, 4]))
        n = int(rng.integers(1, 50))
        codes = np.append(rng.integers(1, nsym + 1, n), 0).astype(np.uint8)
        if case % 4 == 0:
            codes[:n] = ([1, 2] * n)[:n] if nsym > 1 else 1
        isa = oracle.inverse(oracle.sa(codes))
        sa = np.argsort(isa)
        k = int(rng.integers(0, 5))
        p = rng.integers(0, nsym + 2, int(rng.integers(0, 10))).astype(np.uint8)
        want = {}
        for s in range(n):
            for l in range(max(1, len(p) - k), len(p) + k + 1):
                if len(p) and s + l <= n:
                    d = ed(p.tolist(), codes[s:s + l].tolist())
                    if d <= k:
                        want[bytes(codes[s:s + l])] = d
        got = oracle_hits(codes, isa, p, k)
        assert len(got) == len(want), case
        for L, R, ln, d in got:
            q = bytes(codes[sa[L]:sa[L] + ln])
            assert want[q] == d, case
            rows = [r for r in range(len(sa)) if bytes(codes[sa[r]:sa[r] + ln]) == q]
            assert rows == list(range(L, R)), case
        checked += len(got)
    assert checked > 100


@pytest.mark.parametrize("name", TEXTS)
def test_pigeonhole_equals_dp_oracle(oracle, name):
    codes, sigma = text_of(oracle, name)
    isa = oracle.inverse(oracle.sa(codes))
    table = QgramTable(codes, sigma)
    rng = np.random.default_rng(len(codes) + sigma)
    pats = patterns(rng, codes, sigma, 20, 1, 40, 3)
    pats += patterns(rng, codes, sigma, 12, 1, 8, 4)  # (m <= k comes up for the larger k)
    pat, off = _concat(pats), _offsets(pats)
    total = 0
    for k in range(5):
        want = [oracle_hits(codes, isa, p, k) for p in pats]
        got_off, L, R, ln, d = pigeonhole_hits(table, isa, pat, off, k)
        assert got_off.tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), k
        assert list(zip(L.tolist(), R.tolist(), ln.tolist(), d.tolist())) == [h for w in want for h in w], k
        total += len(L)
    assert total > len(pats)  # (the comparison is not vacuous)
