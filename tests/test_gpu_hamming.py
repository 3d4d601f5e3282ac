"""GPU tests of the k-mismatch search (b200sa_hamming_batch) against a brute-force oracle stated here, which uses no
FM machinery: every text window T[s..s+m) at Hamming distance <= k from the pattern P is a hit candidate; windows
are grouped by content, and the string Q of a group has the SA interval [min ISA[s], min ISA[s] + count) over its
positions s (from the oracle's suffix array) and distance Hamming(P, Q).  Hits are sorted by L.  Offsets, L, R and
the distances are compared exactly and in order."""
import ctypes as C

import numpy as np
import pytest

from _hamming_oracle import oracle_hits

pytestmark = pytest.mark.gpu

BAD_ARGUMENT, NOT_BUILT = 2, 5


def _offsets(pats):
    off = np.zeros(len(pats) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    return off


def _concat(pats):
    return np.concatenate(pats).astype(np.uint8) if pats else np.zeros(0, np.uint8)


def _reverse(codes):
    return codes[:-1][::-1].copy()


def fibonacci_codes(n):
    a, b = [1], [1, 2]
    while len(b) < n:
        a, b = b, b + a
    return np.array(b[:n] + [0], np.uint8)


def text_of(oracle, name):
    if name == "dna_4k":
        return oracle.random_codes(1 << 12, 4, seed=12), 5
    if name == "dna_16k":
        return oracle.random_codes(1 << 14, 4, seed=14), 5
    if name == "dna_64k":
        return oracle.random_codes(1 << 16, 4, seed=16), 5
    if name == "binary":
        return oracle.random_codes(3000, 2, seed=2), 3
    if name == "unary":
        return np.array([1] * 2000 + [0], np.uint8), 2
    if name == "acgt_repeat":
        return np.array([1, 2, 3, 4] * 1000 + [0], np.uint8), 5
    if name == "fibonacci":
        return fibonacci_codes(4181), 3
    if name == "byte20":
        return oracle.random_codes(4000, 20, seed=20), 21
    if name == "byte200":
        return oracle.random_codes(1500, 200, seed=200), 201
    raise KeyError(name)


def patterns(rng, codes, sigma, npat, mmin, mmax, kmax):
    """Pieces of the text with 0 .. kmax + 1 substitutions, random patterns, patterns holding 0 or a code >= sigma,
    and one empty pattern."""
    n, nsym = len(codes) - 1, sigma - 1
    pats = [np.zeros(0, np.uint8)]
    for j in range(npat):
        m = int(rng.integers(mmin, mmax + 1))
        kind = j % 5
        if kind == 4 or n < m:
            p = rng.integers(1, nsym + 1, m).astype(np.uint8)
        else:
            s = int(rng.integers(0, n - m + 1))
            p = codes[s:s + m].copy()
            for at in rng.choice(m, size=min(m, int(rng.integers(0, kmax + 2))), replace=False):
                if nsym > 1:
                    p[at] = 1 + (int(p[at]) - 1 + int(rng.integers(1, nsym))) % nsym  # another letter
                else:
                    p[at] = sigma
            if kind == 3:
                p[int(rng.integers(0, m))] = 0 if j % 2 else sigma + int(rng.integers(0, 256 - sigma))
        pats.append(p)
    return pats


def check(idx, rev, codes, isa, pats, ks, fixed_len=0):
    """Both forms of the batch against the oracle for every k in ks; returns the results of the offsets form."""
    runs = [(pats, dict(offsets=_offsets(pats)))]
    if fixed_len:
        runs.append(([p for p in pats if len(p) == fixed_len], dict(fixed_len=fixed_len)))
    out = {}
    for k in ks:
        for batch, form in runs:
            want = [oracle_hits(codes, isa, p, k) for p in batch]
            res = idx.hamming_search(_concat(batch), max_mismatches=k, rev=rev, **form)
            assert res["offsets"].tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), (k, list(form))
            got = list(zip(res["L"].tolist(), res["R"].tolist(), res["mismatches"].tolist()))
            assert got == [h for w in want for h in w], (k, list(form))
            out.setdefault(k, res)
    return out


def check_invariants(idx, codes, pats, res):
    """No interval twice within a pattern, and every located position holds a window at the hit's distance."""
    n = len(codes) - 1
    poff, pos = idx.locate(res["L"], res["R"])
    for q, p in enumerate(pats):
        a, b = int(res["offsets"][q]), int(res["offsets"][q + 1])
        L, R = res["L"][a:b].astype(np.int64), res["R"][a:b].astype(np.int64)
        assert (L < R).all() and (L[1:] >= R[:-1]).all(), q
        for h in range(a, b):
            for s in pos[int(poff[h]):int(poff[h + 1])].tolist():
                assert s + len(p) <= n
                assert int((codes[s:s + len(p)] != p).sum()) == int(res["mismatches"][h]), (q, h, s)


TEXTS = ["dna_4k", "dna_16k", "dna_64k", "binary", "unary", "acgt_repeat", "fibonacci", "byte20", "byte200"]


@pytest.mark.parametrize("name", TEXTS)
def test_hamming_matches_oracle(engine, oracle, name):
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(len(codes) + sigma)
    isa = oracle.inverse(oracle.sa(codes))
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    npat = 40 if len(codes) > 20000 else 80
    pats = patterns(rng, codes, sigma, npat, 1, 60, 3)
    pats += [codes[s:s + 24].copy() for s in range(0, 600, 50)]  # (the fixed-length form)
    res = check(idx, rev, codes, isa, pats, (0, 1, 2, 3), fixed_len=24)
    check_invariants(idx, codes, pats, res[2])
    idx.close()
    rev.close()


@pytest.mark.parametrize("name", ["dna_4k", "binary", "acgt_repeat", "byte20"])
def test_hamming_large_budgets_on_short_patterns(engine, oracle, name):
    """k up to 8 on patterns of 1..12 symbols, so m <= k (empty parts) comes up often."""
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(3 * len(codes) + sigma)
    isa = oracle.inverse(oracle.sa(codes))
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    pats = patterns(rng, codes, sigma, 30, 1, 12, 8)
    res = check(idx, rev, codes, isa, pats, range(4, 9))
    check_invariants(idx, codes, pats, res[8])
    idx.close()
    rev.close()


@pytest.mark.parametrize("name", ["dna_16k", "byte20"])
def test_hamming_same_with_textcmp_and_ktable(engine, oracle, name):
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(5)
    pats = patterns(rng, codes, sigma, 60, 1, 40, 3)
    pat, off = _concat(pats), _offsets(pats)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    builds = [{}, {"textcmp": True}] + ([{"textcmp": True, "ktable": True}] if sigma == 5 else [])
    results = []
    for b in builds:
        idx = engine.SuffixArrayIndex.build(codes[:-1], sigma, **b)
        rv = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True, **b)
        results.append([idx.hamming_search(pat, off, max_mismatches=k, rev=r) for k in (1, 3) for r in (rev, rv)])
        idx.close()
        rv.close()
    for other in results[1:]:
        for a, b in zip(results[0], other):
            assert all(np.array_equal(a[c], b[c]) for c in ("offsets", "L", "R", "mismatches"))
    rev.close()


def test_hamming_k0_is_exact_search(engine, oracle):
    codes, sigma = text_of(oracle, "dna_16k")
    rng = np.random.default_rng(11)
    pats = [p for p in patterns(rng, codes, sigma, 200, 1, 30, 1) if len(p)]
    pat, off = _concat(pats), _offsets(pats)
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    L, R = idx.search(pat, off)
    res = idx.hamming_search(pat, off, max_mismatches=0, rev=rev)
    found = L < R
    assert np.diff(res["offsets"]).tolist() == found.astype(int).tolist()
    assert np.array_equal(res["L"], L[found]) and np.array_equal(res["R"], R[found])
    assert not res["mismatches"].any()
    idx.close()
    rev.close()


def test_hamming_saved_and_loaded_pair(engine, oracle, tmp_path):
    codes, sigma = text_of(oracle, "dna_4k")
    rng = np.random.default_rng(13)
    pats = patterns(rng, codes, sigma, 60, 1, 30, 2)
    pat, off = _concat(pats), _offsets(pats)
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    want = idx.hamming_search(pat, off, max_mismatches=2, rev=rev)
    idx.save(tmp_path / "f.b200sa")
    rev.save(tmp_path / "b.b200sa")
    idx2 = engine.SuffixArrayIndex.load(tmp_path / "f.b200sa")
    rev2 = engine.SuffixArrayIndex.load(tmp_path / "b.b200sa")
    got = idx2.hamming_search(pat, off, max_mismatches=2, rev=rev2)
    assert all(np.array_equal(want[c], got[c]) for c in ("offsets", "L", "R", "mismatches"))
    for h in (idx, rev, idx2, rev2):
        h.close()


def test_hamming_edge_cases(engine, oracle):
    codes, sigma, table = oracle.remap(b"mississippi")
    isa = oracle.inverse(oracle.sa(codes))
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    # no patterns; only empty patterns
    r = idx.hamming_search(np.zeros(0, np.uint8), np.zeros(1, np.uint64), rev=rev)
    assert r["offsets"].tolist() == [0] and len(r["L"]) == 0
    r = idx.hamming_search(np.zeros(0, np.uint8), np.zeros(3, np.uint64), max_mismatches=2, rev=rev)
    assert r["offsets"].tolist() == [0, 0, 0]
    # a pattern of non-letters only: every string of its length is a hit once k >= m
    p = np.array([0, sigma, 255], np.uint8)
    r = idx.hamming_search(p, np.array([0, 3], np.uint64), max_mismatches=3, rev=rev)
    assert list(zip(r["L"].tolist(), r["R"].tolist(), r["mismatches"].tolist())) == oracle_hits(codes, isa, p, 3)
    assert len(r["L"]) == len({bytes(codes[s:s + 3]) for s in range(len(codes) - 3)})
    r = idx.hamming_search(p, np.array([0, 3], np.uint64), max_mismatches=2, rev=rev)
    assert len(r["L"]) == 0
    with pytest.raises(ValueError):
        idx.hamming_search(p, np.array([0, 3], np.uint64))
    idx.close()
    rev.close()


def test_hamming_refusals_of_the_indices(engine, oracle):
    lib = engine.load()
    codes, sigma = text_of(oracle, "dna_4k")
    pats = np.ones(8, np.uint8)

    def refused(code, idx, rev):
        err = C.c_int(-1)
        h = lib.b200sa_hamming_batch(idx._h, rev._h, pats.ctypes.data_as(C.c_void_p), None, 8, 1, 1, C.byref(err))
        assert not h and err.value == code, err.value
        assert lib.b200sa_last_error()

    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    no_occ = engine.SuffixArrayIndex.build(codes[:-1], sigma, occ=False)
    rev_no_occ = engine.SuffixArrayIndex.build(_reverse(codes), sigma, occ=False)
    refused(NOT_BUILT, no_occ, rev)
    refused(NOT_BUILT, idx, rev_no_occ)
    shorter = engine.SuffixArrayIndex.build(_reverse(codes)[1:], sigma, drop_sa=True)
    wider = engine.SuffixArrayIndex.build(_reverse(codes), sigma + 1, drop_sa=True)
    other = codes[:-1].copy()
    other[other == 2] = 1  # the same length and sigma, another C table
    other_counts = engine.SuffixArrayIndex.build(other[::-1].copy(), sigma, drop_sa=True)
    for bad in (shorter, wider, other_counts):
        refused(BAD_ARGUMENT, idx, bad)
    recs = [codes[:2000] + 1, codes[2000:-1] + 1]
    rec_idx = engine.SuffixArrayIndex.build_records(recs, sigma + 1)
    rec_rev = engine.SuffixArrayIndex.build_records([r[::-1].copy() for r in recs[::-1]], sigma + 1, drop_sa=True)
    refused(BAD_ARGUMENT, rec_idx, rec_rev)
    for h in (idx, rev, no_occ, rev_no_occ, shorter, wider, other_counts, rec_idx, rec_rev):
        h.close()
