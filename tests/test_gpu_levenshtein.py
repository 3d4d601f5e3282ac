"""GPU tests of the edit-distance search (b200sa_levenshtein_batch) against the DP oracle of _levenshtein_oracle.py,
which uses no FM machinery: every text window T[s..s+l) with l in [m - k, m + k] at Levenshtein distance <= k from
the pattern is a hit candidate; windows are grouped by content, and the string Q of a group has the SA interval
[min ISA[s], min ISA[s] + count) over its positions s, its length and its distance ED(P, Q).  Hits are sorted by
(L, length).  Offsets, L, R, length and the distances are compared exactly and in order."""
import ctypes as C

import numpy as np
import pytest

from _levenshtein_oracle import oracle_hits
from test_gpu_hamming import TEXTS, _concat, _offsets, _reverse, text_of

pytestmark = pytest.mark.gpu

BAD_ARGUMENT, NOT_BUILT = 2, 5
COLS = ("offsets", "L", "R", "length", "edits")


def edited(rng, p, nsym, edits):
    """p with `edits` random substitutions, insertions and deletions (inserted symbols are letters)."""
    p = [int(x) for x in p]
    for _ in range(edits):
        op = int(rng.integers(0, 3))
        if op == 1 or not p:
            p.insert(int(rng.integers(0, len(p) + 1)), int(rng.integers(1, nsym + 1)))
        elif op == 2:
            del p[int(rng.integers(0, len(p)))]
        else:
            at = int(rng.integers(0, len(p)))
            p[at] = 1 + (p[at] - 1 + int(rng.integers(1, nsym))) % nsym if nsym > 1 else nsym + 1
    return np.array(p, np.uint8)


def patterns(rng, codes, sigma, npat, mmin, mmax, kmax):
    """Pieces of the text with 0 .. kmax + 1 edits, random patterns, patterns holding 0 or a code >= sigma, and one
    empty pattern."""
    n, nsym = len(codes) - 1, sigma - 1
    pats = [np.zeros(0, np.uint8)]
    for j in range(npat):
        m = int(rng.integers(mmin, mmax + 1))
        kind = j % 5
        if kind == 4 or n < m:
            p = rng.integers(1, nsym + 1, m).astype(np.uint8)
        else:
            s = int(rng.integers(0, n - m + 1))
            p = edited(rng, codes[s:s + m], nsym, int(rng.integers(0, kmax + 2)))
            if kind == 3 and len(p):
                p[int(rng.integers(0, len(p)))] = 0 if j % 2 else sigma + int(rng.integers(0, 256 - sigma))
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
            res = idx.levenshtein_search(_concat(batch), max_edits=k, rev=rev, **form)
            assert res["offsets"].tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), (k, list(form))
            got = list(zip(*(res[c].tolist() for c in COLS[1:])))
            assert got == [h for w in want for h in w], (k, list(form))
            out.setdefault(k, res)
    return out


def ed(a, b):
    D = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        prev, D[0] = D[0], i
        for j in range(1, len(b) + 1):
            cur = D[j]
            D[j] = min(D[j] + 1, D[j - 1] + 1, prev + (a[i - 1] != b[j - 1]))
            prev = cur
    return D[len(b)]


def check_invariants(idx, codes, pats, res):
    """No (L, length) twice within a pattern, and every located position holds a window at the hit's distance."""
    n = len(codes) - 1
    poff, pos = idx.locate(res["L"], res["R"])
    for q, p in enumerate(pats):
        a, b = int(res["offsets"][q]), int(res["offsets"][q + 1])
        keys = list(zip(res["L"][a:b].tolist(), res["length"][a:b].tolist()))
        assert len(set(keys)) == len(keys) and keys == sorted(keys), q
        assert (res["L"][a:b] < res["R"][a:b]).all(), q
        for h in range(a, b):
            ln = int(res["length"][h])
            for s in pos[int(poff[h]):int(poff[h + 1])].tolist()[:4]:
                assert s + ln <= n
                assert ed(p.tolist(), codes[s:s + ln].tolist()) == int(res["edits"][h]), (q, h, s)


def _pair(engine, codes, sigma, **build):
    return (engine.SuffixArrayIndex.build(codes[:-1], sigma, **build),
            engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True, **build))


@pytest.mark.parametrize("name", TEXTS)
def test_levenshtein_matches_oracle(engine, oracle, name):
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(len(codes) + sigma)
    isa = oracle.inverse(oracle.sa(codes))
    idx, rev = _pair(engine, codes, sigma)
    npat = 30 if len(codes) > 20000 else 50
    pats = patterns(rng, codes, sigma, npat, 1, 40, 3)
    pats += [codes[s:s + 24].copy() for s in range(0, 600, 50)]  # (the fixed-length form)
    res = check(idx, rev, codes, isa, pats, (0, 1, 2, 3), fixed_len=24)
    check_invariants(idx, codes, pats, res[2])
    idx.close()
    rev.close()


@pytest.mark.parametrize("name", ["dna_4k", "binary", "unary", "acgt_repeat", "fibonacci", "byte20"])
def test_levenshtein_k4_and_short_patterns(engine, oracle, name):
    """k = 4 on patterns of 1..14 symbols, so m <= k (empty parts) comes up often, and k = 3, 4 on 30-symbol reads."""
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(3 * len(codes) + sigma)
    isa = oracle.inverse(oracle.sa(codes))
    idx, rev = _pair(engine, codes, sigma)
    pats = patterns(rng, codes, sigma, 30, 1, 14, 4)
    res = check(idx, rev, codes, isa, pats, (2, 4))
    check_invariants(idx, codes, pats, res[4])
    pats = patterns(rng, codes, sigma, 12, 28, 32, 4)
    check(idx, rev, codes, isa, pats, (4,))
    idx.close()
    rev.close()


@pytest.mark.parametrize("name", ["dna_16k", "byte20"])
def test_levenshtein_same_with_textcmp_and_ktable(engine, oracle, name):
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(5)
    pats = patterns(rng, codes, sigma, 60, 1, 40, 3)
    pat, off = _concat(pats), _offsets(pats)
    rev = engine.SuffixArrayIndex.build(_reverse(codes), sigma, drop_sa=True)
    builds = [{}, {"textcmp": True}] + ([{"textcmp": True, "ktable": True}] if sigma == 5 else [])
    results = []
    for b in builds:
        idx, rv = _pair(engine, codes, sigma, **b)
        results.append([idx.levenshtein_search(pat, off, max_edits=k, rev=r) for k in (1, 3) for r in (rev, rv)])
        idx.close()
        rv.close()
    for other in results[1:]:
        for a, b in zip(results[0], other):
            assert all(np.array_equal(a[c], b[c]) for c in COLS)
    assert len(results[0][1]["L"]) > len(pats)
    rev.close()


def test_levenshtein_k0_is_exact_search(engine, oracle):
    codes, sigma = text_of(oracle, "dna_16k")
    rng = np.random.default_rng(11)
    pats = [p for p in patterns(rng, codes, sigma, 200, 1, 30, 1) if len(p)]
    pat, off = _concat(pats), _offsets(pats)
    idx, rev = _pair(engine, codes, sigma)
    L, R = idx.search(pat, off)
    res = idx.levenshtein_search(pat, off, max_edits=0, rev=rev)
    found = L < R
    assert found.sum() > 50
    assert np.diff(res["offsets"]).tolist() == found.astype(int).tolist()
    assert np.array_equal(res["L"], L[found]) and np.array_equal(res["R"], R[found])
    assert res["length"].tolist() == [len(p) for p, f in zip(pats, found) if f]
    assert not res["edits"].any()
    idx.close()
    rev.close()


@pytest.mark.parametrize("name", ["dna_4k", "acgt_repeat"])
def test_levenshtein_contains_every_approx_hit(engine, oracle, name):
    """Every distinct (L, match length) of the reference's edit-path iterator at max_edits = k is a hit of that
    length: its paths are edit scripts, so the distance is at most their edit count."""
    codes, sigma = text_of(oracle, name)
    rng = np.random.default_rng(17)
    idx, rev = _pair(engine, codes, sigma)
    for k in (1, 2):
        pats = [p for p in patterns(rng, codes, sigma, 40, 8, 20, k)
                if len(p) > k and ((p >= 1) & (p < sigma)).all()]
        pat, off = _concat(pats), _offsets(pats)
        ap = idx.approx_search(pat, off, max_edits=k)
        lv = idx.levenshtein_search(pat, off, max_edits=k, rev=rev)
        seen = 0
        for q in range(len(pats)):
            a, b = int(ap["offsets"][q]), int(ap["offsets"][q + 1])
            want = set(zip(ap["L"][a:b].tolist(), ap["match_length"][a:b].tolist()))
            c, d = int(lv["offsets"][q]), int(lv["offsets"][q + 1])
            got = dict(zip(zip(lv["L"][c:d].tolist(), lv["length"][c:d].tolist()), lv["R"][c:d].tolist()))
            assert want <= set(got), (k, q, want - set(got))
            seen += len(want)
        assert seen > len(pats)
    idx.close()
    rev.close()


def test_levenshtein_saved_and_loaded_pair(engine, oracle, tmp_path):
    codes, sigma = text_of(oracle, "dna_4k")
    rng = np.random.default_rng(13)
    pats = patterns(rng, codes, sigma, 60, 1, 30, 2)
    pat, off = _concat(pats), _offsets(pats)
    idx, rev = _pair(engine, codes, sigma)
    want = idx.levenshtein_search(pat, off, max_edits=2, rev=rev)
    idx.save(tmp_path / "f.b200sa")
    rev.save(tmp_path / "b.b200sa")
    idx2 = engine.SuffixArrayIndex.load(tmp_path / "f.b200sa")
    rev2 = engine.SuffixArrayIndex.load(tmp_path / "b.b200sa")
    got = idx2.levenshtein_search(pat, off, max_edits=2, rev=rev2)
    assert all(np.array_equal(want[c], got[c]) for c in COLS)
    for h in (idx, rev, idx2, rev2):
        h.close()


def test_levenshtein_edge_cases(engine, oracle):
    codes, sigma, table = oracle.remap(b"mississippi")
    isa = oracle.inverse(oracle.sa(codes))
    idx, rev = _pair(engine, codes, sigma)
    # no patterns; only empty patterns
    r = idx.levenshtein_search(np.zeros(0, np.uint8), np.zeros(1, np.uint64), rev=rev)
    assert r["offsets"].tolist() == [0] and len(r["L"]) == 0
    r = idx.levenshtein_search(np.zeros(0, np.uint8), np.zeros(3, np.uint64), max_edits=2, rev=rev)
    assert r["offsets"].tolist() == [0, 0, 0]
    # a pattern of non-letters only matches no letter, so ED(P, Q) = max(m, |Q|): at k = m every non-empty string
    # of up to m symbols is a hit
    p = np.array([0, sigma, 255], np.uint8)
    r = idx.levenshtein_search(p, np.array([0, 3], np.uint64), max_edits=3, rev=rev)
    assert list(zip(*(r[c].tolist() for c in COLS[1:]))) == oracle_hits(codes, isa, p, 3)
    n = len(codes) - 1
    assert len(r["L"]) == len({bytes(codes[s:s + l]) for l in range(1, 4) for s in range(n - l + 1)})
    r = idx.levenshtein_search(p, np.array([0, 3], np.uint64), max_edits=2, rev=rev)
    assert len(r["L"]) == 0
    with pytest.raises(ValueError):
        idx.levenshtein_search(p, np.array([0, 3], np.uint64))
    idx.close()
    rev.close()


def test_levenshtein_refusals_of_the_indices(engine, oracle):
    lib = engine.load()
    codes, sigma = text_of(oracle, "dna_4k")
    pats = np.ones(8, np.uint8)

    def refused(code, idx, rev):
        err = C.c_int(-1)
        h = lib.b200sa_levenshtein_batch(idx._h, rev._h, pats.ctypes.data_as(C.c_void_p), None, 8, 1, 1,
                                         C.byref(err))
        assert not h and err.value == code, err.value
        assert lib.b200sa_last_error()

    idx, rev = _pair(engine, codes, sigma)
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
