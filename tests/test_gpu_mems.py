"""GPU tests of matching statistics and super-maximal exact matches (b200sa_matching_stats, b200sa_smem_batch)
against an oracle stated here from the oracle's dense tables: for every end j of a pattern, backward steps
L = C[a] + O[L, a], R = C[a] + O[R, a] from j until the interval empties; the number of steps taken is ms[j] and the
last non-empty interval is (L[j], R[j]) ((1, 0) when no step succeeds).  SMEMs follow from ms by the rule of
include/b200sa.h.  Everything is compared exactly and in order."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KTABLE_K = "5"  # a small seed table: seeds both hit and miss on these texts


def _tables(oracle, codes, sigma):
    sa = oracle.sa(codes)
    return sa, oracle.c_table(codes, sigma).tolist(), oracle.o_table(oracle.bwt(codes, sa), sigma).tolist()


def oracle_ms(c, o, length, p):
    sigma = len(c)
    m = len(p)
    ms = np.zeros(m, np.uint32)
    L = np.ones(m, np.uint32)
    R = np.zeros(m, np.uint32)
    for j in range(m):
        lo, hi, k = 0, length, 0
        for i in range(j, -1, -1):
            a = int(p[i])
            if a == 0 or a >= sigma:
                break
            nl, nr = c[a] + o[lo][a], c[a] + o[hi][a]
            if nl >= nr:
                break
            lo, hi, k = nl, nr, k + 1
        if k:
            ms[j], L[j], R[j] = k, lo, hi
    return ms, L, R


def oracle_smems(ms, L, R, min_len):
    m = len(ms)
    return [(j + 1 - int(ms[j]), int(ms[j]), int(L[j]), int(R[j])) for j in range(m)
            if ms[j] >= min_len and (j == m - 1 or ms[j + 1] <= ms[j])]


def _offsets(pats):
    off = np.zeros(len(pats) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    return off


def _concat(pats):
    return np.concatenate(pats).astype(np.uint8) if pats else np.zeros(0, np.uint8)


def _patterns(rng, codes, npat, mmin, mmax, lo, hi):
    """Pieces of the text with substitutions, insertions and deletions, and random patterns over codes lo..hi."""
    n = len(codes) - 1
    pats = []
    for k in range(npat):
        m = int(rng.integers(mmin, mmax + 1))
        if k % 4 == 3 or n <= m:
            p = rng.integers(lo, hi + 1, m).tolist()
        else:
            s = int(rng.integers(0, n - m + 1))
            p = codes[s:s + m].tolist()
            for _ in range(int(rng.integers(0, 4))):
                op, at, x = int(rng.integers(0, 3)), int(rng.integers(0, len(p))), int(rng.integers(lo, hi + 1))
                if op == 0:
                    p[at] = x
                elif op == 1:
                    p.insert(at, x)
                elif len(p) > 1:
                    del p[at]
        pats.append(np.array(p, dtype=np.uint8))
    return pats


def check(idx, c, o, length, pats, min_lens=(1, 4), fixed_len=0):
    """Both entry points against the oracle; `fixed_len` also runs the fixed-length form."""
    pat, off = _concat(pats), _offsets(pats)
    expect = [oracle_ms(c, o, length, p) for p in pats]
    forms = [dict(offsets=off)] + ([dict(fixed_len=fixed_len)] if fixed_len else [])
    for form in forms:
        st = idx.matching_stats(pat, **form)
        for k, name in enumerate(("ms", "L", "R")):
            want = np.concatenate([e[k] for e in expect]) if expect else np.zeros(0, np.uint32)
            assert np.array_equal(st[name], want), (name, form)
        for min_len in min_lens:
            res = idx.smems(pat, min_len=min_len, **form)
            want = [oracle_smems(*e, min_len) for e in expect]
            assert res["offsets"].tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), (min_len, form)
            got = list(zip(res["start"].tolist(), res["length"].tolist(), res["L"].tolist(), res["R"].tolist()))
            assert got == [s for w in want for s in w], (min_len, form)
    return idx.smems(pat, off, min_len=1)


def check_invariants(idx, pats, res):
    """Search of every SMEM's substring gives its (L, R); one more symbol on either side, where the pattern has one,
    gives an empty interval."""
    subs, ext = [], []
    for q, p in enumerate(pats):
        for h in range(int(res["offsets"][q]), int(res["offsets"][q + 1])):
            s, n = int(res["start"][h]), int(res["length"][h])
            subs.append(p[s:s + n])
            if s > 0:
                ext.append(p[s - 1:s + n])
            if s + n < len(p):
                ext.append(p[s:s + n + 1])
    if subs:
        L, R = idx.search(_concat(subs), _offsets(subs))
        assert np.array_equal(L, res["L"]) and np.array_equal(R, res["R"])
    if ext:
        L, R = idx.search(_concat(ext), _offsets(ext))
        assert (L >= R).all()


BUILDS = {"occ": {}, "textcmp": {"textcmp": True}, "textcmp_ktable": {"textcmp": True, "ktable": True}}


@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("n", [1 << 12, 1 << 14, 1 << 16])
def test_dna_matches_oracle(engine, oracle, monkeypatch, n, build):
    monkeypatch.setenv("B200SA_KTABLE_K", KTABLE_K)
    rng = np.random.default_rng(n)
    codes = oracle.random_codes(n, 4, seed=n + 3)
    _, c, o = _tables(oracle, codes, 5)
    idx = engine.SuffixArrayIndex.build(codes[:-1], 5, **BUILDS[build])
    pats = _patterns(rng, codes, 120, 1, 150, 1, 4)
    res = check(idx, c, o, len(codes), pats)
    check_invariants(idx, pats, res)
    fixed = _patterns(rng, codes, 40, 100, 100, 1, 4)
    fixed = [p[:100] if len(p) >= 100 else np.concatenate([p, np.ones(100 - len(p), np.uint8)]) for p in fixed]
    check(idx, c, o, len(codes), fixed, fixed_len=100)
    idx.close()


@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("nsym", [20, 200])
def test_byte_layout_matches_oracle(engine, oracle, monkeypatch, nsym, build):
    monkeypatch.setenv("B200SA_KTABLE_K", "2")
    rng = np.random.default_rng(nsym)
    n = 6000
    codes = oracle.random_codes(n, nsym, seed=nsym)
    _, c, o = _tables(oracle, codes, nsym + 1)
    idx = engine.SuffixArrayIndex.build(codes[:-1], nsym + 1, **BUILDS[build])
    pats = _patterns(rng, codes, 100, 1, 40, 1, nsym)
    check_invariants(idx, pats, check(idx, c, o, len(codes), pats))
    idx.close()


def _fibonacci(n):
    a, b = [1], [1, 2]
    while len(b) < n:
        a, b = b, b + a
    return b[:n]


@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("text", ["unary", "acgt_repeat", "fibonacci"])
def test_large_intervals_match_oracle(engine, oracle, monkeypatch, text, build):
    """Texts whose intervals stay wide: the unique-interval shortcut rarely fires and the O steps do the work."""
    monkeypatch.setenv("B200SA_KTABLE_K", KTABLE_K)
    n = 3000
    body = {"unary": [1] * n, "acgt_repeat": [1, 2, 3, 4] * (n // 4), "fibonacci": _fibonacci(n)}[text]
    codes = np.array(body + [0], dtype=np.uint8)
    sigma = int(codes.max()) + 1
    _, c, o = _tables(oracle, codes, sigma)
    idx = engine.SuffixArrayIndex.build(codes[:-1], sigma, **BUILDS[build])
    rng = np.random.default_rng(len(text))
    pats = _patterns(rng, codes, 40, 1, 120, 1, sigma - 1)
    pats += [codes[:200].copy(), codes[100:400].copy()]
    check_invariants(idx, pats, check(idx, c, o, len(codes), pats))
    idx.close()


@pytest.mark.parametrize("build", list(BUILDS))
def test_edge_patterns(engine, oracle, monkeypatch, build):
    """Patterns longer than the text, codes 0 and >= sigma inside patterns, empty patterns; both pattern forms."""
    monkeypatch.setenv("B200SA_KTABLE_K", "4")
    n = 300
    codes = oracle.random_codes(n, 4, seed=11)
    _, c, o = _tables(oracle, codes, 5)
    idx = engine.SuffixArrayIndex.build(codes[:-1], 5, **BUILDS[build])
    text = codes[:-1]
    long1 = np.concatenate([text, text[:50]])
    bad = text[40:100].copy()
    bad[[5, 20, 33]] = [0, 5, 255]
    tail_bad = text[10:30].copy()
    tail_bad[-1] = 7
    pats = [long1, np.zeros(0, np.uint8), bad, np.zeros(0, np.uint8), tail_bad, np.array([0], np.uint8),
            np.array([9, 9], np.uint8), text.copy(), np.zeros(0, np.uint8)]
    res = check(idx, c, o, len(codes), pats)
    assert res["offsets"][1] == res["offsets"][2]  # an empty pattern has no SMEMs
    check_invariants(idx, pats, res)
    fixed = [text[k:k + 64].copy() for k in range(0, 200, 40)]
    fixed[1][[0, 63]] = [0, 6]
    fixed[2][10:20] = 200
    check(idx, c, o, len(codes), fixed, fixed_len=64)
    # no patterns at all
    r = idx.smems(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert r["offsets"].tolist() == [0] and len(r["start"]) == 0
    idx.close()


def test_records_index(engine, oracle, monkeypatch):
    """ms and SMEMs equal the oracle over the assembled text r0 1 r1 1 ... $; code 1 is refused; the positions of
    every SMEM lie inside one record and spell the matched piece."""
    monkeypatch.setenv("B200SA_KTABLE_K", "3")
    rng = np.random.default_rng(5)
    records = [rng.integers(2, 6, int(k)).astype(np.uint8) for k in (500, 0, 37, 900, 1, 260)]
    sigma = 6
    codes = np.concatenate([np.concatenate([r, [1]]) for r in records] + [[0]]).astype(np.uint8)
    _, c, o = _tables(oracle, codes, sigma)
    for flags in ({}, {"textcmp": True, "ktable": True}):
        idx = engine.SuffixArrayIndex.build_records(records, sigma, **flags)
        pats = _patterns(rng, codes, 80, 1, 60, 2, 5)
        pats = [np.where(p == 1, 2, p).astype(np.uint8) for p in pats]  # (pieces across a separator)
        pats.append(np.concatenate([records[0][-20:], records[2][:20]]))  # a piece spanning two records
        res = check(idx, c, o, len(codes), pats)
        check_invariants(idx, pats, res)
        off, rec, pos = idx.locate_records(res["L"], res["R"])
        pat_of = np.repeat(np.arange(len(pats)), np.diff(res["offsets"]).astype(np.int64))
        for h in range(len(res["start"])):
            s, n = int(res["start"][h]), int(res["length"][h])
            piece = pats[pat_of[h]][s:s + n]
            for k in range(int(off[h]), int(off[h + 1])):
                r, p = int(rec[k]), int(pos[k])
                assert p + n <= len(records[r]) and np.array_equal(records[r][p:p + n], piece)
        with pytest.raises(engine.B200saError) as e:
            idx.smems(np.array([2, 1, 3], np.uint8), np.array([0, 3], np.uint64))
        assert e.value.code == 3
        with pytest.raises(engine.B200saError) as e:
            idx.matching_stats(np.array([2, 1, 3], np.uint8), np.array([0, 3], np.uint64))
        assert e.value.code == 3
        idx.close()


def test_save_and_load(engine, oracle, monkeypatch, tmp_path):
    monkeypatch.setenv("B200SA_KTABLE_K", KTABLE_K)
    n = 5000
    codes = oracle.random_codes(n, 4, seed=9)
    idx = engine.SuffixArrayIndex.build(codes[:-1], 5, textcmp=True, ktable=True)
    pats = _patterns(np.random.default_rng(2), codes, 60, 1, 80, 1, 4)
    pat, off = _concat(pats), _offsets(pats)
    path = tmp_path / "ix.b200sa"
    idx.save(str(path))
    back = engine.SuffixArrayIndex.load(str(path))
    for a, b in ((idx.matching_stats(pat, off), back.matching_stats(pat, off)),
                 (idx.smems(pat, off, min_len=3), back.smems(pat, off, min_len=3))):
        assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    back.close()
    idx.close()


def test_errors(engine, oracle):
    lib = engine.load()
    codes = oracle.random_codes(1000, 4, seed=1)
    idx = engine.SuffixArrayIndex.build(codes[:-1], 5)
    p = codes[10:30].copy()
    off = np.array([0, 20], np.uint64)
    err = C.c_int(-1)

    def smem_call(h, pat, offp, npat, min_len):
        err.value = -1
        r = lib.b200sa_smem_batch(h, pat, offp, 0, npat, min_len, C.byref(err))
        if r:
            lib.b200sa_smem_free(r)
        return r, err.value

    pp, op = C.c_void_p(p.ctypes.data), C.c_void_p(off.ctypes.data)
    assert smem_call(idx._h, pp, op, 1, 0) == (None, 2)                 # min_len = 0
    assert smem_call(None, pp, op, 1, 1) == (None, 2)                   # no index
    assert smem_call(idx._h, None, op, 1, 1) == (None, 2)               # no patterns
    ok, code = smem_call(idx._h, pp, op, 1, 1)
    assert ok and code == 0
    out = np.zeros(20, np.uint32)
    assert lib.b200sa_matching_stats(idx._h, pp, op, 0, 1, None, None, None) == 2  # no ms buffer
    assert lib.b200sa_matching_stats(None, pp, op, 0, 1, C.c_void_p(out.ctypes.data), None, None) == 2
    assert lib.b200sa_matching_stats(idx._h, None, op, 0, 1, C.c_void_p(out.ctypes.data), None, None) == 2
    # L and R may be NULL
    assert lib.b200sa_matching_stats(idx._h, pp, op, 0, 1, C.c_void_p(out.ctypes.data), None, None) == 0
    assert out.tolist() == list(range(1, 21))  # a piece of the text: every prefix occurs
    with pytest.raises(engine.B200saError) as e:  # offsets that decrease
        idx.smems(p, np.array([0, 20, 10], np.uint64))
    assert e.value.code == 2
    with pytest.raises(engine.B200saError) as e:
        idx.smems(p, off, min_len=0)
    assert e.value.code == 2
    idx.close()
    plain = engine.SuffixArrayIndex.build(codes[:-1], 5, occ=False)  # no O table
    with pytest.raises(engine.B200saError) as e:
        plain.smems(p, off)
    assert e.value.code == 5
    with pytest.raises(engine.B200saError) as e:
        plain.matching_stats(p, off)
    assert e.value.code == 5
    plain.close()
