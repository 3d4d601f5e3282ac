"""Matching statistics and SMEMs (b200sa_matching_stats, b200sa_smem_batch) at the shapes where the host entry points
and the text comparisons branch:

* a batch of ~460 000 reads of 150 bp, which the host cuts into two pieces of 64 MiB of pattern symbols (the
  per-piece offset rebasing of the SMEM CSR and the `+ b0` of the ms arrays), on random DNA of 2^22 symbols.  The
  dense-table oracle of test_gpu_mems.py is too slow at this size, so ms is checked through its characterisation at
  every end of every read within 2 000 reads of the piece boundary and of a 1 % sample: P[j - ms + 1 .. j] has exactly
  the returned (L, R) and occurs (or ms = 0 and (L, R) = (1, 0)), and P[j - ms .. j] does not occur, where it exists.
  Both are searched with the CPU restatement oracle.search_ck.  The SMEM list of the whole batch equals the one the
  rule of include/b200sa.h derives from the returned ms arrays.
* patterns of 5 000 symbols that are long pieces of a 2^16-symbol text (its start, its end, and its end followed by
  its start), so the unique-interval text comparisons run over long spans and down to suffix 0; compared with the
  dense-table recurrence, all ends at once."""
import os

import numpy as np
import pytest

from test_gpu_hamming_scale import piece_ends
from test_gpu_mems import BUILDS, _concat, _offsets, _patterns, oracle_ms, oracle_smems

pytestmark = pytest.mark.gpu

NEAR = 2000  # reads on each side of a piece boundary whose every end is checked


def smems_from_ms(off, ms, L, R, min_len):
    """The SMEM list of a batch from its ms arrays: end j of a pattern is one when ms[j] >= min_len and j is the last
    end or ms[j + 1] <= ms[j].  Returns (offsets, start, length, L, R) of int64."""
    off = off.astype(np.int64)
    ms = ms.astype(np.int64)
    total = int(off[-1])
    last = np.zeros(total, bool)
    lens = np.diff(off)
    last[off[1:][lens > 0] - 1] = True
    nxt = np.append(ms[1:], 0)
    sel = np.nonzero((ms >= min_len) & (last | (nxt <= ms)))[0]
    q = np.searchsorted(off, sel, "right") - 1
    counts = np.bincount(q, minlength=len(off) - 1)
    return (np.concatenate([[0], np.cumsum(counts)]), sel - off[q] + 1 - ms[sel], ms[sel],
            L[sel].astype(np.int64), R[sel].astype(np.int64))


def check_smems(res, off, st, min_len, what):
    want = smems_from_ms(off, st["ms"], st["L"], st["R"], min_len)
    for name, w in zip(("offsets", "start", "length", "L", "R"), want):
        assert np.array_equal(res[name].astype(np.int64), w), (what, name)


def substrings(pat, begin, length):
    """The concatenated strings pat[begin .. begin + length) and their offsets."""
    offs = np.concatenate([[0], np.cumsum(length)]).astype(np.uint64)
    rows = np.repeat(np.arange(len(begin)), length)
    return pat[np.repeat(begin, length) + np.arange(int(offs[-1])) - offs[:-1][rows].astype(np.int64)], offs


def check_characterisation(oracle, c, bwt, ck, pat, off, st, reads):
    """ms / L / R at every end of the given reads against their characterisation, searched on the CPU."""
    off = off.astype(np.int64)
    lens = off[reads + 1] - off[reads]
    g = np.repeat(off[reads], lens) + np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
    j = g - np.repeat(off[reads], lens)
    ms, L, R = (st[x].astype(np.int64) for x in ("ms", "L", "R"))
    v = ms[g]
    assert (v <= j + 1).all()
    zero = v == 0
    assert (L[g[zero]] == 1).all() and (R[g[zero]] == 0).all()
    threads = os.cpu_count() or 1
    # the match: exactly the returned interval, and not empty
    gm = g[~zero]
    cat, so = substrings(pat, gm - v[~zero] + 1, v[~zero])
    Lm, Rm = oracle.search_ck(c, bwt, ck, 64, cat, so, threads=threads)
    assert np.array_equal(Lm, L[gm]) and np.array_equal(Rm, R[gm])
    assert (Lm < Rm).all()
    # one more symbol to the left, where the pattern has one: no occurrence
    ext = v <= j
    ge = g[ext]
    cat, so = substrings(pat, ge - v[ext], v[ext] + 1)
    Le, Re = oracle.search_ck(c, bwt, ck, 64, cat, so, threads=threads)
    assert (Le >= Re).all()
    return int(len(g)), int(ext.sum())


@pytest.fixture(scope="module")
def batch(oracle):
    """Random DNA of 2^22 symbols with its CPU search tables, and ~460 000 reads of 150 bp with edits in both forms."""
    codes = oracle.random_codes(1 << 22, 4, seed=4022)
    sa = oracle.sa(codes)
    bwt = oracle.bwt(codes, sa)
    rng = np.random.default_rng(22)
    pats = _patterns(rng, codes, 460_000, 150, 150, 1, 4)
    fixed = np.stack([p[:150] if len(p) >= 150 else np.concatenate([p, np.ones(150 - len(p), np.uint8)])
                      for p in pats]).reshape(-1)
    return {"codes": codes, "c": oracle.c_table(codes, 5), "bwt": bwt, "ck": oracle.o_checkpoints(bwt, 5, 64),
            "forms": {"offsets": (_concat(pats), _offsets(pats)),
                      "fixed_len": (fixed, np.arange(0, len(fixed) + 1, 150, dtype=np.uint64))},
            "rng": rng, "verified": {}}


@pytest.mark.parametrize("form", ["offsets", "fixed_len"])
@pytest.mark.parametrize("build", list(BUILDS))
def test_pieces(engine, oracle, batch, build, form):
    """Two pieces of the host batch: ms / L / R by their characterisation around the piece boundary and on a sample
    (the same arrays on every build), and the SMEM list of every read as the rule derives it from them."""
    pat, off = batch["forms"][form]
    npat = len(off) - 1
    call = dict(offsets=off) if form == "offsets" else dict(fixed_len=150)
    ends = piece_ends(np.diff(off.astype(np.int64)), 150 if form == "fixed_len" else 0)
    assert len(ends) == 2, ends
    q1 = ends[0]
    idx = engine.SuffixArrayIndex.build(batch["codes"][:-1], 5, **BUILDS[build])
    st = idx.matching_stats(pat, **call)
    if form in batch["verified"]:
        for name in ("ms", "L", "R"):
            assert np.array_equal(st[name], batch["verified"][form][name]), (build, form, name)
    else:
        reads = np.union1d(np.arange(q1 - NEAR, q1 + NEAR), batch["rng"].choice(npat, npat // 100, replace=False))
        ends_checked, ext_checked = check_characterisation(oracle, batch["c"], batch["bwt"], batch["ck"], pat, off,
                                                           st, reads)
        assert ends_checked == int(np.diff(off.astype(np.int64))[reads].sum()) and ext_checked > 0
        batch["verified"][form] = st
    for min_len in (1, 20):
        res = idx.smems(pat, min_len=min_len, **call)
        assert int(res["offsets"][q1]) > 0 and int(res["offsets"][-1]) > int(res["offsets"][q1])
        check_smems(res, off, st, min_len, (build, form, min_len))
    idx.close()


def oracle_ms_all_ends(c, o, length, p):
    """oracle_ms of test_gpu_mems.py, every end of p stepping at once."""
    m, sigma = len(p), len(c)
    c, o, p = np.asarray(c, np.int64), np.asarray(o, np.int64), np.asarray(p, np.int64)
    j = np.arange(m)
    lo, hi, k = np.zeros(m, np.int64), np.full(m, length, np.int64), np.zeros(m, np.int64)
    active = np.ones(m, bool)
    for i in range(m):
        at = np.nonzero(active & (j >= i))[0]
        if not len(at):
            break
        a = p[at - i]
        letter = (a > 0) & (a < sigma)
        a = np.where(letter, a, 0)
        nl, nr = c[a] + o[lo[at], a], c[a] + o[hi[at], a]
        ok = letter & (nl < nr)
        active[at[~ok]] = False
        at, nl, nr = at[ok], nl[ok], nr[ok]
        lo[at], hi[at], k[at] = nl, nr, k[at] + 1
    return k.astype(np.uint32), np.where(k > 0, lo, 1).astype(np.uint32), np.where(k > 0, hi, 0).astype(np.uint32)


@pytest.mark.parametrize("build", list(BUILDS))
def test_long_pieces_of_the_text(engine, oracle, build):
    """5 000-symbol copies of the start and of the end of a 2^16-symbol text, and its last 2 500 symbols followed by
    its first 2 500, which ms splits at the seam; both entry points, both pattern forms."""
    n = 1 << 16
    codes = oracle.random_codes(n, 4, seed=516)
    sa = oracle.sa(codes)
    c, o = oracle.c_table(codes, 5), oracle.o_table(oracle.bwt(codes, sa), 5)
    text = codes[:-1]
    pats = [text[:5000].copy(), text[n - 5000:].copy(), np.concatenate([text[n - 2500:], text[:2500]])]
    # the all-ends recurrence is oracle_ms itself, on shorter patterns
    rng = np.random.default_rng(1)
    for p in _patterns(rng, codes, 6, 1, 300, 1, 4) + [text[:300].copy(), np.array([1, 0, 2, 7, 3], np.uint8)]:
        assert all(np.array_equal(a, b) for a, b in zip(oracle_ms_all_ends(c, o, len(codes), p),
                                                        oracle_ms(c.tolist(), o.tolist(), len(codes), p)))
    expect = [oracle_ms_all_ends(c, o, len(codes), p) for p in pats]
    assert expect[0][0].tolist() == list(range(1, 5001))  # (every prefix of the text occurs)
    assert int(expect[2][0][2499]) == 2500 and int(expect[2][0][-1]) == 2500
    assert int(expect[2][0][2500]) < 50  # the seam: the text's last symbol and its first do not meet
    idx = engine.SuffixArrayIndex.build(text, 5, **BUILDS[build])
    pat = _concat(pats)
    for form in (dict(offsets=_offsets(pats)), dict(fixed_len=5000)):
        st = idx.matching_stats(pat, **form)
        for k, name in enumerate(("ms", "L", "R")):
            assert np.array_equal(st[name], np.concatenate([e[k] for e in expect])), (name, list(form))
        for min_len in (1, 100):
            res = idx.smems(pat, min_len=min_len, **form)
            want = [oracle_smems(*e, min_len) for e in expect]
            assert res["offsets"].tolist() == np.cumsum([0] + [len(w) for w in want]).tolist(), (min_len, list(form))
            got = list(zip(res["start"].tolist(), res["length"].tolist(), res["L"].tolist(), res["R"].tolist()))
            assert got == [s for w in want for s in w], (min_len, list(form))
    idx.close()
