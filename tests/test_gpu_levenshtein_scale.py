"""Edit-distance search (b200sa_levenshtein_batch) at the shapes where its host and launch logic branch, compared
exactly and in order (offsets, L, R, length, edits) with the pigeonhole oracle of _levenshtein_oracle.py:

* walks split over several launches (a launch holds max(1024, 2^30 / (20 (max_m + 2k + 2))) work units, a unit being
  one (pattern, search) pair, npat (k + 1) in all): patterns of 65 000 symbols next to 3 000 reads;
* host batches cut into pieces of 64 MiB of pattern symbols: 700 000 reads of 100 bp;
* the raw-hit sort at 6 and 7 radix passes (keys of 36 + ceil(log2 npat) bits, 8-bit digits);
* runs of more than two raw hits merged into one: an exact occurrence at k = 3 is found by all four searches.

The texts of test_gpu_hamming_scale.py: random DNA and repeat-rich DNA of 2^20 symbols and a 20-letter text of 2^18,
each on the plain O-table index pair and on the pair built with TEXTCMP (+ KTABLE on DNA)."""
import numpy as np
import pytest

from _levenshtein_oracle import pigeonhole_hits
from test_gpu_hamming import _concat, _offsets
from test_gpu_hamming_scale import MAX_M, Text, piece_ends
from test_gpu_levenshtein import COLS, edited, patterns

pytestmark = pytest.mark.gpu


def launch_units(max_m, k):
    """Work units per launch of the walk (levenshtein_walk in levenshtein.cu)."""
    return max(1024, (1 << 30) // ((max_m + 2 * k + 2) * 20))


def sort_passes(npat):
    return (36 + max(0, int(npat - 1).bit_length()) + 7) // 8


@pytest.fixture(scope="module")
def texts(oracle):
    made = {}

    def get(name):
        if name not in made:
            made[name] = Text(oracle, name)
        return made[name]
    return get


def expect_equal(res, want, what):
    assert np.array_equal(res["offsets"].astype(np.int64), want[0]), what
    for name, w in zip(COLS[1:], want[1:]):
        assert np.array_equal(res[name].astype(np.int64), w), (what, name)


def drawn_reads(rng, codes, sigma, nreads, m, k):
    """Reads of m symbols: 90 % pieces of the text with 0 .. k edits (substitutions, insertions, deletions; the
    piece is cut so the read keeps m symbols), 10 % random; as (codes, offsets)."""
    n, nsym = len(codes) - 1, sigma - 1
    start = rng.integers(k, n - m - k, nreads)
    win = codes[start[:, None] + np.arange(m + k)]
    rand = rng.random(nreads) < 0.1
    win[rand] = rng.integers(1, nsym + 1, (int(rand.sum()), m + k))
    nedit = rng.integers(0, k + 1, nreads)
    pats = win[:, :m].copy()
    for r in np.nonzero((nedit > 0) & ~rand)[0].tolist():
        pats[r] = edited(rng, win[r], nsym, int(nedit[r]))[:m]
    return pats.reshape(-1).astype(np.uint8), np.arange(nreads + 1, dtype=np.uint64) * m


def count_launches(lib, call):
    before = int(lib.b200sa_launch_count())
    res = call()
    return res, int(lib.b200sa_launch_count()) - before


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("name", ["dna", "dna_repeats", "byte20"])
def test_split_walks(engine, texts, name, k):
    """Patterns of 65 000 symbols, the longest taken, among ~3 000 reads: each walk runs as 6 or 12 launches, two
    more per walk than the same reads take without the long patterns."""
    lib = engine.load()
    t = texts(name)
    codes, sigma = t.codes, t.sigma
    n = len(codes) - 1
    rng = np.random.default_rng(100 * k + sigma)
    short = patterns(rng, codes, sigma, 3000, 100, 100, k)
    s = int(rng.integers(0, n - MAX_M - k))
    long_drawn = edited(rng, codes[s:s + MAX_M], sigma - 1, k)[:MAX_M]
    long_random = rng.integers(1, sigma, MAX_M).astype(np.uint8)
    pats = short[:1000] + [long_drawn] + short[1000:] + [long_random]
    pat, off = _concat(pats), _offsets(pats)
    units = len(pats) * (k + 1)
    launches = -(-units // launch_units(MAX_M, k))
    assert launches == (6 if k == 1 else 12) and launch_units(MAX_M, k) == 1024
    assert len(short) * (k + 1) <= launch_units(100, k)  # (without them: one launch a walk)
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    assert want[0][1001] - want[0][1000] >= 1  # the long drawn pattern is found
    spat, soff = _concat(short + [short[0]] * 2), _offsets(short + [short[0]] * 2)
    for idx, rev in t.pairs(engine):
        _, base = count_launches(lib, lambda: idx.levenshtein_search(spat, soff, max_edits=k, rev=rev))
        res, used = count_launches(lib, lambda: idx.levenshtein_search(pat, off, max_edits=k, rev=rev))
        expect_equal(res, want, (name, k, launches))
        assert used - base == 2 * (launches - 1), (used, base, launches)
        idx.close()
        rev.close()


@pytest.mark.parametrize("form", ["fixed_len", "offsets"])
def test_pieces(engine, texts, form):
    """700 000 reads of 100 bp at k = 1: two pieces of the host batch, several launches in each, and raw-hit sorts
    of 7 passes.  The offsets CSR runs on across the piece boundary."""
    t = texts("dna")
    k, nreads, m = 1, 700_000, 100
    rng = np.random.default_rng(7 if form == "fixed_len" else 8)
    pat, off = drawn_reads(rng, t.codes, t.sigma, nreads, m, k)
    ends = piece_ends(np.full(nreads, m), m if form == "fixed_len" else 0)
    assert len(ends) == 2, ends
    q1 = ends[0]
    assert [sort_passes(p) for p in (q1, nreads - q1)] == [7, 7]
    assert q1 * (k + 1) > 2 * launch_units(m, k)  # the first piece takes several launches
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    # both pieces have hits, so a missing rebase of the second piece's offsets would show
    assert want[0][q1] > 0 and want[0][-1] > want[0][q1]
    call = dict(fixed_len=m) if form == "fixed_len" else dict(offsets=off)
    first = None
    for idx, rev in t.pairs(engine):
        res = idx.levenshtein_search(pat, max_edits=k, rev=rev, **call)
        if first is None:
            expect_equal(res, want, form)
            first = res
        else:
            assert all(np.array_equal(first[c], res[c]) for c in COLS)
        idx.close()
        rev.close()


@pytest.mark.parametrize("npat", [257, 65537])
def test_sort_widths(engine, texts, npat):
    """One piece of 257 or 65 537 patterns: 9 or 17 pattern bits in the sort key, 6 or 7 radix passes."""
    t = texts("dna")
    k = 2
    rng = np.random.default_rng(npat)
    pat, off = drawn_reads(rng, t.codes, t.sigma, npat, 100, k)
    assert len(piece_ends(np.full(npat, 100))) == 1
    assert sort_passes(npat) == (6 if npat == 257 else 7)
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    assert want[0][-1] > npat
    for idx, rev in t.pairs(engine):
        expect_equal(idx.levenshtein_search(pat, off, max_edits=k, rev=rev), want, npat)
        expect_equal(idx.levenshtein_search(pat, fixed_len=100, max_edits=k, rev=rev), want, npat)
        idx.close()
        rev.close()


@pytest.mark.parametrize("name", ["dna_repeats", "byte20"])
def test_merged_runs(engine, texts, name):
    """k = 3: a string that holds the whole pattern is found by each of the four searches, and on the repeat-rich
    text a part also recurs inside a hit, so runs of three and more raw hits merge into one hit."""
    t = texts(name)
    k = 3
    rng = np.random.default_rng(33)
    pat, off = drawn_reads(rng, t.codes, t.sigma, 3000, 40, k)
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    assert (want[4] == 0).sum() > 500  # exact occurrences: four raw hits each
    for idx, rev in t.pairs(engine):
        expect_equal(idx.levenshtein_search(pat, off, max_edits=k, rev=rev), want, name)
        idx.close()
        rev.close()
