"""k-mismatch search (b200sa_hamming_batch) at the shapes where its host and launch logic branch, compared exactly and
in order (offsets, L, R, mismatches) with the pigeonhole oracle of _hamming_oracle.py:

* walks split over several launches (a launch holds max(1024, 2^30 / (16 max_m)) work units, a unit being one
  (pattern, search) pair, npat (k + 1) in all): patterns of 65 000 symbols next to 3 000 reads;
* host batches cut into pieces of 64 MiB of pattern symbols: 700 000 reads of 100 bp;
* the hit sort at 6 and 7 radix passes (keys of 32 + ceil(log2 npat) bits, 8-bit digits).

The texts: random DNA of 2^20 symbols, a repeat-rich DNA text of 2^20 symbols (one 3 000-symbol segment tiled with
1 % substitutions: wide intervals, deep walks) and a 20-letter text of 2^18 symbols (the byte layout).  Each runs on
the plain O-table index pair and on the pair built with TEXTCMP (+ KTABLE on DNA); the results are the same."""
import numpy as np
import pytest

from _hamming_oracle import QgramTable, pigeonhole_hits
from test_gpu_hamming import _concat, _offsets, _reverse, patterns

pytestmark = pytest.mark.gpu

MAX_M = 65000
PIECE_SYMBOLS = 64 << 20


def launch_units(max_m):
    """Work units per launch of the walk (hamming_walk in hamming.cu)."""
    return max(1024, (1 << 30) // (max(max_m, 1) * 16))


def piece_ends(lens, fixed_len=0):
    """Where the host entry point cuts a batch: whole patterns of at most 64 MiB of symbols (piece_end in api.cu)."""
    npat = len(lens)
    if fixed_len:
        per = max(1, PIECE_SYMBOLS // fixed_len)
        return list(range(per, npat, per)) + [npat]
    off = np.concatenate([[0], np.cumsum(lens)])
    ends, q0 = [], 0
    while q0 < npat:
        q1 = max(q0 + 1, int(np.searchsorted(off, off[q0] + PIECE_SYMBOLS, "right")) - 1)
        ends.append(q1)
        q0 = q1
    return ends


def sort_passes(npat):
    return (32 + max(0, int(npat - 1).bit_length()) + 7) // 8


def repeat_text(rng, n, seg=3000, rate=0.01):
    base = rng.integers(1, 5, seg).astype(np.uint8)
    t = np.tile(base, n // seg + 1)[:n]
    at = np.nonzero(rng.random(n) < rate)[0]
    t[at] = (t[at] - 1 + rng.integers(1, 4, len(at))) % 4 + 1
    return np.append(t, 0).astype(np.uint8)


class Text:
    def __init__(self, oracle, name):
        rng = np.random.default_rng(20)
        if name == "dna":
            self.codes, self.sigma = oracle.random_codes(1 << 20, 4, seed=1020), 5
        elif name == "dna_repeats":
            self.codes, self.sigma = repeat_text(rng, 1 << 20), 5
        else:
            self.codes, self.sigma = oracle.random_codes(1 << 18, 20, seed=1018), 21
        self.isa = oracle.inverse(oracle.sa(self.codes))
        self.table = QgramTable(self.codes, self.sigma)

    def pairs(self, engine):
        """(F, B) of the plain O-table build, then of the TEXTCMP (+ KTABLE) build."""
        text, rtext = self.codes[:-1], _reverse(self.codes)
        extra = {"textcmp": True, "ktable": True} if self.sigma == 5 else {"textcmp": True}
        for b in ({}, extra):
            yield (engine.SuffixArrayIndex.build(text, self.sigma, **b),
                   engine.SuffixArrayIndex.build(rtext, self.sigma, drop_sa=True, **b))


@pytest.fixture(scope="module")
def texts(oracle):
    """Each text, with its ISA and q-gram table, made once per module."""
    made = {}

    def get(name):
        if name not in made:
            made[name] = Text(oracle, name)
        return made[name]
    return get


def expect_equal(res, want, what):
    off, L, R, d = want
    assert np.array_equal(res["offsets"].astype(np.int64), off), what
    for name, w in (("L", L), ("R", R), ("mismatches", d)):
        assert np.array_equal(res[name].astype(np.int64), w), (what, name)


def drawn_reads(rng, codes, sigma, nreads, lens, k):
    """Reads of the given lengths: 90 % pieces of the text with 0 .. k + 1 substitutions, 10 % random."""
    n, nsym = len(codes) - 1, sigma - 1
    lens = np.broadcast_to(np.asarray(lens, np.int64), (nreads,))
    off = np.concatenate([[0], np.cumsum(lens)])
    q = np.repeat(np.arange(nreads), lens)
    j = np.arange(int(off[-1])) - off[q]
    start = rng.integers(0, n - lens + 1)
    pat = codes[start[q] + j].copy()
    rand = rng.random(nreads) < 0.1
    pat[rand[q]] = rng.integers(1, nsym + 1, int(rand[q].sum()))
    nsub = rng.integers(0, k + 2, nreads)
    for s in range(k + 1):  # substitution s at a distinct position of each read that has more than s
        rows = np.nonzero(nsub > s)[0]
        at = off[rows] + (rng.integers(0, lens[rows] // (k + 1), len(rows)) + s * (lens[rows] // (k + 1)))
        pat[at] = (pat[at] - 1 + rng.integers(1, nsym, len(rows))) % nsym + 1
    return pat.astype(np.uint8), off.astype(np.uint64)


@pytest.mark.parametrize("k", [1, 2, 3, 8])
@pytest.mark.parametrize("name", ["dna", "dna_repeats", "byte20"])
def test_split_walks(engine, texts, name, k):
    """Patterns of 65 000 symbols, the longest taken, among ~3 000 reads: the walk runs as 6 .. 27 launches."""
    t = texts(name)
    codes, sigma = t.codes, t.sigma
    n = len(codes) - 1
    rng = np.random.default_rng(100 * k + sigma)
    pats = patterns(rng, codes, sigma, 3000, 100, 100, k)
    s = int(rng.integers(0, n - MAX_M + 1))
    long_drawn = codes[s:s + MAX_M].copy()
    at = rng.choice(MAX_M, size=k, replace=False)
    long_drawn[at] = (long_drawn[at] - 1 + rng.integers(1, sigma - 1, k)) % (sigma - 1) + 1
    long_random = rng.integers(1, sigma, MAX_M).astype(np.uint8)
    pats[1000:1000] = [long_drawn]
    pats.append(long_random)
    pat, off = _concat(pats), _offsets(pats)
    units = len(pats) * (k + 1)
    launches = -(-units // launch_units(MAX_M))
    assert 6 <= launches <= 27 and launch_units(MAX_M) == 1032
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    assert want[0][1001] - want[0][1000] >= 1  # the long drawn pattern is found
    for idx, rev in t.pairs(engine):
        expect_equal(idx.hamming_search(pat, off, max_mismatches=k, rev=rev), want, (name, k, launches))
        idx.close()
        rev.close()


@pytest.mark.parametrize("form", ["fixed_len", "offsets"])
def test_pieces(engine, texts, form):
    """700 000 reads of 100 bp (or 90 .. 110) at k = 2: two pieces of the host batch, several launches in each, and
    hit sorts of 7 and 6 passes.  The offsets CSR runs on across the piece boundary."""
    t = texts("dna")
    k, nreads = 2, 700_000
    rng = np.random.default_rng(7 if form == "fixed_len" else 8)
    lens = 100 if form == "fixed_len" else rng.integers(90, 111, nreads)
    pat, off = drawn_reads(rng, t.codes, t.sigma, nreads, lens, k)
    lens = np.diff(off.astype(np.int64))
    ends = piece_ends(lens, 100 if form == "fixed_len" else 0)
    assert len(ends) == 2, ends
    q1 = ends[0]
    per_piece = [q1, nreads - q1]
    assert [sort_passes(p) for p in per_piece] == [7, 6]
    assert q1 * (k + 1) > 2 * launch_units(int(lens.max()))  # the first piece takes several launches
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    # both pieces have hits, so a missing rebase of the second piece's offsets would show
    assert want[0][q1] > 0 and want[0][-1] > want[0][q1]
    call = dict(fixed_len=100) if form == "fixed_len" else dict(offsets=off)
    first = None
    for idx, rev in t.pairs(engine):
        res = idx.hamming_search(pat, max_mismatches=k, rev=rev, **call)
        assert int(res["offsets"][q1]) == int(want[0][q1])
        assert np.all(np.diff(res["offsets"].astype(np.int64)) >= 0)
        if first is None:
            expect_equal(res, want, form)
            first = res
        else:
            assert all(np.array_equal(first[c], res[c]) for c in ("offsets", "L", "R", "mismatches"))
        idx.close()
        rev.close()


@pytest.mark.parametrize("npat", [257, 65537])
def test_sort_widths(engine, texts, npat):
    """One piece of 257 or 65 537 patterns: 9 or 17 pattern bits in the sort key, 6 or 7 radix passes."""
    t = texts("dna")
    k = 1
    rng = np.random.default_rng(npat)
    pat, off = drawn_reads(rng, t.codes, t.sigma, npat, 100, k)
    assert len(piece_ends(np.diff(off.astype(np.int64)))) == 1
    assert sort_passes(npat) == (6 if npat == 257 else 7)
    want = pigeonhole_hits(t.table, t.isa, pat, off, k)
    assert want[0][-1] > npat // 2
    for idx, rev in t.pairs(engine):
        expect_equal(idx.hamming_search(pat, off, max_mismatches=k, rev=rev), want, npat)
        expect_equal(idx.hamming_search(pat, fixed_len=100, max_mismatches=k, rev=rev), want, npat)
        idx.close()
        rev.close()
