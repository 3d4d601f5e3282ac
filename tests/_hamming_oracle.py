"""Two oracles of the k-mismatch search (b200sa_hamming_batch), stated without FM machinery (TEST INFRASTRUCTURE).

The hits of a pattern P of m symbols are the distinct text strings Q of length m with Hamming(P, Q) <= k, each as
(L, R, d): L = min ISA[s] over the positions s of Q, R = L + the number of those positions, d = Hamming(P, Q); sorted
by L.  ``codes`` holds the text and its trailing 0; ``isa`` is the oracle's inverse suffix array.

* ``oracle_hits``: every window of the text against P, O(n m) per pattern.
* ``pigeonhole_hits``: a Q at distance <= k from P agrees exactly with at least one of P's k + 1 parts (the split of
  ``part_start`` in hamming.cu).  A sorted table of the text's q-grams gives, for each part that holds letters only,
  the windows that agree with the part on its first min(len, q) symbols; each candidate window is compared with P in
  full.  Batches of 10^5 patterns on 2^20-symbol texts take seconds.
"""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

ROWS = 1 << 24  # symbols compared per numpy step


def oracle_hits(codes, isa, p, k):
    """[(L, R, d)] of pattern p with at most k mismatches, by a scan of every window."""
    n, m = len(codes) - 1, len(p)
    if m == 0 or m > n:
        return []
    win = sliding_window_view(codes[:n], m)
    dist = (win != np.asarray(p, np.uint8)).sum(axis=1)
    sel = np.nonzero(dist <= k)[0]
    if not len(sel):
        return []
    _, first, inv, cnt = np.unique(win[sel], axis=0, return_index=True, return_inverse=True, return_counts=True)
    L = np.full(len(cnt), np.iinfo(np.int64).max, np.int64)
    np.minimum.at(L, inv.reshape(-1), isa[sel].astype(np.int64))
    d = dist[sel][first]
    return sorted(zip(L.tolist(), (L + cnt).tolist(), d.tolist()))


def part_bounds(m, k):
    """(start, length) of the k + 1 parts of a pattern of m symbols: floor(m / (k + 1)) or one more, longer first."""
    m = np.asarray(m, np.int64)
    qs, r = m // (k + 1), m % (k + 1)
    j = np.arange(k + 1, dtype=np.int64)
    st = j * qs[..., None] + np.minimum(j, r[..., None])
    en = (j + 1) * qs[..., None] + np.minimum(j + 1, r[..., None])
    return st, en - st


class QgramTable:
    """The text's q-grams, sorted: each position's next q symbols packed at ceil(log2 sigma) bits per symbol, the
    first symbol highest, 0 past the end."""

    def __init__(self, codes, sigma):
        self.codes = np.ascontiguousarray(codes, np.uint8)
        self.n = len(codes) - 1
        self.sigma = sigma
        self.bits = max(1, int(sigma - 1).bit_length())
        self.q = 64 // self.bits
        padded = np.concatenate([self.codes[:self.n], np.zeros(self.q, np.uint8)]).astype(np.uint64)
        key = np.zeros(self.n, np.uint64)
        for j in range(self.q):
            key = (key << np.uint64(self.bits)) | padded[j:j + self.n]
        self.order = np.argsort(key, kind="stable").astype(np.int64)
        self.keys = key[self.order]

    def ranges(self, pat, start, length):
        """[lo, hi) in the sorted table of the windows that agree with pat[start .. start + length) on its first
        min(length, q) symbols (length >= 1, letters only)."""
        l = np.minimum(length, self.q)
        pre = np.zeros(len(start), np.uint64)
        for j in range(self.q):
            take = j < l
            sym = pat[np.where(take, start + j, 0)].astype(np.uint64)
            pre = np.where(take, (pre << np.uint64(self.bits)) | sym, pre)
        shift = (self.bits * (self.q - l)).astype(np.uint64)
        lo_key = pre << shift
        hi_key = lo_key | ((np.uint64(1) << shift) - np.uint64(1))
        return np.searchsorted(self.keys, lo_key, "left"), np.searchsorted(self.keys, hi_key, "right")


def _distances(codes, pat, q_off, s, m):
    """Hamming distance of pattern symbols pat[q_off + 0 .. m) and text window codes[s + 0 .. m), per row."""
    out = np.empty(len(s), np.int64)
    step = max(1, ROWS // max(m, 1))
    ar = np.arange(m, dtype=np.int64)
    for a in range(0, len(s), step):
        b = min(len(s), a + step)
        out[a:b] = (codes[s[a:b, None] + ar] != pat[q_off[a:b, None] + ar]).sum(axis=1)
    return out


def _same_window(codes, s0, s1, m):
    """Whether codes[s0 .. s0 + m) equals codes[s1 .. s1 + m), per row."""
    out = np.empty(len(s0), bool)
    step = max(1, ROWS // max(m, 1))
    ar = np.arange(m, dtype=np.int64)
    for a in range(0, len(s0), step):
        b = min(len(s0), a + step)
        out[a:b] = (codes[s0[a:b, None] + ar] == codes[s1[a:b, None] + ar]).all(axis=1)
    return out


def pigeonhole_hits(table, isa, pat, offsets, k):
    """Hits of every pattern of a batch (pat: the concatenated codes, offsets[npat + 1]) as (offsets[npat + 1], L, R,
    d) of int64, each pattern's hits in ascending L -- the layout of b200sa_hamming_batch."""
    codes, n, sigma = table.codes, table.n, table.sigma
    pat = np.ascontiguousarray(pat, np.uint8)
    off = np.asarray(offsets, np.int64)
    npat = len(off) - 1
    lens = np.diff(off)
    isa = np.asarray(isa).astype(np.int64)
    bad = np.concatenate([[0], np.cumsum((pat == 0) | (pat >= sigma))])
    pig = np.nonzero((lens > k) & (lens <= n))[0]  # (m <= k: some parts are empty)
    found_q, found_L, found_R, found_d = [], [], [], []
    if len(pig):
        st, ln = part_bounds(lens[pig], k)
        pq = np.repeat(pig, k + 1)
        pst, pln = st.reshape(-1), ln.reshape(-1)
        a = off[pq] + pst
        letters = bad[a + pln] == bad[a]
        pq, pst, a, pln = pq[letters], pst[letters], a[letters], pln[letters]
        lo, hi = table.ranges(pat, a, pln)
        cnt = hi - lo
        cq = np.repeat(pq, cnt)
        at = np.repeat(lo - np.cumsum(cnt) + cnt, cnt) + np.arange(int(cnt.sum()), dtype=np.int64)
        cs = table.order[at] - np.repeat(pst, cnt)
        keep = (cs >= 0) & (cs <= n - lens[cq])
        key = np.unique(cq[keep] * (n + 1) + cs[keep])  # a window that agrees with several parts counts once
        cq, cs = key // (n + 1), key % (n + 1)
        for m in np.unique(lens[cq]).tolist():
            sel = lens[cq] == m
            q, s = cq[sel], cs[sel]
            d = _distances(codes, pat, off[q], s, m)
            ok = d <= k
            q, s, d = q[ok], s[ok], d[ok]
            r = isa[s]
            o = np.lexsort((r, q))
            q, s, d, r = q[o], s[o], d[o], r[o]
            # every occurrence of a kept string is kept (it agrees with the same part), so within a pattern the
            # windows of one string are consecutive in ISA order
            new = np.ones(len(q), bool)
            if len(q) > 1:
                new[1:] = (q[1:] != q[:-1]) | ~_same_window(codes, s[1:], s[:-1], m)
            head = np.nonzero(new)[0]
            size = np.diff(np.append(head, len(q)))
            found_q.append(q[head])
            found_L.append(r[head])
            found_R.append(r[head] + size)
            found_d.append(d[head])
    for q in np.nonzero((lens > 0) & (lens <= k))[0].tolist():
        h = oracle_hits(codes, isa, pat[off[q]:off[q + 1]], k)
        found_q.append(np.full(len(h), q, np.int64))
        found_L.append(np.array([x[0] for x in h], np.int64))
        found_R.append(np.array([x[1] for x in h], np.int64))
        found_d.append(np.array([x[2] for x in h], np.int64))
    if not found_q:
        return np.zeros(npat + 1, np.int64), *(np.zeros(0, np.int64) for _ in range(3))
    q, L, R, d = (np.concatenate(x) for x in (found_q, found_L, found_R, found_d))
    o = np.lexsort((L, q))
    out_off = np.concatenate([[0], np.cumsum(np.bincount(q, minlength=npat))])
    return out_off, L[o], R[o], d[o]
