"""Two oracles of the edit-distance search (b200sa_levenshtein_batch), stated without FM machinery (TEST
INFRASTRUCTURE).

The hits of a pattern P of m symbols are the distinct non-empty text strings Q with ED(P, Q) <= k (unit-cost
Levenshtein distance), each as (L, R, length, d): L = min ISA[s] over the positions s of Q, R = L + the number of
those positions, length = |Q|, d = ED(P, Q); sorted by (L, length).  ``codes`` holds the text and its trailing 0;
``isa`` is the oracle's inverse suffix array.

* ``oracle_hits``: for every start s, a banded DP of P against T[s .. s + m + k), one text symbol per numpy step over
  all starts at once; it gives ED(P, T[s .. s + l)) for every length l in [m - k, m + k].  A start leaves the DP once
  its whole band exceeds k.
* ``pigeonhole_hits``: a Q at distance <= k from P holds one of P's k + 1 parts (the split of ``part_start``) exactly,
  at an offset within k of the part's offset in P.  A sorted table of the text's q-grams gives the occurrences of
  each part that holds letters only; each candidate start runs the same DP.  Batches of 10^5 patterns on 2^20-symbol
  texts take seconds.
"""
import numpy as np

from _hamming_oracle import QgramTable, part_bounds, _same_window  # noqa: F401 (QgramTable: for callers)

ROWS = 1 << 22  # pattern symbols gathered per numpy step


def _window_distances(text, pats, s, k):
    """For rows of patterns pats[r] (all of one length m) and starts s[r]: (row, length, d) of every l in
    [max(1, m - k), m + k] with s + l <= len(text) and d = ED(pats[r], text[s .. s + l)) <= k.  The DP keeps the band
    of 2k + 1 cells around the diagonal (cell b after l text symbols: the pattern prefix of l + b - k symbols),
    saturated at k + 1."""
    n = len(text)
    rows, m = pats.shape
    sat, W = k + 1, 2 * k + 1
    b = np.arange(W, dtype=np.int64)
    j = b - k
    idx = np.arange(rows, dtype=np.int64)
    D = np.broadcast_to(np.where((j >= 0) & (j <= m), np.minimum(np.abs(j), sat), sat).astype(np.int16),
                        (rows, W)).copy()
    P = np.pad(pats, ((0, 0), (k + 1, 2 * k)))  # pattern symbol j - 1 of cell b after l symbols at column l + b
    out_r, out_l, out_d = [], [], []
    for l in range(1, m + k + 1):
        keep = s[idx] + l <= n
        idx, D = idx[keep], D[keep]
        if not len(idx):
            break
        c = text[s[idx] + l - 1]
        j = l + b - k
        diag = D + (P[idx[:, None], l + b] != c[:, None])
        diag[:, j < 1] = sat
        up = np.empty_like(D)
        up[:, :-1] = D[:, 1:] + 1
        up[:, -1] = sat
        D = np.minimum(diag, up)
        for a in range(1, W):  # a pattern symbol against nothing
            np.minimum(D[:, a], D[:, a - 1] + 1, out=D[:, a])
        np.minimum(D, sat, out=D)
        D[:, (j < 0) | (j > m)] = sat
        if l >= m - k:
            end = D[:, m - l + k]
            hit = end <= k
            out_r.append(idx[hit])
            out_l.append(np.full(int(hit.sum()), l, np.int64))
            out_d.append(end[hit].astype(np.int64))
        alive = D.min(axis=1) <= k
        idx, D = idx[alive], D[alive]
    if not out_r:
        return (np.zeros(0, np.int64),) * 3
    return np.concatenate(out_r), np.concatenate(out_l), np.concatenate(out_d)


def _distances(text, pat, off, q, s, m, k):
    """_window_distances in slices of about ROWS pattern symbols; q[r] is the pattern of row r (at off[q])."""
    rr, ll, dd = [], [], []
    step = max(1, ROWS // (m + 1))
    ar = np.arange(m, dtype=np.int64)
    for a in range(0, len(s), step):
        b = min(len(s), a + step)
        pats = pat[off[q[a:b], None] + ar]
        r, l, d = _window_distances(text, pats, s[a:b], k)
        rr.append(r + a)
        ll.append(l)
        dd.append(d)
    return np.concatenate(rr), np.concatenate(ll), np.concatenate(dd)


def _group(codes, isa, q, s, l, d):
    """Hits (q, L, R, length, d) from the windows (q, s, l) at distance d, which hold every occurrence of each of
    their strings; sorted by (q, L, length)."""
    r = isa[s]
    o = np.lexsort((r, l, q))
    q, s, l, d, r = q[o], s[o], l[o], d[o], r[o]
    new = np.ones(len(q), bool)
    if len(q) > 1:
        same = (q[1:] == q[:-1]) & (l[1:] == l[:-1])
        new[1:] = ~same
        for m in np.unique(l[1:][same]).tolist():
            at = np.nonzero(same & (l[1:] == m))[0] + 1
            new[at] = ~_same_window(codes, s[at], s[at - 1], m)
    head = np.nonzero(new)[0]
    size = np.diff(np.append(head, len(q)))
    q, L, R, n, dd = q[head], r[head], r[head] + size, l[head], d[head]
    o = np.lexsort((n, L, q))
    return q[o], L[o], R[o], n[o], dd[o]


def oracle_hits(codes, isa, p, k):
    """[(L, R, length, d)] of pattern p with at most k edits, by the DP from every start."""
    n, m = len(codes) - 1, len(p)
    if m == 0:
        return []
    isa = np.asarray(isa).astype(np.int64)
    s = np.arange(n, dtype=np.int64)
    pat = np.asarray(p, np.uint8)
    r, l, d = _distances(codes[:n], pat, np.zeros(1, np.int64), np.zeros(n, np.int64), s, m, k)
    _, L, R, ln, dd = _group(codes, isa, np.zeros(len(r), np.int64), s[r], l, d)
    return list(zip(L.tolist(), R.tolist(), ln.tolist(), dd.tolist()))


def pigeonhole_hits(table, isa, pat, offsets, k):
    """Hits of every pattern of a batch (pat: the concatenated codes, offsets[npat + 1]) as (offsets[npat + 1], L, R,
    length, d) of int64, each pattern's hits in ascending (L, length) -- the layout of b200sa_levenshtein_batch."""
    codes, n, sigma = table.codes, table.n, table.sigma
    pat = np.ascontiguousarray(pat, np.uint8)
    off = np.asarray(offsets, np.int64)
    npat = len(off) - 1
    lens = np.diff(off)
    isa = np.asarray(isa).astype(np.int64)
    bad = np.concatenate([[0], np.cumsum((pat == 0) | (pat >= sigma))])
    found = []
    pig = np.nonzero(lens > k)[0]  # (m <= k: some parts are empty)
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
        c0 = table.order[at] - np.repeat(pst, cnt)
        # the part at offset o of Q: Q starts k or fewer symbols before or after where P puts it
        cq = np.repeat(cq, 2 * k + 1)
        cs = (c0[:, None] + np.arange(-k, k + 1)).reshape(-1)
        keep = (cs >= 0) & (cs < n)
        key = np.unique(cq[keep] * (n + 1) + cs[keep])
        cq, cs = key // (n + 1), key % (n + 1)
        for m in np.unique(lens[cq]).tolist():
            sel = lens[cq] == m
            q, s = cq[sel], cs[sel]
            r, l, d = _distances(codes[:n], pat, off, q, s, m, k)
            found.append((q[r], s[r], l, d))
    for q in np.nonzero((lens > 0) & (lens <= k))[0].tolist():
        s = np.arange(n, dtype=np.int64)
        r, l, d = _distances(codes[:n], pat, off, np.full(n, q, np.int64), s, int(lens[q]), k)
        found.append((np.full(len(r), q, np.int64), s[r], l, d))
    if not found:
        return np.zeros(npat + 1, np.int64), *(np.zeros(0, np.int64) for _ in range(4))
    q, s, l, d = (np.concatenate(x) for x in zip(*found))
    q, L, R, ln, dd = _group(codes, isa, q, s, l, d)
    out_off = np.concatenate([[0], np.cumsum(np.bincount(q, minlength=npat))])
    return out_off, L, R, ln, dd
