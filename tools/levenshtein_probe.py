"""Edit-distance search of short reads on a 3 Gbp synthetic DNA index pair (b200sa_levenshtein_batch); one JSON line.

The indices: b200sa_synth_codes text, OCC only, and the index of the reversed text (made on the device), OCC only
without its suffix array.  The reads: 100 bp, 90 % drawn from the text with 0 .. k edits (uniform; each edit a
substitution, an insertion or a deletion, one per k-th of the read), 10 % random.  Recorded for k = 1, 2, 3: device
time of the counting walk, the scan, the emitting walk, the sort and the merge, from torch.profiler's CUDA activity
records of one warm call; wall time of the warm host call (reads in, hits out); hits per read (after the merge).
Checked at full size: every drawn read's source window is a hit, so its origin is among the located positions of its
hits (full sensitivity); on a subsample, ED(read, T[pos .. pos + length)) is computed again at the first position of
each hit and must equal the reported distance.  As context, b200sa_hamming_batch on the same reads at the same k, and
b200sa_approx_batch at d = 1 and 2 on the first 10^4 reads.

    python tools/levenshtein_probe.py [--n 3000000000] [--reads 1000000] [--ks 1,2,3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import stralg_b200


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def make_reads(text, n, nreads, m, k, rng):
    """(reads (nreads * m,) uint8, origin per read or -1 for a random read).  Edit j of a read lies in the j-th k-th
    of it: a substitution replaces the source letter, an insertion puts a random letter before the source letter,
    a deletion skips one."""
    nsamp = nreads * 9 // 10
    starts = rng.integers(0, n - m - k, nsamp)
    nedit = rng.integers(0, k + 1, nsamp)
    step = np.zeros((nsamp, m + 1), np.int64)  # source offset increments, by read column
    fresh = np.zeros((nsamp, m), bool)          # read columns that take a random or another letter
    sub = np.zeros((nsamp, m), bool)
    seg = m // max(k, 1)
    for j in range(k):
        rows = np.nonzero(nedit > j)[0]
        at = rng.integers(0, seg, len(rows)) + j * seg
        kind = rng.integers(0, 3, len(rows))
        ins, dele = rows[kind == 1], rows[kind == 2]
        fresh[ins, at[kind == 1]] = True
        step[ins, at[kind == 1] + 1] -= 1
        step[dele, at[kind == 2]] += 1
        sub[rows[kind == 0], at[kind == 0]] = True
    src = np.arange(m)[None, :] + np.cumsum(step, axis=1)[:, :m]
    win = text[torch.from_numpy(starts).cuda()[:, None] + torch.from_numpy(src).cuda()].cpu().numpy()
    win[sub] = (win[sub] - 1 + rng.integers(1, 4, int(sub.sum()))) % 4 + 1  # another letter
    win[fresh] = rng.integers(1, 5, int(fresh.sum()))
    out = np.empty((nreads, m), np.uint8)
    out[:nsamp] = win
    out[nsamp:] = rng.integers(1, 5, (nreads - nsamp, m))
    origin = np.full(nreads, -1, np.int64)
    origin[:nsamp] = starts
    perm = rng.permutation(nreads)
    return np.ascontiguousarray(out[perm].reshape(-1)), origin[perm]


def edit_distance(P, W, wlen):
    """ED(P[r], W[r, :wlen[r]]) per row, by the full DP vectorised over rows."""
    rows, m = P.shape
    j = np.arange(m + 1)
    D = np.broadcast_to(j, (rows, m + 1)).copy()
    out = np.where(wlen == 0, m, 0)
    for l in range(1, W.shape[1] + 1):
        base = np.empty_like(D)
        base[:, 0] = l
        base[:, 1:] = np.minimum(D[:, 1:] + 1, D[:, :-1] + (P != W[:, l - 1:l]))
        D = np.minimum.accumulate(base - j, axis=1) + j
        out = np.where(wlen == l, D[:, m], out)
    return out


WALK = "levenshtein_walk_kernel"


def kernel_ms(fn):
    """Device time (ms) by stage of one call, from the profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    t = {"count": 0.0, "scan": 0.0, "emit": 0.0, "sort": 0.0, "merge": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        ms = ev.device_time_total / 1e3
        key = ev.key
        if WALK in key:
            t["emit" if "true" in key else "count"] += ms
        elif "scan_sum_kernel" in key:
            t["scan"] += ms
        elif any(s in key for s in ("onesweep_pass_kernel", "hist_kernel")):
            t["sort"] += ms
        elif "levenshtein_" in key:
            t["merge"] += ms
        elif "kernel" in key.lower():
            t["other"] += ms
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=100)
    ap.add_argument("--ks", default="1,2,3")
    ap.add_argument("--check", type=int, default=5000, help="hits whose distance is computed again against the text")
    ap.add_argument("--approx-reads", type=int, default=10000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = stralg_b200.load()
    n, m = args.n, args.m
    text = torch.empty(n + 1, dtype=torch.uint8, device="cuda")
    stralg_b200._lib.check(lib.b200sa_synth_codes(C.c_void_p(text.data_ptr()), n, 4, 1, 0, None))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    idx = stralg_b200.SuffixArrayIndex.build(text[:n], 5)
    torch.cuda.synchronize()
    rtext = torch.flip(text[:n], dims=[0]).contiguous()
    rev = stralg_b200.SuffixArrayIndex.build(rtext, 5, drop_sa=True)
    torch.cuda.synchronize()
    del rtext
    build_s = time.perf_counter() - t0
    name, pl = card()
    out = {"probe": "levenshtein", "card": name, "power_limit": pl, "n": n, "reads": args.reads, "read_len": m,
           "flags": "OCC (reverse index: OCC, DROP_SA)", "build_pair_s": round(build_s, 3), "k": {}}
    rng = np.random.default_rng(7)
    ok = True
    first_reads = None
    for k in [int(x) for x in args.ks.split(",")]:
        reads, origin = make_reads(text, n, args.reads, m, k, rng)
        if first_reads is None:
            first_reads = reads[: args.approx_reads * m].copy()
        search = lambda: idx.levenshtein_search(reads, fixed_len=m, max_edits=k, rev=rev)  # noqa: E731
        search()  # warm-up (pool growth, first launches)
        t0 = time.perf_counter()
        res = search()
        wall = time.perf_counter() - t0
        kt = kernel_ms(search)
        hits = len(res["L"])
        poff, pos = idx.locate(res["L"], res["R"])
        read_of_hit = np.repeat(np.arange(args.reads), np.diff(res["offsets"]).astype(np.int64))
        read_of_pos = np.repeat(read_of_hit, np.diff(poff).astype(np.int64))
        found = np.unique(read_of_pos.astype(np.int64) << 32 | pos.astype(np.int64))
        drawn = np.nonzero(origin >= 0)[0]
        want = drawn.astype(np.int64) << 32 | origin[drawn]
        sensitive = bool(np.isin(want, found).all())
        sel = rng.choice(hits, size=min(args.check, hits), replace=False) if hits else np.zeros(0, np.int64)
        p0 = torch.from_numpy(pos[poff[sel].astype(np.int64)].astype(np.int64)).cuda()
        win = text[torch.clamp(p0[:, None] + torch.arange(m + k, device="cuda")[None, :], max=n)].cpu().numpy()
        dist = edit_distance(reads.reshape(-1, m)[read_of_hit[sel]], win, res["length"][sel].astype(np.int64))
        d_ok = bool(np.array_equal(dist, res["edits"][sel]))
        device_ms = kt["count"] + kt["scan"] + kt["emit"] + kt["sort"] + kt["merge"]
        ham = lambda: idx.hamming_search(reads, fixed_len=m, max_mismatches=k, rev=rev)  # noqa: E731
        ham()
        t0 = time.perf_counter()
        hres = ham()
        ham_wall = time.perf_counter() - t0
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ham()
            torch.cuda.synchronize()
        ham_ms = sum(ev.device_time_total for ev in prof.key_averages() if "kernel" in ev.key.lower()) / 1e3
        out["k"][str(k)] = {
            "count_pass_ms": round(kt["count"], 3), "scan_ms": round(kt["scan"], 3), "emit_pass_ms": round(kt["emit"], 3),
            "sort_ms": round(kt["sort"], 3), "merge_ms": round(kt["merge"], 3), "other_kernels_ms": round(kt["other"], 3),
            "device_ms": round(device_ms, 3), "device_reads_per_s": round(args.reads / (device_ms / 1e3), 1),
            "host_call_s": round(wall, 4), "host_reads_per_s": round(args.reads / wall, 1),
            "hits": hits, "hits_per_read": round(hits / args.reads, 4),
            "drawn_reads": int(len(drawn)), "origin_found_for_all": sensitive,
            "distance_rechecked_hits": int(len(sel)), "distance_equal": d_ok,
            "hamming_context": {"device_ms": round(ham_ms, 3), "host_call_s": round(ham_wall, 4),
                                "hits": len(hres["L"])},
        }
        ok = ok and sensitive and d_ok
        print(json.dumps({"k": k, **out["k"][str(k)]}), file=sys.stderr, flush=True)
    out["approx_context"] = {}
    for d in (1, 2):
        idx.approx_search(first_reads[: m * 100], fixed_len=m, max_edits=d, rev=rev)
        t0 = time.perf_counter()
        r = idx.approx_search(first_reads, fixed_len=m, max_edits=d, rev=rev)
        out["approx_context"][f"d{d}"] = {"reads": args.approx_reads, "host_call_s": round(time.perf_counter() - t0, 4),
                                          "intervals": len(r["L"])}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")
    assert ok, "a drawn read's origin is missing or a distance differs"
    idx.close()
    rev.close()


if __name__ == "__main__":
    main()
