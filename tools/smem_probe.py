"""SMEM seeding of divergent reads on a 3 Gbp synthetic DNA index (b200sa_smem_batch); one JSON line.

The index: b200sa_synth_codes text, OCC + TEXTCMP + KTABLE.  The reads: 150 bp, 90 % drawn from the text with about
2 % substitutions and 0.2 % indels, 10 % random.  Recorded: device time of the matching-statistics pass
(mems_stats_kernel) and of the emit pass (mems_emit_kernel), from torch.profiler's CUDA activity records of one warm
call; wall time of the warm host call (reads in, SMEMs out); SMEMs per read; the card and its power limit.  On a
subsample every SMEM's (L, R) is checked against b200sa_search_batch on its substring.

    python tools/smem_probe.py [--n 3000000000] [--reads 1000000] [--approx-d2 0] [--out FILE]
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


def make_reads(text, n, nreads, m, rng):
    """(nreads, m) uint8 codes: 90 % from the text with substitutions (2 %) and indels (0.2 %), 10 % random."""
    pad = 16
    nsamp = nreads * 9 // 10
    starts = torch.from_numpy(rng.integers(0, n - m - pad, nsamp)).cuda()
    win = text[starts[:, None] + torch.arange(m + pad, device="cuda")[None, :]].cpu().numpy()
    sub = rng.random(win.shape) < 0.02
    win[sub] = (win[sub] - 1 + rng.integers(1, 4, int(sub.sum()))) % 4 + 1  # another letter
    out = np.empty((nreads, m), np.uint8)
    nindel = rng.poisson(0.002 * m, nsamp)
    for q in range(nsamp):
        row = win[q]
        for _ in range(int(nindel[q])):
            at = int(rng.integers(0, m))
            if rng.random() < 0.5:
                row = np.insert(row, at, np.uint8(rng.integers(1, 5)))
            else:
                row = np.delete(row, at)
        out[q] = row[:m]
    out[nsamp:] = rng.integers(1, 5, (nreads - nsamp, m))
    return out[rng.permutation(nreads)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def kernel_ms(idx, reads, m):
    """Device time per kernel name (ms) of one smems call, from the profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        idx.smems(reads, fixed_len=m, min_len=19)
        torch.cuda.synchronize()
    t = {}
    for ev in prof.key_averages():
        for k in ("mems_stats_kernel", "mems_emit_kernel", "scan_sum_kernel"):
            if k in ev.key:
                t[k] = t.get(k, 0.0) + ev.device_time_total / 1e3
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=150)
    ap.add_argument("--min-len", type=int, default=19)
    ap.add_argument("--check", type=int, default=2000, help="reads whose SMEMs are checked against exact search")
    ap.add_argument("--approx-d2", type=int, default=0, help="also time approximate search at d = 2 on this many reads")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = stralg_b200.load()
    n, m = args.n, args.m
    text = torch.empty(n + 1, dtype=torch.uint8, device="cuda")
    stralg_b200._lib.check(lib.b200sa_synth_codes(C.c_void_p(text.data_ptr()), n, 4, 1, 0, None))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    idx = stralg_b200.SuffixArrayIndex.build(text[:n], 5, textcmp=True, ktable=True)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    rng = np.random.default_rng(7)
    reads = make_reads(text, n, args.reads, m, rng).reshape(-1)
    del text
    flat = np.ascontiguousarray(reads)
    idx.smems(flat, fixed_len=m, min_len=args.min_len)  # warm-up: the same batch (pool growth, first launches)
    t0 = time.perf_counter()
    res = idx.smems(flat, fixed_len=m, min_len=args.min_len)
    wall = time.perf_counter() - t0
    kt = kernel_ms(idx, flat, m)
    nsm = len(res["start"])
    # every SMEM of the first reads: exact search of its substring gives its (L, R)
    k = min(args.check, args.reads)
    h1 = int(res["offsets"][k])
    q_of = np.repeat(np.arange(k), np.diff(res["offsets"][: k + 1]).astype(np.int64))
    subs = [flat[q * m + s: q * m + s + ln] for q, s, ln in zip(q_of, res["start"][:h1], res["length"][:h1])]
    off = np.zeros(len(subs) + 1, np.uint64)
    off[1:] = np.cumsum([len(x) for x in subs])
    L, R = idx.search(np.concatenate(subs), off)
    checked = bool(np.array_equal(L, res["L"][:h1]) and np.array_equal(R, res["R"][:h1]))
    name, pl = card()
    out = {
        "probe": "smem", "card": name, "power_limit": pl, "n": n, "reads": args.reads, "read_len": m,
        "min_len": args.min_len, "flags": "OCC+TEXTCMP+KTABLE", "ktable_k": idx.stats()["ktable_k"],
        "build_s": round(build_s, 3),
        "stats_pass_ms": round(kt.get("mems_stats_kernel", float("nan")), 3),
        "scan_ms": round(kt.get("scan_sum_kernel", float("nan")), 3),
        "emit_pass_ms": round(kt.get("mems_emit_kernel", float("nan")), 3),
        "device_reads_per_s": round(args.reads / ((kt.get("mems_stats_kernel", 0) + kt.get("mems_emit_kernel", 0)) / 1e3), 1),
        "host_call_s": round(wall, 4), "host_reads_per_s": round(args.reads / wall, 1),
        "smems": nsm, "smems_per_read": round(nsm / args.reads, 3),
        "checked_reads": k, "checked_smems": h1, "L_R_equal_search": checked,
    }
    if args.approx_d2:
        t0 = time.perf_counter()
        r = idx.approx_search(flat[: args.approx_d2 * m], fixed_len=m, max_edits=2)
        out["approx_d2"] = {"reads": args.approx_d2, "host_call_s": round(time.perf_counter() - t0, 3),
                            "intervals": len(r["L"])}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")
    assert checked, "SMEM intervals differ from exact search"
    idx.close()


if __name__ == "__main__":
    main()
