"""Records index against one index per record, on a synthetic multi-record reference.  One JSON line.

    python tools/records_probe.py [--records 10000] [--min-len 1000] [--max-len 100000]
                                  [--reads 1000000] [--reads-d1 100000]
                                  [--baseline-reads 20000] [--baseline-reads-d1 2000] [--out DIR]

Input: `--records` ACGT records of uniform random length in [min-len, max-len] (seeded), and 100 bp reads
sampled from them with about one substitution in twenty reads.

* build: one b200sa_build_records over all records against the sum of one b200sa_build per record
  (both with the O table, wall clock around the synchronous calls).
* mapping: bwt_map_fastq_records (it builds its own records index inside the call; that build is included)
  and bwt_map_fastq (one table per record, built beforehand with its reverse O rows, as `bwt_readmapper -p`
  leaves them), at d = 0 and d = 1.  bwt_map_fastq remaps and searches every batch once per record, so at
  thousands of records it maps only the first `--baseline-reads` (`--baseline-reads-d1`) reads; the records
  path maps the same prefix once more, and the two SAM outputs of that prefix are asserted identical.
  Rates are reads per second of each measured run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import stralg_b200  # noqa: E402
from _oracle import RefBwtTable, bind_stralg_api, u8p  # noqa: E402

COMPAT_SO = os.path.join(ROOT, "stralg_b200", "lib", "libstralg_b200.so")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def bind(lib):
    bind_stralg_api(lib)
    tp = C.POINTER(C.POINTER(RefBwtTable))
    for fn in ("bwt_map_fastq", "bwt_map_fastq_records"):
        f = getattr(lib, fn)
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_char_p), tp, C.c_int, C.c_uint64]
        f.restype = C.c_uint64
    return lib


def write_reads(path, records, nreads, m, seed):
    rng = np.random.default_rng(seed)
    lens = np.array([len(r) for r in records])
    ok = np.nonzero(lens >= m)[0]
    which = rng.choice(ok, nreads, p=lens[ok] / lens[ok].sum())
    letters = np.frombuffer(b"ACGT", np.uint8)
    with open(path, "wb") as f:
        for q in range(nreads):
            rec = records[which[q]]
            s = int(rng.integers(0, len(rec) - m + 1))
            read = bytearray(rec[s:s + m])
            if q % 20 == 0:
                read[int(rng.integers(0, m))] = int(letters[rng.integers(0, 4)])
            f.write(b"@r%d\n%s\n+\n%s\n" % (q, bytes(read), b"I" * m))


def head_fastq(src, dst, nreads):
    with open(src, "rb") as f, open(dst, "wb") as g:
        for _ in range(4 * nreads):
            g.write(f.readline())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10000)
    ap.add_argument("--min-len", type=int, default=1000)
    ap.add_argument("--max-len", type=int, default=100000)
    ap.add_argument("--reads", type=int, default=1000000)
    ap.add_argument("--reads-d1", type=int, default=100000)
    ap.add_argument("--baseline-reads", type=int, default=20000)
    ap.add_argument("--baseline-reads-d1", type=int, default=2000)
    ap.add_argument("--out", default=None, help="directory for the FASTQ / SAM files (default: a temporary one)")
    a = ap.parse_args()
    rng = np.random.default_rng(2026)
    letters = np.frombuffer(b"ACGT", np.uint8)
    records = [letters[rng.integers(0, 4, int(rng.integers(a.min_len, a.max_len + 1)))].tobytes()
               for _ in range(a.records)]
    total = sum(len(r) for r in records)
    res = {"probe": "records", "gpu": gpu_info(), "records": a.records, "symbols": total}

    # ---- build: one records index against one index per record ----
    remap = stralg_b200.RecordsRemap(records)
    codes = [remap.remap(r) for r in records]
    stralg_b200.SuffixArrayIndex.build_records(codes[:50], remap.alphabet_size).close()  # warm-up
    t0 = time.perf_counter()
    idx = stralg_b200.SuffixArrayIndex.build_records(codes, remap.alphabet_size)
    res["records_build_s"] = time.perf_counter() - t0
    idx.close()
    own = [c - np.uint8(1) for c in codes]  # every record holds all four letters: its own codes are 1..4
    t0 = time.perf_counter()
    for c in own:
        stralg_b200.SuffixArrayIndex.build(c, 5).close()
    res["per_record_builds_s"] = time.perf_counter() - t0
    del own, codes
    print(json.dumps(res), file=sys.stderr, flush=True)  # (progress)

    # ---- mapping ----
    lib = bind(C.CDLL(COMPAT_SO))
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    t0 = time.perf_counter()
    tbls = []
    for r in records:
        buf = C.create_string_buffer(r, len(r) + 1)
        tbls.append(lib.build_complete_table(C.cast(buf, u8p), True))  # (it keeps a remapped copy of the string)
    res["tables_s"] = time.perf_counter() - t0
    names = (C.c_char_p * len(records))(*[b"rec%d" % k for k in range(len(records))])
    tarr = (C.POINTER(RefBwtTable) * len(records))(*tbls)

    def run(fn, fq, sam, edits):
        f, o = libc.fopen(fq.encode(), b"r"), libc.fopen(sam.encode(), b"w")
        t = time.perf_counter()
        lines = getattr(lib, fn)(f, o, len(records), names, tarr, edits, 0)
        t = time.perf_counter() - t
        libc.fclose(f)
        libc.fclose(o)
        return t, int(lines)

    with tempfile.TemporaryDirectory() as tmp:
        d = a.out or tmp
        os.makedirs(d, exist_ok=True)
        for edits, nreads, nbase in ((0, a.reads, a.baseline_reads), (1, a.reads_d1, a.baseline_reads_d1)):
            fq = os.path.join(d, f"reads_d{edits}.fq")
            write_reads(fq, records, nreads, 100, 7 + edits)
            t, lines = run("bwt_map_fastq_records", fq, os.path.join(d, f"records_d{edits}.sam"), edits)
            res[f"d{edits}"] = {"reads": nreads, "records_s": t, "records_reads_per_s": nreads / t, "sam_lines": lines}
            print(json.dumps(res), file=sys.stderr, flush=True)
            fqb = os.path.join(d, f"reads_d{edits}_head.fq")
            head_fastq(fq, fqb, nbase)
            tb, lb = run("bwt_map_fastq", fqb, os.path.join(d, f"per_record_d{edits}.sam"), edits)
            tr, lr = run("bwt_map_fastq_records", fqb, os.path.join(d, f"records_head_d{edits}.sam"), edits)
            same = open(os.path.join(d, f"per_record_d{edits}.sam"), "rb").read() == \
                open(os.path.join(d, f"records_head_d{edits}.sam"), "rb").read()
            assert same and lb == lr, f"d={edits}: the SAM outputs differ"
            res[f"d{edits}"].update({"baseline_reads": nbase, "per_record_s": tb, "per_record_reads_per_s": nbase / tb,
                                     "records_same_reads_s": tr, "sam_identical": same})
    for t in tbls:
        lib.completely_free_bwt_table(t)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
