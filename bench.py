#!/usr/bin/env python
"""bench.py -- headline benchmark of the stralg hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

N = 1  -> workload "build": SA + BWT + C + sampled O of a 3 Gbp synthetic DNA text (BASELINE.json
          configs[2]; the text is resident in HBM before the timed region).  value = Mchars/s.
          (`scaling_series` repeats the N = 1 point of the search series at the top level.)
          The same line carries `search` (FM exact search of 100-bp reads at 1 GPU),
          `roofline` (dominant kernel of the build), `e2e` (host buffers through the C ABI, copies
          inside the timed region), `cpu_baseline` (the unmodified reference on the box's host
          cores, bounded sample), and the same build on NON-UNIFORM texts, each verified with the
          suffix-array checker: `build_repeat_rich` (SURVEY 8(d) C3 repeat-rich), `build_hg38_like`
          (the reference's genome sample tiled with mutations), `build_dna_with_n` (ACGT with 5 % N in runs, the
          alphabet A C G N T), `config5_stress` (BASELINE
          configs[4]: five texts at 2^30), plus `compat` (numbers through libstralg_b200.so, the
          reference's own function names).
N > 1  -> workload "search" (BASELINE.json configs[3]): the index is replicated (every rank builds
          it), 100 M 2-bit packed reads are split over the ranks (strong scaling), (L, R) pairs
          reach rank 0 inside the timed region.  value = patterns/s, whole job.
Launched by torch.distributed.run with ONE rank (the N = 1 point of a scaling series) the line's
headline is the search metric as well (build nested as `build`), so that efficiency v_N / (N v_1)
is computable from the lines of one series.
--impl reference times the reference's own CPU implementation (oracle/_ref, else the oracle
port) on a bounded sample of the same workload; rank 0 only.
--dump-outputs DIR (rank 0) writes, after the timed steps, a fixed seeded sample of what the last timed step
computed: the build's suffix array, C table and O table, and the (L, R) intervals of the timed search.  The
inputs are generated from fixed seeds, so two builds of the project can be compared file by file.  The one
difference in what is timed: the last build step's index is released after the timed region instead of inside it
(one host-side release of its device buffers per run), so that its tables can be read afterwards.

One JSON line on stdout (rank 0).  Timing: W >= 3 warm-up steps, CUDA events on the launching
stream, barrier + synchronize on both sides, max over ranks; inputs are far larger than L2.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC_BUILD = "SA+BWT build Mchars/s on 1 B200"
METRIC_SEARCH = "FM exact-search patterns/s"
N_FULL = 3_000_000_000
READS_FULL = 100_000_000
READ_LEN = 100
MISS_PER_1024 = 102  # ~10 % of the reads are uniform random (SURVEY 8d, C4)
SEED = 88172645463325252
CPU_SAMPLE = 1 << 24
DUMP_ROWS = 1 << 19  # rows per sampled array of --dump-outputs: all of them come to about 32 MB in float64
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 20261020


def env_int(name, dflt):
    v = os.environ.get(name)
    return int(v) if v else dflt


def dump_rows(count, seed):
    """The fixed, seeded, sorted rows of an output of `count` rows that --dump-outputs writes (all rows when the
    output is small), so that two builds of the project dump the same entries."""
    if count <= DUMP_ROWS:
        return np.arange(count, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).integers(0, count, DUMP_ROWS, dtype=np.int64))


def build_outputs(idx, torch, device):
    """What a caller of the timed build receives, sampled: SA rows, the C table and O(a, i) (the sampled O table
    answers through the library's occ query)."""
    from stralg_b200 import texts as T
    rows = dump_rows(idx.length, DUMP_SEED)
    sa = T.device_view(idx.device_ptr("sa"), idx.length, 4, device)
    sa_rows = sa[torch.from_numpy(rows).to(sa.device)].cpu().numpy().view(np.uint32)
    occ_i = dump_rows(idx.length + 1, DUMP_SEED + 1).astype(np.uint32)
    occ_a = np.random.default_rng(DUMP_SEED + 2).integers(0, idx.sigma, len(occ_i)).astype(np.uint8)
    return {"build_sa_rows": rows, "build_sa": sa_rows, "build_c_table": idx.c_table(),
            "build_occ_i": occ_i, "build_occ_a": occ_a, "build_occ": idx.occ(occ_a, occ_i)}


def search_outputs(L, R, torch):
    """(L, R) of the timed search's last step (int32 tensors holding uint32 values), sampled by read."""
    rows = dump_rows(L.numel(), DUMP_SEED + 3)
    sel = torch.from_numpy(rows).to(L.device)
    return {"search_read_rows": rows, "search_L": L[sel].cpu().numpy().view(np.uint32),
            "search_R": R[sel].cpu().numpy().view(np.uint32)}


def write_outputs(out_dir, arrays):
    """DIR/<name>.npy in float64 (every value here is an integer below 2^53, so the conversion is exact)."""
    arrays = {k: np.asarray(v).astype(np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [ln for (t, ln) in self.lines if t0 <= t <= t1] or [ln for (_, ln) in self.lines]
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
                for k, nm in enumerate(names):
                    if f[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm)}


# build stage (library timer name) -> the kernel it brackets
STAGE_KERNELS = {
    "msd_local_sort": "msd_local_sort_kernel (in-SM sort of the final buckets; emits SA, BWT rows, ranks of shared keys)",
    "msd_part1": "msd_partition_kernel<FROM_TEXT> (level-1 partition, elements formed from the packed text)",
    "msd_part": "msd_partition_kernel (level-2 partition of 8-byte elements)",
    "msd_hist": "msd_hist_elems_kernel (level-2 digit histogram)",
    "radix_pass0": "onesweep_pass_kernel (LSD round 0, one digit)",
    "radix_pass": "onesweep_pass_kernel (doubling round, one digit)",
}


def load_traffic(kernel_key, n=None):
    """ncu dram__bytes_read.sum + dram__bytes_write.sum of the kernel behind a build stage, per launch,
    from the capture summarised in profiles/roofline_traffic.json (scaled linearly when this run's
    text length differs from the captured one).  None when there is no capture for the stage."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        ent = json.load(open(p)).get(kernel_key)
        if ent is None:
            return None
        if isinstance(ent, dict):
            v = float(ent["dram_bytes_per_launch"])
            if n is not None and ent.get("n") and int(ent["n"]) != int(n):
                v *= float(n) / float(ent["n"])
            return v
        return float(ent)
    except Exception:
        return None


def search_traffic(reads):
    """ncu DRAM bytes of the search kernel for `reads` reads of this workload (captured at 10^8 reads on
    the 3 Gbp index, profiles/r1_search_dram_3g.csv; per-read traffic does not depend on the batch size)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        ent = json.load(open(p))["fm_search"]
        return float(ent["dram_bytes_per_launch"]) * float(reads) / float(ent["reads"])
    except Exception:
        return None


# =================================================================================================
# reference arm / cpu baseline (the only place bench.py touches oracle/)
# =================================================================================================
def cpu_reference_build(codes_sample, sigma):
    """One pass of the reference's CPU path over a bounded sample: sa_is_construction
    (stralg/sa_is.c:466-509) + init_bwt_table (stralg/bwt.c:22-89).  Returns seconds, kind."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    n = len(codes_sample) - 1
    if _oracle.Ref.available():
        ref = _oracle.Ref()
        lib = ref.lib
        buf = np.ascontiguousarray(codes_sample, dtype=np.uint8)
        remap = _oracle.RefRemapTable()
        remap.alphabet_size = sigma
        t0 = time.perf_counter()
        sa = lib.sa_is_construction(buf.ctypes.data_as(_oracle.u8p), C.c_uint32(sigma))
        tab = lib.alloc_bwt_table(sa, None, C.byref(remap))
        dt = time.perf_counter() - t0
        lib.free_bwt_table(tab)
        lib.free_suffix_array(sa)
        return dt, "reference"
    o = _oracle.Oracle()
    t0 = time.perf_counter()
    sa = o.sa(codes_sample)
    bwt = o.bwt(codes_sample, sa)
    o.c_table(codes_sample, sigma)
    o.o_checkpoints(bwt, sigma, 64)
    return time.perf_counter() - t0, "port"


def cpu_reference_search(codes_sample, sigma, reads, m, threads):
    """Reference exact iterator (stralg/bwt.c:164-199) over a dense O table, pattern shards on
    `threads` host threads.  Returns (seconds for the search only, kind)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    npat = len(reads) // m
    L = np.empty(npat, dtype=np.uint32)
    R = np.empty(npat, dtype=np.uint32)
    o = _oracle.Oracle()
    if _oracle.Ref.available():
        ref = _oracle.Ref()
        lib = ref.lib
        buf = np.ascontiguousarray(codes_sample, dtype=np.uint8)
        remap = _oracle.RefRemapTable()
        remap.alphabet_size = sigma
        sa = lib.sa_is_construction(buf.ctypes.data_as(_oracle.u8p), C.c_uint32(sigma))
        tab = lib.alloc_bwt_table(sa, None, C.byref(remap))
        fn = C.cast(lib.init_bwt_exact_match_iter, C.c_void_p)
        t0 = time.perf_counter()
        o.lib.oracle_ref_search_threads(fn, tab, reads.ctypes.data_as(_oracle.u8p), C.c_uint32(m),
                                        C.c_uint64(npat), C.c_uint32(threads), L.ctypes.data_as(_oracle.u32p),
                                        R.ctypes.data_as(_oracle.u32p))
        dt = time.perf_counter() - t0
        lib.free_bwt_table(tab)
        lib.free_suffix_array(sa)
        return dt, "reference", L, R
    sa = o.sa(codes_sample)
    bwt = o.bwt(codes_sample, sa)
    c = o.c_table(codes_sample, sigma)
    ck = o.o_checkpoints(bwt, sigma, 64)
    off = np.arange(0, (npat + 1) * m, m, dtype=np.uint64)
    t0 = time.perf_counter()
    L, R = o.search_ck(c, bwt, ck, 64, reads, off, threads=threads)
    return time.perf_counter() - t0, "port", L, R


def cpu_reference_approx(text, ns, m, d, nreads):
    """The unmodified reference's approximate iterator over its own tables (build_complete_table with the
    reverse tables) on the first `ns` symbols; `nreads` reads of length m, edit distance d, one core."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    if not _oracle.Ref.available():
        return {"unavailable": "oracle/_ref/libstralg_ref.so is not present"}
    ref = _oracle.Ref()
    o = _oracle.Oracle()
    sample = np.concatenate([text[:ns].cpu().numpy(), np.zeros(1, np.uint8)])
    raw = (np.frombuffer(b"ACGT", dtype=np.uint8)[sample[:-1] - 1]).tobytes()
    t = ref.tables(raw, include_reverse=True)
    hr = np.empty(nreads * m, dtype=np.uint8)
    o.lib.oracle_synth_reads(sample.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(ns), C.c_uint32(4),
                             hr.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(nreads), C.c_uint32(m),
                             C.c_uint32(MISS_PER_1024), C.c_uint64(SEED + 1))
    t0 = time.perf_counter()
    hits = 0
    for q in range(nreads):
        hits += len(ref.approx_matches(t["handle"], hr[q * m:(q + 1) * m], d)[0])
    dt = time.perf_counter() - t0
    ref.free_tables(t["handle"])
    return {"value": nreads / dt, "unit": "reads/s", "cores": 1, "kind": "reference", "intervals": hits,
            "sample": f"{nreads} reads x {m} bp, edit distance {d}, against the first {ns} symbols (dense O + RO "
                      f"tables of the reference), {dt:.2f} s"}


def host_synth(n, nsym, seed):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    o = _oracle.Oracle()
    out = np.empty(n + 1, dtype=np.uint8)
    o.lib.oracle_synth_codes(out.ctypes.data_as(_oracle.u8p), C.c_uint64(n), C.c_uint32(nsym), C.c_uint64(seed))
    return out, o


def run_reference_arm(args, rank):
    if rank != 0:
        return
    under_torchrun = "TORCHELASTIC_RUN_ID" in os.environ or ("RANK" in os.environ and "LOCAL_RANK" in os.environ)
    workload = args.workload if args.workload != "auto" else ("build" if (args.gpus == 1 and not under_torchrun) else "search")
    cores = os.cpu_count() or 1
    n = min(args.cpu_sample, args.n)
    codes, o = host_synth(n, 4, SEED)
    times = []
    if workload == "build":
        for step in range(args.warmup_ref + args.steps):
            dt, kind = cpu_reference_build(codes, 5)
            if step >= args.warmup_ref:
                times.append(dt)
        per = float(np.mean(times))
        value = n / per / 1e6
        line = {
            "impl": "reference", "metric": METRIC_BUILD, "value": value, "unit": "Mchars/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup_ref, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "build: SA + C + dense O (sa_is_construction + init_bwt_table) of random ACGT",
                       "n": n, "sigma": 5, "full_workload_n": args.n},
            "cpu_baseline": {"value": value, "unit": "Mchars/s", "cores": 1, "kind": kind,
                             "sample": f"first {n} symbols of the {args.n}-symbol synthetic text, per step"},
            "e2e": {"value": value, "unit": "Mchars/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
    else:
        npat = args.cpu_reads
        reads = np.empty(npat * READ_LEN, dtype=np.uint8)
        o.lib.oracle_synth_reads(codes.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(n), C.c_uint32(4),
                                 reads.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(npat), C.c_uint32(READ_LEN),
                                 C.c_uint32(MISS_PER_1024), C.c_uint64(SEED + 1))
        for step in range(args.warmup_ref + args.steps):
            dt, kind, _, _ = cpu_reference_search(codes, 5, reads, READ_LEN, cores)
            if step >= args.warmup_ref:
                times.append(dt)
        per = float(np.mean(times))
        value = npat / per
        line = {
            "impl": "reference", "metric": METRIC_SEARCH, "value": value, "unit": "patterns/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup_ref, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "search: reference exact iterator over its dense O table", "n": n, "sigma": 5,
                       "reads": npat, "read_len": READ_LEN, "full_workload_n": args.n,
                       "full_workload_reads": args.reads},
            "cpu_baseline": {"value": value, "unit": "patterns/s", "cores": cores, "kind": kind,
                             "sample": f"{npat} reads x {READ_LEN} bp against a {n}-symbol text (dense O limit of "
                                       f"the reference, bwt.c:50), {cores} threads"},
            "e2e": {"value": value, "unit": "patterns/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
    print(json.dumps(line), flush=True)



def numa_pin(local_rank):
    """Run this process (and allocate its pinned staging) on the CPUs next to its GPU: VERDICT r1 found all
    ranks of the 8-GPU run on NUMA node 0.  Best effort; returns what was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # 00000000:1B:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        base = f"/sys/bus/pci/devices/{bus}"
        node = open(base + "/numa_node").read().strip()
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
        return {"numa_node": node, "cpus": cpus}
    except Exception as ex:
        return {"error": str(ex)[:120]}


def timed_build(stralg_b200, torch, src, sigma, local_rank, stream, reps=2, **kw):
    """Best of `reps` device-timed builds of one text; returns (ms, stats, stage ms, index of the last build)."""
    best, idx = None, None
    for _ in range(reps):
        if idx is not None:
            idx.close()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        idx = stralg_b200.SuffixArrayIndex.build(src, sigma, profile=True, device=local_rank, stream=stream, **kw)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if best is None or ms < best[0]:
            agg = {}
            for name, sms, _ in idx.profile():
                agg[name] = agg.get(name, 0.0) + sms
            best = (ms, idx.stats(), agg)
        if ms > 6000.0:
            break
    return best[0], best[1], best[2], idx


def nonuniform_builds(args, lib, stralg_b200, torch, local_rank, stream, n):
    """VERDICT r1 items 1-2: the same build on texts that are NOT uniform -- SURVEY 8(d)'s repeat-rich C3 variant,
    a genome-like text (the reference's hg38 sample tiled with point mutations) and the five config-5 stress texts
    at 2^30 (BASELINE configs[4]) -- each verified with the suffix-array checker of stralg_b200/texts.py
    (permutation + adjacent order: pins the array uniquely), independent of the product kernels."""
    from stralg_b200 import texts as T
    out = {}

    def one(label, make, nn, sigma_hint=None, occ=True, reps=2):
        try:
            text, sigma, info = make()
            ms, st, stages, idx = timed_build(stralg_b200, torch, text[:nn], sigma, local_rank, stream, reps=reps, occ=occ)
            lib.b200sa_release_workspace(local_rank)
            sa = T.device_view(idx.device_ptr("sa"), nn + 1, 4, local_rank)
            ok, why = T.check_suffix_array(text, sa, nn)
            idx.close()
            top = sorted(stages.items(), key=lambda kv: -kv[1])[:6]
            rec = {"n": nn, "sigma": sigma, "ms_per_build": ms, "Mchars_per_s": nn / (ms / 1e3) / 1e6,
                   "doubling_rounds": st["rounds"], "round0_mode": st["round0_mode"], "partition_levels": st["passes0"],
                   "k0": st["k0"], "shallow_buckets": st["shallow_buckets"], "chain_rounds": st["chain_rounds"],
                   "pivot_rounds": st["pivot_rounds"], "pivot_elems_over_len": st["pivot_elems"] / (nn + 1),
                   "pair_placed": st["pair_placed"], "resolved_by_text": st["resolved_small"], "dense_keys": st["dense_keys"],
                   "sorted_total_over_len": st["sorted_total"] / (nn + 1), "sa_verified": ok, "checker": why,
                   "tables": "SA + BWT + C + sampled O" if occ else "SA",
                   "top_stages_ms": {k: round(v, 2) for k, v in top}}
            rec.update(info)
            del text, sa
            torch.cuda.empty_cache()
            return rec
        except Exception as ex:
            torch.cuda.empty_cache()
            return {"error": str(ex)[:300]}

    def make_repeat():
        t = T.random_codes(lib, n, 4, SEED, local_rank)
        return t, 5, {"text": "random ACGT + copies of random 300-6000 bp segments (SURVEY 8d, C3 repeat-rich)",
                      **T.add_repeats(t, n)}

    def make_hg38():
        return T.hg38_like(n, local_rank, mut_inv=64), 5, {
            "text": "hg38-10000.fa sample (499 950 bp) tiled to n with 1/64 point mutations per copy"}

    def make_dna_n():
        t, frac = T.dna_with_n(lib, n, local_rank)
        return t, 6, {"text": "random ACGT with 5 % N in runs of 10^3-10^6 plus single N (alphabet A C G N T: dense initial keys)",
                      "N_fraction": round(frac, 4)}

    out["build_repeat_rich"] = one("repeat", make_repeat, n)
    out["build_hg38_like"] = one("hg38", make_hg38, n, reps=2)
    out["build_dna_with_n"] = one("dna_n", make_dna_n, n, reps=2)
    n5 = min(1 << 30, n)
    stress = {}
    names = {"byte": "C5a random bytes 1..255", "unary": "C5b a^n", "acgt4": "C5c (ACGT)^(n/4)",
             "period1000": "C5d period-1000 random block", "fib": "C5e Fibonacci string"}
    for kind in T.STRESS_KINDS:
        def mk(kind=kind):
            t, sigma = T.stress_text(lib, kind, n5, local_rank)
            return t, sigma, {"text": names[kind]}
        stress[kind] = one(kind, mk, n5, occ=False, reps=2)
    out["config5_stress"] = stress
    return out


def compat_bench(args, n_text_avail):
    """VERDICT r1 item 4: numbers THROUGH the drop-in library (libstralg_b200.so, the reference's own names):
    build_complete_table (bwt.c:134-161) on 2^24 and 2^28 symbols including the copies into malloc'd host arrays,
    and the protocol of performance/suffix_array_search.c:122-143 (n = 10^6, m = 100, one iterator per pattern,
    patterns sampled from the text), next to the unmodified reference on one host core."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    so = os.path.join(ROOT, "stralg_b200", "lib", "libstralg_b200.so")
    shim = _oracle.bind_stralg_api(C.CDLL(so))
    shim.bwt_exact_match_loop.restype = C.c_uint64
    shim.bwt_exact_match_loop.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64]
    o = _oracle.Oracle()
    ref = _oracle.Ref() if _oracle.Ref.available() else None
    res = {"library": "stralg_b200/lib/libstralg_b200.so"}
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)

    def ascii_text(n, seed):
        codes, _ = host_synth(n, 4, seed)
        t = letters[codes[:-1] - 1]
        return np.concatenate([t, np.zeros(1, np.uint8)])

    # ---- build_complete_table ----
    for logn in (24, 28):
        n = 1 << logn
        if n > n_text_avail:
            continue
        txt = ascii_text(n, SEED + logn)
        ts = []
        for it in range(3 if logn == 24 else 2):
            t0 = time.perf_counter()
            tab = shim.build_complete_table(txt.ctypes.data_as(_oracle.u8p), False)
            ts.append(time.perf_counter() - t0)
            shim.completely_free_bwt_table(tab)
        rec = {"n": n, "seconds": float(min(ts)), "Mchars_per_s": n / min(ts) / 1e6,
               "includes": "remap + H2D + GPU build + D2H of SA (and of the dense O table where it is representable) "
                           "into malloc'd host arrays"}
        if ref is not None and logn == 24 and not args.no_cpu:
            t0 = time.perf_counter()
            tab = ref.lib.build_complete_table(txt.ctypes.data_as(_oracle.u8p), False)
            rec["reference_seconds"] = time.perf_counter() - t0
            rec["reference_Mchars_per_s"] = n / rec["reference_seconds"] / 1e6
            ref.lib.completely_free_bwt_table(tab)
        elif logn == 28:
            rec["reference"] = "not runnable: the reference's dense O size overflows uint32 at this length (bwt.c:50)"
        res[f"build_complete_table_2p{logn}"] = rec
        del txt

    # ---- one iterator per pattern ----
    n, m = 1_000_000, 100
    txt = ascii_text(n, SEED + 99)
    rng = np.random.default_rng(3)
    for npat in (200, 20000):
        starts = rng.integers(0, n - m, npat)
        tab = shim.build_complete_table(txt.ctypes.data_as(_oracle.u8p), False)
        rt = tab.contents.remap_table.contents
        codes = np.frombuffer(bytes(rt.table), dtype=np.int8)[txt[:-1]].astype(np.uint8)
        pats = np.zeros((npat, m + 1), dtype=np.uint8)
        for k, s0 in enumerate(starts):
            pats[k, :m] = codes[s0:s0 + m]
        ts = []
        for it in range(4):
            t0 = time.perf_counter()
            hits = shim.bwt_exact_match_loop(tab, pats.ctypes.data_as(C.c_void_p), m, npat)
            ts.append(time.perf_counter() - t0)
        rec = {"n": n, "m": m, "patterns": npat, "matches": int(hits), "seconds": float(min(ts[1:])),
               "patterns_per_s": npat / min(ts[1:]), "us_per_pattern": min(ts[1:]) / npat * 1e6,
               "path": "init_bwt_exact_match_iter -> one-pattern b200sa_search_batch through mapped pinned memory "
                       "(one kernel launch + one stream synchronisation per pattern); positions from the host copy of SA"}
        shim.completely_free_bwt_table(tab)
        if ref is not None and not args.no_cpu:
            rtab = ref.lib.build_complete_table(txt.ctypes.data_as(_oracle.u8p), False)
            o.lib.oracle_ref_iter_loop.restype = C.c_uint64
            o.lib.oracle_ref_iter_loop.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64]
            fi = C.cast(ref.lib.init_bwt_exact_match_iter, C.c_void_p)
            fn = C.cast(ref.lib.next_bwt_exact_match_iter, C.c_void_p)
            tr = []
            for it in range(4):
                t0 = time.perf_counter()
                rh = o.lib.oracle_ref_iter_loop(fi, fn, rtab, pats.ctypes.data_as(C.c_void_p), m, npat)
                tr.append(time.perf_counter() - t0)
            rec["reference_patterns_per_s"] = npat / min(tr[1:])
            rec["reference_us_per_pattern"] = min(tr[1:]) / npat * 1e6
            rec["reference_matches"] = int(rh)
            rec["same_matches"] = int(rh) == int(hits)
            ref.lib.completely_free_bwt_table(rtab)
        res[f"iterator_per_pattern_{npat}"] = rec
    res["note"] = ("a single dependent chain of ~100 random lookups per pattern is latency-bound: the CPU's cache "
                   "beats a kernel launch per pattern; the batched entry points (bwt_exact_match_batch, "
                   "b200sa_search_batch[_packed]) are the ones that use the GPU")
    return res


# =================================================================================================
# GPU arm
# =================================================================================================
def gpu_arm(args, rank, local_rank, world):
    # stdout carries the ONE JSON line only: libraries (NCCL's version banner) write to fd 1 too
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import stralg_b200
    lib = stralg_b200.load()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    # launched by torch.distributed.run (the driver's scaling series), one rank included: the line's headline is the
    # SEARCH metric at every N, so that a scaling efficiency can be computed from the per-N values; the build
    # (BASELINE configs[2]) is then nested as `build`.  Plain `python bench.py` (N = 1): the build is the headline.
    under_torchrun = "TORCHELASTIC_RUN_ID" in os.environ or ("RANK" in os.environ and "LOCAL_RANK" in os.environ)
    workload = args.workload if args.workload != "auto" else ("build" if (world == 1 and not under_torchrun) else "search")
    stream = torch.cuda.current_stream().cuda_stream
    peak, peak_src = measured_peak()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic text in HBM ----
    n = args.n
    text = None
    while text is None:
        try:
            text = torch.empty(n + 1, dtype=torch.uint8, device=dev)
        except torch.OutOfMemoryError:
            n //= 2
    assert lib.b200sa_synth_codes(C.c_void_p(text.data_ptr()), n, 4, SEED, local_rank, C.c_void_p(stream)) == 0
    torch.cuda.synchronize()

    def build(profile=False, drop_sa=False, src=None, textcmp=False, ktable=False):
        return stralg_b200.SuffixArrayIndex.build(text[:n] if src is None else src, 5, occ=True, profile=profile,
                                                  drop_sa=drop_sa, textcmp=textcmp, ktable=ktable, device=local_rank,
                                                  stream=stream)

    sampler = ClockSampler(local_rank)
    out = {}
    dump = {} if (args.dump_outputs and rank == 0) else None  # name -> array of the last timed step

    if workload == "build":
        # ------------------------------------------------------------------ device-resident build
        for _ in range(args.warmup):
            build().close()
        barrier()
        sampler.start()
        launches0 = lib.b200sa_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage_ms = {}
        t_wall0 = time.time()
        ev0.record()
        stats = None
        for step in range(args.steps):
            idx = build(profile=True)
            for name, ms, by in idx.profile():
                a = stage_ms.setdefault(name, [0, 0.0, 0.0])
                a[0] += 1
                a[1] += ms
                a[2] += by
            stats = idx.stats()
            if not (dump is not None and step == args.steps - 1):  # --dump-outputs reads the last index below
                idx.close()
        ev1.record()
        barrier()
        t_wall1 = time.time()
        sampler.stop()
        if dump is not None:
            dump.update(build_outputs(idx, torch, local_rank))
            idx.close()
        launches = lib.b200sa_launch_count() - launches0
        ms_total = max_over_ranks(ev0.elapsed_time(ev1))
        ms_step = ms_total / args.steps
        value = n / (ms_step / 1e3) / 1e6
        clocks = sampler.summary(t_wall0, t_wall1)

        # roofline of the dominant kernel = the build stage with the largest share of the step; its
        # algorithmic bytes per launch are what the library's stage timer records (DESIGN.md section 4),
        # its duration comes from CUDA events on the launching stream around that launch.
        dom = max(stage_ms.items(), key=lambda kv: kv[1][1])
        dname, (dlaunch, dms, dbytes) = dom[0], dom[1]
        pass_ms = dms / dlaunch
        pass_bytes = dbytes / dlaunch
        achieved = pass_bytes / (pass_ms / 1e3) / 1e9
        traffic = load_traffic(dname, n)
        roofline = {"bound": "hbm", "kernel": STAGE_KERNELS.get(dname, dname), "stage": dname,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": pass_bytes, "avg_launch_ms": pass_ms,
                    "launches_timed": dlaunch, "share_of_step": dms / ms_total}
        model_bytes = 244.5 * n  # SURVEY 8d: 237 B/char SA + 7.5 B/char BWT/C/O
        stages = {k: {"launches": v[0], "ms_per_step": v[1] / args.steps,
                      "algorithmic_GBps": (v[2] / v[1] / 1e6) if v[1] else None} for k, v in stage_ms.items()}

        # ------------------------------------------------------------------ e2e: host buffers via the C ABI
        # Every step: b200sa_build from a pinned HOST text (H2D inside), then SA + O + C back into pinned host
        # memory.  Steps are issued the way a caller that builds index after index would: the copies of step i
        # (b200sa_copy_async on a second stream, two sets of host buffers) run while step i + 1 uploads its text
        # and builds; the timed region covers all steps including the last copy.  `serial_ms_per_step` is the
        # same step with nothing overlapped (build, then blocking copies).
        e2e = None
        try:
            h_text = torch.empty(n, dtype=torch.uint8, pin_memory=True)
            h_text.copy_(text[:n])
            occ_bytes = stats["occ_bytes"]
            h_c = np.empty(5, dtype=np.uint32)
            nbuf = 2
            try:
                h_sa = [torch.empty(n + 1, dtype=torch.int32, pin_memory=True) for _ in range(nbuf)]
                h_occ = [torch.empty(occ_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(nbuf)]
            except Exception:
                nbuf = 1
                h_sa = [torch.empty(n + 1, dtype=torch.int32, pin_memory=True)]
                h_occ = [torch.empty(occ_bytes, dtype=torch.uint8, pin_memory=True)]
            torch.cuda.synchronize()
            chk = stralg_b200._lib.check

            def build_host():
                return stralg_b200.SuffixArrayIndex.build(h_text.numpy(), 5, occ=True, device=local_rank, stream=stream)

            # serial reference point (also warms the stream-ordered pool: cuMemMap of the outputs)
            t_ser = []
            for it in range(3):
                t0 = time.perf_counter()
                idx = build_host()
                chk(lib.b200sa_copy_sa(idx._h, C.c_void_p(h_sa[0].data_ptr())))
                chk(lib.b200sa_copy_occ(idx._h, C.c_void_p(h_occ[0].data_ptr())))
                chk(lib.b200sa_copy_c_table(idx._h, C.c_void_p(h_c.ctypes.data)))
                torch.cuda.synchronize()
                t_ser.append(time.perf_counter() - t0)
                idx.close()
            serial = float(np.mean(t_ser[1:]))
            e_steps = max(args.steps, 6) if nbuf == 2 else max(1, min(args.steps, 2))
            copy_stream = torch.cuda.Stream(device=dev)
            cs = copy_stream.cuda_stream
            def run_steps(count):
                pending = []  # (index, event) whose copies are in flight
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for it in range(count):
                    k = it % nbuf
                    if len(pending) >= nbuf:  # the host buffers of step it - nbuf must have been filled
                        old, ev = pending.pop(0)
                        ev.synchronize()
                        old.close()
                    t_w = time.perf_counter()
                    idx = build_host()  # returns when the build is complete (text uploaded inside)
                    if os.environ.get("B200SA_BENCH_DEBUG"):
                        print(f"[e2e] step {it}: waited until {(t_w - t0) * 1e3:.0f} ms, built by "
                              f"{(time.perf_counter() - t0) * 1e3:.0f} ms", file=sys.stderr)
                    if nbuf == 2:
                        chk(lib.b200sa_copy_async(idx._h, 0, C.c_void_p(h_sa[k].data_ptr()), C.c_void_p(cs)))
                        chk(lib.b200sa_copy_async(idx._h, 4, C.c_void_p(h_occ[k].data_ptr()), C.c_void_p(cs)))
                        chk(lib.b200sa_copy_c_table(idx._h, C.c_void_p(h_c.ctypes.data)))
                        ev = torch.cuda.Event()
                        ev.record(copy_stream)
                        pending.append((idx, ev))
                    else:
                        chk(lib.b200sa_copy_sa(idx._h, C.c_void_p(h_sa[0].data_ptr())))
                        chk(lib.b200sa_copy_occ(idx._h, C.c_void_p(h_occ[0].data_ptr())))
                        chk(lib.b200sa_copy_c_table(idx._h, C.c_void_p(h_c.ctypes.data)))
                        idx.close()
                for old, ev in pending:
                    ev.synchronize()
                    old.close()
                torch.cuda.synchronize()
                return time.perf_counter() - t0

            run_steps(2)  # untimed: the pool grows to two live indices once
            e_per = run_steps(e_steps) / e_steps
            # the overlapped loop keeps two indices alive, and the stream-ordered pool may have to map fresh
            # memory for it on some runs; the headline is the better of the two ways to call the API
            overlapped = e_per
            best = min(e_per, serial)
            e2e = {"value": n / best / 1e6, "unit": "Mchars/s", "h2d_bytes_per_step": int(n),
                   "d2h_bytes_per_step": int(4 * (n + 1) + occ_bytes + 20), "ms_per_step": best * 1e3,
                   "steps": e_steps, "serial_ms_per_step": serial * 1e3, "serial_value": n / serial / 1e6,
                   "overlapped_ms_per_step": overlapped * 1e3, "mode": "overlapped" if e_per <= serial else "serial",
                   "api": "b200sa_build(pinned host codes) + b200sa_copy_async(SA, O) / b200sa_copy_c_table into pinned "
                          "host buffers; the copies of a step overlap the next step's upload and build (two buffer sets)"
                          if nbuf == 2 else "b200sa_build(host codes) + b200sa_copy_sa/_occ/_c_table (pinned host)"}
            del h_text, h_sa, h_occ
        except Exception as ex:  # pinned-memory shortage must not kill the device-timed number
            e2e = {"value": None, "unit": "Mchars/s", "error": str(ex)[:200]}

        # ------------------------------------------------------------------ CPU baseline (bounded sample)
        cpu_baseline = None
        if not args.no_cpu:
            ns = min(args.cpu_sample, n)
            sample = np.concatenate([text[:ns].cpu().numpy(), np.zeros(1, np.uint8)])
            dt, kind = cpu_reference_build(sample, 5)
            cpu_baseline = {"value": ns / dt / 1e6, "unit": "Mchars/s", "cores": 1, "kind": kind,
                            "host_cores_available": os.cpu_count(),
                            "sample": f"first {ns} symbols of the text: sa_is_construction + init_bwt_table, "
                                      f"{dt:.2f} s"}

        out = {
            "metric": METRIC_BUILD, "value": value, "unit": "Mchars/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "build: SA + BWT + C + sampled O of random ACGT (BASELINE configs[2])"
                       if n == N_FULL else "build: SA + BWT + C + sampled O of random ACGT",
                       "n": n, "sigma": 5, "sa_dtype": "uint32", "l2": "inputs larger than L2 (no flush needed)",
                       "k0": stats["k0"], "radix_bits": stats["radix_bits"], "passes0": stats["passes0"],
                       "doubling_rounds": stats["rounds"]},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline,
            "model": {"algorithmic_bytes_per_char": 244.5, "whole_build_GBps": model_bytes / (ms_step / 1e3) / 1e9,
                      "whole_build_frac_of_peak": model_bytes / (ms_step / 1e3) / 1e9 / peak},
            "cpu_baseline": cpu_baseline, "stages": stages,
        }
        # BASELINE configs[1]: SA + LCP of a 256 Mi random ACGT text (device-resident, same timing rules)
        try:
            n2 = min(1 << 28, n)
            for _ in range(2):
                stralg_b200.SuffixArrayIndex.build(text[:n2], 5, occ=False, lcp=True, device=local_rank,
                                                   stream=stream).close()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            c0.record()
            reps2 = 3
            lcp_stages = {}
            for _ in range(reps2):
                i2 = stralg_b200.SuffixArrayIndex.build(text[:n2], 5, occ=False, lcp=True, profile=True,
                                                        device=local_rank, stream=stream)
                for name, ms, by in i2.profile():
                    lcp_stages[name] = lcp_stages.get(name, 0.0) + ms / reps2
                i2.close()
            c1.record()
            torch.cuda.synchronize()
            ms2 = c0.elapsed_time(c1) / reps2
            out["config2_sa_lcp"] = {"workload": "SA + LCP of random ACGT (BASELINE configs[1])", "n": n2,
                                     "ms_per_build": ms2, "Mchars_per_s": n2 / (ms2 / 1e3) / 1e6,
                                     "lcp_stage_ms": {k: round(v, 3) for k, v in lcp_stages.items()
                                                      if k.startswith(("phi", "plcp", "lcp", "inverse"))}}
        except Exception as ex:
            out["config2_sa_lcp"] = {"error": str(ex)[:200]}
        # BASELINE configs[0]: SA + LCP + BWT + C/O of a 1 Mi random ACGT text and exact search of 10 k random
        # 20-mers (the reference's own performance/ harness case): small-input latency, host buffers in and out
        try:
            n1 = min(1 << 20, n)
            h1 = text[:n1].cpu().numpy()
            rng = np.random.default_rng(1)
            starts = rng.integers(0, n1 - 20, 10000)
            pats = np.concatenate([h1[s0:s0 + 20] if k % 2 else rng.integers(1, 5, 20).astype(np.uint8)
                                   for k, s0 in enumerate(starts)])
            tb, ts = [], []
            for it in range(6):
                t0 = time.perf_counter()
                i1 = stralg_b200.SuffixArrayIndex.build(h1, 5, lcp=True, bwt=True, occ=True, device=local_rank,
                                                        stream=stream)
                sa1 = i1.sa()
                lcp1 = i1.lcp()
                t1 = time.perf_counter()
                L1, R1 = i1.search(pats, fixed_len=20)
                _, pos1 = i1.locate(L1, R1)
                t2 = time.perf_counter()
                i1.close()
                if it:
                    tb.append(t1 - t0)
                    ts.append(t2 - t1)
            c1 = {"workload": "SA + LCP + BWT + C/O of 1 Mi random ACGT, then exact search + locate of 10 k 20-mers "
                              "(BASELINE configs[0]); host buffers in and out, wall clock",
                  "n": n1, "build_ms": float(np.median(tb)) * 1e3, "search_locate_ms": float(np.median(ts)) * 1e3,
                  "matches": int(len(pos1))}
            if not args.no_cpu:
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import _oracle
                if _oracle.Ref.available():
                    ref = _oracle.Ref()
                    cz = np.concatenate([h1, np.zeros(1, np.uint8)])
                    t0 = time.perf_counter()
                    ref.sa_lcp(cz, 5)
                    c1["cpu_reference_sa_lcp_ms"] = (time.perf_counter() - t0) * 1e3
            out["config1_small"] = c1
        except Exception as ex:
            out["config1_small"] = {"error": str(ex)[:200]}
        torch.cuda.empty_cache()
        if not args.no_nonuniform:
            out.update(nonuniform_builds(args, lib, stralg_b200, torch, local_rank, stream, n))
        if not args.no_compat:
            try:
                lib.b200sa_release_workspace(local_rank)
                out["compat"] = compat_bench(args, n)
            except Exception as ex:
                out["compat"] = {"error": str(ex)[:300]}
        if not args.no_search:
            out["search"] = search_bench(args, lib, stralg_b200, torch, dev, local_rank, stream, text, n, None, 0, 1,
                                         peak, peak_src, build, dump=dump)
            # BASELINE.json's metric has two parts: the build on 1 GPU (this line's `value`) and the search at
            # 1/2/4/8 GPUs (the `value` of the N > 1 lines).  The N = 1 point of the SEARCH series is repeated
            # here at the top level so that a scaling table can be read off the lines of one run.
            out["scaling_series"] = {"metric": METRIC_SEARCH, "unit": "patterns/s", "n_gpus": 1,
                                     "value": out["search"]["value"],
                                     "note": "compare with `value` of the --gpus 2/4/8 lines (same 10^8 reads, strong scaling)"}
    else:
        nested_build = None
        if world == 1:
            for _ in range(2):
                build().close()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(3):
                build().close()
            b1.record()
            torch.cuda.synchronize()
            bms = b0.elapsed_time(b1) / 3
            nested_build = {"metric": METRIC_BUILD, "value": n / (bms / 1e3) / 1e6, "unit": "Mchars/s", "ms_per_step": bms,
                            "n": n, "note": "the full build line is what `python bench.py --gpus 1` prints"}
        res = search_bench(args, lib, stralg_b200, torch, dev, local_rank, stream, text, n, dist, rank, world, peak,
                           peak_src, build, dump=dump)
        out = res
        if nested_build:
            out["build"] = nested_build
        out["scaling_series"] = {"metric": METRIC_SEARCH, "unit": "patterns/s", "n_gpus": world, "value": res["value"],
                                 "note": "the N = 1 point of this series is `scaling_series.value` of the --gpus 1 line"}
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())


def search_bench(args, lib, stralg_b200, torch, dev, local_rank, stream, text, n, dist, rank, world, peak, peak_src,
                 build, dump=None):
    """Replicated index, reads split over ranks, (L, R) delivered on rank 0 in the timed region.  The reads are
    2-bit packed (b200sa_search_device_packed / _batch_packed; VERDICT r1 item 3); the one-byte-per-base entry
    points are measured beside them (`byte_api`)."""
    total_reads = args.reads
    m = READ_LEN
    stride = (m + 3) // 4
    chk = stralg_b200._lib.check
    # search index: C + sampled O, plus SA / ISA / packed text for the unique-interval shortcut
    idx = build(textcmp=True, ktable=True)
    kk = idx.stats()["ktable_k"]
    lib.b200sa_release_workspace(local_rank)
    # contiguous shards of the read set, one per rank; (L, R) reach rank 0 inside the step
    from stralg_b200.shard import ShardedSearch
    ss = ShardedSearch(total_reads, stride, dev, dist, chunks=1, transport=args.transport)
    shard = ss.count

    def gen_reads(count, seed):
        r = torch.empty(count * m, dtype=torch.uint8, device=dev)
        assert lib.b200sa_synth_reads(C.c_void_p(text.data_ptr()), n, 4, C.c_void_p(r.data_ptr()), count, m,
                                      MISS_PER_1024, seed, local_rank, C.c_void_p(stream)) == 0
        return r

    def pack(r, count):
        p = torch.zeros(count * stride + 8, dtype=torch.uint8, device=dev)
        chk(lib.b200sa_pack_reads_device(C.c_void_p(r.data_ptr()), m, stride, count, C.c_void_p(p.data_ptr()), local_rank,
                                         C.c_void_p(stream)))
        return p

    reads = gen_reads(shard, SEED + 1 + rank * 7919)
    preads = pack(reads, shard)

    def search_fn(r, _stride, count, Lo, Ro):
        idx.search_device_packed(r, m, count, Lo, Ro, stride, stream)

    def step():
        ss.step(search_fn, preads)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.b200sa_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    tw1 = time.time()
    sampler.stop()
    if dump is not None:
        dump.update(search_outputs(*ss.result(), torch))
    ms_total = ev0.elapsed_time(ev1)
    if dist is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    launches = lib.b200sa_launch_count() - launches0
    value = total_reads / (ms_step / 1e3)

    # N > 1: rank 0 re-creates every rank's reads (same seeded generator), searches them on its own index through
    # the BYTE entry point and compares with what the step delivered -- the sharded packed path checked bit for
    # bit against the other kernel, outside the timed region
    verified = None
    if dist is not None:
        if rank == 0:
            Lall, Rall = ss.result()
            verified = True
            from stralg_b200.shard import shard_bounds
            for g in range(world):
                glo, ghi = shard_bounds(total_reads, world, g)
                rg = gen_reads(ghi - glo, SEED + 1 + g * 7919)
                Lg = torch.empty(ghi - glo, dtype=torch.int32, device=dev)
                Rg = torch.empty(ghi - glo, dtype=torch.int32, device=dev)
                idx.search_device(rg, None, m, ghi - glo, Lg, Rg, stream)
                torch.cuda.synchronize()
                verified = verified and bool(torch.equal(Lg, Lall[glo:ghi])) and bool(torch.equal(Rg, Rall[glo:ghi]))
                del rg, Lg, Rg
        dist.barrier()

    Lt, Rt = ss.local_result()
    Lh = Lt.cpu().numpy().view(np.uint32)
    Rh = Rt.cpu().numpy().view(np.uint32)
    LR = torch.empty((2, max(shard, 1)), dtype=torch.int32, device=dev)
    hit_frac = float((Rh > Lh).mean())

    def time_kernel(fn):
        fn()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(args.steps):
            fn()
        k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / args.steps

    # kernel-only timing of one rank's shard, both read formats; the byte kernel's (L, R) must equal the packed one's
    kernel_ms = time_kernel(lambda: idx.search_device_packed(preads, m, shard, LR[0], LR[1], stride, stream))
    byte_ms = time_kernel(lambda: idx.search_device(reads, None, m, shard, LR[0], LR[1], stream))
    same_as_bytes = bool(torch.equal(LR[0][:shard], Lt)) and bool(torch.equal(LR[1][:shard], Rt))
    # algorithmic bytes of the launch = the memory operations the kernel issues for this batch, counted by the
    # counting variant of the same kernel: 32-byte O-block loads, 8-byte words of packed reads and packed text,
    # 4-byte SA / ISA loads (8 per k-mer table entry), plus the 8-byte (L, R) result per read.
    counts = (C.c_uint64 * 4)()
    chk(lib.b200sa_search_traffic_packed(idx._h, C.c_void_p(preads.data_ptr()), m, stride, shard,
                                         C.c_void_p(LR[0].data_ptr()), C.c_void_p(LR[1].data_ptr()), counts,
                                         C.c_void_p(stream)))
    issued_bytes = 32.0 * counts[0] + 8.0 * counts[1] + 8.0 * counts[2] + 4.0 * counts[3] + 8.0 * shard
    achieved = issued_bytes / (kernel_ms / 1e3) / 1e9
    miss_steps = 16.0
    survey_bytes_per_read = hit_frac * (m + 2 * m * 32 + 8) + (1 - hit_frac) * (m + 2 * miss_steps * 32 + 8)
    survey_gbps = survey_bytes_per_read * shard / (kernel_ms / 1e3) / 1e9
    roofline = {"bound": "hbm", "kernel": "fm_search_dna_packed_kernel (one lane per read, 2-bit packed reads, k-mer seed "
                "table, unique intervals finished by a 32-symbols-per-step text comparison)", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": search_traffic(shard),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": issued_bytes,
                "avg_launch_ms": kernel_ms, "hit_fraction": hit_frac,
                "ops_per_read": {"o_block_loads_32B": counts[0] / shard, "read_words_8B": counts[1] / shard,
                                 "text_words_8B": counts[2] / shard, "sa_isa_ktable_loads_4B": counts[3] / shard},
                "survey_model": {"bytes_per_read": survey_bytes_per_read, "GBps": survey_gbps,
                                 "frac": survey_gbps / peak,
                                 "note": "SURVEY 8(d) bytes of the plain recurrence (every step two 32-byte O "
                                         "fetches); random accesses, bounded by sector rate rather than bytes"}}

    # e2e: host reads in, host (L, R) out through the C ABI, pinned host buffers allocated next to the GPU
    numa = numa_pin(local_rank)
    e2e, e2e_bytes = None, None
    try:
        e_reads = min(shard, args.e2e_reads)
        hp = torch.empty(e_reads * stride + 8, dtype=torch.uint8, pin_memory=True)
        hp.copy_(preads[: e_reads * stride + 8])
        hL = torch.empty(e_reads, dtype=torch.int32, pin_memory=True)
        hR = torch.empty(e_reads, dtype=torch.int32, pin_memory=True)
        torch.cuda.synchronize()

        def timed_calls(fn):
            ts = []
            for it in range(4):
                if dist is not None:
                    dist.barrier()
                t0 = time.perf_counter()
                fn()
                dt = time.perf_counter() - t0
                if it > 0:
                    ts.append(dt)
            dt = float(np.mean(ts))
            if dist is not None:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt

        dt = timed_calls(lambda: chk(lib.b200sa_search_batch_packed(idx._h, C.c_void_p(hp.data_ptr()), m, stride, e_reads,
                                                                    C.c_void_p(hL.data_ptr()), C.c_void_p(hR.data_ptr()))))
        e2e_ok = bool(np.array_equal(hL.numpy().view(np.uint32), Lh[:e_reads]))
        e2e = {"value": e_reads * world / dt, "unit": "patterns/s", "h2d_bytes_per_step": int(e_reads * stride),
               "d2h_bytes_per_step": int(e_reads * 8), "reads_per_rank": e_reads, "equals_device_result": e2e_ok,
               "numa": numa,
               "api": "b200sa_search_batch_packed (pinned host packed reads in, host (L, R) out), all ranks concurrently"}
        del hp
        hb = torch.empty(e_reads * m, dtype=torch.uint8, pin_memory=True)
        hb.copy_(reads[: e_reads * m])
        torch.cuda.synchronize()
        dtb = timed_calls(lambda: chk(lib.b200sa_search_batch(idx._h, C.c_void_p(hb.data_ptr()), None, m, e_reads,
                                                              C.c_void_p(hL.data_ptr()), C.c_void_p(hR.data_ptr()))))
        e2e_bytes = {"value": e_reads * world / dtb, "unit": "patterns/s", "h2d_bytes_per_step": int(e_reads * m),
                     "d2h_bytes_per_step": int(e_reads * 8),
                     "api": "b200sa_search_batch (one byte per base)"}
        del hb
    except Exception as ex:
        e2e = e2e or {"value": None, "unit": "patterns/s", "error": str(ex)[:200]}

    res = {
        "metric": METRIC_SEARCH, "value": value, "unit": "patterns/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "search: batched FM exact search, replicated 3 Gbp index (BASELINE configs[3])"
                   if n == N_FULL else "search: batched FM exact search, replicated index",
                   "n": n, "sigma": 5, "reads": total_reads, "read_len": m, "reads_per_gpu": shard,
                   "read_format": "2 bits per base, 25 bytes per 100-bp read",
                   "miss_fraction": MISS_PER_1024 / 1024.0, "gather": ("search kernels store (L,R) into rank 0's HBM through NVLink peer memory (symmetric memory) + one "
                              "device-side barrier" if ss.transport == "p2p" else
                              f"NCCL gather of (L,R) to rank 0, {ss.chunks} piece(s) per shard") if world > 1
                   else "none (1 GPU)", "ktable_k": kk, "l2": f"index (1.5 GB O + {8 * 4 ** kk / 1e9:.1f} GB k-mer table, k = {kk}) and reads larger than L2"},
        "clocks": sampler.summary(tw0, tw1), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "kernel_only_patterns_per_s_per_gpu": shard / (kernel_ms / 1e3),
        "byte_api": {"kernel_only_patterns_per_s_per_gpu": shard / (byte_ms / 1e3), "kernel_ms": byte_ms,
                     "same_intervals_as_packed": same_as_bytes, "e2e": e2e_bytes},
        "delivered_equals_single_gpu_search": verified,
    }
    if world == 1 and not args.no_extras:
        # ---- locate (SURVEY 8f rank 3): positions of the first reads through the full suffix array and
        # through the sampled one (LF walk), device buffers, CUDA events; results compared bit for bit
        try:
            nloc = min(shard, args.locate_reads)
            Ld, Rd = LR[0][:nloc].contiguous(), LR[1][:nloc].contiguous()
            poff = torch.empty(nloc + 1, dtype=torch.int64, device=dev)
            total = idx.locate_device(Ld, Rd, nloc, poff, None, 0, stream)
            pos_full = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
            pos_ssa = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
            loc = {"reads": nloc, "positions": total}
            t_b0, t_b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_b0.record()
            idx.sample_sa(args.sa_rate, drop_sa=False)
            t_b1.record()
            torch.cuda.synchronize()
            loc["sample_build_ms"] = t_b0.elapsed_time(t_b1)
            loc["sa_sample_rate"] = args.sa_rate
            for name, buf, env in (("full_sa", pos_full, None), ("sampled_sa", pos_ssa, "1")):
                if env:
                    os.environ["B200SA_LOCATE_SAMPLED"] = env
                else:
                    os.environ.pop("B200SA_LOCATE_SAMPLED", None)
                idx.locate_device(Ld, Rd, nloc, poff, buf, total, stream)  # warm-up
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(args.steps):
                    idx.locate_device(Ld, Rd, nloc, poff, buf, total, stream)
                a1.record()
                torch.cuda.synchronize()
                ms = a0.elapsed_time(a1) / args.steps
                loc[name] = {"ms": ms, "positions_per_s": total / (ms / 1e3)}
            os.environ.pop("B200SA_LOCATE_SAMPLED", None)
            loc["sampled_equals_full"] = bool(torch.equal(pos_full, pos_ssa))
            loc["bytes_per_row"] = {"full_sa": 4.0, "sampled_sa": 0.25 + 4.0 / args.sa_rate}
            res_locate = loc
            del pos_full, pos_ssa, poff
        except Exception as ex:
            res_locate = {"error": str(ex)[:200]}
        # ---- approximate search (SURVEY 8f rank 4): edit distance 1 through the host API (reads in, interval
        # lists + CIGARs out), D table from an index of the reversed text
        try:
            na = min(shard, args.approx_reads)
            rev_text = torch.flip(text[:n], dims=[0]).contiguous()
            rev = build(src=rev_text, drop_sa=True)
            del rev_text
            h_reads = reads[: na * m].cpu().numpy()
            ap = {}
            for d in (1, 2) if args.approx_d2 else (1,):
                cnt = na if d == 1 else max(1, na // 20)
                idx.approx_search(h_reads[: min(cnt, 1000) * m], fixed_len=m, max_edits=d, rev=rev)  # warm-up
                t0 = time.perf_counter()
                r = idx.approx_search(h_reads[: cnt * m], fixed_len=m, max_edits=d, rev=rev)
                dt = time.perf_counter() - t0
                ap[f"d{d}"] = {"reads": cnt, "seconds": dt, "reads_per_s": cnt / dt, "intervals": int(len(r["L"])),
                               "reads_with_a_match": int((np.diff(r["offsets"].astype(np.int64)) > 0).sum())}
            if not args.no_cpu and rank == 0:
                # the reference's own iterator (init_bwt_approx_iter, bwt.c:302-382) on one host core, on a
                # text small enough for its dense O / RO tables; reads drawn from that text the same way
                try:
                    ap["cpu_baseline"] = cpu_reference_approx(text, min(1 << 22, n), m, 1, 4000)
                except Exception as ex:
                    ap["cpu_baseline"] = {"error": str(ex)[:200]}
            ap["api"] = "b200sa_approx_batch (host reads in; intervals, matched lengths and CIGARs out)"
            ap["read_len"] = m
            rev.close()
            res_approx = ap
        except Exception as ex:
            res_approx = {"error": str(ex)[:200]}
        res["locate"] = res_locate
        res["approx"] = res_approx
    if not args.no_cpu and rank == 0 and world == 1:
        ns = min(args.cpu_sample, n)
        sample = np.concatenate([text[:ns].cpu().numpy(), np.zeros(1, np.uint8)])
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import _oracle
        o = _oracle.Oracle()
        npat = args.cpu_reads
        hr = np.empty(npat * m, dtype=np.uint8)
        o.lib.oracle_synth_reads(sample.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(ns), C.c_uint32(4),
                                 hr.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_uint64(npat), C.c_uint32(m),
                                 C.c_uint32(MISS_PER_1024), C.c_uint64(SEED + 1))
        cores = os.cpu_count() or 1
        what = (f"{{}} reads x {m} bp against the first {ns} symbols (the reference's dense O cannot be built beyond "
                f"~214 M rows, bwt.c:50)")
        dt, kind, _, _ = cpu_reference_search(sample, 5, hr, m, cores)
        res["cpu_baseline"] = {"value": npat / dt, "unit": "patterns/s", "cores": cores, "kind": kind,
                               "sample": what.format(npat)}
        n1 = max(1, npat // 8)  # SURVEY 8(d): one core AND all cores
        dt1, kind1, _, _ = cpu_reference_search(sample, 5, hr[: n1 * m], m, 1)
        res["cpu_baseline_1core"] = {"value": n1 / dt1, "unit": "patterns/s", "cores": 1, "kind": kind1,
                                     "sample": what.format(n1)}
    idx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "build", "search"])
    ap.add_argument("--n", type=int, default=env_int("B200SA_BENCH_N", N_FULL))
    ap.add_argument("--reads", type=int, default=env_int("B200SA_BENCH_READS", READS_FULL))
    ap.add_argument("--e2e-reads", type=int, default=20_000_000)
    ap.add_argument("--gather-chunks", type=int, default=1,
                    help="N > 1, gather transport: pieces per shard whose gathers are issued asynchronously")
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "gather"],
                    help="N > 1: how (L, R) reach rank 0: kernel stores through NVLink peer memory, or one NCCL gather")
    ap.add_argument("--cpu-sample", type=int, default=CPU_SAMPLE)
    ap.add_argument("--cpu-reads", type=int, default=1_000_000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-search", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the locate / approximate-search lines")
    ap.add_argument("--no-nonuniform", action="store_true", help="skip the repeat-rich / genome-like / config-5 builds")
    ap.add_argument("--no-compat", action="store_true", help="skip the numbers through libstralg_b200.so")
    ap.add_argument("--locate-reads", type=int, default=20_000_000)
    ap.add_argument("--sa-rate", type=int, default=32)
    ap.add_argument("--approx-reads", type=int, default=200_000)
    ap.add_argument("--approx-d2", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed, seeded sample of what the last step computed (suffix "
                         "array rows, C table, O(a, i), search intervals) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    args.warmup_ref = min(args.warmup, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
