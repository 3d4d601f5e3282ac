"""A/B timing of build-stage variants selected by environment variables that the library reads per
build (not cached): alternates the settings inside one process and prints per-stage medians.
    python tools/ab_probe.py B200SA_MSD_AVG 3000,1500 msd_part [n] [reps]"""
import ctypes as C
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import stralg_b200

var, values, stage = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
n = int(float(sys.argv[4])) if len(sys.argv) > 4 else 3_000_000_000
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 5
lib = stralg_b200.load()
text = torch.empty(n + 1, dtype=torch.uint8, device="cuda")
lib.b200sa_synth_codes(C.c_void_p(text.data_ptr()), n, 4, 12345, 0, None)
res = {v: [] for v in values}
tot = {v: [] for v in values}
for rep in range(reps + 1):
    for v in values:
        os.environ[var] = v
        idx = stralg_b200.SuffixArrayIndex.build(text[:n], 5, profile=True, bwt=True, occ=True)
        prof = idx.profile()
        idx.close()
        if rep:
            res[v].append(sum(ms for name, ms, _ in prof if name == stage))
            tot[v].append(sum(ms for _, ms, _ in prof))
for v in values:
    print(f"{var}={v}: {stage} median {statistics.median(res[v]):.3f} ms (min {min(res[v]):.3f}, max {max(res[v]):.3f}); "
          f"all stages median {statistics.median(tot[v]):.2f} ms")
