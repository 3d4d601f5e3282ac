"""End-to-end times of b200sa_approx_batch on a synthetic DNA index."""
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import stralg_b200

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 28
reads_n = int(sys.argv[2]) if len(sys.argv) > 2 else 200000
m = 100
lib = stralg_b200.load()
text = torch.empty(n + 1, dtype=torch.uint8, device="cuda")
lib.b200sa_synth_codes(C.c_void_p(text.data_ptr()), n, 4, 1, 0, None)
reads = torch.empty(reads_n * m, dtype=torch.uint8, device="cuda")
lib.b200sa_synth_reads(C.c_void_p(text.data_ptr()), n, 4, C.c_void_p(reads.data_ptr()), reads_n, m, 102, 2, 0, None)
idx = stralg_b200.SuffixArrayIndex.build(text[:n], 5)
rev = stralg_b200.SuffixArrayIndex.build(torch.flip(text[:n], dims=[0]).contiguous(), 5, drop_sa=True)
h = reads.cpu().numpy()
for d, cnt in ((1, reads_n), (1, reads_n), (2, reads_n // 20)):
    for use_rev in (True, False):
        t0 = time.perf_counter()
        r = idx.approx_search(h[: cnt * m], fixed_len=m, max_edits=d, rev=rev if use_rev else None)
        print(f"d={d} reads={cnt} rev={use_rev}: {time.perf_counter() - t0:.3f} s, {len(r['L'])} intervals", flush=True)
