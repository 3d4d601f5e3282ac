"""Short workloads to run UNDER ncu (one GPU):  python tools/ncu_target.py build|search|repeat|stress:<kind> [n] [reads]
build : two builds of n random ACGT symbols (SA + BWT + C + O)          -> round-0 kernels
repeat: one build of the repeat-rich text (SURVEY 8(d) C3)               -> doubling / chain kernels
stress:<kind>: one build (SA only) of a config-5 text (unary, acgt4, period1000, fib)      -> pivot path kernels
search: index of n symbols (k-mer table + text comparison), `reads` 100-bp reads, byte and packed kernels
Numbers printed by a run under ncu are never bench values."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import stralg_b200  # noqa: E402
from stralg_b200 import texts as T  # noqa: E402

lib = stralg_b200.load()
what = sys.argv[1] if len(sys.argv) > 1 else "build"
n = int(float(sys.argv[2])) if len(sys.argv) > 2 else 3_000_000_000
reads_n = int(float(sys.argv[3])) if len(sys.argv) > 3 else 100_000_000
text = None if what.startswith("stress:") else T.random_codes(lib, n, 4, T.SEED)
if what.startswith("stress:"):
    text, sigma = T.stress_text(lib, what.split(":")[1], n)
    torch.cuda.synchronize()
    idx = stralg_b200.SuffixArrayIndex.build(text[:n], sigma, occ=False)
    print(idx.stats())
    idx.close()
elif what == "build":
    for _ in range(2):
        stralg_b200.SuffixArrayIndex.build(text[:n], 5, occ=True).close()
elif what == "repeat":
    T.add_repeats(text, n)
    torch.cuda.synchronize()
    stralg_b200.SuffixArrayIndex.build(text[:n], 5, occ=True).close()
else:
    idx = stralg_b200.SuffixArrayIndex.build(text[:n], 5, occ=True, textcmp=True, ktable=True)
    lib.b200sa_release_workspace(0)
    m, stride = 100, 25
    r = torch.empty(reads_n * m, dtype=torch.uint8, device="cuda")
    assert lib.b200sa_synth_reads(C.c_void_p(text.data_ptr()), n, 4, C.c_void_p(r.data_ptr()), reads_n, m, 102, 7, 0, None) == 0
    p = torch.zeros(reads_n * stride + 8, dtype=torch.uint8, device="cuda")
    assert lib.b200sa_pack_reads_device(C.c_void_p(r.data_ptr()), m, stride, reads_n, C.c_void_p(p.data_ptr()), 0, None) == 0
    L = torch.empty(reads_n, dtype=torch.int32, device="cuda")
    R = torch.empty(reads_n, dtype=torch.int32, device="cuda")
    for _ in range(2):
        idx.search_device(r, None, m, reads_n, L, R)
        idx.search_device_packed(p, m, reads_n, L, R, stride)
    torch.cuda.synchronize()
    for name, fn in (("byte", lambda: idx.search_device(r, None, m, reads_n, L, R)),
                     ("packed", lambda: idx.search_device_packed(p, m, reads_n, L, R, stride))):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        print(f"{name} kernel: {e0.elapsed_time(e1) / 5:.3f} ms for {reads_n} reads")
    idx.close()
torch.cuda.synchronize()
print("done", what, n)
