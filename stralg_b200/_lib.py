"""ctypes loader for libb200sa.so (the C ABI of include/b200sa.h).

The library is built in-tree by ``make -C stralg_b200/csrc`` (``__graft_entry__.build()``).
There is no fallback: if the shared object is missing, importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200sa.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)

# build flags (include/b200sa.h)
BUILD_ISA = 0x1
BUILD_LCP = 0x2
BUILD_BWT = 0x4
BUILD_OCC = 0x8
BUILD_TEXTCMP = 0x10
BUILD_KTABLE = 0x20
TEXT_ON_DEVICE = 0x100
PROFILE = 0x200
DROP_SA = 0x400

ERROR_NAMES = {
    0: "OK", 1: "CUDA", 2: "BAD_ARGUMENT", 3: "BAD_SYMBOL", 4: "TOO_LARGE",
    5: "NOT_BUILT", 6: "OUT_OF_MEMORY", 7: "INTERNAL",
}


class Stats(C.Structure):
    _fields_ = [
        ("length", C.c_uint32), ("sigma", C.c_uint32), ("primary", C.c_uint32), ("rounds", C.c_uint32),
        ("k0", C.c_uint32), ("radix_bits", C.c_uint32), ("passes0", C.c_uint32), ("occ_layout", C.c_uint32),
        ("sorted_total", C.c_uint64), ("passes_elems", C.c_uint64), ("occ_bytes", C.c_uint64),
        ("round0_mode", C.c_uint32), ("bucket_bits", C.c_uint32),
        ("sa_sample_rate", C.c_uint32), ("sa_resident", C.c_uint32),
        ("shallow_buckets", C.c_uint32), ("chain_rounds", C.c_uint32), ("shallow_elems", C.c_uint64),
        ("chain_elems", C.c_uint64), ("lazy_lookups", C.c_uint64), ("resolved_small", C.c_uint64),
        ("small_path_elems", C.c_uint64), ("pivot_elems", C.c_uint64), ("pivot_rounds", C.c_uint32),
        ("pair_placed", C.c_uint32),
        ("ktable_k", C.c_uint32), ("dense_keys", C.c_uint32),
    ]


# every symbol include/b200sa.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "b200sa_build": (C.c_void_p, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                  C.POINTER(C.c_int)]),
    "b200sa_extend": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "b200sa_free": (None, [C.c_void_p]),
    "b200sa_last_error": (C.c_char_p, []),
    "b200sa_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "b200sa_profile": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_float),
                                 C.POINTER(C.c_double), C.c_int]),
    "b200sa_device_sa": (C.c_void_p, [C.c_void_p]),
    "b200sa_device_isa": (C.c_void_p, [C.c_void_p]),
    "b200sa_device_lcp": (C.c_void_p, [C.c_void_p]),
    "b200sa_device_bwt": (C.c_void_p, [C.c_void_p]),
    "b200sa_device_occ": (C.c_void_p, [C.c_void_p]),
    "b200sa_copy_sa": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_isa": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_lcp": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_bwt": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_c_table": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_occ": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_copy_async": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "b200sa_launch_count": (C.c_uint64, []),
    "b200sa_workspace_bytes": (C.c_uint64, [C.c_int]),
    "b200sa_release_workspace": (C.c_int, [C.c_int]),
    "b200sa_plan_round0": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "b200sa_copy_o_dense": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_occ": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200sa_search_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64,
                                      C.c_void_p, C.c_void_p]),
    "b200sa_search_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sa_search_traffic": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64,
                                        C.c_void_p, C.c_void_p, u64p, C.c_void_p]),
    "b200sa_search_batch_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64,
                                             C.c_void_p, C.c_void_p]),
    "b200sa_search_device_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64,
                                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sa_search_traffic_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64,
                                               C.c_void_p, C.c_void_p, u64p, C.c_void_p]),
    "b200sa_replicate": (C.c_void_p, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "b200sa_search_sharded_packed": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_uint32, C.c_uint32,
                                               C.c_uint64, C.c_void_p, C.c_void_p]),
    "b200sa_pack_reads": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]),
    "b200sa_pack_reads_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_int,
                                           C.c_void_p]),
    "b200sa_locate_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                      C.c_void_p, C.c_uint64, u64p]),
    "b200sa_locate_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                       C.c_void_p, C.c_uint64, u64p, C.c_void_p]),
    "b200sa_locate_batch_sorted": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                             C.c_void_p, C.c_uint64, u64p]),
    "b200sa_sort_positions_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                               C.c_void_p]),
    "b200sa_sample_sa": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int]),
    "b200sa_sa_lookup": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]),
    "b200sa_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "b200sa_load": (C.c_void_p, [C.c_char_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "b200sa_approx_batch": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                         C.c_uint64, C.c_int, C.POINTER(C.c_int)]),
    "b200sa_approx_hits": (C.c_uint64, [C.c_void_p]),
    "b200sa_approx_hit_offsets": (u64p, [C.c_void_p]),
    "b200sa_approx_L": (u32p, [C.c_void_p]),
    "b200sa_approx_R": (u32p, [C.c_void_p]),
    "b200sa_approx_match_length": (u32p, [C.c_void_p]),
    "b200sa_approx_cigar_offsets": (u64p, [C.c_void_p]),
    "b200sa_approx_cigars": (C.POINTER(C.c_char), [C.c_void_p]),
    "b200sa_approx_free": (None, [C.c_void_p]),
    "b200sa_matching_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "b200sa_smem_batch": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32,
                                       C.POINTER(C.c_int)]),
    "b200sa_smem_count": (C.c_uint64, [C.c_void_p]),
    "b200sa_smem_offsets": (u64p, [C.c_void_p]),
    "b200sa_smem_start": (u32p, [C.c_void_p]),
    "b200sa_smem_length": (u32p, [C.c_void_p]),
    "b200sa_smem_L": (u32p, [C.c_void_p]),
    "b200sa_smem_R": (u32p, [C.c_void_p]),
    "b200sa_smem_free": (None, [C.c_void_p]),
    "b200sa_synth_codes": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]),
    "b200sa_synth_reads": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint32,
                                     C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]),
    "b200sa_device_count": (C.c_int, []),
    "b200sa_build_records": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                          C.c_void_p, C.POINTER(C.c_int)]),
    "b200sa_records": (C.c_int, [C.c_void_p, u32p, C.c_void_p]),
    "b200sa_copy_record_sas": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200sa_record_sas_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sa_locate_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_uint64, u64p]),
    "b200sa_locate_records_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_uint64, u64p, C.c_void_p]),
}


class B200saError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"b200sa error {ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


_lib = None


def load():
    """Load libb200sa.so and bind every declared entry point.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C stralg_b200/csrc` "
            "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise B200saError(rc, load().b200sa_last_error().decode())
