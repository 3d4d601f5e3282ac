"""CPU tests of the C ABI's refusals that come before any CUDA call (include/b200sa.h).

Each call runs on a fresh host thread: b200sa_last_error() is per thread and starts empty there, so a
non-empty message proves the refusal wrote one.  Without a device these refusals must still come back
as their own code, not as B200SA_ERR_CUDA: the argument checks run before the library touches a device.
"""
import ctypes as C
import threading

import numpy as np
import pytest

OK, CUDA, BAD_ARGUMENT, BAD_SYMBOL, TOO_LARGE, NOT_BUILT = 0, 1, 2, 3, 4, 5


@pytest.fixture(scope="module")
def lib():
    import stralg_b200
    return stralg_b200.load()


def on_fresh_thread(lib, fn, *args):
    """(return value, last error) of fn(*args) called on a new host thread."""
    out = {}

    def run():
        try:
            out["ret"] = fn(*args)
            out["msg"] = lib.b200sa_last_error()
        except Exception as e:  # (raised again on the test's thread)
            out["exc"] = e

    t = threading.Thread(target=run)
    t.start()
    t.join()
    if "exc" in out:
        raise out["exc"]
    return out["ret"], out["msg"]


def refused(lib, code, fn, *args):
    rc, msg = on_fresh_thread(lib, fn, *args)
    assert rc == code, (fn.__name__, rc, msg)
    assert msg, fn.__name__


def refused_handle(lib, code, fn, *args):
    """A pointer-returning entry point: nullptr, `err` written with `code`, and a message."""
    err = C.c_int(-1)
    h, msg = on_fresh_thread(lib, fn, *args, C.byref(err))
    assert not h, fn.__name__
    assert err.value == code, (fn.__name__, err.value, msg)
    assert msg, fn.__name__


def ptr(a):
    return C.c_void_p(a.ctypes.data)


# A handle for the refusals that happen before the handle is read: zeroed host memory, never dereferenced.
_UNREAD = np.zeros(1 << 20, np.uint8)


def test_null_index_is_refused_by_every_entry_point(lib):
    buf = np.zeros(64, np.uint64)
    p = ptr(buf)
    n = None
    calls = [
        (lib.b200sa_stats, n, n), (lib.b200sa_records, n, C.cast(p, C.POINTER(C.c_uint32)), p), (lib.b200sa_extend, n, p, 0),
        (lib.b200sa_copy_sa, n, p), (lib.b200sa_copy_isa, n, p), (lib.b200sa_copy_lcp, n, p),
        (lib.b200sa_copy_bwt, n, p), (lib.b200sa_copy_occ, n, p), (lib.b200sa_copy_c_table, n, p),
        (lib.b200sa_copy_o_dense, n, p), (lib.b200sa_copy_async, n, 0, p, n),
        (lib.b200sa_occ, n, p, p, 1, p),
        (lib.b200sa_search_batch, n, p, p, 0, 1, p, p),
        (lib.b200sa_search_device, n, p, p, 0, 1, p, p, n),
        (lib.b200sa_search_traffic, n, p, p, 0, 1, p, p, C.cast(p, C.POINTER(C.c_uint64)), n),
        (lib.b200sa_search_batch_packed, n, p, 8, 0, 1, p, p),
        (lib.b200sa_search_device_packed, n, p, 8, 0, 1, p, p, n),
        (lib.b200sa_search_traffic_packed, n, p, 8, 0, 1, p, p, C.cast(p, C.POINTER(C.c_uint64)), n),
        (lib.b200sa_locate_batch, n, p, p, 1, p, p, 8, n),
        (lib.b200sa_locate_batch_sorted, n, p, p, 1, p, p, 8, n),
        (lib.b200sa_locate_device, n, p, p, 1, p, p, 8, n, n),
        (lib.b200sa_sort_positions_device, n, 1, p, 1, p, n),
        (lib.b200sa_sample_sa, n, 8, 0), (lib.b200sa_sa_lookup, n, p, 1, p, 0),
        (lib.b200sa_save, n, b"/dev/null"),
        (lib.b200sa_record_sas_device, n, p, n), (lib.b200sa_copy_record_sas, n, p),
        (lib.b200sa_locate_records, n, p, p, 1, p, p, p, 8, n),
        (lib.b200sa_locate_records_device, n, p, p, 1, p, p, p, 8, n, n),
    ]
    for fn, *args in calls:
        refused(lib, BAD_ARGUMENT, fn, *args)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_replicate, n, 0, n)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_approx_batch, n, n, n, p, n, 4, 1, 1)


def test_null_buffers_without_an_index(lib):
    codes = np.ones(64, np.uint8)
    p = ptr(codes)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_build, None, 10, 5, 0, 0, None)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, None, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads, None, 8, 0, 1, p)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads, p, 8, 0, 1, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads, p, 0, 0, 1, p)  # empty reads
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads_device, None, 8, 0, 1, p, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads_device, p, 8, 0, 1, None, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads_device, p, 0, 0, 1, p, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_synth_codes, None, 10, 4, 1, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_synth_codes, p, 10, 0, 1, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_synth_codes, p, 10, 256, 1, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_synth_reads, None, 10, 4, p, 1, 4, 0, 1, 0, None)
    refused(lib, BAD_ARGUMENT, lib.b200sa_synth_reads, p, 10, 4, None, 1, 4, 0, 1, 0, None)


def test_build_refusals(lib):
    codes = np.ones(8, np.uint8)
    p = ptr(codes)
    for sigma in (0, 257):
        refused_handle(lib, BAD_ARGUMENT, lib.b200sa_build, p, 8, sigma, 0, 0, None)
    refused_handle(lib, TOO_LARGE, lib.b200sa_build, p, 2 ** 32 - 1, 5, 0, 0, None)
    refused_handle(lib, TOO_LARGE, lib.b200sa_build, p, 2 ** 40, 5, 0, 0, None)


def test_build_records_refusals(lib):
    from stralg_b200._lib import BUILD_BWT, BUILD_ISA, BUILD_LCP, BUILD_OCC
    codes = np.full(16, 2, np.uint8)
    off = [0, 5, 16]

    def records(code, codes, off, nrec, sigma, flags=BUILD_OCC):
        off = None if off is None else np.array(off, np.uint64)
        refused_handle(lib, code, lib.b200sa_build_records, None if codes is None else ptr(codes),
                       None if off is None else ptr(off), nrec, sigma, flags, 0, None)

    records(BAD_ARGUMENT, codes, None, 2, 6)  # null offsets
    records(BAD_ARGUMENT, codes, off, 0, 6)  # no record
    for sigma in (0, 1, 2, 257):
        records(BAD_ARGUMENT, codes, off, 2, sigma)
    for flag in (BUILD_ISA, BUILD_LCP, BUILD_BWT, 0x8000):
        records(BAD_ARGUMENT, codes, off, 2, 6, BUILD_OCC | flag)
    records(BAD_ARGUMENT, codes, [1, 5, 16], 2, 6)  # rec_off[0] != 0
    records(BAD_ARGUMENT, codes, [0, 9, 5], 2, 6)  # decreasing offsets
    records(BAD_ARGUMENT, None, off, 2, 6)  # null codes
    records(TOO_LARGE, codes, [0, 2 ** 32 - 1], 1, 6)  # the codes alone
    records(TOO_LARGE, codes, [0, 2 ** 32 - 2], 1, 6)  # codes and one separator
    records(TOO_LARGE, codes, [0, 5, 2 ** 32 - 3], 2, 6)


def test_pack_reads_stride_and_symbols(lib):
    reads = np.array([1, 2, 3, 4, 4, 3, 2, 1, 1], np.uint8)  # one read of 9 bases: 3 bytes
    out = np.full(8, 0xEE, np.uint8)
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads, ptr(reads), 9, 2, 1, ptr(out))
    refused(lib, BAD_ARGUMENT, lib.b200sa_pack_reads_device, ptr(reads), 9, 2, 1, ptr(out), 0, None)
    rc, _ = on_fresh_thread(lib, lib.b200sa_pack_reads, ptr(reads), 9, 4, 1, ptr(out))
    assert rc == OK
    # 2 bits per base, first base in the high bits, code c packed as c - 1, zero padding up to the stride
    assert out[:4].tolist() == [0b00011011, 0b11100100, 0b00000000, 0]
    assert out[4:].tolist() == [0xEE] * 4
    rc, _ = on_fresh_thread(lib, lib.b200sa_pack_reads, ptr(reads), 9, 0, 1, ptr(out))  # stride 0: ceil(9 / 4)
    assert rc == OK and out[:3].tolist() == [0b00011011, 0b11100100, 0]
    for bad in (0, 5, 255):
        r = reads.copy()
        r[4] = bad
        refused(lib, BAD_SYMBOL, lib.b200sa_pack_reads, ptr(r), 9, 0, 1, ptr(out))


def test_refusals_before_the_handle_is_read(lib):
    h = ptr(_UNREAD)
    pats = np.ones(8, np.uint8)
    for edits in (-1, 256):
        refused_handle(lib, BAD_ARGUMENT, lib.b200sa_approx_batch, h, None, None, ptr(pats), None, 8, 1, edits)
    refused(lib, BAD_ARGUMENT, lib.b200sa_sample_sa, h, 0, 0)


def test_bad_replica_lists(lib):
    reads = np.zeros(8, np.uint8)
    L = np.zeros(2, np.uint32)
    arr = (C.c_void_p * 2)(None, None)
    for reps, nrep in ((None, 1), (arr, 0), (arr, 65), (arr, 2)):
        refused(lib, BAD_ARGUMENT, lib.b200sa_search_sharded_packed, reps, nrep, ptr(reads), 8, 0, 1, ptr(L), ptr(L))


def test_load_refusals(lib, tmp_path):
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, None, 0, None)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, str(tmp_path / "missing.b200sa").encode(), 0, None)
