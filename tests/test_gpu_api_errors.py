"""The C ABI's refusals that need a real index (include/b200sa.h), each with its error code, and the
`err` out-parameter of the pointer-returning entry points on success.  Refusals that come before any
CUDA call are in test_api_errors.py; the records-index refusals are in test_gpu_records.py."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OK, BAD_ARGUMENT, BAD_SYMBOL, TOO_LARGE, NOT_BUILT, INTERNAL = 0, 2, 3, 4, 5, 7
TABLE_SA, TABLE_ISA, TABLE_LCP, TABLE_BWT, TABLE_OCC = range(5)


def ptr(a):
    return C.c_void_p(a.ctypes.data)


def dptr(t):
    return C.c_void_p(t.data_ptr())


def refused(lib, code, fn, *args):
    rc = fn(*args)
    assert rc == code, (fn.__name__, rc, lib.b200sa_last_error())
    assert lib.b200sa_last_error(), fn.__name__


def refused_handle(lib, code, fn, *args):
    err = C.c_int(-1)
    h = fn(*args, C.byref(err))
    assert not h, fn.__name__
    assert err.value == code, (fn.__name__, err.value, lib.b200sa_last_error())
    assert lib.b200sa_last_error(), fn.__name__


@pytest.fixture(scope="module")
def dna(oracle):
    return oracle.random_codes(5000, 4, seed=11)


def test_tables_that_were_not_built(engine, dna):
    lib = engine.load()
    host = np.zeros(1 << 16, np.uint64)
    h = ptr(host)
    bare = engine.SuffixArrayIndex.build(dna[:-1], 5, occ=False)
    for fn in (lib.b200sa_copy_isa, lib.b200sa_copy_lcp, lib.b200sa_copy_bwt, lib.b200sa_copy_occ,
               lib.b200sa_copy_o_dense):
        refused(lib, NOT_BUILT, fn, bare._h, h)
    for table in (TABLE_ISA, TABLE_LCP, TABLE_BWT, TABLE_OCC):
        refused(lib, NOT_BUILT, lib.b200sa_copy_async, bare._h, table, h, None)
    for table in (-1, 5):
        refused(lib, BAD_ARGUMENT, lib.b200sa_copy_async, bare._h, table, h, None)
    a = np.array([1, 2], np.uint8)
    i = np.array([3, 4], np.uint32)
    refused(lib, NOT_BUILT, lib.b200sa_occ, bare._h, ptr(a), ptr(i), 2, h)
    pats = np.array([1, 2, 3, 4] * 4, np.uint8)
    L = np.zeros(4, np.uint32)
    R = np.zeros(4, np.uint32)
    refused(lib, NOT_BUILT, lib.b200sa_search_batch, bare._h, ptr(pats), None, 4, 4, ptr(L), ptr(R))
    import torch
    d_pats = torch.from_numpy(pats).cuda()
    d_L = torch.empty(4, dtype=torch.int32, device="cuda")
    d_R = torch.empty_like(d_L)
    refused(lib, NOT_BUILT, lib.b200sa_search_device, bare._h, dptr(d_pats), None, 4, 4, dptr(d_L), dptr(d_R), None)
    refused_handle(lib, NOT_BUILT, lib.b200sa_approx_batch, bare._h, None, None, ptr(pats), None, 4, 4, 1)
    refused(lib, NOT_BUILT, lib.b200sa_sample_sa, bare._h, 8, 0)
    assert np.array_equal(bare.sa(), engine.SuffixArrayIndex.build(dna[:-1], 5).sa())  # still usable
    bare.close()

    dropped = engine.SuffixArrayIndex.build(dna[:-1], 5, drop_sa=True)
    refused(lib, NOT_BUILT, lib.b200sa_copy_sa, dropped._h, h)
    refused(lib, NOT_BUILT, lib.b200sa_copy_async, dropped._h, TABLE_SA, h, None)
    refused(lib, NOT_BUILT, lib.b200sa_extend, dropped._h, ptr(dna), 0x1)
    refused(lib, NOT_BUILT, lib.b200sa_sample_sa, dropped._h, 8, 0)
    dropped.close()


def test_null_buffers_with_an_index(engine, dna):
    lib = engine.load()
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5, isa=True, lcp=True, bwt=True)
    host = np.zeros(1 << 16, np.uint64)
    h = ptr(host)
    n = None
    for fn in (lib.b200sa_copy_sa, lib.b200sa_copy_isa, lib.b200sa_copy_lcp, lib.b200sa_copy_bwt, lib.b200sa_copy_occ,
               lib.b200sa_copy_c_table, lib.b200sa_copy_o_dense, lib.b200sa_copy_record_sas):
        refused(lib, BAD_ARGUMENT, fn, idx._h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_copy_async, idx._h, TABLE_SA, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_stats, idx._h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_records, idx._h, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_save, idx._h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_occ, idx._h, n, h, 1, h)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_batch, idx._h, n, n, 4, 1, h, h)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_batch, idx._h, h, n, 4, 1, n, h)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_device, idx._h, n, n, 4, 1, h, h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_batch_packed, idx._h, n, 8, 0, 1, h, h)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_device_packed, idx._h, n, 8, 0, 1, h, h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_traffic, idx._h, h, n, 4, 1, h, h, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_traffic_packed, idx._h, h, 8, 0, 1, h, h, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_batch, idx._h, h, h, 1, n, n, 0, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_batch_sorted, idx._h, n, h, 1, h, n, 0, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_device, idx._h, h, h, 1, n, n, 0, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_sort_positions_device, idx._h, 1, n, 1, h, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_sort_positions_device, idx._h, 1, h, 1, n, n)
    refused(lib, BAD_ARGUMENT, lib.b200sa_sa_lookup, idx._h, n, 1, h, 0)
    refused(lib, BAD_ARGUMENT, lib.b200sa_extend, idx._h, n, 0x1)
    refused(lib, BAD_ARGUMENT, lib.b200sa_record_sas_device, idx._h, n, n)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_approx_batch, idx._h, n, n, n, n, 4, 1, 1)
    # a packed read of zero length, and a packed buffer off the 8-byte grid
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_batch_packed, idx._h, h, 0, 0, 1, h, h)
    import torch
    d = torch.zeros(64, dtype=torch.uint8, device="cuda")
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_device_packed, idx._h, C.c_void_p(d.data_ptr() + 1), 8, 0, 1,
            dptr(d), dptr(d), n)
    # out-of-range queries
    sym, row, end = np.array([5], np.uint8), np.array([0], np.uint32), np.array([idx.length], np.uint32)
    refused(lib, BAD_ARGUMENT, lib.b200sa_occ, idx._h, ptr(sym), ptr(row), 1, h)
    refused(lib, BAD_ARGUMENT, lib.b200sa_sa_lookup, idx._h, ptr(end), 1, h, 0)
    assert np.array_equal(idx.c_table(), engine.SuffixArrayIndex.build(dna[:-1], 5).c_table())
    idx.close()


def test_traffic_counters_need_the_dna_kernel(engine, oracle):
    import torch
    lib = engine.load()
    codes = oracle.random_codes(5000, 20, seed=4)
    big = engine.SuffixArrayIndex.build(codes[:-1], 21)
    d = torch.zeros(64, dtype=torch.uint8, device="cuda") + 1
    d_L = torch.empty(4, dtype=torch.int32, device="cuda")
    counts = (C.c_uint64 * 4)()
    refused(lib, NOT_BUILT, lib.b200sa_search_traffic, big._h, dptr(d), None, 4, 4, dptr(d_L), dptr(d_L), counts, None)
    refused(lib, NOT_BUILT, lib.b200sa_search_traffic_packed, big._h, dptr(d), 8, 0, 4, dptr(d_L), dptr(d_L), counts,
            None)
    big.close()
    dna = engine.SuffixArrayIndex.build(oracle.random_codes(5000, 4, seed=4)[:-1], 5)
    # (the DNA kernel reads its patterns in 8-byte words)
    refused(lib, NOT_BUILT, lib.b200sa_search_traffic, dna._h, C.c_void_p(d.data_ptr() + 1), None, 4, 4, dptr(d_L),
            dptr(d_L), counts, None)
    assert lib.b200sa_search_traffic(dna._h, dptr(d), None, 4, 4, dptr(d_L), dptr(d_L), counts, None) == OK
    dna.close()


def test_two_replicas_on_one_device(engine, dna):
    lib = engine.load()
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5)
    packed = engine.pack_reads(dna[:64], 8)
    L = np.zeros(8, np.uint32)
    arr = (C.c_void_p * 2)(idx._h.value, idx._h.value)
    refused(lib, BAD_ARGUMENT, lib.b200sa_search_sharded_packed, arr, 2, ptr(packed), 8, 0, 8, ptr(L), ptr(L))
    idx.close()


def test_extend_with_another_text(engine, dna, oracle):
    from stralg_b200 import B200saError
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5)
    other = oracle.random_codes(5000, 4, seed=12)
    with pytest.raises(B200saError) as e:
        idx.extend(other[:-1], isa=True)
    assert e.value.code == BAD_ARGUMENT
    bad = dna[:-1].copy()
    bad[100] = 7
    with pytest.raises(B200saError) as e:
        idx.extend(bad, isa=True)
    assert e.value.code == BAD_SYMBOL
    # the index is what it was: it still searches, and extends with its own text
    sa = oracle.sa(dna)
    pat = dna[200:212].copy()
    L, R = idx.search(pat, fixed_len=12)
    off, pos = idx.locate(L, R)
    assert 200 in pos.tolist() and np.array_equal(np.sort(pos), np.sort(oracle.locate(sa, L, R)[1]))
    idx.extend(dna[:-1], isa=True)
    assert np.array_equal(idx.isa(), oracle.inverse(sa))
    L2, R2 = idx.search(pat, fixed_len=12)
    assert np.array_equal(L2, L) and np.array_equal(R2, R)
    idx.close()


def test_locate_capacity_too_small(engine, dna):
    import torch
    lib = engine.load()
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5)
    pat = np.array([1, 2], np.uint8)  # a 2-mer of a 5000-symbol text: many positions
    L, R = idx.search(pat, fixed_len=2)
    total = int(R[0] - L[0])
    assert total > 1
    off = np.zeros(2, np.uint64)
    pos = np.zeros(total, np.uint32)
    for fn in (lib.b200sa_locate_batch, lib.b200sa_locate_batch_sorted):
        refused(lib, BAD_ARGUMENT, fn, idx._h, ptr(L), ptr(R), 1, ptr(off), ptr(pos), total - 1, None)
    d_L = torch.from_numpy(L.view(np.int32)).cuda()
    d_R = torch.from_numpy(R.view(np.int32)).cuda()
    d_off = torch.zeros(2, dtype=torch.int64, device="cuda")
    d_pos = torch.zeros(total, dtype=torch.int32, device="cuda")
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_device, idx._h, dptr(d_L), dptr(d_R), 1, dptr(d_off), dptr(d_pos),
            total - 1, None, None)
    idx.close()
    rec = engine.SuffixArrayIndex.build_records([dna[:2000] + 1, dna[2000:4000] + 1], 6)
    pat = np.array([2, 3], np.uint8)
    L, R = rec.search(pat, fixed_len=2)
    total = int(R[0] - L[0])
    assert total > 1
    rpos = np.zeros(total, np.uint32)
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_records, rec._h, ptr(L), ptr(R), 1, ptr(off), ptr(rpos), ptr(rpos),
            total - 1, None)
    d_L = torch.from_numpy(L.view(np.int32)).cuda()
    d_R = torch.from_numpy(R.view(np.int32)).cuda()
    refused(lib, BAD_ARGUMENT, lib.b200sa_locate_records_device, rec._h, dptr(d_L), dptr(d_R), 1, dptr(d_off),
            dptr(d_pos), dptr(d_pos), total - 1, None, None)
    rec.close()


def test_sort_positions_beyond_u32(engine, dna):
    import torch
    lib = engine.load()
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5)
    d = torch.zeros(16, dtype=torch.int64, device="cuda")
    refused(lib, TOO_LARGE, lib.b200sa_sort_positions_device, idx._h, 1, dptr(d), 2 ** 32, dptr(d), None)
    refused(lib, TOO_LARGE, lib.b200sa_sort_positions_device, idx._h, 2 ** 32, dptr(d), 1, dptr(d), None)
    idx.close()


def _sa_only_file(engine, tmp_path, codes):
    """An index file that holds one section, the suffix array, at its end: (bytes, offset of the section header)."""
    idx = engine.SuffixArrayIndex.build(codes, 5, occ=False)
    path = tmp_path / "sa_only.b200sa"
    idx.save(path)
    blob = bytearray(path.read_bytes())
    data = 4 * idx.length
    at = len(blob) - (data + (-data) % 8) - 24  # {tag[8], elem_bytes, count}, the array, its padding
    assert bytes(blob[at:at + 8]) == b"SA" + bytes(6)
    assert int.from_bytes(blob[at + 16:at + 24], "little") == idx.length
    idx.close()
    return blob, at


def test_load_refusals(engine, dna, tmp_path):
    lib = engine.load()
    blob, at = _sa_only_file(engine, tmp_path, dna[:-1])

    def load(b):
        p = tmp_path / "case.b200sa"
        p.write_bytes(bytes(b))
        return str(p).encode()

    good = load(blob)
    err = C.c_int(-1)
    h = lib.b200sa_load(good, 0, None, C.byref(err))
    assert h and err.value == OK
    lib.b200sa_free(C.c_void_p(h))

    magic = bytearray(blob)
    magic[:8] = b"B200SAIY"
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, load(magic), 0, None)
    version = bytearray(blob)
    version[8:12] = (3).to_bytes(4, "little")
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, load(version), 0, None)
    unknown = bytearray(blob)
    unknown[at:at + 8] = b"XA" + bytes(6)
    refused_handle(lib, BAD_ARGUMENT, lib.b200sa_load, load(unknown), 0, None)
    # cut off inside the suffix array's data: a short read of a section is an INTERNAL error
    refused_handle(lib, INTERNAL, lib.b200sa_load, load(blob[:at + 24 + 4000]), 0, None)
    # a section of the wrong shape: INTERNAL as well
    shape = bytearray(blob)
    shape[at + 16:at + 24] = (int.from_bytes(blob[at + 16:at + 24], "little") - 1).to_bytes(8, "little")
    refused_handle(lib, INTERNAL, lib.b200sa_load, load(shape), 0, None)


def test_save_to_an_unopenable_path(engine, dna, tmp_path):
    lib = engine.load()
    idx = engine.SuffixArrayIndex.build(dna[:-1], 5)
    refused(lib, BAD_ARGUMENT, lib.b200sa_save, idx._h, str(tmp_path / "no_such_dir" / "x.b200sa").encode())
    idx.close()


def test_err_is_written_on_success(engine, dna, tmp_path):
    lib = engine.load()
    text = np.ascontiguousarray(dna[:-1])
    err = C.c_int(-1)
    h = lib.b200sa_build(ptr(text), text.size, 5, 0x8, 0, None, C.byref(err))
    assert h and err.value == OK
    err.value = -1
    rep = lib.b200sa_replicate(C.c_void_p(h), 0, None, C.byref(err))
    assert rep and err.value == OK
    lib.b200sa_free(C.c_void_p(rep))
    path = str(tmp_path / "ok.b200sa").encode()
    assert lib.b200sa_save(C.c_void_p(h), path) == OK
    err.value = -1
    back = lib.b200sa_load(path, 0, None, C.byref(err))
    assert back and err.value == OK
    lib.b200sa_free(C.c_void_p(back))
    pats = np.ascontiguousarray(text[:32])
    for npat in (0, 2):
        err.value = -1
        res = lib.b200sa_approx_batch(C.c_void_p(h), None, None, ptr(pats), None, 16, npat, 1, C.byref(err))
        assert res and err.value == OK
        assert lib.b200sa_approx_hits(res) >= npat
        lib.b200sa_approx_free(res)
    lib.b200sa_free(C.c_void_p(h))
    recs = np.ascontiguousarray(dna[:300] + 1)
    off = np.array([0, 100, 300], np.uint64)
    err.value = -1
    h = lib.b200sa_build_records(ptr(recs), ptr(off), 2, 6, 0x8, 0, None, C.byref(err))
    assert h and err.value == OK
    lib.b200sa_free(C.c_void_p(h))
