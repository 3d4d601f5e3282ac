"""GPU tests of the records index (include/b200sa.h: b200sa_build_records): one build over many records
answers for every record exactly like that record's own index -- suffix arrays, exact search + locate,
approximate search + locate in report order -- and bwt_map_fastq_records writes the SAM of
bwt_map_fastq byte for byte."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ACGT = np.array([2, 3, 4, 5], np.uint8)


def own(rec):
    """A record's codes in its own alphabet (the letters it holds, 1.., in code order) and that sigma; the
    map union code -> own code (0 = absent)."""
    rec = np.asarray(rec, np.uint8)
    letters = np.unique(rec)
    m = np.zeros(256, np.uint8)
    m[letters] = np.arange(1, len(letters) + 1)
    return m[rec], len(letters) + 1, m


def own_index(engine, rec, **kw):
    codes, sigma, m = own(rec)
    return engine.SuffixArrayIndex.build(codes, max(sigma, 2), **kw), m


def records_case(name, rng):
    if name == "one":
        return [rng.choice(ACGT, 5000)]
    if name == "two":
        return [rng.choice(ACGT, 3000), rng.choice(ACGT, 1700)]
    if name == "random300":
        return [rng.choice(ACGT, int(rng.integers(0, 2001))) for _ in range(300)]
    if name == "copies100":
        r = rng.choice(ACGT, 700)
        return [r] * 100
    if name == "alphabets":  # ACGT, ACGTN, 20 letters
        return [rng.choice(ACGT, 4000), rng.choice(np.arange(2, 7, dtype=np.uint8), 3000),
                rng.integers(2, 22, 5000).astype(np.uint8), rng.choice(ACGT, 10)]
    if name == "periodic":
        return [np.tile(np.array([2, 3, 3, 5], np.uint8), 3000), rng.choice(ACGT, 9000)]
    if name == "large":  # >= 2^20 symbols: the bucketed initial sort
        return [rng.choice(ACGT, int(rng.integers(20000, 60000))) for _ in range(30)]
    raise KeyError(name)


def sigma_of(records):
    return int(max(int(r.max()) for r in records if len(r))) + 1


@pytest.mark.parametrize("mode", ["default", "lsd"])
@pytest.mark.parametrize("case", ["one", "two", "random300", "copies100", "alphabets", "periodic", "large"])
def test_record_sas_equal_own_builds(engine, case, mode, monkeypatch):
    if mode == "lsd":
        monkeypatch.setenv("B200SA_ROUND0", "lsd")
    rng = np.random.default_rng(sum(case.encode()))
    records = records_case(case, rng)
    idx = engine.SuffixArrayIndex.build_records(records, sigma_of(records), occ=False)
    off = idx.record_offsets()
    assert np.array_equal(off, np.concatenate([[0], np.cumsum([len(r) for r in records])]).astype(np.uint64))
    assert idx.length == sum(len(r) for r in records) + len(records) + 1
    sas = idx.record_sas()
    assert len(sas) == len(records)
    cache = {}
    for r, rec in enumerate(records):
        if len(rec) == 0:
            assert np.array_equal(sas[r], [0])
            continue
        key = rec.tobytes()
        if key not in cache:
            oi, _ = own_index(engine, rec, occ=False)
            cache[key] = oi.sa()
        assert np.array_equal(sas[r], cache[key]), (case, r)


def expected_exact(engine, records, owns, pats):
    """Per pattern: [(record, position)] from every record's own index, records ascending, own SA order."""
    out = [[] for _ in pats]
    for r, (oi, m) in enumerate(owns):
        if oi is None:
            continue
        ok = [k for k, p in enumerate(pats) if (m[p] > 0).all()]
        if not ok:
            continue
        mp = [m[pats[k]] for k in ok]
        off = np.zeros(len(ok) + 1, np.uint64)
        off[1:] = np.cumsum([len(p) for p in mp])
        L, R = oi.search(np.concatenate(mp), off)
        poff, pos = oi.locate(L, R)
        for j, k in enumerate(ok):
            out[k].extend((r, int(x)) for x in pos[poff[j]:poff[j + 1]])
    return [sorted(e, key=lambda t: t[0]) for e in out]  # (stable: SA order kept inside a record)


def got_exact(off, rec, pos):
    return [[(int(rec[e]), int(pos[e])) for e in range(int(off[k]), int(off[k + 1]))] for k in range(len(off) - 1)]


def exact_patterns(rng, records, n_in=600, n_span=100, n_miss=100):
    pats, span = [], []
    nonempty = [r for r in records if len(r) > 0]
    for _ in range(n_in):
        rec = nonempty[int(rng.integers(0, len(nonempty)))]
        m = int(rng.integers(1, min(20, len(rec)) + 1))
        s = int(rng.integers(0, len(rec) - m + 1))
        pats.append(rec[s:s + m].copy())
    for _ in range(n_span):  # the end of one record followed by the start of the next, without the separator
        k = int(rng.integers(0, len(records) - 1))
        a, b = records[k], records[k + 1]
        if len(a) < 15 or len(b) < 15:
            continue
        span.append(len(pats))
        pats.append(np.concatenate([a[-15:], b[:15]]))
    for _ in range(n_miss):
        pats.append(rng.choice(ACGT, int(rng.integers(18, 30))))
    return pats, span


@pytest.mark.parametrize("sampled,textcmp", [(False, False), (True, False), (False, True)],
                         ids=["full_sa", "sampled_sa", "textcmp"])
def test_exact_search_and_locate_records(engine, sampled, textcmp):
    rng = np.random.default_rng(11)
    records = [rng.choice(ACGT, int(rng.integers(0, 3000))) for _ in range(40)]
    records[5] = rng.choice(ACGT[:3], 2000)                       # no T
    records[6] = rng.choice(np.arange(2, 7, dtype=np.uint8), 2500)  # ACGTN
    records[7] = records[8].copy()                                 # identical records
    idx = engine.SuffixArrayIndex.build_records(records, 7, textcmp=textcmp, ktable=textcmp)
    if sampled:
        idx.sample_sa(8, drop_sa=True)
        assert idx.stats()["sa_resident"] == 0
    owns = [own_index(engine, r) if len(r) else (None, None) for r in records]
    pats, span = exact_patterns(rng, records)
    off = np.zeros(len(pats) + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    L, R = idx.search(np.concatenate(pats), off)
    poff, rec, pos = idx.locate_records(L, R)
    got = got_exact(poff, rec, pos)
    assert got == expected_exact(engine, records, owns, pats)
    assert span and all(got[k] == [] for k in span)
    assert sum(len(g) for g in got) > len(pats) // 2


def approx_by_record(engine, idx, rev, records, owns, pats, d):
    off = np.zeros(len(pats) + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    res = idx.approx_search(np.concatenate(pats), off, max_edits=d, rev=rev)
    poff, rec, pos = idx.locate_records(res["L"], res["R"])
    for r, (oi, m) in enumerate(owns):
        if oi is None:
            continue
        for k, p in enumerate(pats):
            if not (m[p] > 0).all():  # the skip rule: the record's own table has no code for a letter of p
                continue
            want = []
            o = oi.approx_search(m[p], np.array([0, len(p)], np.uint64), max_edits=d)
            ooff, opos = oi.locate(o["L"], o["R"])
            for h in range(len(o["L"])):
                want.append((o["cigars"][h], int(o["match_length"][h]), opos[ooff[h]:ooff[h + 1]].tolist()))
            have = []
            for h in range(int(res["offsets"][k]), int(res["offsets"][k + 1])):
                e = range(int(poff[h]), int(poff[h + 1]))
                ps = [int(pos[x]) for x in e if rec[x] == r]
                if ps:
                    have.append((res["cigars"][h], int(res["match_length"][h]), ps))
            assert have == want, (r, k, d)


@pytest.mark.parametrize("d", [1, 2])
@pytest.mark.parametrize("use_rev", [False, True], ids=["no_dtable", "dtable"])
def test_approx_search_per_record_equals_own_index(engine, d, use_rev):
    rng = np.random.default_rng(20 + d)
    records = [rng.choice(ACGT, int(rng.integers(200, 1500))) for _ in range(7)]
    records[2] = rng.choice(ACGT[:3], 900)  # no T
    records[4] = records[3][:400].copy()     # a prefix of another record
    sigma = 6
    idx = engine.SuffixArrayIndex.build_records(records, sigma)
    rev = None
    if use_rev:  # index of the reversed text, separators included
        text = np.concatenate([np.concatenate([r, [1]]) for r in records]).astype(np.uint8)
        rev = engine.SuffixArrayIndex.build(text[::-1].copy(), sigma)
    owns = [own_index(engine, r) for r in records]
    pats = []
    for k in range(120):
        rec = records[k % len(records)]
        m = int(rng.integers(6, 16))
        s = int(rng.integers(0, len(rec) - m))
        p = rec[s:s + m].copy()
        for _ in range(int(rng.integers(0, d + 2))):
            p[int(rng.integers(0, m))] = ACGT[int(rng.integers(0, 4))]
        pats.append(p)
    approx_by_record(engine, idx, rev, records, owns, pats, d)


# ---- the drop-in --------------------------------------------------------------------------------
def _compat(engine):
    from test_compat import COMPAT_SO, bind_extra, bind_mapper
    from _oracle import RefBwtTable
    lib = bind_mapper(bind_extra(C.CDLL(COMPAT_SO)))
    lib.bwt_map_fastq_records.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_char_p),
                                          C.POINTER(C.POINTER(RefBwtTable)), C.c_int, C.c_uint64]
    lib.bwt_map_fastq_records.restype = C.c_uint64
    return lib


def _map(compat, fn, recs, tbls, fq_path, out_path, edits, batch_reads=0):
    from _oracle import RefBwtTable
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    names = (C.c_char_p * len(recs))(*[n.encode() for n, _ in recs])
    tarr = (C.POINTER(RefBwtTable) * len(recs))(*tbls)
    fq = libc.fopen(str(fq_path).encode(), b"r")
    out = libc.fopen(str(out_path).encode(), b"w")
    lines = getattr(compat, fn)(fq, out, len(recs), names, tarr, edits, batch_reads)
    libc.fclose(fq)
    libc.fclose(out)
    return lines, open(out_path, "rb").read()


@pytest.mark.parametrize("edits,expected", [(0, "expected.sam"), (1, "expected_d1.sam"), (2, "expected_d2.sam")])
def test_map_fastq_records_reproduces_reference_tool(engine, tmp_path, edits, expected):
    from test_compat import cbuf, read_fasta
    from _oracle import u8p
    from conftest import ROOT
    compat = _compat(engine)
    gdir = os.path.join(ROOT, "tests", "golden", "readmapper")
    recs = read_fasta(os.path.join(gdir, "ref.fa"))
    tbls = [compat.build_complete_table(C.cast(cbuf(seq.encode()), u8p), True) for _, seq in recs]
    fq = os.path.join(gdir, "reads.fq" if edits == 0 else f"reads_d{edits}.fq")
    lines, sam = _map(compat, "bwt_map_fastq_records", recs, tbls, fq, tmp_path / "out.sam", edits)
    assert sam == open(os.path.join(gdir, expected), "rb").read()
    assert lines == sam.count(b"\n")
    for t in tbls:
        compat.completely_free_bwt_table(t)


def test_map_fastq_records_equals_per_record_mapping(engine, tmp_path):
    from test_compat import cbuf
    from _oracle import u8p
    compat = _compat(engine)
    rng = np.random.default_rng(7)
    recs = []
    for k in range(200):
        letters = list(b"ACG") if k == 17 else list(b"ACGT")  # record 17 holds no T
        recs.append((f"rec{k}", bytes(rng.choice(letters, int(rng.integers(40, 700))).tolist()).decode()))
    recs[30] = ("rec30", recs[31][1][:200])  # a prefix of its neighbour: the same hits in two records
    with open(tmp_path / "reads.fq", "w") as f:
        for q in range(400):
            name, seq = recs[17 if q % 5 == 0 else int(rng.integers(0, len(recs)))]
            m = int(rng.integers(12, 30))
            s = int(rng.integers(0, len(seq) - m))
            read = list(seq[s:s + m])
            for _ in range(int(rng.integers(0, 3))):
                read[int(rng.integers(0, m))] = "ACGT"[int(rng.integers(0, 4))]
            if q % 37 == 0:
                read[0] = "N"  # a letter no record holds
            f.write(f"@r{q}\n{''.join(read)}\n+\n{'I' * m}\n")
    for with_ro in (True, False):
        tbls = [compat.build_complete_table(C.cast(cbuf(seq.encode()), u8p), with_ro) for _, seq in recs]
        for edits in (0, 1, 2):
            n1, a = _map(compat, "bwt_map_fastq", recs, tbls, tmp_path / "reads.fq", tmp_path / "a.sam", edits, 150)
            n2, b = _map(compat, "bwt_map_fastq_records", recs, tbls, tmp_path / "reads.fq", tmp_path / "b.sam", edits,
                         150)
            assert n1 == n2 and a == b, (with_ro, edits)
            assert n1 > 100
        for t in tbls:
            compat.completely_free_bwt_table(t)


# ---- lifecycle and errors -------------------------------------------------------------------------
def _small(rng):
    return [rng.choice(ACGT, int(rng.integers(0, 800))) for _ in range(25)]


def _query(idx, rng, records):
    pats, _ = exact_patterns(rng, records, 300, 0, 30)
    off = np.zeros(len(pats) + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    L, R = idx.search(np.concatenate(pats), off)
    return (L, R) + idx.locate_records(L, R)


def test_save_load_and_replicate_keep_records(engine, tmp_path):
    rng = np.random.default_rng(3)
    records = _small(rng)
    idx = engine.SuffixArrayIndex.build_records(records, 6)
    idx.sample_sa(4)
    want = _query(idx, np.random.default_rng(1), records)
    idx.save(tmp_path / "rec.b200sa")
    back = engine.SuffixArrayIndex.load(tmp_path / "rec.b200sa")
    assert np.array_equal(back.record_offsets(), idx.record_offsets())
    for a, b in zip(_query(back, np.random.default_rng(1), records), want):
        assert np.array_equal(a, b)
    assert all(np.array_equal(a, b) for a, b in zip(back.record_sas(), idx.record_sas()))
    # a plain index saved and loaded is still a plain one
    plain = engine.SuffixArrayIndex.build(np.concatenate(records) - 1, 5)
    plain.save(tmp_path / "plain.b200sa")
    assert engine.SuffixArrayIndex.load(tmp_path / "plain.b200sa").record_offsets().size == 0
    if engine.load().b200sa_device_count() > 1:
        rep = idx.replicate(1)
        assert np.array_equal(rep.record_offsets(), idx.record_offsets())
        for a, b in zip(_query(rep, np.random.default_rng(1), records), want):
            assert np.array_equal(a, b)


def test_errors_leave_the_index_untouched(engine):
    from stralg_b200 import B200saError
    from stralg_b200._lib import BUILD_BWT, BUILD_ISA, BUILD_LCP, BUILD_OCC
    lib = engine.load()
    rng = np.random.default_rng(9)
    records = _small(rng)
    codes = np.concatenate(records).astype(np.uint8)
    off = np.concatenate([[0], np.cumsum([len(r) for r in records])]).astype(np.uint64)
    err = C.c_int(0)

    def build(c, o, nrec, sigma, flags):
        h = lib.b200sa_build_records(C.c_void_p(c.ctypes.data), C.c_void_p(o.ctypes.data), nrec, sigma, flags, 0,
                                     None, C.byref(err))
        if h:
            lib.b200sa_free(C.c_void_p(h))
        return err.value if not h else 0

    for f in (BUILD_ISA, BUILD_LCP, BUILD_BWT):
        assert build(codes, off, len(records), 6, BUILD_OCC | f) == 2
    for bad in (0, 1, 6, 200):
        c = codes.copy()
        c[len(c) // 2] = bad
        assert build(c, off, len(records), 6, BUILD_OCC) == 3, bad
    dec = off.copy()
    dec[3] = off[4] + 1  # record 3 would end before it starts
    assert build(codes, dec, len(records), 6, BUILD_OCC) == 2
    shifted = off + np.uint64(1)
    assert build(codes, shifted, len(records), 6, BUILD_OCC) == 2  # rec_off[0] != 0
    assert build(codes, np.array([0, 2 ** 32 - 2], np.uint64), 1, 6, BUILD_OCC) == 4
    assert build(codes, np.array([0, 5, 2 ** 32], np.uint64), 2, 6, BUILD_OCC) == 4
    assert build(codes[:7], np.array([0, 7], np.uint64), 1, 6, BUILD_OCC) == 0  # one record is legal

    idx = engine.SuffixArrayIndex.build_records(records, 6)
    want = _query(idx, np.random.default_rng(2), records)
    sas = idx.record_sas()
    with pytest.raises(B200saError) as e:
        idx.search(np.array([2, 1, 3], np.uint8), np.array([0, 3], np.uint64))
    assert e.value.code == 3
    with pytest.raises(B200saError) as e:
        idx.approx_search(np.array([2, 3, 1, 4], np.uint8), np.array([0, 4], np.uint64), max_edits=1)
    assert e.value.code == 3
    with pytest.raises(B200saError) as e:
        idx.extend(np.zeros(1, np.uint8), isa=True)
    assert e.value.code == 2
    with pytest.raises(B200saError) as e:
        idx.search_packed(engine.pack_reads(np.ones(8, np.uint8), 8), 8, 1)
    assert e.value.code == 5
    plain = engine.SuffixArrayIndex.build(np.concatenate(records) - 1, 5)
    with pytest.raises(B200saError) as e:
        plain.locate_records([0], [3])
    assert e.value.code == 2
    with pytest.raises(B200saError) as e:
        plain.record_sas()
    assert e.value.code == 2
    for a, b in zip(_query(idx, np.random.default_rng(2), records), want):
        assert np.array_equal(a, b)
    assert all(np.array_equal(a, b) for a, b in zip(idx.record_sas(), sas))
    dropped = engine.SuffixArrayIndex.build_records(records, 6, drop_sa=True)
    with pytest.raises(B200saError) as e:
        dropped.record_sas()
    assert e.value.code == 5
    # row 0 (the global sentinel) belongs to no record: the empty pattern's whole interval is every record's array
    o, r, p = idx.locate_records([0], [idx.length])
    assert int(o[1]) == idx.length - 1
    for k in range(len(records)):
        assert np.array_equal(p[r == k], sas[k])


def test_packed_reads_refuse_a_dna_records_index(engine):
    """Records over three letters (codes 2..4) with the separator are sigma 5, the 2-bit O layout: the packed
    read kernels would run, and packed base 0 is code 1, the separator.  They must refuse the index."""
    import torch
    from stralg_b200 import B200saError
    rng = np.random.default_rng(12)
    records = [rng.choice(ACGT[:3], int(rng.integers(50, 400))) for _ in range(8)]
    idx = engine.SuffixArrayIndex.build_records(records, 5)
    assert idx.stats()["occ_layout"] == 1  # (the DNA layout: this is the case the refusal has to cover)
    reads = np.concatenate([r[:12] - 1 for r in records]).astype(np.uint8)  # codes 1..3 as packed bases
    packed = engine.pack_reads(reads, 12)
    calls = [lambda: idx.search_packed(packed, 12, len(records)),
             lambda: engine.search_sharded_packed([idx], packed, 12, len(records))]
    d_packed = torch.from_numpy(packed).cuda()
    d_L = torch.empty(len(records), dtype=torch.int32, device="cuda")
    d_R = torch.empty_like(d_L)
    calls.append(lambda: idx.search_device_packed(d_packed, 12, len(records), d_L, d_R))
    for call in calls:
        with pytest.raises(B200saError) as e:
            call()
        assert e.value.code == 5
    lib = engine.load()
    counts = (C.c_uint64 * 4)()
    rc = lib.b200sa_search_traffic_packed(idx._h, C.c_void_p(d_packed.data_ptr()), 12, 0, len(records),
                                          C.c_void_p(d_L.data_ptr()), C.c_void_p(d_R.data_ptr()), counts, None)
    assert rc == 5
    # the byte entry points still answer, per record exactly as the records' own indices
    owns = [own_index(engine, r) for r in records]
    pats = [r[k:k + 6].copy() for r in records for k in (0, 17, 33)]
    off = np.zeros(len(pats) + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in pats])
    L, R = idx.search(np.concatenate(pats), off)
    assert got_exact(*idx.locate_records(L, R)) == expected_exact(engine, records, owns, pats)


def test_device_entry_points_equal_host_ones(engine):
    import torch
    rng = np.random.default_rng(13)
    records = _small(rng)
    idx = engine.SuffixArrayIndex.build_records(records, 6)
    d_out = torch.empty(idx.length - 1, dtype=torch.int32, device="cuda")
    idx.record_sas_device(d_out)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy().view(np.uint32), np.concatenate(idx.record_sas()))
    L, R, off, rec, pos = _query(idx, np.random.default_rng(4), records)
    npat = len(L)
    d_L = torch.from_numpy(L.view(np.int32)).cuda()
    d_R = torch.from_numpy(R.view(np.int32)).cuda()
    d_off = torch.empty(npat + 1, dtype=torch.int64, device="cuda")
    total = idx.locate_records_device(d_L, d_R, npat, d_off)
    assert total == len(pos) and np.array_equal(d_off.cpu().numpy().view(np.uint64), off)
    d_rec = torch.empty(total, dtype=torch.int32, device="cuda")
    d_pos = torch.empty(total, dtype=torch.int32, device="cuda")
    assert idx.locate_records_device(d_L, d_R, npat, d_off, d_rec, d_pos, total) == total
    torch.cuda.synchronize()
    assert np.array_equal(d_rec.cpu().numpy().view(np.uint32), rec)
    assert np.array_equal(d_pos.cpu().numpy().view(np.uint32), pos)


def test_map_fastq_records_with_a_shared_remap_table(engine, tmp_path):
    """Tables made with init_bwt_table over one remap table for all records (its letters a superset of each
    record's): bwt_map_fastq searches a read whose letters the table codes even where the record's string lacks
    one, so the records path must as well -- same SAM at d = 0, 1, 2."""
    from test_compat import cbuf
    from _oracle import RefBwtTable, u8p
    compat = _compat(engine)
    rng = np.random.default_rng(14)
    recs = []
    for k in range(40):
        letters = list(b"ACG") if k % 7 == 3 else list(b"ACGT") if k % 5 else list(b"ACGTN")
        recs.append((f"s{k}", bytes(rng.choice(letters, int(rng.integers(60, 500))).tolist()).decode()))
    rt = compat.alloc_remap_table(C.cast(cbuf(b"ACGNT"), u8p))
    keep, tbls, sas = [], [], []
    for _, seq in recs:
        buf = C.create_string_buffer(len(seq) + 1)
        assert compat.remap(C.cast(buf, u8p), C.cast(cbuf(seq.encode()), u8p), rt)
        sa = compat.sa_is_construction(C.cast(buf, u8p), rt.contents.alphabet_size)
        keep.append(buf)
        sas.append(sa)
        tbls.append(compat.alloc_bwt_table(sa, None, rt))
    with open(tmp_path / "reads.fq", "w") as f:
        for q in range(300):
            seq = recs[int(rng.integers(0, len(recs)))][1]
            m = int(rng.integers(10, 25))
            s = int(rng.integers(0, len(seq) - m))
            read = list(seq[s:s + m])
            for _ in range(int(rng.integers(0, 3))):
                read[int(rng.integers(0, m))] = "ACGTN"[int(rng.integers(0, 5))]
            f.write(f"@q{q}\n{''.join(read)}\n+\n{'I' * m}\n")
    for edits in (0, 1, 2):
        n1, a = _map(compat, "bwt_map_fastq", recs, tbls, tmp_path / "reads.fq", tmp_path / "a.sam", edits)
        n2, b = _map(compat, "bwt_map_fastq_records", recs, tbls, tmp_path / "reads.fq", tmp_path / "b.sam", edits)
        assert n1 == n2 and a == b and n1 > 50, edits
    for t, sa in zip(tbls, sas):
        compat.free_bwt_table(t)
        compat.free_suffix_array(sa)
    compat.free_remap_table(rt)
    # no record with a letter, and no record at all: no line, the stream is read to its end, like bwt_map_fastq
    empty_rt = _empty_remap_table()
    empty_sa = _identity_sa(b"")
    fake = RefBwtTable(remap_table=C.pointer(empty_rt), sa=C.pointer(empty_sa))
    for recs_, tbls_ in ((recs[:2], [C.pointer(fake)] * 2), ([], [])):
        for fn in ("bwt_map_fastq", "bwt_map_fastq_records"):
            assert _map(compat, fn, recs_, tbls_, tmp_path / "reads.fq", tmp_path / "c.sam", 1) == (0, b"")


def _empty_remap_table():
    from _oracle import RefRemapTable
    t = RefRemapTable()
    t.alphabet_size = 1
    for b in range(1, 256):
        t.table[b] = -1
    for b in range(1, 128):
        t.rev_table[b] = -1
    return t


_keep = []


def _identity_sa(text: bytes):
    from _oracle import RefSuffixArray, u8p
    buf = C.create_string_buffer(text, len(text) + 1)
    arr = (C.c_uint32 * (len(text) + 1))(*range(len(text) + 1))
    _keep.extend([buf, arr])
    return RefSuffixArray(string=C.cast(buf, u8p), length=len(text) + 1, array=C.cast(arr, C.POINTER(C.c_uint32)))
