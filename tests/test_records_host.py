"""CPU tests of the records-index argument (include/b200sa.h: b200sa_build_records): with the oracle's
suffix array, the concatenation r0 1 r1 1 ... r(k-1) 1 $ restricted to one record's positions is that
record's own suffix array, and RecordsRemap orders letters and masks records like RemapTable."""
import numpy as np
import pytest

from stralg_b200 import RecordsRemap, RemapTable


def concat(records):
    """Records over codes 2.. -> text with separator 1 after every record and the sentinel 0, record starts."""
    parts, starts, at = [], [], 0
    for r in records:
        starts.append(at)
        parts.append(np.asarray(r, dtype=np.uint8))
        parts.append(np.ones(1, np.uint8))
        at += len(r) + 1
    starts.append(at)
    return np.concatenate(parts + [np.zeros(1, np.uint8)]), np.array(starts, dtype=np.int64)


def own_sa(oracle, rec):
    """Suffix array of one record alone, over its codes shifted down to 1.. (order-preserving)."""
    codes = np.concatenate([np.asarray(rec, dtype=np.uint8) - 1, np.zeros(1, np.uint8)]) if len(rec) else \
        np.zeros(1, np.uint8)
    return oracle.sa(codes)


def check_partition(oracle, records):
    text, starts = concat(records)
    sa = oracle.sa(text).astype(np.int64)
    assert sa[0] == len(text) - 1  # the global sentinel
    rec_of = np.searchsorted(starts, sa[1:], side="right") - 1
    for r, rec in enumerate(records):
        got = sa[1:][rec_of == r] - starts[r]
        assert np.array_equal(got, own_sa(oracle, rec).astype(np.int64)), r


def dna(rng, n):
    return rng.integers(2, 6, n).astype(np.uint8)


def test_random_acgt_records(oracle):
    rng = np.random.default_rng(1)
    check_partition(oracle, [dna(rng, int(rng.integers(1, 400))) for _ in range(40)])


def test_identical_records(oracle):
    rng = np.random.default_rng(2)
    r = dna(rng, 300)
    check_partition(oracle, [r] * 12)


def test_records_that_are_prefixes_of_one_another(oracle):
    rng = np.random.default_rng(3)
    r = dna(rng, 500)
    check_partition(oracle, [r[:k] for k in (500, 1, 250, 499, 3, 250, 0, 100)])


def test_empty_records(oracle):
    rng = np.random.default_rng(4)
    check_partition(oracle, [np.zeros(0, np.uint8), dna(rng, 50), np.zeros(0, np.uint8), np.zeros(0, np.uint8),
                             dna(rng, 7), np.zeros(0, np.uint8)])
    check_partition(oracle, [np.zeros(0, np.uint8)] * 5)


def test_unary_records(oracle):
    check_partition(oracle, [np.full(k, 2, np.uint8) for k in (100, 1, 37, 100, 0, 64)])
    check_partition(oracle, [np.full(50, 2, np.uint8), np.full(50, 3, np.uint8), np.full(20, 2, np.uint8)])


def test_periodic_record_next_to_random_one(oracle):
    rng = np.random.default_rng(5)
    check_partition(oracle, [np.tile(np.array([2, 3, 3], np.uint8), 200), dna(rng, 600),
                             np.tile(np.array([2, 3, 3], np.uint8), 199)])


@pytest.mark.parametrize("seed", range(3))
def test_records_remap_matches_remap_table_per_record(seed):
    rng = np.random.default_rng(seed)
    alphabets = [b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY", b"ac", b"T"]
    raw = [bytes(rng.choice(list(alphabets[k % len(alphabets)]), int(rng.integers(1, 300))).tolist())
           for k in range(12)] + [b""]
    rr = RecordsRemap(raw)
    union = RemapTable(b"".join(raw))
    assert rr.alphabet_size == union.alphabet_size + 1
    # union letters in byte order, shifted up by one for the separator
    present = union.table > 0
    assert np.array_equal(rr.table[present], union.table[present] + 1)
    assert (rr.table[~present][1:] == -1).all() and rr.table[0] == 0
    for r, rec in enumerate(raw):
        own = RemapTable(rec)
        # the mask is exactly the set of bytes record r's own table can remap, and the letter order agrees
        assert np.array_equal(rr.masks[r][1:], own.table[1:] > 0)
        mine = np.nonzero(own.table[1:] > 0)[0] + 1
        assert np.array_equal(np.argsort(rr.table[mine]), np.argsort(own.table[mine]))
        for probe in (rec[:20], b"ACGT", b"N", b"acgt", b"W"):
            assert rr.in_record(probe, r) == (own.remap(probe) is not None)
        codes = rr.remap(rec)
        assert codes is not None and (codes >= 2).all()
        assert rr.remap(b"\x01") is None
