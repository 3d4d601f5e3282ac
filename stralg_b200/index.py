"""Host-side mirror of the reference's suffix_array.h / bwt.h surface over the B200 engine.

Names follow the reference: ``remap`` (stralg/remap.c), ``sa_is_construction`` and friends
(stralg/suffix_array.h:22-41), ``compute_inverse`` / ``compute_lcp`` (suffix_array.h:96-101),
``build_complete_table`` (stralg/bwt.c:134-161), the exact-match iterator
(stralg/bwt.c:164-217).  All compute runs in libb200sa.so on the GPU; numpy arrays are only the
host-side carriers the reference's structs would be.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (BUILD_BWT, BUILD_ISA, BUILD_KTABLE, BUILD_LCP, BUILD_OCC, BUILD_TEXTCMP, DROP_SA, PROFILE, TEXT_ON_DEVICE, B200saError,
                   Stats, check)


def _np_ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _is_torch_tensor(x) -> bool:
    return type(x).__module__.startswith("torch")


class RemapTable:
    """Alphabet remap table (stralg/remap.h:9-19, remap.c:8-58): bytes present in the text get
    dense codes 1..sigma-1 in byte order, 0 is the sentinel."""

    def __init__(self, text: bytes):
        seen = np.zeros(256, dtype=bool)
        seen[np.frombuffer(text, dtype=np.uint8)] = True
        seen[0] = False
        letters = np.nonzero(seen)[0]
        self.table = np.full(256, -1, dtype=np.int16)
        self.rev_table = np.full(256, -1, dtype=np.int16)
        self.table[0] = 0
        self.rev_table[0] = 0
        self.table[letters] = np.arange(1, len(letters) + 1, dtype=np.int16)
        self.rev_table[1:len(letters) + 1] = letters
        self.alphabet_size = len(letters) + 1

    def remap(self, text: bytes) -> Optional[np.ndarray]:
        """remap() (remap.c:102-114): codes for ``text``; None if a letter has no code
        (the reference returns a NULL pointer, remap.c:80-84)."""
        codes = self.table[np.frombuffer(text, dtype=np.uint8)]
        if (codes < 0).any() or (codes == 0).any():
            return None
        return codes.astype(np.uint8)

    def rev_remap(self, codes: np.ndarray) -> bytes:
        return self.rev_table[np.asarray(codes, dtype=np.uint8)].astype(np.uint8).tobytes()


class RecordsRemap:
    """Alphabet of a records index (include/b200sa.h, b200sa_build_records): the bytes present in any
    record get codes 2..sigma-1 in byte order, code 1 is the separator the library inserts after every
    record, 0 the sentinel.  ``masks[r]`` is the 256-entry set of bytes record r holds: a read with a
    byte outside it has no code in record r's own ``RemapTable`` (the reference skips such a read for
    that record, remap.c:80-84)."""

    def __init__(self, records: Sequence[bytes]):
        self.masks = np.zeros((len(records), 256), dtype=bool)
        for r, rec in enumerate(records):
            self.masks[r, np.frombuffer(bytes(rec), dtype=np.uint8)] = True
        self.masks[:, 0] = False
        seen = self.masks.any(axis=0)
        letters = np.nonzero(seen)[0]
        self.table = np.full(256, -1, dtype=np.int16)
        self.rev_table = np.full(256, -1, dtype=np.int16)
        self.table[0] = 0
        self.rev_table[0] = 0
        self.table[letters] = np.arange(2, len(letters) + 2, dtype=np.int16)
        self.rev_table[2:len(letters) + 2] = letters
        self.alphabet_size = len(letters) + 2  # sentinel + separator + letters

    def remap(self, text: bytes) -> Optional[np.ndarray]:
        """Codes 2..sigma-1 for ``text``; None if a byte is in no record."""
        codes = self.table[np.frombuffer(bytes(text), dtype=np.uint8)]
        if (codes <= 0).any():
            return None
        return codes.astype(np.uint8)

    def in_record(self, text: bytes, r: int) -> bool:
        """Whether every byte of ``text`` occurs in record r (its own RemapTable can remap it)."""
        return bool(self.masks[r, np.frombuffer(bytes(text), dtype=np.uint8)].all())


class SuffixArrayIndex:
    """Device-resident suffix array + optional ISA / LCP / BWT / C / O tables for one text.

    The analogue of ``struct suffix_array`` (suffix_array.h:10-20) plus ``struct bwt_table``
    (bwt.h:36-44); ``length`` is n + 1 like the reference's ``sa->length``.
    """

    def __init__(self, handle: int, device: int, keepalive=None):
        self._h = C.c_void_p(handle)
        self.device = device
        self._keepalive = keepalive
        st = Stats()
        check(_lib.load().b200sa_stats(self._h, C.byref(st)))
        self.length = int(st.length)
        self.sigma = int(st.sigma)
        self.primary = int(st.primary)

    # ---- construction ---------------------------------------------------------------------
    @classmethod
    def build(cls, codes, sigma: int, *, isa=False, lcp=False, bwt=False, occ=True, textcmp=False, ktable=False,
              drop_sa=False,
              profile=False, device: int = 0, stream: int = 0) -> "SuffixArrayIndex":
        """codes: remapped text WITHOUT the sentinel -- numpy uint8 array / bytes (host), or a
        CUDA uint8 torch tensor (device-resident, borrowed during the call)."""
        lib = _lib.load()
        flags = (BUILD_ISA if isa else 0) | (BUILD_LCP if lcp else 0) | (BUILD_BWT if bwt else 0) | \
                (BUILD_OCC if occ else 0) | (BUILD_TEXTCMP if textcmp else 0) | (BUILD_KTABLE if ktable else 0) | (DROP_SA if drop_sa else 0) | (PROFILE if profile else 0)
        keep = None
        if _is_torch_tensor(codes):
            assert codes.is_cuda and codes.dtype.itemsize == 1 and codes.is_contiguous()
            ptr, n = C.c_void_p(codes.data_ptr()), codes.numel()
            flags |= TEXT_ON_DEVICE
            device = codes.device.index
        else:
            keep = np.ascontiguousarray(np.frombuffer(codes, dtype=np.uint8) if isinstance(codes, (bytes, bytearray))
                                        else codes, dtype=np.uint8)
            ptr, n = _np_ptr(keep), keep.size
        err = C.c_int(0)
        h = lib.b200sa_build(ptr, n, sigma, flags, device, C.c_void_p(stream), C.byref(err))
        if not h:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        return cls(h, device)

    @classmethod
    def build_records(cls, records, sigma: int, *, occ=True, textcmp=False, ktable=False, drop_sa=False,
                      profile=False, device: int = 0, stream: int = 0) -> "SuffixArrayIndex":
        """One index over many records (b200sa_build_records): ``records`` is a sequence of code arrays /
        bytes over 2..sigma-1 (code 1 is the separator the library inserts after every record)."""
        lib = _lib.load()
        flags = (BUILD_OCC if occ else 0) | (BUILD_TEXTCMP if textcmp else 0) | (BUILD_KTABLE if ktable else 0) | \
                (DROP_SA if drop_sa else 0) | (PROFILE if profile else 0)
        parts = [np.frombuffer(r, dtype=np.uint8) if isinstance(r, (bytes, bytearray)) else np.asarray(r, dtype=np.uint8)
                 for r in records]
        off = np.zeros(len(parts) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([p.size for p in parts], dtype=np.uint64)
        codes = np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(0, np.uint8), dtype=np.uint8)
        err = C.c_int(0)
        h = lib.b200sa_build_records(_np_ptr(codes), _np_ptr(off), len(parts), sigma, flags, device,
                                     C.c_void_p(stream), C.byref(err))
        if not h:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        return cls(h, device)

    def extend(self, codes, *, isa=False, lcp=False, bwt=False, occ=False, textcmp=False, ktable=False) -> None:
        """Adds tables that were not requested at build time (b200sa_extend: the reference's lazy compute_inverse /
        compute_lcp, suffix_array.c:55-85, and init_bwt_table over an existing suffix array, bwt.c:22-89).  `codes` is
        the text the index was built from (host array or CUDA tensor)."""
        flags = (BUILD_ISA if isa else 0) | (BUILD_LCP if lcp else 0) | (BUILD_BWT if bwt else 0) | \
                (BUILD_OCC if occ else 0) | (BUILD_TEXTCMP if textcmp else 0) | (BUILD_KTABLE if ktable else 0)
        if _is_torch_tensor(codes):
            assert codes.is_cuda and codes.dtype.itemsize == 1 and codes.is_contiguous()
            ptr = C.c_void_p(codes.data_ptr())
            flags |= TEXT_ON_DEVICE
        else:
            keep = np.ascontiguousarray(codes, dtype=np.uint8)
            ptr = _np_ptr(keep)
        check(_lib.load().b200sa_extend(self._h, ptr, flags))

    # ---- native index file (include/b200sa.h: b200sa_save / b200sa_load) ------------------------
    def save(self, path: str) -> None:
        check(_lib.load().b200sa_save(self._h, str(path).encode()))

    @classmethod
    def load(cls, path: str, device: int = 0, stream: int = 0) -> "SuffixArrayIndex":
        lib = _lib.load()
        err = C.c_int(0)
        h = lib.b200sa_load(str(path).encode(), device, C.c_void_p(stream), C.byref(err))
        if not h:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        return cls(h, device)

    def replicate(self, device: int, stream: int = 0) -> "SuffixArrayIndex":
        """A copy of this index on another device of the same process (peer copies, no rebuild)."""
        lib = _lib.load()
        err = C.c_int(0)
        h = lib.b200sa_replicate(self._h, device, C.c_void_p(stream), C.byref(err))
        if not h:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        return SuffixArrayIndex(h, device)

    def close(self):
        if self._h:
            _lib.load().b200sa_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- tables to host (the arrays of struct suffix_array / struct bwt_table) -----------------
    def _copy(self, fn, dtype, count):
        out = np.empty(count, dtype=dtype)
        check(fn(self._h, _np_ptr(out)))
        return out

    def sa(self) -> np.ndarray:
        return self._copy(_lib.load().b200sa_copy_sa, np.uint32, self.length)

    def isa(self) -> np.ndarray:
        return self._copy(_lib.load().b200sa_copy_isa, np.uint32, self.length)

    def lcp(self) -> np.ndarray:
        return self._copy(_lib.load().b200sa_copy_lcp, np.uint32, self.length)

    def bwt(self) -> np.ndarray:
        return self._copy(_lib.load().b200sa_copy_bwt, np.uint8, self.length)

    def c_table(self) -> np.ndarray:
        return self._copy(_lib.load().b200sa_copy_c_table, np.uint32, self.sigma)

    def o_dense(self) -> np.ndarray:
        """Dense O table in the reference layout, shape (length + 1, sigma) (bwt.c:47-65)."""
        out = np.empty((self.length + 1, self.sigma), dtype=np.uint32)
        check(_lib.load().b200sa_copy_o_dense(self._h, _np_ptr(out)))
        return out

    def occ(self, a: Sequence[int], i: Sequence[int]) -> np.ndarray:
        """O(a[q], i[q]) (the O(a,i) macro of bwt.h:48-50)."""
        a = np.ascontiguousarray(a, dtype=np.uint8)
        i = np.ascontiguousarray(i, dtype=np.uint32)
        out = np.empty(len(a), dtype=np.uint32)
        check(_lib.load().b200sa_occ(self._h, _np_ptr(a), _np_ptr(i), len(a), _np_ptr(out)))
        return out

    # ---- device views ---------------------------------------------------------------------------
    def device_ptr(self, what: str) -> int:
        fn = getattr(_lib.load(), f"b200sa_device_{what}")
        return fn(self._h) or 0

    def stats(self) -> dict:
        st = Stats()
        check(_lib.load().b200sa_stats(self._h, C.byref(st)))
        return {k: int(getattr(st, k)) for k, _ in Stats._fields_}

    def profile(self):
        """[(stage, ms, algorithmic_bytes)] of the build (needs profile=True)."""
        cap = 1024
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        by = (C.c_double * cap)()
        n = _lib.load().b200sa_profile(self._h, names, ms, by, cap)
        return [(names[k].decode(), float(ms[k]), float(by[k])) for k in range(min(n, cap))]

    # ---- exact search (init_bwt_exact_match_iter, bwt.c:164-199) ----------------------------------
    def search(self, patterns, offsets=None, fixed_len: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """Host buffers in, host (L, R) out.  patterns: concatenated remapped codes."""
        pat = np.ascontiguousarray(patterns, dtype=np.uint8)
        if offsets is not None:
            off = np.ascontiguousarray(offsets, dtype=np.uint64)
            npat = len(off) - 1
            offp = _np_ptr(off)
        else:
            assert fixed_len > 0
            npat = pat.size // fixed_len
            offp = None
        L = np.empty(npat, dtype=np.uint32)
        R = np.empty(npat, dtype=np.uint32)
        check(_lib.load().b200sa_search_batch(self._h, _np_ptr(pat), offp, fixed_len, npat, _np_ptr(L), _np_ptr(R)))
        return L, R

    def search_device(self, d_patterns, d_offsets, fixed_len: int, npat: int, d_L, d_R, stream: int = 0):
        """Device buffers (torch CUDA tensors) in and out; asynchronous on ``stream``."""
        check(_lib.load().b200sa_search_device(
            self._h, C.c_void_p(d_patterns.data_ptr()),
            C.c_void_p(d_offsets.data_ptr()) if d_offsets is not None else None, fixed_len, npat,
            C.c_void_p(d_L.data_ptr()), C.c_void_p(d_R.data_ptr()), C.c_void_p(stream)))

    def search_packed(self, packed, read_len: int, npat: int, stride_bytes: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """Packed reads (2 bits per base, see ``pack_reads``) in host memory -> host (L, R)."""
        pk = np.ascontiguousarray(packed, dtype=np.uint8)
        L = np.empty(npat, dtype=np.uint32)
        R = np.empty(npat, dtype=np.uint32)
        check(_lib.load().b200sa_search_batch_packed(self._h, _np_ptr(pk), read_len, stride_bytes, npat, _np_ptr(L),
                                                     _np_ptr(R)))
        return L, R

    def search_device_packed(self, d_packed, read_len: int, npat: int, d_L, d_R, stride_bytes: int = 0,
                             stream: int = 0):
        """Packed reads in device memory (torch CUDA tensor, 8-byte aligned); asynchronous on ``stream``."""
        check(_lib.load().b200sa_search_device_packed(
            self._h, C.c_void_p(d_packed.data_ptr()), read_len, stride_bytes, npat, C.c_void_p(d_L.data_ptr()),
            C.c_void_p(d_R.data_ptr()), C.c_void_p(stream)))

    def search_one(self, pattern_codes) -> Tuple[int, int]:
        p = np.ascontiguousarray(pattern_codes, dtype=np.uint8)
        L, R = self.search(p, np.array([0, len(p)], dtype=np.uint64))
        return int(L[0]), int(R[0])

    # ---- locate (next_bwt_exact_match_iter, bwt.c:201-217) -------------------------------------
    def locate(self, L, R, sorted: bool = False) -> Tuple[np.ndarray, np.ndarray]:
        """CSR (offsets[npat + 1], positions) in suffix-array order, like the reference iterator;
        ``sorted=True`` orders the positions of every pattern ascending (match_test.c:608)."""
        L = np.ascontiguousarray(L, dtype=np.uint32)
        R = np.ascontiguousarray(R, dtype=np.uint32)
        npat = len(L)
        off = np.empty(npat + 1, dtype=np.uint64)
        total = C.c_uint64(0)
        lib = _lib.load()
        fn = lib.b200sa_locate_batch_sorted if sorted else lib.b200sa_locate_batch
        check(fn(self._h, _np_ptr(L), _np_ptr(R), npat, _np_ptr(off), None, 0, C.byref(total)))
        pos = np.empty(total.value, dtype=np.uint32)
        if total.value:
            check(fn(self._h, _np_ptr(L), _np_ptr(R), npat, _np_ptr(off), _np_ptr(pos), total.value, C.byref(total)))
        return off, pos

    # ---- approximate search (init_bwt_approx_iter / next_bwt_approx_match, bwt.c:226-409) -------
    def approx_search(self, patterns, offsets=None, fixed_len: int = 0, max_edits: int = 1,
                      rev: "Optional[SuffixArrayIndex]" = None, d_table=None) -> dict:
        """All intervals within ``max_edits`` edits, per pattern in the reference's report order.
        ``rev``: index of the reversed text (the reference's RO table -> D table pruning).
        Returns dict(offsets[npat+1], L, R, match_length, cigars[list of str])."""
        lib = _lib.load()
        pat = np.ascontiguousarray(patterns, dtype=np.uint8)
        if offsets is not None:
            off = np.ascontiguousarray(offsets, dtype=np.uint64)
            npat = len(off) - 1
            offp = _np_ptr(off)
        else:
            assert fixed_len > 0
            npat = pat.size // fixed_len
            offp = None
        dt = None
        if d_table is not None:
            dt = np.ascontiguousarray(d_table, dtype=np.uint8)
            assert dt.size == pat.size
        err = C.c_int(0)
        r = lib.b200sa_approx_batch(self._h, rev._h if rev is not None else None, _np_ptr(dt) if dt is not None else None,
                                    _np_ptr(pat), offp, fixed_len, npat, max_edits, C.byref(err))
        if not r:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        r = C.c_void_p(r)
        try:
            nh = int(lib.b200sa_approx_hits(r))
            hoff = np.ctypeslib.as_array(lib.b200sa_approx_hit_offsets(r), shape=(npat + 1,)).copy()
            if nh:
                L = np.ctypeslib.as_array(lib.b200sa_approx_L(r), shape=(nh,)).copy()
                R = np.ctypeslib.as_array(lib.b200sa_approx_R(r), shape=(nh,)).copy()
                ml = np.ctypeslib.as_array(lib.b200sa_approx_match_length(r), shape=(nh,)).copy()
                coff = np.ctypeslib.as_array(lib.b200sa_approx_cigar_offsets(r), shape=(nh + 1,))
                raw = C.string_at(lib.b200sa_approx_cigars(r), int(coff[nh]))
                cig = [x.decode() for x in raw.split(b"\0")[:-1]]
            else:
                L = R = ml = np.zeros(0, np.uint32)
                cig = []
        finally:
            lib.b200sa_approx_free(r)
        return {"offsets": hoff, "L": L, "R": R, "match_length": ml, "cigars": cig}

    # ---- matching statistics and super-maximal exact matches (include/b200sa.h) ----------------------
    @staticmethod
    def _batch(patterns, offsets, fixed_len):
        pat = np.ascontiguousarray(patterns, dtype=np.uint8)
        if offsets is not None:
            off = np.ascontiguousarray(offsets, dtype=np.uint64)
            return pat, off, len(off) - 1, _np_ptr(off)
        assert fixed_len > 0
        return pat, None, pat.size // fixed_len, None

    def matching_stats(self, patterns, offsets=None, fixed_len: int = 0) -> dict:
        """Per pattern symbol, laid out like ``patterns``: ms (the length of the longest substring of the pattern that
        ends there and occurs in the text) and the SA interval [L, R) of that substring ((1, 0) where ms = 0).
        Returns dict(ms, L, R)."""
        pat, _, npat, offp = self._batch(patterns, offsets, fixed_len)
        ms = np.zeros(pat.size, dtype=np.uint32)
        L = np.zeros(pat.size, dtype=np.uint32)
        R = np.zeros(pat.size, dtype=np.uint32)
        check(_lib.load().b200sa_matching_stats(self._h, _np_ptr(pat), offp, fixed_len, npat, _np_ptr(ms), _np_ptr(L),
                                                _np_ptr(R)))
        return {"ms": ms, "L": L, "R": R}

    def smems(self, patterns, offsets=None, fixed_len: int = 0, min_len: int = 1) -> dict:
        """Super-maximal exact matches of at least ``min_len`` symbols, per pattern in ascending start.
        Returns dict(offsets[npat+1], start, length, L, R)."""
        lib = _lib.load()
        pat, _, npat, offp = self._batch(patterns, offsets, fixed_len)
        err = C.c_int(0)
        r = lib.b200sa_smem_batch(self._h, _np_ptr(pat), offp, fixed_len, npat, min_len, C.byref(err))
        if not r:
            raise B200saError(err.value, lib.b200sa_last_error().decode())
        r = C.c_void_p(r)
        try:
            n = int(lib.b200sa_smem_count(r))
            soff = np.ctypeslib.as_array(lib.b200sa_smem_offsets(r), shape=(npat + 1,)).copy()
            cols = {}
            for k, fn in (("start", lib.b200sa_smem_start), ("length", lib.b200sa_smem_length),
                          ("L", lib.b200sa_smem_L), ("R", lib.b200sa_smem_R)):
                cols[k] = np.ctypeslib.as_array(fn(r), shape=(n,)).copy() if n else np.zeros(0, np.uint32)
        finally:
            lib.b200sa_smem_free(r)
        return {"offsets": soff, **cols}

    # ---- sampled suffix array (SURVEY 8f rank 3) -----------------------------------------------
    def sample_sa(self, rate: int = 32, drop_sa: bool = False) -> None:
        """Keep SA only at text positions that are multiples of ``rate``; with ``drop_sa`` the full
        array is released and locate walks LF to the nearest sampled row (same positions)."""
        check(_lib.load().b200sa_sample_sa(self._h, rate, 1 if drop_sa else 0))

    def sa_lookup(self, rows, force_sampled: bool = False) -> np.ndarray:
        """SA[rows] (``sa->array[i]`` of suffix_array.h:10-20) without copying the whole array."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        out = np.empty(len(rows), dtype=np.uint32)
        check(_lib.load().b200sa_sa_lookup(self._h, _np_ptr(rows), len(rows), _np_ptr(out), 1 if force_sampled else 0))
        return out

    def locate_device(self, d_L, d_R, npat: int, d_pos_off, d_pos=None, capacity: int = 0, stream: int = 0) -> int:
        """Device buffers (torch CUDA tensors): fills d_pos_off[npat + 1] and, when given, d_pos; returns
        the number of positions."""
        total = C.c_uint64(0)
        check(_lib.load().b200sa_locate_device(
            self._h, C.c_void_p(d_L.data_ptr()), C.c_void_p(d_R.data_ptr()), npat, C.c_void_p(d_pos_off.data_ptr()),
            C.c_void_p(d_pos.data_ptr()) if d_pos is not None else None, capacity, C.byref(total), C.c_void_p(stream)))
        return int(total.value)

    # ---- records index (b200sa_build_records) ----------------------------------------------------
    def record_offsets(self) -> np.ndarray:
        """rec_off[nrec + 1] of a records index (b200sa_records); an empty array for a plain index."""
        lib = _lib.load()
        nrec = C.c_uint32(0)
        check(lib.b200sa_records(self._h, C.byref(nrec), None))
        if not nrec.value:
            return np.zeros(0, dtype=np.uint64)
        off = np.empty(nrec.value + 1, dtype=np.uint64)
        check(lib.b200sa_records(self._h, C.byref(nrec), _np_ptr(off)))
        return off

    def record_sas(self) -> list:
        """Every record's own suffix array (b200sa_copy_record_sas), one array per record in local positions."""
        off = self.record_offsets()
        flat = self._copy(_lib.load().b200sa_copy_record_sas, np.uint32, self.length - 1)
        start = off + np.arange(len(off), dtype=np.uint64)
        return [flat[int(start[r]):int(start[r + 1])] for r in range(len(off) - 1)]

    def record_sas_device(self, d_out, stream: int = 0) -> None:
        """b200sa_record_sas_device: every record's own suffix array into ``d_out`` (a CUDA uint32 tensor of
        length - 1 entries, record r at rec_off[r] + r); asynchronous on ``stream``."""
        check(_lib.load().b200sa_record_sas_device(self._h, C.c_void_p(d_out.data_ptr()), C.c_void_p(stream)))

    def locate_records_device(self, d_L, d_R, npat: int, d_pos_off, d_rec=None, d_pos=None, capacity: int = 0,
                              stream: int = 0) -> int:
        """b200sa_locate_records_device (torch CUDA tensors): fills d_pos_off[npat + 1] and, when given, d_rec and
        d_pos; returns the number of entries."""
        total = C.c_uint64(0)
        check(_lib.load().b200sa_locate_records_device(
            self._h, C.c_void_p(d_L.data_ptr()), C.c_void_p(d_R.data_ptr()), npat, C.c_void_p(d_pos_off.data_ptr()),
            C.c_void_p(d_rec.data_ptr()) if d_rec is not None else None,
            C.c_void_p(d_pos.data_ptr()) if d_pos is not None else None, capacity, C.byref(total), C.c_void_p(stream)))
        return int(total.value)

    def locate_records(self, L, R) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(offsets[npat + 1], rec, pos) (b200sa_locate_records): per pattern, records ascending, the
        local positions of one record in that record's suffix-array order."""
        L = np.ascontiguousarray(L, dtype=np.uint32)
        R = np.ascontiguousarray(R, dtype=np.uint32)
        npat = len(L)
        off = np.empty(npat + 1, dtype=np.uint64)
        total = C.c_uint64(0)
        fn = _lib.load().b200sa_locate_records
        check(fn(self._h, _np_ptr(L), _np_ptr(R), npat, _np_ptr(off), None, None, 0, C.byref(total)))
        rec = np.empty(total.value, dtype=np.uint32)
        pos = np.empty(total.value, dtype=np.uint32)
        if total.value:
            check(fn(self._h, _np_ptr(L), _np_ptr(R), npat, _np_ptr(off), _np_ptr(rec), _np_ptr(pos), total.value,
                     C.byref(total)))
        return off, rec, pos

    def exact_matches(self, pattern_codes) -> np.ndarray:
        """All match positions of one pattern in SA order (the iterator loop of match_test.c:599-603)."""
        L, R = self.search_one(pattern_codes)
        _, pos = self.locate([L], [R])
        return pos


def pack_reads(codes, read_len: int, stride_bytes: int = 0) -> np.ndarray:
    """One-byte-per-base codes 1..4 (reads of ``read_len`` bases back to back) -> 2-bit packed reads:
    four bases per byte, the first base in the two most significant bits; read q starts at byte
    q * stride (default ceil(read_len / 4)).  Eight zero bytes of padding follow the last read."""
    c = np.ascontiguousarray(codes, dtype=np.uint8)
    npat = c.size // read_len
    stride = stride_bytes or (read_len + 3) // 4
    out = np.zeros(npat * stride + 8, dtype=np.uint8)
    check(_lib.load().b200sa_pack_reads(_np_ptr(c), read_len, stride, npat, _np_ptr(out)))
    return out


def search_sharded_packed(replicas, packed, read_len: int, npat: int, stride_bytes: int = 0):
    """b200sa_search_sharded_packed: one process, one replica of the index per device, the packed reads
    split into contiguous shards; (L, R) of all reads in input order."""
    pk = np.ascontiguousarray(packed, dtype=np.uint8)
    L = np.empty(npat, dtype=np.uint32)
    R = np.empty(npat, dtype=np.uint32)
    arr = (C.c_void_p * len(replicas))(*[r._h for r in replicas])
    check(_lib.load().b200sa_search_sharded_packed(arr, len(replicas), _np_ptr(pk), read_len, stride_bytes, npat,
                                                   _np_ptr(L), _np_ptr(R)))
    return L, R


# ---- reference-named constructors -----------------------------------------------------------------
def sa_is_construction(remapped_codes, alphabet_size: int, **kw) -> SuffixArrayIndex:
    """suffix_array.h:29-33.  The sentinel must NOT be included in ``remapped_codes``."""
    return SuffixArrayIndex.build(remapped_codes, alphabet_size, occ=False, **kw)


sa_is_mem_construction = sa_is_construction  # suffix_array.h:35-39: same array, one GPU builder


def skew_sa_construction(text_bytes, **kw) -> SuffixArrayIndex:
    """suffix_array.h:26-28: any bytes 1..255, fixed alphabet of 256."""
    return SuffixArrayIndex.build(text_bytes, 256, occ=False, **kw)


qsort_sa_construction = skew_sa_construction  # suffix_array.h:22-25


def build_complete_table(text: bytes, **kw) -> Tuple[SuffixArrayIndex, RemapTable]:
    """bwt.c:134-161: remap -> suffix array -> C and O tables (exact-match tables only)."""
    table = RemapTable(text)
    codes = table.remap(text)
    if codes is None:
        raise ValueError("text contains a NUL byte")
    return SuffixArrayIndex.build(codes, table.alphabet_size, occ=True, **kw), table
