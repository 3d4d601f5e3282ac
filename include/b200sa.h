/*
 * b200sa.h -- C ABI of the B200-native suffix-array / BWT / FM-index engine.
 *
 * This is the drop-in boundary for the hot path of mailund/stralg: the functions a binding of
 * stralg's suffix_array.h / bwt.h would call (reference file:line cited per entry point; paths
 * are relative to the stralg checkout).  Plain pointers and sizes only, no CUDA or torch types.
 * The reference-named shims (sa_is_construction, compute_lcp, init_bwt_table,
 * init_bwt_exact_match_iter, ...) are declared in include/stralg_compat.h and implemented on top of
 * this header by libstralg_b200.so.
 *
 * Conventions (stralg README.md:106-134, stralg/error.h:7-21): an `enum b200sa_error *err`
 * out-parameter is the LAST argument, 0 means success, it is written on every call and may be
 * NULL.  Functions returning int return the same code.  b200sa_last_error() gives a
 * thread-local message.  There is no CPU fallback: without a CUDA device every call fails with
 * B200SA_ERR_CUDA.
 *
 * Texts are "remapped codes" (stralg/remap.c:73-114): n bytes in 1..sigma-1; the sentinel 0 is
 * implicit (text[n] is never read).  All tables have len = n + 1 entries/rows because the
 * sentinel suffix is a real suffix (stralg/suffix_array_internal.c:7-19); n <= 2^32 - 2.
 */
#ifndef B200SA_H
#define B200SA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200sa_index b200sa_index;

enum b200sa_error {
    B200SA_OK = 0,
    B200SA_ERR_CUDA = 1,          /* CUDA runtime failure or no device */
    B200SA_ERR_BAD_ARGUMENT = 2,
    B200SA_ERR_BAD_SYMBOL = 3,    /* text holds a code 0 or >= sigma (remap.c:80-84 returns NULL) */
    B200SA_ERR_TOO_LARGE = 4,     /* n > 2^32 - 2, or a dense table that cannot be indexed in u32 */
    B200SA_ERR_NOT_BUILT = 5,     /* table was not requested at build time */
    B200SA_ERR_OUT_OF_MEMORY = 6,
    B200SA_ERR_INTERNAL = 7
};

/* build flags */
#define B200SA_BUILD_ISA 0x1u        /* keep the inverse suffix array   (suffix_array.c:55-62)  */
#define B200SA_BUILD_LCP 0x2u        /* LCP array                       (suffix_array.c:64-85)  */
#define B200SA_BUILD_BWT 0x4u        /* keep the BWT rows               (bwt.c:13-20)           */
#define B200SA_BUILD_OCC 0x8u        /* C table + sampled O table       (bwt.c:35-65)           */
#define B200SA_BUILD_TEXTCMP 0x10u   /* keep ISA + packed text: exact search finishes a unique interval
                                        (R - L == 1) by comparing the remaining pattern symbols with the
                                        text directly instead of one O lookup per symbol; results are
                                        identical to the plain recurrence (needs OCC, keeps SA); any alphabet */
#define B200SA_BUILD_KTABLE 0x20u    /* table of the (L, R) interval the recurrence of bwt.c:185-195 reaches on
                                        every k-mer; other alphabets than DNA: (sigma - 1)^k entries under the
                                        same budget, fewer than 2^32.  DNA index (sigma <= 5): the largest k <= 15 whose table
                                        stays under 3 bytes per text symbol: 15 at 3 Gbp; with TEXTCMP, which
                                        keeps 8 bytes per symbol anyway, k <= 16 under 12 bytes: 16, 34 GB, at
                                        3 Gbp; B200SA_KTABLE_K overrides); exact search starts from the entry of the pattern's last k
                                        symbols instead of running those k steps; results are identical
                                        (needs OCC)                                                      */
#define B200SA_TEXT_ON_DEVICE 0x100u /* `codes` is a device pointer (borrowed during the call)  */
#define B200SA_PROFILE 0x200u        /* record per-stage device times (b200sa_profile)          */
#define B200SA_DROP_SA 0x400u        /* release the suffix array after the tables are built     */

struct b200sa_stats {
    uint32_t length;       /* n + 1 */
    uint32_t sigma;
    uint32_t primary;      /* row r with SA[r] == 0 (BWT row holding the sentinel) */
    uint32_t rounds;       /* prefix-doubling rounds after the initial sort */
    uint32_t k0;           /* symbols packed into the initial sort key */
    uint32_t radix_bits;   /* digit bits: LSD passes, or the first partition level of the bucket sort */
    uint32_t passes0;      /* radix passes (LSD) or partition levels (bucket sort) of the initial sort */
    uint32_t occ_layout;   /* 1 = 32-byte DNA blocks, 2 = byte blocks */
    uint64_t sorted_total; /* elements sorted, summed over rounds */
    uint64_t passes_elems; /* elements moved, summed over all radix passes */
    uint64_t occ_bytes;
    uint32_t round0_mode;  /* initial sort: 0 = LSD radix passes, 1 = MSD bucket sort of 8-byte elements */
    uint32_t bucket_bits;  /* bucket sort: leading key bits that select a bucket */
    uint32_t sa_sample_rate; /* b200sa_sample_sa: text-position sampling rate of the sampled SA, 0 = none */
    uint32_t sa_resident;    /* 1 while the full suffix array is held in HBM */
    uint32_t shallow_buckets; /* bucket sort: buckets too large for one SM, handed to the doubling rounds unsorted
                                 as groups that share bucket_bits leading key bits (repeats, poly-A runs) */
    uint32_t chain_rounds;    /* doubling rounds that ordered groups by their chain offset (the distance to the
                                 position where the copies of a repeat part) instead of the doubling offset */
    uint64_t shallow_elems;   /* suffixes in them (upper bound) */
    uint64_t chain_elems;     /* suffixes in groups that "continued", summed over those rounds */
    uint64_t lazy_lookups;    /* ranks of retired suffixes recovered on demand */
    uint64_t resolved_small;  /* suffixes in groups of 2..4 equal initial keys decided by the next 64 bits of text */
    uint64_t small_path_elems; /* list elements of doubling rounds ordered inside their tile (groups of <= 32) */
    uint64_t pivot_elems;      /* list elements of doubling rounds that stayed with their group's pivot key and
                                  skipped the radix sort (periodic texts: nearly all), summed over rounds */
    uint32_t pivot_rounds;     /* doubling rounds that split their groups around a pivot key */
    uint32_t pair_placed;      /* suffixes in groups of two equal initial keys (a position of a repeat and the same
                                  position of its copy) decided by one text comparison per repeat */
    uint32_t ktable_k;         /* symbols per entry of the k-mer seed table (B200SA_BUILD_KTABLE), 0 = none */
    uint32_t dense_keys;       /* initial keys formed as base-(letters) numbers (alphabets that do not fill their symbol
                                  width, e.g. DNA + N or amino acids): the number of letters, 0 = raw keys */
};

/* ---- construction ------------------------------------------------------------------------
 * Replaces sa_is_construction / sa_is_mem_construction / skew_sa_construction /
 * qsort_sa_construction (suffix_array.h:22-41), compute_inverse / compute_lcp
 * (suffix_array.h:96-101) and init_bwt_table (bwt.h:73-76) in one call.
 * `stream` is a cudaStream_t (NULL = default stream).  */
b200sa_index *b200sa_build(const uint8_t *codes, uint64_t n, uint32_t sigma, uint32_t flags,
                           int device, void *stream, enum b200sa_error *err);
/* Adds tables that were not requested at build time to an existing index (the reference's lazy
 * compute_inverse / compute_lcp, suffix_array.c:55-85, and init_bwt_table over an existing
 * suffix array, bwt.c:22-89).  `codes` is the same text again (host, or device with
 * B200SA_TEXT_ON_DEVICE); flags is a subset of B200SA_BUILD_{ISA,LCP,BWT,OCC,TEXTCMP,KTABLE}.  Fails with
 * B200SA_ERR_BAD_SYMBOL / _BAD_ARGUMENT (index untouched) when `codes` holds a code outside
 * 1..sigma-1 or is not the text the index was built from (symbol counts differ). */
int b200sa_extend(b200sa_index *idx, const uint8_t *codes, uint32_t flags);
void b200sa_free(b200sa_index *idx);
const char *b200sa_last_error(void);

int b200sa_stats(const b200sa_index *idx, struct b200sa_stats *out);
/* per-stage device times of the last build (needs B200SA_PROFILE): fills up to `cap` entries,
 * returns the number of stages.  bytes[] = algorithmic bytes of the stage (SURVEY 8d model). */
int b200sa_profile(const b200sa_index *idx, const char **names, float *ms, double *bytes, int cap);

/* ---- device-resident views (valid until b200sa_free) --------------------------------------- */
const uint32_t *b200sa_device_sa(const b200sa_index *idx);   /* struct suffix_array.array   */
const uint32_t *b200sa_device_isa(const b200sa_index *idx);  /* .inverse                    */
const uint32_t *b200sa_device_lcp(const b200sa_index *idx);  /* .lcp                        */
const uint8_t *b200sa_device_bwt(const b200sa_index *idx);
const uint8_t *b200sa_device_occ(const b200sa_index *idx);

/* ---- copies into caller-owned HOST memory (len entries each) ------------------------------- */
int b200sa_copy_sa(const b200sa_index *idx, uint32_t *host);
int b200sa_copy_isa(const b200sa_index *idx, uint32_t *host);
int b200sa_copy_lcp(const b200sa_index *idx, uint32_t *host);
int b200sa_copy_bwt(const b200sa_index *idx, uint8_t *host);
int b200sa_copy_c_table(const b200sa_index *idx, uint32_t *host /* sigma entries */);
/* The sampled O table as stored (b200sa_stats.occ_bytes bytes; layout in stralg_b200/csrc/occ.cuh). */
int b200sa_copy_occ(const b200sa_index *idx, uint8_t *host);
/* Asynchronous variant: enqueues the copy of one table on `stream` (a cudaStream_t) and returns;
 * `host` should be pinned memory, and the index must stay alive until the stream has passed the
 * copy.  Lets a caller that builds index after index overlap the transfer of one result with the
 * construction of the next (bench.py's end-to-end loop). */
enum b200sa_table { B200SA_TABLE_SA = 0, B200SA_TABLE_ISA = 1, B200SA_TABLE_LCP = 2, B200SA_TABLE_BWT = 3,
                    B200SA_TABLE_OCC = 4 };
int b200sa_copy_async(const b200sa_index *idx, int what, void *host, void *stream);
/* Dense O table in the reference layout o[i * sigma + a], i in [0, len] (bwt.c:47-65).
 * Fails with B200SA_ERR_TOO_LARGE where the reference's own u32 size computation overflows. */
int b200sa_copy_o_dense(const b200sa_index *idx, uint32_t *host /* (len + 1) * sigma */);
/* O(a[q], i[q]) for q < count (the O(a,i) macro of bwt.h:48-50); host buffers. */
int b200sa_occ(const b200sa_index *idx, const uint8_t *a, const uint32_t *i, uint64_t count,
               uint32_t *out);

/* ---- batched exact search (init_bwt_exact_match_iter, bwt.c:164-199) -----------------------
 * Patterns are remapped codes, concatenated; pattern p is patterns[offsets[p] .. offsets[p+1]).
 * With offsets == NULL every pattern has fixed_len symbols.  Results: half-open SA intervals
 * [L[p], R[p]); L >= R means no match.  Host-buffer and device-buffer variants.
 * A call with ONE pattern of up to 186 symbols on a DNA index (the drop-in's one-iterator-per-pattern use) is served
 * by a one-warp kernel that stays resident on the index's device while such calls keep coming and polls a request
 * slot in mapped pinned memory: no launch and no synchronisation per call.  It leaves by itself after a few
 * milliseconds without a request (B200SA_MAIL_IDLE polls, default 2000) and when its index is freed or extended;
 * B200SA_MAIL_SERVER=0 turns it off. */
int b200sa_search_batch(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets,
                        uint32_t fixed_len, uint64_t npat, uint32_t *L, uint32_t *R);
int b200sa_search_device(const b200sa_index *idx, const uint8_t *d_patterns,
                         const uint64_t *d_offsets, uint32_t fixed_len, uint64_t npat,
                         uint32_t *d_L, uint32_t *d_R, void *stream);
/* ---- packed reads (DNA index, sigma <= 5) ---------------------------------------------------------
 * The consuming application streams FASTQ (bioinf/fastq.c:16-34, bwt_readmapper.c:128-161): reads are
 * short, of one length, over ACGT.  Packed, a read of read_len bases is read_len 2-bit symbols
 * (code - 1), four to a byte, the FIRST base in the two most significant bits of its byte; read q
 * starts at byte q * stride_bytes (stride_bytes >= ceil(read_len / 4); 0 selects exactly that).
 * A quarter of the bytes over PCIe and through the kernel; (L, R) are bit-identical to
 * b200sa_search_batch on the unpacked reads.  The device variant reads whole aligned 8-byte words:
 * d_packed must be 8-byte aligned and readable up to the next 8-byte boundary after the last read.
 * b200sa_pack_reads / _device convert one-byte-per-base codes (1..4; anything else fails with
 * B200SA_ERR_BAD_SYMBOL -- the reference skips such reads, remap.c:80-84, bwt_readmapper.c:136-142). */
int b200sa_search_batch_packed(const b200sa_index *idx, const uint8_t *packed, uint32_t read_len,
                               uint32_t stride_bytes, uint64_t npat, uint32_t *L, uint32_t *R);
int b200sa_search_device_packed(const b200sa_index *idx, const uint8_t *d_packed, uint32_t read_len,
                                uint32_t stride_bytes, uint64_t npat, uint32_t *d_L, uint32_t *d_R,
                                void *stream);
int b200sa_pack_reads(const uint8_t *codes, uint32_t read_len, uint32_t stride_bytes, uint64_t npat,
                      uint8_t *packed);
int b200sa_pack_reads_device(const uint8_t *d_codes, uint32_t read_len, uint32_t stride_bytes,
                             uint64_t npat, uint8_t *d_packed, int device, void *stream);

/* ---- multi-GPU search behind the C ABI (SURVEY 8e; one process, several devices) ------------------
 * The index is replicated, the reads are split into contiguous shards, one per replica, nothing is
 * exchanged on the data path of the search; the (L, R) pairs of every shard are stored by the search
 * kernel itself into the result array in the FIRST replica's HBM through NVLink peer memory (or, where
 * peer access is unavailable, copied from each device), and return to the host from there.
 * b200sa_replicate copies an index to another device (peer copies of the tables it holds) instead of
 * rebuilding it there.  (L, R) are those of b200sa_search_batch_packed on one device. */
b200sa_index *b200sa_replicate(const b200sa_index *src, int device, void *stream, enum b200sa_error *err);
int b200sa_search_sharded_packed(const b200sa_index *const *replicas, int nreplicas, const uint8_t *packed,
                                 uint32_t read_len, uint32_t stride_bytes, uint64_t npat, uint32_t *L,
                                 uint32_t *R);

/* Measurement aid: the same search (DNA index, 8-byte aligned device patterns), run by a counting
 * variant of the kernel.  counts[0] = 32-byte O-block loads, [1] = 8-byte pattern words,
 * [2] = 8-byte packed-text words, [3] = 4-byte SA / ISA loads issued for the whole batch:
 * the algorithmic bytes behind bench.py's search roofline.  Synchronises the stream. */
int b200sa_search_traffic(const b200sa_index *idx, const uint8_t *d_patterns,
                          const uint64_t *d_offsets, uint32_t fixed_len, uint64_t npat,
                          uint32_t *d_L, uint32_t *d_R, uint64_t counts[4], void *stream);
/* the same for packed reads (counts[1] = 8-byte words of packed reads) */
int b200sa_search_traffic_packed(const b200sa_index *idx, const uint8_t *d_packed, uint32_t read_len,
                                 uint32_t stride_bytes, uint64_t npat, uint32_t *d_L, uint32_t *d_R,
                                 uint64_t counts[4], void *stream);

/* ---- locate (next_bwt_exact_match_iter, bwt.c:201-217) -------------------------------------
 * pos_off[npat + 1] receives a CSR; positions of pattern p are pos[pos_off[p] .. pos_off[p+1]),
 * in suffix-array order like the reference iterator.  Call with pos == NULL to size the output
 * (*total is always written); pos_capacity is in entries.  Host buffers. */
int b200sa_locate_batch(const b200sa_index *idx, const uint32_t *L, const uint32_t *R,
                        uint64_t npat, uint64_t *pos_off, uint32_t *pos, uint64_t pos_capacity,
                        uint64_t *total);
int b200sa_locate_device(const b200sa_index *idx, const uint32_t *d_L, const uint32_t *d_R,
                         uint64_t npat, uint64_t *d_pos_off, uint32_t *d_pos,
                         uint64_t pos_capacity, uint64_t *total, void *stream);

/* Same, with the positions of every pattern in ascending order: the order the reference's tests
 * compare in (tests/stralg/match_test.c:608 sorts the iterator's output before checking it). */
int b200sa_locate_batch_sorted(const b200sa_index *idx, const uint32_t *L, const uint32_t *R,
                               uint64_t npat, uint64_t *pos_off, uint32_t *pos,
                               uint64_t pos_capacity, uint64_t *total);
/* Sorts the positions of every pattern of an existing CSR in place (device buffers). */
int b200sa_sort_positions_device(const b200sa_index *idx, uint64_t npat, const uint64_t *d_pos_off,
                                 uint64_t total, uint32_t *d_pos, void *stream);

/* ---- sampled suffix array (SURVEY 8f rank 3) ------------------------------------------------
 * Keeps SA[r] only for the rows whose suffix starts at a multiple of `rate` (a bitmap with rank
 * directory + the sampled values: 0.25 + 4/rate bytes per row instead of 4); every other entry
 * is recovered by at most rate - 1 LF steps over the O table (stralg_b200/csrc/locate.cu), so
 * next_bwt_exact_match_iter's positions (bwt.c:201-217) come out identical.  With drop_sa != 0
 * the full array is released (12 GB at 3 Gbp) and locate uses the sampled one.  Needs OCC. */
int b200sa_sample_sa(b200sa_index *idx, uint32_t rate, int drop_sa);
/* out[q] = SA[rows[q]] (struct suffix_array.array[rows[q]]), host buffers; force_sampled != 0
 * answers through the sampled array even when the full one is resident. */
int b200sa_sa_lookup(const b200sa_index *idx, const uint32_t *rows, uint64_t count, uint32_t *out,
                     int force_sampled);

/* ---- native index file (SURVEY 8f rank 1, large n) --------------------------------------------
 * The reference's own files (write_complete_bwt_info, serialise.c:7-49; served by the shim) hold the
 * dense O table and u32 element counts (bwt.c:430) and cannot represent a 3 Gbp index.  This
 * format stores what is resident in HBM: a fixed header (magic "B200SAIX", version, byte-order
 * mark, n, sigma, primary, C table, O layout) followed by tagged sections {tag[8], element bytes,
 * count, raw array}: SA, ISA, LCP, BWT, OCC (sampled O blocks), TEXT (packed text), KTABLE,
 * SSAMARK / SSAVAL (sampled suffix array), RECOFF (record offsets of a records index).  b200sa_load returns an index that answers search /
 * locate / approximate search exactly like the one that was saved, without rebuilding. */
int b200sa_save(const b200sa_index *idx, const char *path);
b200sa_index *b200sa_load(const char *path, int device, void *stream, enum b200sa_error *err);

/* ---- records index: many records in one build ------------------------------------------------
 * A multi-record reference (chromosomes and contigs, transcript sets) in ONE index.  The records are
 * codes 2..sigma-1; code 1 is the separator, which the library inserts after every record, the last
 * one included:  r0 1 r1 1 ... r(k-1) 1 $.  Record r has len_r = rec_off[r+1] - rec_off[r] >= 0
 * symbols and starts at text position start_r = rec_off[r] + r; its separator at start_r + len_r
 * plays its own sentinel.  n = rec_off[nrec] + nrec <= 2^32 - 2; sigma (b200sa_stats) counts the
 * separator.  The separator sorts below every letter, so the global suffix array restricted to one
 * record's positions is that record's own suffix array, in the same order: one build serves every
 * record, and an exact match never crosses a record (patterns never hold code 1).
 *
 * b200sa_build_records: `codes` holds the records back to back without separators, rec_off[nrec + 1]
 * (host; rec_off[0] = 0) the record boundaries, so `codes` has rec_off[nrec] symbols (a host array, or a
 * device array with B200SA_TEXT_ON_DEVICE).  The separators are inserted on the device; the text then
 * takes the path of b200sa_build.  Flags: OCC, TEXTCMP, KTABLE, DROP_SA, PROFILE, TEXT_ON_DEVICE; ISA,
 * LCP or BWT -> B200SA_ERR_BAD_ARGUMENT (per-record tables of that kind do not exist).  A code 0, 1 or
 * >= sigma -> _BAD_SYMBOL; offsets that decrease or rec_off[0] != 0 -> _BAD_ARGUMENT; n > 2^32 - 2 ->
 * _TOO_LARGE.
 *
 * On a records index every other entry point works on the whole text and returns global rows
 * (search, locate, sample_sa, sa_lookup).  b200sa_search_batch and b200sa_approx_batch refuse a
 * pattern holding code 1 (_BAD_SYMBOL); with b200sa_search_device keeping code 1 out is the caller's
 * duty.  The packed-read entry points refuse a records index whatever its sigma (_NOT_BUILT): packed
 * base 0 would be code 1, the separator (a DNA records index, ACGT and the separator, has the byte
 * O-table layout anyway).  b200sa_extend -> _BAD_ARGUMENT.  The approximate
 * search never consumes the separator: same report order per record as the record's own index.
 * b200sa_replicate and b200sa_save / b200sa_load carry the record offsets (file section RECOFF;
 * builds of the library from before records indices refuse such a file as an unknown section).
 *
 * b200sa_records: *nrec (0 for a plain index) and, when rec_off is not NULL, its nrec + 1 offsets.
 * b200sa_copy_record_sas / _device: every record's own suffix array back to back -- record r's
 * len_r + 1 entries, in local positions, at offset start_r; n entries in all (the global sentinel row
 * belongs to no record).  Each equals b200sa_copy_sa of b200sa_build on that record alone.  Needs the
 * full suffix array (_NOT_BUILT after DROP_SA).
 * b200sa_locate_records / _device: like b200sa_locate_batch, a CSR pos_off[npat + 1] over entries that
 * are (rec[k], pos[k]) pairs: the record and the local position.  Within a pattern, records ascend and
 * the positions of one record come in that record's suffix-array order (the reference iterator's order
 * on the record's own index).  Row 0 (the global sentinel) is skipped.  rec and pos are both NULL to
 * size the output (*total).  A plain index -> _BAD_ARGUMENT. */
b200sa_index *b200sa_build_records(const uint8_t *codes, const uint64_t *rec_off, uint32_t nrec, uint32_t sigma,
                                   uint32_t flags, int device, void *stream, enum b200sa_error *err);
int b200sa_records(const b200sa_index *idx, uint32_t *nrec, uint64_t *rec_off /* NULL or nrec + 1 entries */);
int b200sa_copy_record_sas(const b200sa_index *idx, uint32_t *host /* n entries */);
int b200sa_record_sas_device(const b200sa_index *idx, uint32_t *d_out, void *stream);
int b200sa_locate_records(const b200sa_index *idx, const uint32_t *L, const uint32_t *R, uint64_t npat,
                          uint64_t *pos_off, uint32_t *rec, uint32_t *pos, uint64_t capacity, uint64_t *total);
int b200sa_locate_records_device(const b200sa_index *idx, const uint32_t *d_L, const uint32_t *d_R, uint64_t npat,
                                 uint64_t *d_pos_off, uint32_t *d_rec, uint32_t *d_pos, uint64_t capacity,
                                 uint64_t *total, void *stream);

/* ---- batched approximate search (SURVEY 8f rank 4) -------------------------------------------
 * Replaces init_bwt_approx_iter / next_bwt_approx_match (bwt.h:246-333, bwt.c:226-409): all
 * intervals whose suffixes match the pattern within `max_edits` edits (substitutions, insertions,
 * deletions), per pattern in the order the reference's depth-first recursion reports them,
 * duplicates included, each with its matched text length and CIGAR (cigar.c:8-31).
 * `rev_idx` (may be NULL) is an index (B200SA_BUILD_OCC) of the REVERSED text: it provides the
 * reference's D table (bwt.c:319-337), which only prunes -- results are the same without it.
 * `d_table` (may be NULL) passes a precomputed D table instead: one byte per pattern symbol, laid
 * out like `patterns`.  Positions: b200sa_locate_batch over the returned (L, R) arrays; the
 * reference reports position SA[L..R) for every interval in turn (bwt.c:384-401).
 * Accessors return host arrays owned by the result (valid until b200sa_approx_free). */
typedef struct b200sa_approx_result b200sa_approx_result;
b200sa_approx_result *b200sa_approx_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                          const uint8_t *d_table, const uint8_t *patterns,
                                          const uint64_t *offsets, uint32_t fixed_len, uint64_t npat,
                                          int max_edits, enum b200sa_error *err);
uint64_t b200sa_approx_hits(const b200sa_approx_result *r);              /* intervals in total   */
const uint64_t *b200sa_approx_hit_offsets(const b200sa_approx_result *r);/* npat + 1 (CSR)       */
const uint32_t *b200sa_approx_L(const b200sa_approx_result *r);
const uint32_t *b200sa_approx_R(const b200sa_approx_result *r);
const uint32_t *b200sa_approx_match_length(const b200sa_approx_result *r);
const uint64_t *b200sa_approx_cigar_offsets(const b200sa_approx_result *r); /* hits + 1          */
const char *b200sa_approx_cigars(const b200sa_approx_result *r);  /* NUL-terminated, back to back */
void b200sa_approx_free(b200sa_approx_result *r);

/* ---- matching statistics and super-maximal exact matches (SMEMs) ----------------------------
 * Seeds for reads that do not occur whole (sequencing errors, SNPs, long reads), as BWA-MEM seeds.
 * Patterns take the form of b200sa_search_batch (patterns / offsets / fixed_len, host buffers).
 * For a pattern P[0..m) in remapped codes and every end j (0 <= j < m):
 *   s_j   = the smallest s such that P[s..j] occurs in the text; j + 1 when no suffix of P[0..j] does;
 *   ms[j] = j + 1 - s_j, the length of the longest substring of P that ends at j and occurs in the text;
 *   [L[j], R[j]) = the SA interval of P[s_j..j], what b200sa_search_batch returns for that substring;
 *                  (1, 0), the search's no-match pair, when ms[j] = 0.
 * An SMEM is (start = s_j, length = ms[j], L[j], R[j]) for every j with ms[j] >= min_len and
 * (j = m - 1 or ms[j+1] <= ms[j]), i.e. s_{j+1} > s_j: since s never decreases, exactly the occurring
 * pieces of P that no other occurring piece contains.  Per pattern, SMEMs come in ascending start.
 * A code 0 or >= sigma in a pattern occurs nowhere: it gets ms = 0 and breaks every match across it
 * (not an error, as the search answers (1, 0) for it).  On a records index a pattern holding code 1,
 * the separator, is refused with B200SA_ERR_BAD_SYMBOL, so an SMEM never crosses a record; its
 * positions come from b200sa_locate_records over (L, R).  An empty pattern has no entries and no
 * SMEMs.  min_len = 0 -> B200SA_ERR_BAD_ARGUMENT; an index without OCC -> B200SA_ERR_NOT_BUILT.
 * TEXTCMP and KTABLE make the computation faster; results are identical with and without them.
 * b200sa_matching_stats: ms, L and R are laid out like `patterns` (entry offsets[p] + j); L and R may
 * be NULL.  b200sa_smem_batch: accessors return host arrays owned by the result (valid until
 * b200sa_smem_free).  Both stage long batches in pieces of about 64 MB of pattern symbols. */
int b200sa_matching_stats(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets,
                          uint32_t fixed_len, uint64_t npat, uint32_t *ms, uint32_t *L, uint32_t *R);
typedef struct b200sa_smem_result b200sa_smem_result;
b200sa_smem_result *b200sa_smem_batch(const b200sa_index *idx, const uint8_t *patterns,
                                      const uint64_t *offsets, uint32_t fixed_len, uint64_t npat,
                                      uint32_t min_len, enum b200sa_error *err);
uint64_t b200sa_smem_count(const b200sa_smem_result *r);             /* SMEMs in total        */
const uint64_t *b200sa_smem_offsets(const b200sa_smem_result *r);    /* npat + 1 (CSR)        */
const uint32_t *b200sa_smem_start(const b200sa_smem_result *r);
const uint32_t *b200sa_smem_length(const b200sa_smem_result *r);
const uint32_t *b200sa_smem_L(const b200sa_smem_result *r);
const uint32_t *b200sa_smem_R(const b200sa_smem_result *r);
void b200sa_smem_free(b200sa_smem_result *r);

/* ---- batched k-mismatch search on a bidirectional FM index -----------------------------------
 * Every distinct text string within Hamming distance k of a read, each reported once: for short
 * reads, barcodes, primers and off-target scans that need substitutions only.  (b200sa_approx_batch
 * is the edit-distance search of the reference: it reports every edit path, so the same interval
 * many times, in the reference's order.)
 * Patterns take the form of b200sa_search_batch: remapped codes, concatenated, in host buffers, with
 * `offsets` or `fixed_len`.  For a pattern P of length m >= 1 and k = max_mismatches, the hits are
 * every distinct string Q with
 *   |Q| = m,  Q over the letters 1..sigma-1,  Q occurs in the text,  Hamming(P, Q) <= k;
 * each hit is one triple (L, R, d): [L, R) is Q's SA interval in `idx` (what b200sa_search_batch
 * returns for Q) and d = Hamming(P, Q).  Hits of one pattern come in ascending L: the intervals of
 * distinct strings of one length are disjoint, so the order is total and does not depend on how the
 * search runs.  A pattern symbol 0 or >= sigma is not an error: it differs from every letter and costs
 * one mismatch there.  An empty pattern has no hits; k = 0 gives exactly the non-empty results of
 * b200sa_search_batch, each with d = 0.  Positions: b200sa_locate_batch / _sorted over (L, R).
 * `rev_idx` is required: an index (B200SA_BUILD_OCC) of the reversed text (codes n-1 .. 0) on the same
 * device, as for b200sa_approx_batch's D table; it may drop its suffix array.  Only the checks below
 * are made: beyond them the caller guarantees that it really is the reversed text.
 * Refusals, all before any CUDA call: NULL idx or rev_idx, NULL patterns with npat > 0, decreasing
 * offsets, max_mismatches > 8 -> B200SA_ERR_BAD_ARGUMENT; a pattern longer than 65000 symbols ->
 * B200SA_ERR_TOO_LARGE; either index without OCC -> B200SA_ERR_NOT_BUILT; rev_idx of another length,
 * sigma, device or C table, or either index a records index -> B200SA_ERR_BAD_ARGUMENT.
 * TEXTCMP and KTABLE do not change the results.  Long batches are staged in pieces of about 64 MB of
 * pattern symbols; a piece with more than 2^32 - 1 hits -> B200SA_ERR_TOO_LARGE.  Accessors return
 * host arrays owned by the result (valid until b200sa_hamming_free). */
typedef struct b200sa_hamming_result b200sa_hamming_result;
b200sa_hamming_result *b200sa_hamming_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                            const uint8_t *patterns, const uint64_t *offsets,
                                            uint32_t fixed_len, uint64_t npat, uint32_t max_mismatches,
                                            enum b200sa_error *err);
uint64_t b200sa_hamming_hits(const b200sa_hamming_result *r);          /* hits in total         */
const uint64_t *b200sa_hamming_offsets(const b200sa_hamming_result *r);/* npat + 1 (CSR)        */
const uint32_t *b200sa_hamming_L(const b200sa_hamming_result *r);
const uint32_t *b200sa_hamming_R(const b200sa_hamming_result *r);
const uint32_t *b200sa_hamming_mismatches(const b200sa_hamming_result *r);
void b200sa_hamming_free(b200sa_hamming_result *r);

/* ---- batched edit-distance search on a bidirectional FM index -------------------------------
 * Every distinct text string within Levenshtein distance k of a read, each reported once: for primers
 * and guides with bulges, barcodes with synthesis indels and short reads from indel-prone platforms.
 * (b200sa_approx_batch reports every edit path in the reference's order; b200sa_hamming_batch takes
 * substitutions only.)  Patterns take the form of b200sa_search_batch.  For a pattern P of length
 * m >= 1 and k = max_edits, the hits are every distinct string Q with
 *   Q non-empty,  Q over the letters 1..sigma-1,  Q occurs in the text,  ED(P, Q) <= k,
 * where ED is the Levenshtein distance with unit cost for substitution, insertion and deletion; so
 * m - k <= |Q| <= m + k.  Each hit is (L, R, length, d): [L, R) is Q's SA interval in `idx` (what
 * b200sa_search_batch returns for Q), length = |Q| and d = ED(P, Q).  Hits of one pattern come in
 * ascending L, then ascending length: distinct strings of one length have disjoint intervals, so
 * (L, length) identifies Q and the order does not depend on how the search runs.  A pattern symbol 0
 * or >= sigma matches no letter (substituting or deleting it costs 1); it is not an error.  An empty
 * pattern has no hits; k = 0 gives exactly the non-empty results of b200sa_search_batch, with
 * length = m and d = 0.
 * The set holds near-duplicates of every occurrence by design: an exact occurrence of P at position p
 * also yields T[p+a .. p+m+b) for |a| + |b| <= k, up to 2k^2 + 2k + 1 hits (13 at k = 2).  Callers
 * locate the hits (b200sa_locate_batch / _sorted over (L, R)) and choose among them.
 * `rev_idx` and the refusals are those of b200sa_hamming_batch, all before any CUDA call, with
 * max_edits > 4 -> B200SA_ERR_BAD_ARGUMENT.  TEXTCMP and KTABLE do not change the results.  Long
 * batches are staged in pieces of about 64 MB of pattern symbols and at most 2^28 patterns; a piece
 * with more than 2^32 - 1 raw hits (before the near-identical hits of several searches are merged)
 * -> B200SA_ERR_TOO_LARGE.  Accessors return host arrays owned by the result (valid until
 * b200sa_levenshtein_free). */
typedef struct b200sa_levenshtein_result b200sa_levenshtein_result;
b200sa_levenshtein_result *b200sa_levenshtein_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                                    const uint8_t *patterns, const uint64_t *offsets,
                                                    uint32_t fixed_len, uint64_t npat, uint32_t max_edits,
                                                    enum b200sa_error *err);
uint64_t b200sa_levenshtein_hits(const b200sa_levenshtein_result *r);           /* hits in total  */
const uint64_t *b200sa_levenshtein_offsets(const b200sa_levenshtein_result *r); /* npat + 1 (CSR) */
const uint32_t *b200sa_levenshtein_L(const b200sa_levenshtein_result *r);
const uint32_t *b200sa_levenshtein_R(const b200sa_levenshtein_result *r);
const uint32_t *b200sa_levenshtein_length(const b200sa_levenshtein_result *r);
const uint32_t *b200sa_levenshtein_distance(const b200sa_levenshtein_result *r);
void b200sa_levenshtein_free(b200sa_levenshtein_result *r);

/* ---- synthetic inputs on the device (bench / tests; mirrors performance/suffix_array_search.c:13-32)
 * d_text must hold n + 1 bytes; symbols are 1 + hash(seed + i) % nsym, d_text[n] = 0. */
int b200sa_synth_codes(uint8_t *d_text, uint64_t n, uint32_t nsym, uint64_t seed, int device,
                       void *stream);
int b200sa_synth_reads(const uint8_t *d_text, uint64_t n, uint32_t nsym, uint8_t *d_reads,
                       uint64_t nreads, uint32_t m, uint32_t miss_per_1024, uint64_t seed,
                       int device, void *stream);

int b200sa_device_count(void);
/* The build workspace (a few large device allocations) persists per device between builds so that
 * steady-state builds never call cudaMalloc; release it explicitly when memory is needed. */
uint64_t b200sa_workspace_bytes(int device);
int b200sa_release_workspace(int device);
/* kernels launched by this library in this process so far (bench accounting) */
uint64_t b200sa_launch_count(void);
/* Diagnostic, host only (no GPU needed): the plan of the bucketed initial sort for a text of `len` = n + 1 symbols
 * over `sigma` codes; sym_counts (256 entries, occurrences per code) may be NULL.  out[16] = {applies, levels,
 * D1, D2, D3, bucket bits, key symbols K, key bits, bits of the preceding symbol carried, remainder bits,
 * dense letters (0 = raw keys), Khi, Klo, nsym^Klo, symbol width, 0}.  Returns 0. */
int b200sa_plan_round0(uint32_t len, uint32_t sigma, const uint64_t *sym_counts, uint64_t out[16]);

#ifdef __cplusplus
}
#endif
#endif /* B200SA_H */
