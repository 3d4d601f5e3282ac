/*
 * stralg_compat.h -- drop-in declarations for the hot-path surface of mailund/stralg, served by
 * the B200 engine (libstralg_b200.so, built from stralg_b200/csrc/compat.cpp on top of b200sa.h).
 *
 * Every name, argument list and struct layout below is the reference's (file:line cited, paths
 * relative to the stralg checkout), so a caller compiled against stralg's own suffix_array.h /
 * bwt.h / remap.h links against this library unchanged.  Only the hot path is covered: alphabet
 * remap, the four suffix-array constructors (all served by ONE GPU constructor), inverse + LCP,
 * the SA binary searches (host code over the copied array), BWT C/O tables, and the exact-match
 * iterator.  The approximate iterator, suffix trees etc. are out of scope (SURVEY.md section 8).
 *
 * Ownership follows the reference: arrays hanging off these structs are malloc()'d host memory,
 * free_suffix_array() frees array/inverse/lcp with free(), the string is borrowed unless the
 * *_complete_* variants are used (suffix_array.c:11-23, bwt.c:91-132).
 * Failure convention: these signatures have no error channel (the reference never checks
 * malloc either); on a CUDA failure the shim prints b200sa_last_error() to stderr and aborts.
 */
#ifndef STRALG_COMPAT_H
#define STRALG_COMPAT_H

#include <stdbool.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- remap.h:9-19 ------------------------------------------------------------------------ */
struct remap_table {
    uint32_t alphabet_size;
    signed char table[256];
    signed char rev_table[128];
};
struct remap_table *alloc_remap_table(const uint8_t *string);                 /* remap.h:21-23 */
void init_remap_table(struct remap_table *table, const uint8_t *string);      /* remap.h:24-27 */
void dealloc_remap_table(struct remap_table *table);                          /* remap.h:28-30 */
void free_remap_table(struct remap_table *table);                             /* remap.h:31-33 */
uint8_t *remap(uint8_t *output, const uint8_t *input, struct remap_table *table);      /* :43-47 */
uint8_t *rev_remap(uint8_t *output, const uint8_t *input, struct remap_table *table);  /* :48-52 */
uint8_t *remap_between(uint8_t *output, const uint8_t *from, const uint8_t *to,
                       struct remap_table *table);                                     /* :54-59 */
uint8_t *rev_remap_between(uint8_t *output, const uint8_t *from, const uint8_t *to,
                           struct remap_table *table);                                 /* :60-65 */
uint8_t *remap_between0(uint8_t *output, const uint8_t *from, const uint8_t *to,
                        struct remap_table *table);                                    /* :66-71 */
uint8_t *rev_remap_between0(uint8_t *output, const uint8_t *from, const uint8_t *to,
                            struct remap_table *table);                                /* :72-77 */
uint32_t remap_string(uint8_t *output, uint8_t *input);                                /* :83-86 */
bool identical_remap_tables(const struct remap_table *a, const struct remap_table *b); /* :116-119 */

/* ---- suffix_array.h:10-20 ----------------------------------------------------------------- */
struct suffix_array {
    uint8_t *string;   /* borrowed, NUL terminated */
    uint32_t length;   /* strlen(string) + 1: the sentinel suffix is a real suffix */
    uint32_t *array;
    uint32_t *inverse; /* NULL until compute_inverse() */
    uint32_t *lcp;     /* NULL until compute_lcp() */
};
/* suffix_array.h:22-41 -- four names, one GPU prefix-doubling constructor */
struct suffix_array *qsort_sa_construction(uint8_t *string);
struct suffix_array *skew_sa_construction(uint8_t *string);
struct suffix_array *sa_is_construction(uint8_t *remapped_string, uint32_t alphabet_size);
struct suffix_array *sa_is_mem_construction(uint8_t *remapped_string, uint32_t alphabet_size);
void free_suffix_array(struct suffix_array *sa);                     /* suffix_array.h:45-47 */
void free_complete_suffix_array(struct suffix_array *sa);            /* suffix_array.h:49-51 */
void compute_inverse(struct suffix_array *sa);                       /* suffix_array.h:96-98 */
void compute_lcp(struct suffix_array *sa);                           /* suffix_array.h:99-101 */
bool identical_suffix_arrays(const struct suffix_array *sa1, const struct suffix_array *sa2);

/* suffix_array.h:54-94 -- binary searches over the (host copy of the) suffix array */
uint32_t lower_bound_search(struct suffix_array *sa, const uint8_t *key);
uint32_t upper_bound_search(struct suffix_array *sa, const uint8_t *key);
uint32_t lower_bound_k(struct suffix_array *sa, uint32_t k, uint8_t a, uint32_t L, uint32_t R);
uint32_t upper_bound_k(struct suffix_array *sa, uint32_t k, uint8_t a, uint32_t L, uint32_t R);
struct sa_match_iter {
    struct suffix_array *sa;
    uint32_t L;
    uint32_t R;
    uint32_t i;
};
struct sa_match {
    uint32_t position;
};
void init_sa_match_iter(struct sa_match_iter *iter, const uint8_t *pattern, struct suffix_array *sa);
bool next_sa_match(struct sa_match_iter *iter, struct sa_match *match);
void dealloc_sa_match_iter(struct sa_match_iter *iter);

/* ---- bwt.h:36-50 ---------------------------------------------------------------------------- */
struct bwt_table {
    struct remap_table *remap_table;
    struct suffix_array *sa;
    uint32_t *c_table;
    uint32_t *o_table;     /* dense (length+1) x sigma, row-major by position; NULL when the   */
    uint32_t **o_indices;  /* reference's own u32 size computation would overflow (bwt.c:50)   */
    uint32_t *ro_table;
    uint32_t **ro_indices;
};
#ifndef STRALG_COMPAT_NO_MACROS
#define C(a) (bwt_table->c_table[(a)])
#define O(a, i) (bwt_table->o_indices[i][a])
#define RO(a, i) (bwt_table->ro_indices[i][a])
#endif
void init_bwt_table(struct bwt_table *bwt_table, struct suffix_array *sa, struct suffix_array *rsa,
                    struct remap_table *remap_table);                               /* bwt.h:73-76 */
struct bwt_table *alloc_bwt_table(struct suffix_array *sa, struct suffix_array *rsa,
                                  struct remap_table *remap_table);                 /* bwt.h:97-99 */
void dealloc_bwt_table(struct bwt_table *bwt_table);                                /* bwt.h:109 */
void free_bwt_table(struct bwt_table *bwt_table);                                   /* bwt.h:119 */
void completely_dealloc_bwt_table(struct bwt_table *bwt_table);                     /* bwt.h:129 */
void completely_free_bwt_table(struct bwt_table *bwt_table);                        /* bwt.h:138 */
struct bwt_table *build_complete_table(const uint8_t *string, bool include_reverse); /* bwt.h:156-160 */
bool equivalent_bwt_tables(struct bwt_table *table1, struct bwt_table *table2);

/* bwt.h:168-234 -- exact-match iterator (stack allocated by callers, so the layout is ABI) */
struct bwt_exact_match_iter {
    const struct suffix_array *sa;
    uint32_t L;
    int64_t i;
    uint32_t R;
};
struct bwt_exact_match {
    uint32_t pos;
};
void init_bwt_exact_match_iter(struct bwt_exact_match_iter *iter, struct bwt_table *bwt_table,
                               const uint8_t *remapped_pattern);
bool next_bwt_exact_match_iter(struct bwt_exact_match_iter *iter, struct bwt_exact_match *match);
void dealloc_bwt_exact_match_iter(struct bwt_exact_match_iter *iter);

/* ---- extension: the batched entry point a read mapper should call instead of one iterator per
 * read (tools/readmappers/bwt_readmapper/bwt_readmapper.c:128-161 maps one read at a time). */
void bwt_exact_match_batch(struct bwt_table *bwt_table, const uint8_t *remapped_patterns,
                           const uint64_t *offsets, uint64_t npatterns, uint32_t *L, uint32_t *R);
/* The same for reads of ONE length over a DNA alphabet, packed to 2 bits per base (four bases per byte, first
 * base in the high bits, read q at byte q * stride_bytes; b200sa.h: b200sa_pack_reads). */
void bwt_exact_match_batch_packed(struct bwt_table *bwt_table, const uint8_t *packed_reads, uint32_t read_len,
                                  uint32_t stride_bytes, uint64_t nreads, uint32_t *L, uint32_t *R);
/* Measurement aid: one iterator per pattern (the loop of performance/suffix_array_search.c:127-141) over
 * npat NUL-terminated remapped patterns laid out with a stride of m + 1 bytes; returns the matches. */
uint64_t bwt_exact_match_loop(struct bwt_table *tbl, const uint8_t *patterns, uint32_t m, uint64_t npat);

/* bwt.h:246-333 -- approximate-match iterator (SURVEY 8f rank 4).  Layouts are the reference's
 * (vectors.h:29-33, 153-157; bwt.h:246-259, 277-281); callers stack-allocate the iterator.
 * init runs the whole D-table-pruned search (bwt.c:226-382) on the GPU and fills Ls / Rs /
 * match_lengths / cigars in the reference's report order; next walks them (bwt.c:384-401). */
struct index_vector {
    uint32_t *data;
    uint32_t size;
    uint32_t used;
};
struct string_vector {
    uint8_t **data;
    uint32_t size;
    uint32_t used;
};
struct bwt_approx_iter {
    struct bwt_table *bwt_table;
    const uint8_t *remapped_pattern;
    uint32_t L, R, next_interval;
    struct index_vector Ls;
    struct index_vector Rs;
    struct string_vector cigars;
    struct index_vector match_lengths;
    uint32_t m;
    char *edits_buf;
    int *D_table;
};
struct bwt_approx_match {
    const char *cigar;
    uint32_t position;
    uint32_t match_length;
};
void init_bwt_approx_iter(struct bwt_approx_iter *iter, struct bwt_table *bwt_table,
                          const uint8_t *remapped_pattern, int edits);             /* bwt.h:290-295 */
bool next_bwt_approx_match(struct bwt_approx_iter *iter, struct bwt_approx_match *match); /* :311-314 */
void dealloc_bwt_approx_iter(struct bwt_approx_iter *iter);                        /* :329-331 */

/* ---- index files (SURVEY 8f rank 1): the reference's own on-disk layouts, byte for byte ----------
 * Raw host-endian dumps without header (suffix_array.c:238-267, remap.c:168-201, bwt.c:425-503,
 * serialise.c:7-49, string_utils.c:48-82).  A file written by either library is read by the other.
 * Tables whose dense O the reference itself cannot size (u32 overflow, bwt.c:430) cannot be
 * written in this format: write_bwt_table aborts with a message.  What is read back is host
 * memory; the device index is rebuilt from the string on first use (same arrays by uniqueness). */
void write_suffix_array(FILE *f, const struct suffix_array *sa);                      /* suffix_array.h:109 */
void write_suffix_array_fname(const char *fname, const struct suffix_array *sa);      /* :113 */
struct suffix_array *read_suffix_array(FILE *f, uint8_t *string);                     /* :118 */
struct suffix_array *read_suffix_array_fname(const char *fname, uint8_t *string);     /* :123 */
void write_remap_table(FILE *f, const struct remap_table *table);                     /* remap.h:89 */
void write_remap_table_fname(const char *fname, const struct remap_table *table);     /* :93 */
struct remap_table *read_remap_table(FILE *f);                                        /* :98 */
struct remap_table *read_remap_table_fname(const char *fname);                        /* :102 */
void write_bwt_table(FILE *f, const struct bwt_table *bwt_table);                     /* bwt.h:337 */
void write_bwt_table_fname(const char *fname, const struct bwt_table *bwt_table);     /* :341 */
struct bwt_table *read_bwt_table(FILE *f, struct suffix_array *sa, struct remap_table *remap_table);  /* :346 */
struct bwt_table *read_bwt_table_fname(const char *fname, struct suffix_array *sa,
                                       struct remap_table *remap_table);              /* :351 */
void write_complete_bwt_info(FILE *f, const struct bwt_table *bwt_table);             /* serialise.h:23 */
void write_complete_bwt_info_fname(const char *fname, const struct bwt_table *bwt_table);  /* :24 */
struct bwt_table *read_complete_bwt_info(FILE *f);                                    /* :32 */
struct bwt_table *read_complete_bwt_info_fname(const char *fname);                    /* :33 */

/* ---- reads in, SAM out (SURVEY 8f rank 2): `bwt_readmapper -d 0`, batched --------------------------
 * The reference maps one read at a time (map_read, tools/readmappers/bwt_readmapper/bwt_readmapper.c:
 * 128-161): for every FASTQ record (bioinf/fastq.c:16-34), for every reference record in list order,
 * remap the read with that record's table (skipped when remap() returns NULL), enumerate the matches
 * and print one SAM line each (bioinf/sam.c:4-10; position 1-based, CIGAR "<m>M").  With zero edits
 * its approximate iterator yields exactly the interval of the exact iterator, in suffix-array order.
 * bwt_map_fastq_exact does the same for a whole FASTQ stream, `batch_reads` reads per GPU batch
 * (one backward-search launch per batch and record); the output is byte-identical to the
 * reference tool's.  Returns the number of SAM lines written. */
uint64_t bwt_map_fastq_exact(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                             struct bwt_table *const *tables, uint64_t batch_reads);
/* `bwt_readmapper -d <edits>` for any edit distance: the approximate search of every batch runs as
 * one GPU call per reference record (b200sa_approx_batch, D table from the table's RO rows when it
 * has them, bwt.c:319-337), SAM lines in the tool's order (reads, records, intervals in report
 * order, positions in suffix-array order) with the tool's CIGARs.  Byte-identical to the tool. */
uint64_t bwt_map_fastq(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                       struct bwt_table *const *tables, int edits, uint64_t batch_reads);
/* The same mapping against ONE records index (include/b200sa.h: b200sa_build_records) over all the tables'
 * strings, turned back into bytes with their remap tables and remapped with one union alphabet: per batch
 * one search or approximate-search call and one b200sa_locate_records call, however many records there
 * are, where bwt_map_fastq makes one call per record and remaps every read once per record on the host.
 * Same contract, byte-identical SAM: a read with a letter missing from record r's own alphabet gives no
 * line for r (the tool's remap() skip), lines in the tool's order.  With edits > 0 and reverse O tables in
 * every table, the D table comes from an index of the reversed text (it prunes, the results are the same).
 * A record's letters are those its remap table codes (as for bwt_map_fastq's remap of a read); the tables'
 * codes must follow byte order, as init_remap_table / build_complete_table make them, so that the union
 * alphabet takes a record's letters in the order its own table does (the approximate search's report order). */
uint64_t bwt_map_fastq_records(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                               struct bwt_table *const *tables, int edits, uint64_t batch_reads);
/* The multi-record index file of `bwt_readmapper -p` (bwt_readmapper.c:48-61): [u32 records], then per
 * record [u32 len][name incl. NUL] (string_utils.c:48-65) + write_complete_bwt_info.  The tool writes
 * the FASTA records in REVERSE file order (bioinf/fasta.c:131 prepends) and maps in the reverse of
 * the order read (bwt_readmapper.c:107 prepends again).  read_bwt_tables_file returns file order;
 * names[i] and tables[i] are malloc'd (free the arrays with free(), tables with
 * completely_free_bwt_table). */
void write_bwt_tables_file(const char *fname, uint32_t nrecords, const char *const *record_names,
                           struct bwt_table *const *tables);
uint32_t read_bwt_tables_file(const char *fname, char ***record_names, struct bwt_table ***tables);

#ifdef __cplusplus
}
#endif
#endif /* STRALG_COMPAT_H */
