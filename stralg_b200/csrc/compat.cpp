// compat.cpp -- libstralg_b200.so: the reference-named hot-path functions of mailund/stralg
// (include/stralg_compat.h) implemented on top of the B200 engine's C ABI (include/b200sa.h).
//
// Every array these functions hand out is malloc()'d host memory with the reference's layout and
// ownership; every computation that the reference does in sa_is.c / skew.c / suffix_array.c:55-85 /
// bwt.c:22-89 / bwt.c:164-199 runs on the GPU.  A side registry maps each `struct suffix_array *`
// to its device-resident index so that later calls (compute_lcp, init_bwt_table, the exact
// iterator) reuse the suffix array already in HBM.  Host-only pieces: the alphabet remap
// (remap.c), the SA binary searches (suffix_array.c:90-233, kept on the host by design, SURVEY
// 8a row a16), the comparison helpers and the index-file readers / writers (SURVEY 8f rank 1).
#include "../../include/b200sa.h"
#define STRALG_COMPAT_NO_MACROS
#include "../../include/stralg_compat.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

std::mutex g_mu;
std::unordered_map<const void *, b200sa_index *> g_index;  // struct suffix_array* -> device index

[[noreturn]] void die(const char *where) {
    fprintf(stderr, "stralg_b200: %s failed: %s\n", where, b200sa_last_error());
    abort();
}

b200sa_index *lookup(const struct suffix_array *sa) {
    std::lock_guard<std::mutex> lock(g_mu);
    auto it = g_index.find(sa);
    return it == g_index.end() ? nullptr : it->second;
}

void remember(const struct suffix_array *sa, b200sa_index *idx) {
    std::lock_guard<std::mutex> lock(g_mu);
    g_index[sa] = idx;
}

void forget(const struct suffix_array *sa) {
    b200sa_index *idx = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        auto it = g_index.find(sa);
        if (it != g_index.end()) {
            idx = it->second;
            g_index.erase(it);
        }
    }
    b200sa_free(idx);
}

int device_id() {
    const char *e = getenv("STRALG_B200_DEVICE");
    return e && *e ? atoi(e) : 0;
}

// STRALG_B200_TRACE=1: at exit, one line on stderr with the number of calls the drop-in served (how a
// test that runs the reference's own binaries knows which library did the work)
struct Trace {
    unsigned long constructions = 0, tables = 0, exact_iters = 0, approx_iters = 0;
    ~Trace() {
        const char *e = getenv("STRALG_B200_TRACE");
        if (e && *e && *e != '0')
            fprintf(stderr, "stralg_b200: served constructions=%lu tables=%lu exact_iters=%lu approx_iters=%lu\n",
                    constructions, tables, exact_iters, approx_iters);
    }
} g_trace;

// One GPU constructor behind the four reference names.
struct suffix_array *construct(uint8_t *string, uint32_t sigma, const char *who) {
    struct suffix_array *sa = (struct suffix_array *)malloc(sizeof *sa);
    size_t n = strlen((const char *)string);
    sa->string = string;
    sa->length = (uint32_t)n + 1;  // suffix_array_internal.c:12
    sa->array = (uint32_t *)malloc((size_t)sa->length * sizeof(uint32_t));
    sa->inverse = nullptr;
    sa->lcp = nullptr;
    enum b200sa_error err;
    ++g_trace.constructions;
    b200sa_index *idx = b200sa_build(string, n, sigma, 0, device_id(), nullptr, &err);
    if (!idx) die(who);
    if (b200sa_copy_sa(idx, sa->array)) die(who);
    remember(sa, idx);
    return sa;
}

// The device index of `sa`; rebuilt from sa->string if the array did not come from us
// (e.g. read_suffix_array) -- the result is the same array by uniqueness.
b200sa_index *index_of(struct suffix_array *sa, uint32_t sigma, bool exact_sigma = false) {
    b200sa_index *idx = lookup(sa);
    if (idx && exact_sigma) {
        // e.g. qsort_sa_construction(remapped) built with sigma 256, tables want the remapped sigma
        struct b200sa_stats st;
        b200sa_stats(idx, &st);
        if (st.sigma != sigma) {
            forget(sa);
            idx = nullptr;
        }
    }
    if (idx) return idx;
    enum b200sa_error err;
    idx = b200sa_build(sa->string, sa->length - 1, sigma, 0, device_id(), nullptr, &err);
    if (!idx) die("b200sa_build");
    remember(sa, idx);
    return idx;
}

uint32_t sigma_guess(const struct suffix_array *sa) {
    // largest code + 1; only used when an index has to be rebuilt without a remap table
    uint32_t mx = 0;
    for (uint32_t i = 0; i + 1 < sa->length; ++i)
        if (sa->string[i] > mx) mx = sa->string[i];
    return mx + 1;
}

// dense O rows in the reference layout (bwt.c:47-65); returns false where its u32 size overflows
bool dense_o(b200sa_index *idx, uint32_t sigma, uint32_t length, uint32_t **table, uint32_t ***rows) {
    uint64_t entries = ((uint64_t)length + 1) * sigma;
    if (entries * 4 > 0xFFFFFFFFull) {
        *table = nullptr;
        *rows = nullptr;
        return false;
    }
    *table = (uint32_t *)malloc(entries * sizeof(uint32_t));
    *rows = (uint32_t **)malloc(((size_t)length + 1) * sizeof(uint32_t *));
    if (b200sa_copy_o_dense(idx, *table)) die("b200sa_copy_o_dense");
    for (uint64_t i = 0; i <= length; ++i) (*rows)[i] = *table + i * sigma;
    return true;
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------
// remap.c (host side, tiny): letters present get codes 1..sigma-1 in byte order, 0 = sentinel
// ------------------------------------------------------------------------------------------------
void init_remap_table(struct remap_table *t, const uint8_t *string) {
    bool present[256] = {false};
    for (const uint8_t *p = string; *p; ++p) present[*p] = true;
    memset(t->table, -1, sizeof t->table);
    memset(t->rev_table, -1, sizeof t->rev_table);
    t->table[0] = 0;
    t->rev_table[0] = 0;
    uint32_t next = 1;
    for (int c = 1; c < 256; ++c) {
        if (!present[c]) continue;
        t->table[c] = (signed char)next;
        if (next < 128) t->rev_table[next] = (signed char)c;
        ++next;
    }
    t->alphabet_size = next;
}

struct remap_table *alloc_remap_table(const uint8_t *string) {
    struct remap_table *t = (struct remap_table *)malloc(sizeof *t);
    init_remap_table(t, string);
    return t;
}

void dealloc_remap_table(struct remap_table *) {}
void free_remap_table(struct remap_table *t) { free(t); }

static uint8_t *map_range(uint8_t *out, const uint8_t *from, const uint8_t *to, const signed char *tab) {
    for (const uint8_t *p = from; p != to; ++p, ++out) {
        signed char code = tab[*p];
        *out = (uint8_t)code;
        if (code < 0) return nullptr;  // letter without a code (remap.c:80-84)
    }
    return out;
}

uint8_t *remap_between(uint8_t *output, const uint8_t *from, const uint8_t *to, struct remap_table *t) {
    return map_range(output, from, to, t->table);
}
uint8_t *rev_remap_between(uint8_t *output, const uint8_t *from, const uint8_t *to, struct remap_table *t) {
    // codes >= 128 cannot index the 128-entry reverse table
    for (const uint8_t *p = from; p != to; ++p)
        if (*p >= 128) return nullptr;
    return map_range(output, from, to, t->rev_table);
}
uint8_t *remap_between0(uint8_t *output, const uint8_t *from, const uint8_t *to, struct remap_table *t) {
    uint8_t *end = remap_between(output, from, to, t);
    if (!end) return nullptr;
    *end = 0;
    return end + 1;
}
uint8_t *rev_remap_between0(uint8_t *output, const uint8_t *from, const uint8_t *to, struct remap_table *t) {
    uint8_t *end = rev_remap_between(output, from, to, t);
    if (!end) return nullptr;
    *end = 0;
    return end + 1;
}
uint8_t *remap(uint8_t *output, const uint8_t *input, struct remap_table *t) {
    // the terminating NUL is mapped too (0 -> 0), so the output is sentinel-terminated (remap.c:102-114)
    return remap_between(output, input, input + strlen((const char *)input) + 1, t);
}
uint8_t *rev_remap(uint8_t *output, const uint8_t *input, struct remap_table *t) {
    return rev_remap_between(output, input, input + strlen((const char *)input) + 1, t);
}
uint32_t remap_string(uint8_t *output, uint8_t *input) {
    struct remap_table t;
    init_remap_table(&t, input);
    remap(output, input, &t);
    return t.alphabet_size;
}
bool identical_remap_tables(const struct remap_table *a, const struct remap_table *b) {
    if (a->alphabet_size != b->alphabet_size) return false;
    return memcmp(a->table, b->table, a->alphabet_size) == 0;  // same prefix the reference compares
}

// ------------------------------------------------------------------------------------------------
// suffix arrays
// ------------------------------------------------------------------------------------------------
struct suffix_array *qsort_sa_construction(uint8_t *string) { return construct(string, 256, "qsort_sa_construction"); }
struct suffix_array *skew_sa_construction(uint8_t *string) { return construct(string, 256, "skew_sa_construction"); }
struct suffix_array *sa_is_construction(uint8_t *s, uint32_t sigma) { return construct(s, sigma, "sa_is_construction"); }
struct suffix_array *sa_is_mem_construction(uint8_t *s, uint32_t sigma) {
    return construct(s, sigma, "sa_is_mem_construction");
}

void free_suffix_array(struct suffix_array *sa) {
    forget(sa);
    free(sa->array);
    free(sa->inverse);
    free(sa->lcp);
    free(sa);
}
void free_complete_suffix_array(struct suffix_array *sa) {
    free(sa->string);
    free_suffix_array(sa);
}

void compute_inverse(struct suffix_array *sa) {
    if (sa->inverse) return;  // idempotent like suffix_array.c:57
    b200sa_index *idx = index_of(sa, sigma_guess(sa));
    if (b200sa_extend(idx, sa->string, B200SA_BUILD_ISA)) die("compute_inverse");
    sa->inverse = (uint32_t *)malloc((size_t)sa->length * sizeof(uint32_t));
    if (b200sa_copy_isa(idx, sa->inverse)) die("compute_inverse");
}

void compute_lcp(struct suffix_array *sa) {
    if (sa->lcp) return;  // suffix_array.c:66
    compute_inverse(sa);  // the reference fills both (suffix_array.c:70)
    b200sa_index *idx = index_of(sa, sigma_guess(sa));
    if (b200sa_extend(idx, sa->string, B200SA_BUILD_LCP)) die("compute_lcp");
    sa->lcp = (uint32_t *)malloc((size_t)sa->length * sizeof(uint32_t));
    if (b200sa_copy_lcp(idx, sa->lcp)) die("compute_lcp");
}

bool identical_suffix_arrays(const struct suffix_array *a, const struct suffix_array *b) {
    if (a->length != b->length) return false;
    if (strcmp((const char *)a->string, (const char *)b->string) != 0) return false;
    if (memcmp(a->array, b->array, (size_t)a->length * sizeof(uint32_t)) != 0) return false;
    return strlen((const char *)a->string) + 1 == a->length;
}

// ---- binary searches over the host copy (suffix_array.c:90-233); return values are pinned by
// ---- tests/stralg/suffix_array_test.c:33-126 and reproduced in tests/test_compat.py
uint32_t lower_bound_search(struct suffix_array *sa, const uint8_t *key) {
    const size_t klen = strlen((const char *)key);
    uint32_t lo = 0, hi = sa->length;
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (strncmp((const char *)key, (const char *)sa->string + sa->array[mid], klen) > 0) lo = mid + 1;
        else hi = mid;
    }
    return lo <= hi ? lo : hi;
}

uint32_t upper_bound_search(struct suffix_array *sa, const uint8_t *key) {
    const size_t klen = strlen((const char *)key);
    uint32_t lo = 0, hi = sa->length;
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (strncmp((const char *)key, (const char *)sa->string + sa->array[mid], klen) < 0) hi = mid - 1;
        else lo = mid + 1;
    }
    uint32_t r = hi > lo ? hi : lo;
    if (r == sa->length) return r;
    return strncmp((const char *)key, (const char *)sa->string + sa->array[r], klen) >= 0 ? r + 1 : r;
}

uint32_t lower_bound_k(struct suffix_array *sa, uint32_t k, uint8_t a, uint32_t L, uint32_t R) {
    while (L < R) {
        uint32_t mid = L + (R - L) / 2;
        uint32_t at = sa->array[mid] + k;
        // a suffix that ends before offset k is smaller than any letter
        if (at >= sa->length || sa->string[at] < a) L = mid + 1;
        else R = mid;
    }
    return L <= R ? L : R;
}

uint32_t upper_bound_k(struct suffix_array *sa, uint32_t k, uint8_t a, uint32_t L, uint32_t R) {
    const uint32_t end = R;
    while (L < R) {
        uint32_t mid = L + (R - L) / 2;
        uint32_t at = sa->array[mid] + k;
        if (at >= sa->length) L = mid + 1;
        else if (a < sa->string[at]) R = mid - 1;
        else L = mid + 1;
    }
    uint32_t r = R > L ? R : L;
    if (r == end) return r;
    return a >= sa->string[sa->array[r] + k] ? r + 1 : r;
}

void init_sa_match_iter(struct sa_match_iter *iter, const uint8_t *pattern, struct suffix_array *sa) {
    iter->sa = sa;
    const uint32_t m = (uint32_t)strlen((const char *)pattern);
    uint32_t L = 0, R = sa->length;
    for (uint32_t i = 0; i < m && L < R; ++i) {
        L = lower_bound_k(sa, i, pattern[i], L, R);
        R = upper_bound_k(sa, i, pattern[i], L, R);
    }
    // closed interval [L, R-1] as in suffix_array.c:216-218 (an empty one has R - 1 < L)
    iter->L = L;
    iter->R = R - 1;
    iter->i = L;
}
bool next_sa_match(struct sa_match_iter *iter, struct sa_match *match) {
    if (iter->i > iter->R) return false;
    match->position = iter->sa->array[iter->i++];
    return true;
}
void dealloc_sa_match_iter(struct sa_match_iter *) {}

// ------------------------------------------------------------------------------------------------
// BWT tables
// ------------------------------------------------------------------------------------------------
void init_bwt_table(struct bwt_table *tbl, struct suffix_array *sa, struct suffix_array *rsa,
                    struct remap_table *remap_table) {
    const uint32_t sigma = remap_table->alphabet_size;
    tbl->remap_table = remap_table;
    tbl->sa = sa;
    ++g_trace.tables;
    b200sa_index *idx = index_of(sa, sigma, true);
    if (b200sa_extend(idx, sa->string, B200SA_BUILD_OCC)) die("init_bwt_table");
    tbl->c_table = (uint32_t *)calloc(sigma, sizeof(uint32_t));
    if (b200sa_copy_c_table(idx, tbl->c_table)) die("init_bwt_table");
    dense_o(idx, sigma, sa->length, &tbl->o_table, &tbl->o_indices);
    tbl->ro_table = nullptr;
    tbl->ro_indices = nullptr;
    if (rsa) {  // O table of the reversed text (bwt.c:67-84); only the approximate search reads it
        b200sa_index *ridx = index_of(rsa, sigma, true);
        if (b200sa_extend(ridx, rsa->string, B200SA_BUILD_OCC)) die("init_bwt_table(rsa)");
        dense_o(ridx, sigma, rsa->length, &tbl->ro_table, &tbl->ro_indices);
    }
}

struct bwt_table *alloc_bwt_table(struct suffix_array *sa, struct suffix_array *rsa, struct remap_table *rt) {
    struct bwt_table *tbl = (struct bwt_table *)malloc(sizeof *tbl);
    init_bwt_table(tbl, sa, rsa, rt);
    return tbl;
}

void dealloc_bwt_table(struct bwt_table *tbl) {
    free(tbl->c_table);
    free(tbl->o_table);
    free(tbl->o_indices);
    free(tbl->ro_table);
    free(tbl->ro_indices);
}
void free_bwt_table(struct bwt_table *tbl) {
    dealloc_bwt_table(tbl);
    free(tbl);
}
void completely_dealloc_bwt_table(struct bwt_table *tbl) {
    free_complete_suffix_array(tbl->sa);
    free_remap_table(tbl->remap_table);
    dealloc_bwt_table(tbl);
}
void completely_free_bwt_table(struct bwt_table *tbl) {
    completely_dealloc_bwt_table(tbl);
    free(tbl);
}

struct bwt_table *build_complete_table(const uint8_t *string, bool include_reverse) {
    const size_t n = strlen((const char *)string);
    struct remap_table *rt = alloc_remap_table(string);
    uint8_t *codes = (uint8_t *)malloc(n + 1);
    remap(codes, string, rt);
    struct suffix_array *sa = sa_is_construction(codes, rt->alphabet_size);
    struct suffix_array *rsa = nullptr;
    if (include_reverse) {
        uint8_t *rev = (uint8_t *)malloc(n + 1);
        for (size_t i = 0; i < n; ++i) rev[i] = codes[n - 1 - i];
        rev[n] = 0;
        rsa = sa_is_construction(rev, rt->alphabet_size);
    }
    struct bwt_table *tbl = alloc_bwt_table(sa, rsa, rt);
    if (rsa) free_complete_suffix_array(rsa);  // bwt.c:156-158
    return tbl;
}

bool equivalent_bwt_tables(struct bwt_table *t1, struct bwt_table *t2) {
    if (!identical_remap_tables(t1->remap_table, t2->remap_table)) return false;
    if (!identical_suffix_arrays(t1->sa, t2->sa)) return false;
    const uint32_t sigma = t1->remap_table->alphabet_size;
    if (memcmp(t1->c_table, t2->c_table, (size_t)sigma * 4) != 0) return false;
    const size_t o_entries = (size_t)sigma * t1->sa->length;  // the reference compares this many (bwt.c:579)
    if (!t1->o_table != !t2->o_table) return false;
    if (t1->o_table && memcmp(t1->o_table, t2->o_table, o_entries * 4) != 0) return false;
    if (!t1->ro_table != !t2->ro_table) return false;
    if (t1->ro_table && memcmp(t1->ro_table, t2->ro_table, o_entries * 4) != 0) return false;
    return true;
}

// ------------------------------------------------------------------------------------------------
// exact search (bwt.c:164-217): the backward search runs on the GPU, positions come from sa->array
// ------------------------------------------------------------------------------------------------
void bwt_exact_match_batch(struct bwt_table *tbl, const uint8_t *patterns, const uint64_t *offsets,
                           uint64_t npatterns, uint32_t *L, uint32_t *R) {
    b200sa_index *idx = index_of(tbl->sa, tbl->remap_table->alphabet_size, true);
    // (first search on this table: also the k-mer seed table and the text-comparison shortcut -- they cut the
    // chain of dependent lookups of one pattern from its length to about a dozen)
    if (b200sa_extend(idx, tbl->sa->string, B200SA_BUILD_OCC | B200SA_BUILD_TEXTCMP | B200SA_BUILD_KTABLE))
        die("bwt_exact_match_batch");
    if (b200sa_search_batch(idx, patterns, offsets, 0, npatterns, L, R)) die("bwt_exact_match_batch");
}

// the same for reads of one length packed to 2 bits per base (include/b200sa.h: b200sa_search_batch_packed)
void bwt_exact_match_batch_packed(struct bwt_table *tbl, const uint8_t *packed, uint32_t read_len, uint32_t stride_bytes,
                                  uint64_t nreads, uint32_t *L, uint32_t *R) {
    b200sa_index *idx = index_of(tbl->sa, tbl->remap_table->alphabet_size, true);
    if (b200sa_extend(idx, tbl->sa->string, B200SA_BUILD_OCC | B200SA_BUILD_TEXTCMP | B200SA_BUILD_KTABLE))
        die("bwt_exact_match_batch_packed");
    if (b200sa_search_batch_packed(idx, packed, read_len, stride_bytes, nreads, L, R)) die("bwt_exact_match_batch_packed");
}

void init_bwt_exact_match_iter(struct bwt_exact_match_iter *iter, struct bwt_table *tbl,
                               const uint8_t *remapped_pattern) {
    iter->sa = tbl->sa;
    ++g_trace.exact_iters;
    const uint64_t off[2] = {0, (uint64_t)strlen((const char *)remapped_pattern)};
    uint32_t L = 0, R = 0;
    bwt_exact_match_batch(tbl, remapped_pattern, off, 1, &L, &R);
    iter->L = L;
    iter->R = R;
    iter->i = L;
}

// Measurement aid (bench.py `compat`): the loop of performance/suffix_array_search.c:127-141 -- ONE
// iterator per pattern, every match fetched -- over `npat` NUL-terminated remapped patterns laid out
// with a stride of m + 1 bytes.  Returns the number of matches.
uint64_t bwt_exact_match_loop(struct bwt_table *tbl, const uint8_t *patterns, uint32_t m, uint64_t npat) {
    uint64_t hits = 0;
    for (uint64_t q = 0; q < npat; ++q) {
        struct bwt_exact_match_iter it;
        struct bwt_exact_match mt;
        init_bwt_exact_match_iter(&it, tbl, patterns + q * ((uint64_t)m + 1));
        while (next_bwt_exact_match_iter(&it, &mt)) ++hits;
        dealloc_bwt_exact_match_iter(&it);
    }
    return hits;
}

bool next_bwt_exact_match_iter(struct bwt_exact_match_iter *iter, struct bwt_exact_match *match) {
    if (iter->i < 0 || iter->i >= (int64_t)iter->R) return false;
    match->pos = iter->sa->array[iter->i++];
    return true;
}
void dealloc_bwt_exact_match_iter(struct bwt_exact_match_iter *) {}

// ------------------------------------------------------------------------------------------------
// approximate search (bwt.c:226-409): the recursion runs on the GPU for a whole batch of patterns
// ------------------------------------------------------------------------------------------------
namespace {
// D table from the dense RO rows (bwt.c:319-337), one byte per pattern symbol
void host_d_table(const struct bwt_table *tbl, const uint8_t *pat, uint64_t m, uint8_t *out) {
    const uint32_t sigma = tbl->remap_table->alphabet_size, len = tbl->sa->length;
    uint32_t L = 0, R = len, need = 0;
    for (uint64_t i = 0; i < m; ++i) {
        const uint8_t a = pat[i];
        if (a == 0 || a >= sigma) {
            L = 1;
            R = 0;
        } else {
            L = tbl->c_table[a] + tbl->ro_indices[L][a];
            R = tbl->c_table[a] + tbl->ro_indices[R][a];
        }
        if (L >= R) {
            ++need;
            L = 0;
            R = len;
        }
        out[i] = (uint8_t)(need > 255 ? 255 : need);
    }
}

b200sa_approx_result *approx_batch(struct bwt_table *tbl, const uint8_t *patterns, const uint64_t *offsets,
                                   uint64_t npatterns, int edits, const char *who) {
    b200sa_index *idx = index_of(tbl->sa, tbl->remap_table->alphabet_size, true);
    if (b200sa_extend(idx, tbl->sa->string, B200SA_BUILD_OCC)) die(who);
    std::vector<uint8_t> dt;
    if (tbl->ro_indices) {
        dt.resize(offsets[npatterns] + 1);
        for (uint64_t q = 0; q < npatterns; ++q)
            host_d_table(tbl, patterns + offsets[q], offsets[q + 1] - offsets[q], dt.data() + offsets[q]);
    }
    enum b200sa_error err;
    b200sa_approx_result *r = b200sa_approx_batch(idx, nullptr, tbl->ro_indices ? dt.data() : nullptr, patterns, offsets,
                                                  0, npatterns, edits, &err);
    if (!r) die(who);
    return r;
}
}  // namespace

void init_bwt_approx_iter(struct bwt_approx_iter *iter, struct bwt_table *tbl, const uint8_t *remapped_pattern,
                          int edits) {
    const uint64_t m = strlen((const char *)remapped_pattern);
    const uint64_t off[2] = {0, m};
    ++g_trace.approx_iters;
    b200sa_approx_result *r = approx_batch(tbl, remapped_pattern, off, 1, edits < 0 ? 0 : edits, "init_bwt_approx_iter");
    const uint64_t k = edits < 0 ? 0 : b200sa_approx_hits(r);
    iter->bwt_table = tbl;
    iter->remapped_pattern = remapped_pattern;
    iter->m = (uint32_t)m;
    iter->edits_buf = nullptr;
    iter->D_table = nullptr;
    struct index_vector *vecs[3] = {&iter->Ls, &iter->Rs, &iter->match_lengths};
    const uint32_t *src[3] = {b200sa_approx_L(r), b200sa_approx_R(r), b200sa_approx_match_length(r)};
    for (int v = 0; v < 3; ++v) {
        vecs[v]->data = (uint32_t *)malloc((k ? k : 1) * sizeof(uint32_t));
        vecs[v]->size = (uint32_t)(k ? k : 1);
        vecs[v]->used = (uint32_t)k;
        if (k) memcpy(vecs[v]->data, src[v], k * sizeof(uint32_t));
    }
    iter->cigars.data = (uint8_t **)malloc((k ? k : 1) * sizeof(uint8_t *));
    iter->cigars.size = (uint32_t)(k ? k : 1);
    iter->cigars.used = (uint32_t)k;
    const uint64_t *coff = b200sa_approx_cigar_offsets(r);
    const char *cig = b200sa_approx_cigars(r);
    for (uint64_t h = 0; h < k; ++h) iter->cigars.data[h] = (uint8_t *)strdup(cig + coff[h]);
    b200sa_approx_free(r);
    iter->L = (uint32_t)m;  // bwt.c:379-381: start before the first interval
    iter->R = 0;
    iter->next_interval = 0;
}

bool next_bwt_approx_match(struct bwt_approx_iter *iter, struct bwt_approx_match *match) {
    if (iter->L >= iter->R) {
        if (iter->next_interval >= iter->Ls.used) return false;
        iter->L = iter->Ls.data[iter->next_interval];
        iter->R = iter->Rs.data[iter->next_interval];
        iter->next_interval++;
    }
    match->cigar = (const char *)iter->cigars.data[iter->next_interval - 1];
    match->match_length = iter->match_lengths.data[iter->next_interval - 1];
    match->position = iter->bwt_table->sa->array[iter->L++];
    return true;
}

void dealloc_bwt_approx_iter(struct bwt_approx_iter *iter) {
    free(iter->Ls.data);
    free(iter->Rs.data);
    free(iter->match_lengths.data);
    for (uint32_t h = 0; h < iter->cigars.used; ++h) free(iter->cigars.data[h]);
    free(iter->cigars.data);
    free(iter->edits_buf);
    free(iter->D_table);
}

// ------------------------------------------------------------------------------------------------
// Index files: the reference's raw layouts (no header, host endianness).  Host-side I/O only; a
// structure read from a file has no device index yet -- index_of() rebuilds it from the string
// the first time the GPU is needed, which yields the same arrays by uniqueness.
// ------------------------------------------------------------------------------------------------
static void must(bool ok, const char *what) {
    if (!ok) {
        fprintf(stderr, "stralg_b200: %s\n", what);
        abort();
    }
}
static FILE *open_or_die(const char *fname, const char *mode) {
    FILE *f = fopen(fname, mode);
    if (!f) {
        fprintf(stderr, "stralg_b200: cannot open %s\n", fname);
        abort();
    }
    return f;
}

void write_suffix_array(FILE *f, const struct suffix_array *sa) {  // suffix_array.c:238-241: length u32 entries
    must(fwrite(sa->array, sizeof(uint32_t), sa->length, f) == sa->length, "write_suffix_array: short write");
}
void write_suffix_array_fname(const char *fname, const struct suffix_array *sa) {
    FILE *f = open_or_die(fname, "wb");
    write_suffix_array(f, sa);
    fclose(f);
}
struct suffix_array *read_suffix_array(FILE *f, uint8_t *string) {  // suffix_array.c:250-257
    struct suffix_array *sa = (struct suffix_array *)malloc(sizeof *sa);
    sa->string = string;
    sa->length = (uint32_t)strlen((const char *)string) + 1;
    sa->array = (uint32_t *)malloc((size_t)sa->length * sizeof(uint32_t));
    sa->inverse = nullptr;
    sa->lcp = nullptr;
    must(fread(sa->array, sizeof(uint32_t), sa->length, f) == sa->length, "read_suffix_array: short read");
    return sa;
}
struct suffix_array *read_suffix_array_fname(const char *fname, uint8_t *string) {
    FILE *f = open_or_die(fname, "rb");
    struct suffix_array *sa = read_suffix_array(f, string);
    fclose(f);
    return sa;
}

void write_remap_table(FILE *f, const struct remap_table *t) {  // remap.c:168-173: the raw struct
    must(fwrite(t, sizeof(struct remap_table), 1, f) == 1, "write_remap_table: short write");
}
void write_remap_table_fname(const char *fname, const struct remap_table *t) {
    FILE *f = open_or_die(fname, "wb");
    write_remap_table(f, t);
    fclose(f);
}
struct remap_table *read_remap_table(FILE *f) {
    struct remap_table *t = (struct remap_table *)malloc(sizeof *t);
    must(fread(t, sizeof(struct remap_table), 1, f) == 1, "read_remap_table: short read");
    return t;
}
struct remap_table *read_remap_table_fname(const char *fname) {
    FILE *f = open_or_die(fname, "rb");
    struct remap_table *t = read_remap_table(f);
    fclose(f);
    return t;
}

// bwt.c:425-440: C[sigma], O[sigma * (length + 1)], bool has_ro, RO[...] when present
void write_bwt_table(FILE *f, const struct bwt_table *tbl) {
    const uint32_t sigma = tbl->remap_table->alphabet_size;
    const uint64_t o_entries = (uint64_t)sigma * ((uint64_t)tbl->sa->length + 1);
    must(tbl->o_table != nullptr && o_entries <= 0xFFFFFFFFull,
         "write_bwt_table: the dense O table of this text does not fit the reference's format (bwt.c:430)");
    must(fwrite(tbl->c_table, sizeof(uint32_t), sigma, f) == sigma, "write_bwt_table: short write");
    must(fwrite(tbl->o_table, sizeof(uint32_t), o_entries, f) == o_entries, "write_bwt_table: short write");
    const bool has_ro = tbl->ro_table != nullptr;
    must(fwrite(&has_ro, sizeof(bool), 1, f) == 1, "write_bwt_table: short write");
    if (has_ro) must(fwrite(tbl->ro_table, sizeof(uint32_t), o_entries, f) == o_entries, "write_bwt_table: short write");
}
void write_bwt_table_fname(const char *fname, const struct bwt_table *tbl) {
    FILE *f = open_or_die(fname, "wb");
    write_bwt_table(f, tbl);
    fclose(f);
}
static void read_dense(FILE *f, uint32_t sigma, uint32_t length, uint32_t **table, uint32_t ***rows) {
    const uint64_t o_entries = (uint64_t)sigma * ((uint64_t)length + 1);
    *table = (uint32_t *)malloc(o_entries * sizeof(uint32_t));
    must(fread(*table, sizeof(uint32_t), o_entries, f) == o_entries, "read_bwt_table: short read");
    *rows = (uint32_t **)malloc(((size_t)length + 1) * sizeof(uint32_t *));
    for (uint64_t i = 0; i <= length; ++i) (*rows)[i] = *table + i * sigma;
}
struct bwt_table *read_bwt_table(FILE *f, struct suffix_array *sa, struct remap_table *remap_table) {  // bwt.c:451-492
    struct bwt_table *tbl = (struct bwt_table *)malloc(sizeof *tbl);
    const uint32_t sigma = remap_table->alphabet_size;
    tbl->remap_table = remap_table;
    tbl->sa = sa;
    tbl->c_table = (uint32_t *)malloc((size_t)sigma * sizeof(uint32_t));
    must(fread(tbl->c_table, sizeof(uint32_t), sigma, f) == sigma, "read_bwt_table: short read");
    read_dense(f, sigma, sa->length, &tbl->o_table, &tbl->o_indices);
    tbl->ro_table = nullptr;
    tbl->ro_indices = nullptr;
    bool has_ro = false;
    must(fread(&has_ro, sizeof(bool), 1, f) == 1, "read_bwt_table: short read");
    if (has_ro) read_dense(f, sigma, sa->length, &tbl->ro_table, &tbl->ro_indices);
    return tbl;
}
struct bwt_table *read_bwt_table_fname(const char *fname, struct suffix_array *sa, struct remap_table *remap_table) {
    FILE *f = open_or_die(fname, "rb");
    struct bwt_table *tbl = read_bwt_table(f, sa, remap_table);
    fclose(f);
    return tbl;
}

// serialise.c:7-18: [u32 n][n bytes of the remapped string] SA remap_table bwt_table
void write_complete_bwt_info(FILE *f, const struct bwt_table *tbl) {
    const struct suffix_array *sa = tbl->sa;
    const uint32_t n = sa->length - 1;  // string_utils.c:48-52 (write_string_len)
    must(fwrite(&n, sizeof n, 1, f) == 1 && fwrite(sa->string, 1, n, f) == n, "write_complete_bwt_info: short write");
    write_suffix_array(f, sa);
    write_remap_table(f, tbl->remap_table);
    write_bwt_table(f, tbl);
}
void write_complete_bwt_info_fname(const char *fname, const struct bwt_table *tbl) {
    FILE *f = open_or_die(fname, "wb");
    write_complete_bwt_info(f, tbl);
    fclose(f);
}
struct bwt_table *read_complete_bwt_info(FILE *f) {  // serialise.c:29-41; the table owns everything it read
    uint32_t n = 0;
    must(fread(&n, sizeof n, 1, f) == 1, "read_complete_bwt_info: short read");
    uint8_t *str = (uint8_t *)malloc((size_t)n + 1);  // string_utils.c:73-82 (read_string_len)
    must(fread(str, 1, n, f) == n, "read_complete_bwt_info: short read");
    str[n] = 0;
    struct suffix_array *sa = read_suffix_array(f, str);
    struct remap_table *rt = read_remap_table(f);
    return read_bwt_table(f, sa, rt);
}
struct bwt_table *read_complete_bwt_info_fname(const char *fname) {
    FILE *f = open_or_die(fname, "rb");
    struct bwt_table *tbl = read_complete_bwt_info(f);
    fclose(f);
    return tbl;
}

// ------------------------------------------------------------------------------------------------
// Reads in, SAM out: the loop of bwt_readmapper -d 0 with the backward searches batched on the GPU
// ------------------------------------------------------------------------------------------------
namespace {
const int kFastqLine = 2048;  // MAX_STRING_LEN, bioinf/fastq.h:9

// one line without its newline, the way next_fastq_record takes it (fgets + strtok(..., "\n"))
bool fastq_line(FILE *f, char *buf, std::string *out, int skip) {
    if (!fgets(buf, kFastqLine, f)) return false;
    char *p = buf + skip;
    while (*p == '\n') ++p;  // strtok skips leading delimiters
    size_t n = strcspn(p, "\n");
    out->assign(p, n);
    return true;
}
}  // namespace

uint64_t bwt_map_fastq_exact(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                             struct bwt_table *const *tables, uint64_t batch_reads) {
    return bwt_map_fastq(fastq, samfile, nrecords, record_names, tables, 0, batch_reads);
}

uint64_t bwt_map_fastq(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                       struct bwt_table *const *tables, int edits, uint64_t batch_reads) {
    if (batch_reads == 0) batch_reads = edits > 0 ? 1u << 16 : 1u << 20;
    // per record and read: the read's intervals are hits [hit_lo, hit_hi) of that record's result
    std::vector<b200sa_approx_result *> results(nrecords, nullptr);
    std::vector<std::vector<uint64_t>> hit_lo(nrecords), hit_hi(nrecords);
    std::vector<char> line(kFastqLine + 1);
    std::vector<std::string> names, seqs, quals;
    std::vector<uint8_t> pat, packed;
    std::vector<uint64_t> off;
    std::vector<uint32_t> which;
    std::vector<std::vector<uint32_t>> Ls(nrecords), Rs(nrecords);
    uint64_t lines = 0;
    bool more = true;
    while (more) {
        names.clear(); seqs.clear(); quals.clear();
        while (names.size() < batch_reads) {
            std::string name, seq, plus, qual;
            if (!fastq_line(fastq, line.data(), &name, 1)) {  // name: the text after '@'
                more = false;
                break;
            }
            fastq_line(fastq, line.data(), &seq, 0);
            fastq_line(fastq, line.data(), &plus, 0);
            fastq_line(fastq, line.data(), &qual, 0);
            names.push_back(name); seqs.push_back(seq); quals.push_back(qual);
        }
        const size_t nreads = names.size();
        if (!nreads) break;
        // one batched backward search per reference record; (1, 0) marks a read that record skips
        for (uint32_t r = 0; r < nrecords; ++r) {
            struct remap_table *rt = tables[r]->remap_table;
            pat.clear(); off.assign(1, 0); which.clear();
            Ls[r].assign(nreads, 1); Rs[r].assign(nreads, 0);
            for (size_t q = 0; q < nreads; ++q) {
                const std::string &sq = seqs[q];
                if (sq.empty()) continue;
                const size_t at = pat.size();
                pat.resize(at + sq.size());
                bool ok = true;
                for (size_t k = 0; k < sq.size() && ok; ++k) {
                    const signed char c = rt->table[(unsigned char)sq[k]];
                    ok = c > 0;  // remap() returns NULL on a letter without a code (remap.c:80-84)
                    pat[at + k] = (uint8_t)c;
                }
                if (!ok) {
                    pat.resize(at);
                    continue;
                }
                off.push_back(pat.size());
                which.push_back((uint32_t)q);
            }
            if (which.empty()) continue;
            if (edits > 0) {
                results[r] = approx_batch(tables[r], pat.data(), off.data(), which.size(), edits, "bwt_map_fastq");
                const uint64_t *ho = b200sa_approx_hit_offsets(results[r]);
                hit_lo[r].assign(nreads, 0);
                hit_hi[r].assign(nreads, 0);
                for (size_t k = 0; k < which.size(); ++k) {
                    hit_lo[r][which[k]] = ho[k];
                    hit_hi[r][which[k]] = ho[k + 1];
                }
                continue;
            }
            std::vector<uint32_t> L(which.size()), R(which.size());
            // reads of one length over a DNA alphabet (the usual FASTQ): packed to 2 bits per base right after
            // the remap -- a quarter of the bytes cross PCIe (b200sa_search_batch_packed, same intervals)
            bool one_len = rt->alphabet_size <= 5;
            const uint64_t m0 = off[1] - off[0];
            for (size_t k = 1; k < which.size() && one_len; ++k) one_len = off[k + 1] - off[k] == m0;
            if (one_len && m0 > 0 && m0 < (1ull << 31)) {
                const uint32_t stride = (uint32_t)((m0 + 3) / 4);
                packed.assign((size_t)stride * which.size() + 8, 0);
                if (b200sa_pack_reads(pat.data(), (uint32_t)m0, stride, which.size(), packed.data())) die("bwt_map_fastq");
                bwt_exact_match_batch_packed(tables[r], packed.data(), (uint32_t)m0, stride, which.size(), L.data(), R.data());
            } else {
                bwt_exact_match_batch(tables[r], pat.data(), off.data(), which.size(), L.data(), R.data());
            }
            for (size_t k = 0; k < which.size(); ++k) {
                Ls[r][which[k]] = L[k];
                Rs[r][which[k]] = R[k];
            }
        }
        // SAM lines in the reference's order: reads, then records, then suffix-array order
        for (size_t q = 0; q < nreads; ++q)
            for (uint32_t r = 0; r < nrecords; ++r) {
                const uint32_t *sa = tables[r]->sa->array;
                if (edits > 0) {
                    if (!results[r]) continue;
                    const uint32_t *aL = b200sa_approx_L(results[r]), *aR = b200sa_approx_R(results[r]);
                    const uint64_t *coff = b200sa_approx_cigar_offsets(results[r]);
                    const char *cig = b200sa_approx_cigars(results[r]);
                    for (uint64_t h = hit_lo[r][q]; h < hit_hi[r][q]; ++h)
                        for (uint32_t i = aL[h]; i < aR[h]; ++i) {
                            fprintf(samfile, "%s\t0\t%s\t%u\t0\t%s\t*\t0\t0\t%s\t%s\n", names[q].c_str(),
                                    record_names[r], sa[i] + 1, cig + coff[h], seqs[q].c_str(), quals[q].c_str());
                            ++lines;
                        }
                    continue;
                }
                for (uint32_t i = Ls[r][q]; i < Rs[r][q]; ++i) {
                    fprintf(samfile, "%s\t0\t%s\t%u\t0\t%zuM\t*\t0\t0\t%s\t%s\n", names[q].c_str(), record_names[r],
                            sa[i] + 1, seqs[q].size(), seqs[q].c_str(), quals[q].c_str());
                    ++lines;
                }
            }
        for (uint32_t r = 0; r < nrecords; ++r) {
            b200sa_approx_free(results[r]);
            results[r] = nullptr;
        }
    }
    return lines;
}

// The same mapping against ONE records index (include/b200sa.h: b200sa_build_records) built from all the tables'
// strings: one search or approximate-search call and one b200sa_locate_records call per batch, whatever the number
// of records.  A read is remapped once, with the union alphabet; the tool's rule that a read with a letter missing
// from record r's own alphabet produces no line for r is applied per (read, record) through letter masks -- with
// edits, a substitution could otherwise align such a read to r.
uint64_t bwt_map_fastq_records(FILE *fastq, FILE *samfile, uint32_t nrecords, const char *const *record_names,
                               struct bwt_table *const *tables, int edits, uint64_t batch_reads) {
    if (batch_reads == 0) batch_reads = edits > 0 ? 1u << 16 : 1u << 20;
    // The records as bytes (rev_table of each table).  A record's letters are the letters its remap table codes, as
    // bwt_map_fastq remaps a read with that table: mask[r] is that set (it may hold letters the string lacks, when the
    // table was made for a wider alphabet), and the union table gives codes 2..sigma-1 to the letters of all tables.
    std::vector<std::vector<uint8_t>> raw(nrecords);
    std::vector<std::vector<bool>> mask(nrecords, std::vector<bool>(256, false));
    bool present[256] = {false};
    bool all_ro = true;
    for (uint32_t r = 0; r < nrecords; ++r) {
        const struct suffix_array *sa = tables[r]->sa;
        const struct remap_table *rt = tables[r]->remap_table;
        all_ro = all_ro && tables[r]->ro_table != nullptr;
        for (int b = 1; b < 256; ++b)
            if (rt->table[b] > 0) mask[r][b] = present[b] = true;
        raw[r].resize(sa->length - 1);
        for (uint32_t i = 0; i + 1 < sa->length; ++i) {
            const uint8_t c = sa->string[i];
            const int b = c < 128 ? rt->rev_table[c] : -1;
            if (b <= 0 || !mask[r][b]) {
                fprintf(stderr, "stralg_b200: bwt_map_fastq_records: record %u holds a code without a letter\n", r);
                abort();
            }
            raw[r][i] = (uint8_t)b;
        }
    }
    int16_t code[256];
    uint32_t sigma = 2;
    for (int b = 0; b < 256; ++b) code[b] = b > 0 && present[b] ? (int16_t)sigma++ : (int16_t)-1;
    if (sigma == 2) {  // no record has a letter (or there is no record): no read maps, as with bwt_map_fastq
        std::vector<char> line(kFastqLine + 1);
        while (fgets(line.data(), kFastqLine, fastq)) {
        }
        return 0;
    }
    if (sigma > 256) {
        fprintf(stderr, "stralg_b200: bwt_map_fastq_records: more than 254 letters\n");
        abort();
    }
    std::vector<uint64_t> rec_off(nrecords + 1, 0);
    for (uint32_t r = 0; r < nrecords; ++r) rec_off[r + 1] = rec_off[r] + raw[r].size();
    std::vector<uint8_t> codes(rec_off[nrecords]);
    for (uint32_t r = 0; r < nrecords; ++r)
        for (size_t i = 0; i < raw[r].size(); ++i) codes[rec_off[r] + i] = (uint8_t)code[raw[r][i]];
    raw.clear();
    enum b200sa_error err;
    const uint32_t flags = edits > 0 ? B200SA_BUILD_OCC : B200SA_BUILD_OCC | B200SA_BUILD_TEXTCMP | B200SA_BUILD_KTABLE;
    b200sa_index *idx = b200sa_build_records(codes.data(), rec_off.data(), nrecords, sigma, flags, device_id(), nullptr, &err);
    if (!idx) die("bwt_map_fastq_records");
    // the tool's D table comes from the tables' reverse O rows; here from an index of the reversed text, separators
    // included: it bounds every record's D table from below, so it prunes less and changes no result
    b200sa_index *rev = nullptr;
    if (edits > 0 && all_ro) {
        const uint64_t n = rec_off[nrecords] + nrecords;
        std::vector<uint8_t> text(n);
        for (uint32_t r = 0; r < nrecords; ++r) {
            std::copy(codes.begin() + rec_off[r], codes.begin() + rec_off[r + 1], text.begin() + rec_off[r] + r);
            text[rec_off[r + 1] + r] = 1;
        }
        std::reverse(text.begin(), text.end());
        rev = b200sa_build(text.data(), n, sigma, B200SA_BUILD_OCC, device_id(), nullptr, &err);
        if (!rev) die("bwt_map_fastq_records");
    }
    codes.clear();
    codes.shrink_to_fit();

    std::vector<char> line(kFastqLine + 1);
    std::vector<std::string> names, seqs, quals;
    std::vector<uint8_t> pat;
    std::vector<uint64_t> off, hit_off, pos_off;
    std::vector<uint32_t> which, L, R, rec, pos;
    std::vector<std::string> cigars;
    std::vector<uint64_t> order;
    uint64_t lines = 0;
    bool more = true;
    while (more) {
        names.clear(); seqs.clear(); quals.clear();
        while (names.size() < batch_reads) {
            std::string name, seq, plus, qual;
            if (!fastq_line(fastq, line.data(), &name, 1)) {
                more = false;
                break;
            }
            fastq_line(fastq, line.data(), &seq, 0);
            fastq_line(fastq, line.data(), &plus, 0);
            fastq_line(fastq, line.data(), &qual, 0);
            names.push_back(name); seqs.push_back(seq); quals.push_back(qual);
        }
        const size_t nreads = names.size();
        if (!nreads) break;
        // every read once through the union table; a letter that no record holds skips the read for all of them
        pat.clear(); off.assign(1, 0); which.clear();
        for (size_t q = 0; q < nreads; ++q) {
            const std::string &sq = seqs[q];
            if (sq.empty()) continue;
            const size_t at = pat.size();
            pat.resize(at + sq.size());
            bool ok = true;
            for (size_t k = 0; k < sq.size() && ok; ++k) {
                const int16_t c = code[(unsigned char)sq[k]];
                ok = c > 0;
                pat[at + k] = (uint8_t)c;
            }
            if (!ok) {
                pat.resize(at);
                continue;
            }
            off.push_back(pat.size());
            which.push_back((uint32_t)q);
        }
        const size_t nvalid = which.size();
        // hits of read which[k]: [hit_off[k], hit_off[k + 1]), each an interval with its CIGAR
        L.clear(); R.clear(); cigars.clear();
        hit_off.assign(nvalid + 1, 0);
        if (nvalid && edits > 0) {
            b200sa_approx_result *res = b200sa_approx_batch(idx, rev, nullptr, pat.data(), off.data(), 0, nvalid, edits, &err);
            if (!res) die("bwt_map_fastq_records");
            const uint64_t nh = b200sa_approx_hits(res);
            const uint64_t *ho = b200sa_approx_hit_offsets(res), *coff = b200sa_approx_cigar_offsets(res);
            const char *cig = b200sa_approx_cigars(res);
            L.assign(b200sa_approx_L(res), b200sa_approx_L(res) + nh);
            R.assign(b200sa_approx_R(res), b200sa_approx_R(res) + nh);
            hit_off.assign(ho, ho + nvalid + 1);
            cigars.resize(nh);
            for (uint64_t h = 0; h < nh; ++h) cigars[h] = cig + coff[h];
            b200sa_approx_free(res);
        } else if (nvalid) {
            L.resize(nvalid);
            R.resize(nvalid);
            if (b200sa_search_batch(idx, pat.data(), off.data(), 0, nvalid, L.data(), R.data())) die("bwt_map_fastq_records");
            for (size_t k = 0; k <= nvalid; ++k) hit_off[k] = k;
        }
        // (record, local position) of every interval: records ascending, each record's suffix-array order
        const uint64_t nh = L.size();
        pos_off.assign(nh + 1, 0);
        uint64_t total = 0;
        if (b200sa_locate_records(idx, L.data(), R.data(), nh, pos_off.data(), nullptr, nullptr, 0, &total))
            die("bwt_map_fastq_records");
        rec.resize(total);
        pos.resize(total);
        if (total && b200sa_locate_records(idx, L.data(), R.data(), nh, pos_off.data(), rec.data(), pos.data(), total, &total))
            die("bwt_map_fastq_records");
        // SAM lines in the tool's order: reads, records, intervals in report order, positions in suffix-array order
        for (size_t k = 0; k < nvalid; ++k) {
            const size_t q = which[k];
            const std::string &sq = seqs[q];
            order.clear();
            for (uint64_t h = hit_off[k]; h < hit_off[k + 1]; ++h)
                for (uint64_t e = pos_off[h]; e < pos_off[h + 1]; ++e) order.push_back(e);
            std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return rec[a] < rec[b]; });
            char exact_cigar[32];
            snprintf(exact_cigar, sizeof exact_cigar, "%zuM", sq.size());
            for (size_t j = 0; j < order.size();) {
                const uint32_t r = rec[order[j]];
                size_t j1 = j;
                while (j1 < order.size() && rec[order[j1]] == r) ++j1;
                bool in_r = true;
                for (size_t c = 0; c < sq.size() && in_r; ++c) in_r = mask[r][(unsigned char)sq[c]];
                for (; in_r && j < j1; ++j) {
                    const uint64_t e = order[j];
                    // the interval of entry e: the last hit of this read whose entries start at or before e
                    const uint64_t h = std::upper_bound(pos_off.begin() + hit_off[k], pos_off.begin() + hit_off[k + 1],
                                                        e) - pos_off.begin() - 1;
                    fprintf(samfile, "%s\t0\t%s\t%u\t0\t%s\t*\t0\t0\t%s\t%s\n", names[q].c_str(), record_names[r],
                            pos[e] + 1, edits > 0 ? cigars[h].c_str() : exact_cigar, sq.c_str(), quals[q].c_str());
                    ++lines;
                }
                j = j1;
            }
        }
    }
    b200sa_free(rev);
    b200sa_free(idx);
    return lines;
}

void write_bwt_tables_file(const char *fname, uint32_t nrecords, const char *const *record_names,
                           struct bwt_table *const *tables) {
    FILE *f = open_or_die(fname, "wb");
    must(fwrite(&nrecords, sizeof nrecords, 1, f) == 1, "write_bwt_tables_file: short write");
    for (uint32_t r = 0; r < nrecords; ++r) {
        const uint32_t len = (uint32_t)strlen(record_names[r]) + 1;  // write_string: the NUL is stored
        must(fwrite(&len, sizeof len, 1, f) == 1 && fwrite(record_names[r], 1, len, f) == len,
             "write_bwt_tables_file: short write");
        write_complete_bwt_info(f, tables[r]);
    }
    fclose(f);
}

uint32_t read_bwt_tables_file(const char *fname, char ***record_names, struct bwt_table ***tables) {
    FILE *f = open_or_die(fname, "rb");
    uint32_t nrecords = 0;
    must(fread(&nrecords, sizeof nrecords, 1, f) == 1, "read_bwt_tables_file: short read");
    *record_names = (char **)malloc((size_t)nrecords * sizeof(char *));
    *tables = (struct bwt_table **)malloc((size_t)nrecords * sizeof(struct bwt_table *));
    for (uint32_t r = 0; r < nrecords; ++r) {
        uint32_t len = 0;
        must(fread(&len, sizeof len, 1, f) == 1, "read_bwt_tables_file: short read");
        char *name = (char *)malloc((size_t)len + 1);
        must(fread(name, 1, len, f) == len, "read_bwt_tables_file: short read");
        name[len] = 0;
        (*record_names)[r] = name;
        (*tables)[r] = read_complete_bwt_info(f);
    }
    fclose(f);
    return nrecords;
}

}  // extern "C"
