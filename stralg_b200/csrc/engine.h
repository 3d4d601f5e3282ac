// engine.h -- internal C++ interface between the C ABI (api.cu) and the kernel files.
#pragma once
#include "common.cuh"

#include <vector>

namespace b200sa {

// Text packing parameters derived from the alphabet size (sentinel included in sigma).
struct Packing {
    int bits;   // bits per packed symbol (1, 2, 4 or 8); packed symbol = code - 1
    int cpw;    // symbols per 64-bit word
};
static inline Packing packing_for_sigma(u32 sigma) {
    u32 nsym = sigma > 1 ? sigma - 1 : 1;  // codes 1..sigma-1
    Packing p;
    p.bits = nsym <= 2 ? 1 : nsym <= 4 ? 2 : nsym <= 16 ? 4 : 8;
    p.cpw = 64 / p.bits;
    return p;
}

struct BuildStats {
    u32 rounds;          // doubling rounds after the initial K-character sort
    u32 k0;              // characters packed into the round-0 key
    u32 radix_bits;
    u32 passes0;         // radix passes in round 0
    u64 sorted_total;    // sum over rounds of elements sorted
    u64 passes_elems;    // sum over all radix passes of elements moved
    u32 round0_mode;     // 0: LSD radix passes, 1: MSD bucket sort (round0_msd.cu)
    u32 bucket_bits;     // MSD: leading key bits that select a bucket
    u32 shallow_buckets; // MSD: oversize buckets emitted unsorted as groups of depth bucket_bits / bits
    u64 shallow_elems;   // suffixes in them
    u64 lazy_lookups;    // ranks of retired suffixes recovered on demand by the doubling rounds
    u32 chain_rounds;    // doubling rounds that used chain offsets (sa_build.cu: chain_flags_kernel)
    u64 chain_elems;     // suffixes whose group "continued", summed over those rounds
    u32 resolved_small;  // suffixes in groups of 2..4 equal keys that the next 64 bits of text decided after round 0
    u64 small_path_elems; // list elements ordered inside their tile (groups of up to 32), summed over rounds
    u32 pivot_rounds;     // doubling rounds that split their groups around a pivot key (sa_build.cu: pivot path)
    u64 pivot_elems;      // list elements that stayed with the pivot key and skipped the sort, summed over rounds
    u32 pair_placed;      // suffixes in groups of two that one text comparison per repeat decided after round 0
    u32 dense_keys;       // bucketed round 0 formed dense keys (round0_msd.cuh DenseKey): the number of letters
};

// Occurrence-table layouts
enum OccLayout { OCC_NONE = 0, OCC_DNA32 = 1, OCC_BYTE = 2 };

struct DeviceIndex {
    cudaStream_t stream = 0;
    int device = 0;
    u32 n = 0, len = 0, sigma = 0;
    Packing pk{};
    // owned device arrays (may be null when not requested / released)
    DevBuf<u8> text;        // len bytes of codes (text[n] = 0), only when we own a copy
    const u8 *text_ptr = nullptr;
    u64 *packed = nullptr;  // packed text (workspace arena), padded with zero words
    Arena *arena = nullptr; // per-device build workspace (valid during the build only)
    DevBuf<u32> sa, isa, lcp;
    DevBuf<u64> text_packed;  // kept copy of the packed text (B200SA_BUILD_TEXTCMP: search shortcut)
    DevBuf<uint2> ktable;     // (L, R) after the recurrence on every k-mer (B200SA_BUILD_KTABLE)
    int ktable_k = 0;
    DevBuf<uint4> ssa_marks;  // sampled suffix array (locate.cu): 16 bytes per 64 rows
    DevBuf<u32> ssa_vals;     // SA values of the sampled rows
    u32 ssa_rate = 0;         // 0: none
    DevBuf<u8> bwt;
    DevBuf<u32> c_table;    // sigma entries (device)
    u32 c_host[256];
    u64 sym_counts_host[256];
    u32 primary = 0;        // row r with sa[r] == 0
    OccLayout occ_layout = OCC_NONE;
    DevBuf<u8> occ;         // occurrence blocks
    u64 occ_blocks = 0;
    u32 occ_block_bytes = 0;
    BuildStats stats{};
    StageTimer timer;
    // records index (records.cu): nrec records, record r at text positions start[r] .. start[r] + len_r (its separator)
    u32 nrec = 0;                 // 0: a plain index
    std::vector<u64> rec_off;     // nrec + 1 offsets into the records without separators
    DevBuf<u64> rec_start;        // nrec + 1 entries: start[r] = rec_off[r] + r, start[nrec] = n
};

// sa_build.cu
void pack_text(DeviceIndex &ix, int *d_err);
size_t build_workspace_estimate(u32 len, int bits);
void build_suffix_array(DeviceIndex &ix, bool want_bwt);  // fills ix.sa (+ ix.bwt, ix.primary)
void build_inverse(DeviceIndex &ix);
// lcp.cu
void build_lcp(DeviceIndex &ix);
// bwt_occ.cu
void gather_bwt(DeviceIndex &ix);  // ix.bwt + ix.primary from an existing SA
void build_bwt_tables(DeviceIndex &ix, bool keep_bwt);
void occ_probe(const DeviceIndex &ix, const u8 *d_a, const u32 *d_i, u64 count, u32 *d_out);
void occ_dense(const DeviceIndex &ix, u32 *d_out);  // (len+1)*sigma entries, reference layout
// fm_search.cu
void build_ktable(DeviceIndex &ix);  // fills ix.ktable (DNA layout only)
void fm_search(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 *d_L,
               u32 *d_R, cudaStream_t st, unsigned long long *d_stats = nullptr);
// resident one-pattern search (the drop-in's iterator): a one-warp kernel that polls `d_slot` (mapped pinned memory)
void fm_mailbox_server_launch(const DeviceIndex &ix, void *d_slot, u32 tag, u32 idle_limit, cudaStream_t st);
// packed reads: 2 bits per base, four to a byte, first base in the high bits; read q at q * stride bytes
void fm_search_packed(const DeviceIndex &ix, const u8 *d_packed, u32 m, u32 stride, u64 npat, u32 *d_L, u32 *d_R,
                      cudaStream_t st, unsigned long long *d_stats = nullptr);
void pack_reads(const u8 *d_codes, u32 m, u32 stride, u64 npat, u8 *d_out, int *d_err, cudaStream_t st);
u64 fm_locate_count(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, u64 *d_pos_off,
                    cudaStream_t st);
void fm_locate_fill(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, const u64 *d_pos_off,
                    u64 total, u32 *d_pos, cudaStream_t st);
void scan_u64(u64 *d_vals, u64 count, cudaStream_t st);  // exclusive scan in place; d_vals[count] = the total
// locate.cu
void build_sampled_sa(DeviceIndex &ix, u32 rate);  // fills ix.ssa_* from ix.sa
void fm_locate_fill_ssa(const DeviceIndex &ix, const u32 *d_L, u64 npat, const u64 *d_pos_off, u64 total,
                        u32 *d_pos, cudaStream_t st);
void sa_lookup_rows(const DeviceIndex &ix, const u32 *d_rows, u64 count, u32 *d_out, bool force_sampled,
                    cudaStream_t st);
void sort_positions(const DeviceIndex &ix, u64 npat, const u64 *d_pos_off, u64 total, u32 *d_pos, cudaStream_t st);
// approx.cu
void approx_dtable(const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u8 *d_dtab,
                   cudaStream_t st);
void approx_count(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m,
                  const u8 *d_dtab, int max_edits, u64 *d_hit_off, u64 *d_ops_off, u64 *hits, u64 *ops,
                  cudaStream_t st);
void approx_emit(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m,
                 const u8 *d_dtab, int max_edits, const u64 *d_hit_off, const u64 *d_ops_off, u32 *d_L, u32 *d_R,
                 u32 *d_mlen, u64 *d_hit_ops_off, char *d_ops, cudaStream_t st);
// mems.cu: matching statistics (ms / L / R per pattern symbol, laid out like d_pat) and, with d_count, the SMEMs of
// each pattern counted; mems_emit writes them at d_smem_off (exclusive scan of the counts)
void mems_stats(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 min_len,
                u32 *d_ms, u32 *d_L, u32 *d_R, u64 *d_count, cudaStream_t st);
void mems_emit(const DeviceIndex &ix, const u64 *d_off, u32 fixed_len, u64 npat, u32 min_len, const u32 *d_ms,
               const u32 *d_L, const u32 *d_R, const u64 *d_smem_off, u32 *d_start, u32 *d_len, u32 *d_sL, u32 *d_sR,
               cudaStream_t st);
// records.cu
void records_assemble(const u8 *d_codes, u64 ncodes, const u64 *d_rec_off, u32 nrec, u32 sigma, u8 *d_text,
                      int *d_err, cudaStream_t st);  // d_text: ncodes + nrec + 1 bytes
void record_sas(const DeviceIndex &ix, u32 *d_out, cudaStream_t st);  // needs ix.sa; n entries
void records_clamp_rows(const u32 *d_L, u64 npat, u32 *d_out, cudaStream_t st);  // max(L, 1)
void locate_records_group(const DeviceIndex &ix, u64 npat, const u64 *d_pos_off, u64 total, const u32 *d_pos,
                          u32 *d_rec, u32 *d_local, cudaStream_t st);
// synth.cu
void synth_codes(u8 *d_text, u64 n, u32 nsym, u64 seed, cudaStream_t st);
void synth_reads(const u8 *d_text, u64 n, u32 nsym, u8 *d_reads, u64 nreads, u32 m, u32 miss_per_1024,
                 u64 seed, cudaStream_t st);

}  // namespace b200sa
