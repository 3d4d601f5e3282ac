// locate.cu -- locate through a SAMPLED suffix array, and per-pattern sorted positions (sm_100a).
//
// The reference iterator reports SA[i] for i in [L, R) (stralg/bwt.c:201-217), which needs the
// whole suffix array next to the O table: 12 GB at 3 Gbp on every GPU that holds a replica of the
// index.  Here only the rows whose suffix starts at a multiple of `rate` keep their entry:
//
//   marks[w]  (16 bytes per 64 rows)   u64 bits  -- row 64w+k is sampled <=> bit k
//                                      u32 rank  -- sampled rows before row 64w
//   vals[j]                            SA value of the j-th sampled row
//
// SA[r] for any other row is recovered by walking LF(r) = C(a) + O(a, r), a = bwt[r] (the suffix
// one position to the left) until a sampled row is met, at most rate - 1 steps later:
// SA[r] = vals[...] + steps.  The row that holds the sentinel (SA == 0) is always sampled, so the
// walk never steps over the start of the text.  Both the symbol of a row and its rank come out of
// the same O block, i.e. one 32-byte sector per step with the DNA layout (occ.cuh).
//
// The values are those of the full array, so parity with the reference iterator is unchanged:
// same positions, same (suffix-array) order.  sort_positions() reorders the positions of every
// pattern ascending -- the order the reference's tests compare in (tests/stralg/match_test.c:608).
#include "engine.h"
#include "occ.cuh"
#include "radix_sort.cuh"

#include <algorithm>

namespace b200sa {

static constexpr int SS_TILE_WORDS = 1024;  // mark words per scan tile (65 536 rows)

// one warp per 64 rows: two ballots form the mark word; tile totals by one atomic per word
__global__ void __launch_bounds__(256) ssa_mark_kernel(const u32 *__restrict__ sa, u32 len, u32 rate, u64 nwords,
                                                       uint4 *__restrict__ marks, u32 *__restrict__ tile_tot) {
    const u64 warp0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const u32 lane = lane_id();
    for (u64 w = warp0; w < nwords; w += nwarps) {
        const u64 r0 = w * 64 + lane, r1 = r0 + 32;
        const bool m0 = r0 < len && ld_stream_u32(sa + r0) % rate == 0;
        const bool m1 = r1 < len && ld_stream_u32(sa + r1) % rate == 0;
        const u32 b0 = __ballot_sync(0xffffffffu, m0), b1 = __ballot_sync(0xffffffffu, m1);
        if (lane == 0) {
            const u32 c = (u32)__popc(b0) + (u32)__popc(b1);
            marks[w] = make_uint4(b0, b1, c, 0u);  // .z: count for now, rank after the scan
            if (c) atomicAdd(&tile_tot[w / SS_TILE_WORDS], c);
        }
    }
}

// one CTA per tile of mark words: counts -> ranks, then the sampled values are stored
__global__ void __launch_bounds__(SS_TILE_WORDS) ssa_fill_kernel(const u32 *__restrict__ sa, u64 nwords,
                                                                 const u32 *__restrict__ tile_prefix,
                                                                 uint4 *__restrict__ marks, u32 *__restrict__ vals) {
    __shared__ u32 wsum[32];
    const u64 w = (u64)blockIdx.x * SS_TILE_WORDS + threadIdx.x;
    uint4 mk = make_uint4(0, 0, 0, 0);
    if (w < nwords) mk = marks[w];
    const u32 excl = block_exclusive<SS_TILE_WORDS>(mk.z, wsum);
    if (w >= nwords) return;
    const u32 rank = tile_prefix[blockIdx.x] + excl;
    mk.z = rank;
    marks[w] = mk;
    u64 bits = ((u64)mk.y << 32) | mk.x;
    u32 j = rank;
    while (bits) {
        const int k = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        vals[j++] = sa[w * 64 + (u64)k];
    }
}

void build_sampled_sa(DeviceIndex &ix, u32 rate) {
    cudaStream_t st = ix.stream;
    const u64 nwords = ((u64)ix.len + 63) / 64;
    const u64 nsamp = (u64)ix.n / rate + 1;  // text positions 0, rate, 2 rate, ... <= n
    const u32 ntiles = div_up_u(nwords, SS_TILE_WORDS);
    ix.ssa_marks.alloc(nwords, st);
    ix.ssa_vals.alloc(nsamp, st);
    DevBuf<u32> tile_tot(ntiles, st);
    CUDA_CHECK(cudaMemsetAsync(tile_tot.ptr, 0, (size_t)ntiles * 4, st));
    unsigned blocks = std::max(1u, std::min(div_up_u(nwords, 8), 148u * 16u));
    ssa_mark_kernel<<<blocks, 256, 0, st>>>(ix.sa.ptr, ix.len, rate, nwords, ix.ssa_marks.ptr, tile_tot.ptr);
    KERNEL_CHECK();
    scan_sum(tile_tot.ptr, ntiles, st);
    ssa_fill_kernel<<<ntiles, SS_TILE_WORDS, 0, st>>>(ix.sa.ptr, nwords, tile_tot.ptr, ix.ssa_marks.ptr, ix.ssa_vals.ptr);
    KERNEL_CHECK();
    ix.ssa_rate = rate;  // (tile_tot is released in stream order)
}

struct SsaView {
    const uint4 *marks;
    const u32 *vals;
};

// SA[row] through the sampled array (see the header of this file)
template <int LAYOUT>
__device__ __forceinline__ u32 ssa_lookup(const OccView &ov, const SsaView &sv, const u32 *__restrict__ c_tab, u32 row) {
    u32 steps = 0;
    while (true) {
        const uint4 mk = __ldg(sv.marks + (row >> 6));
        const u64 bits = ((u64)mk.y << 32) | mk.x;
        const u32 k = row & 63u;
        if ((bits >> k) & 1ull) return __ldg(sv.vals + mk.z + (u32)__popcll(bits & ((1ull << k) - 1ull))) + steps;
        u32 a;
        if (LAYOUT == 1) {
            const DnaBlock *blk = (const DnaBlock *)ov.blocks + (row >> 6);
            const uint4 h = __ldg((const uint4 *)blk);
            const uint4 p = __ldg((const uint4 *)blk + 1);
            const u64 w0 = ((u64)p.y << 32) | p.x, w1 = ((u64)p.w << 32) | p.z;
            a = (u32)(((k < 32 ? w0 : w1) >> (2 * (k & 31u))) & 3ull) + 1u;
            const u32 base = a == 1 ? h.x : a == 2 ? h.y : a == 3 ? h.z : h.w;
            u32 c = base + dna_match_count(w0, w1, a - 1, k);
            // the sentinel row is stored as value 0 (code 1); it is sampled, so `row` is never it
            if (a == 1 && ov.primary >= (row & ~63u) && ov.primary < row) c -= 1;
            row = c_tab[a] + c;
        } else {
            const u8 *blk = ov.blocks + (size_t)(row >> 6) * ov.block_bytes;
            a = blk[(size_t)ov.hdr_words * 4 + k];
            row = c_tab[a] + occ_byte(ov, a, row);
        }
        ++steps;
    }
}

template <int LAYOUT>
__global__ void __launch_bounds__(256) locate_fill_ssa_kernel(OccView ov, SsaView sv, const u32 *__restrict__ c_dev,
                                                              const u32 *__restrict__ L,
                                                              const u64 *__restrict__ pos_off, u64 npat, u64 total,
                                                              u32 *__restrict__ pos) {
    __shared__ u32 c_sh[256];
    for (u32 i = threadIdx.x; i < 256; i += blockDim.x) c_sh[i] = i < ov.sigma ? c_dev[i] : 0;
    __syncthreads();
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    u64 lo = 0, hi = npat;  // largest q with pos_off[q] <= t  (pos_off[npat] = total > t)
    while (hi - lo > 1) {
        const u64 mid = lo + (hi - lo) / 2;
        if (pos_off[mid] <= t) lo = mid;
        else hi = mid;
    }
    const u32 row = (u32)((u64)L[lo] + (t - pos_off[lo]));
    pos[t] = ssa_lookup<LAYOUT>(ov, sv, c_sh, row);
}

void fm_locate_fill_ssa(const DeviceIndex &ix, const u32 *d_L, u64 npat, const u64 *d_pos_off, u64 total,
                        u32 *d_pos, cudaStream_t st) {
    if (!total) return;
    OccView ov = occ_view(ix);
    SsaView sv{ix.ssa_marks.ptr, ix.ssa_vals.ptr};
    const unsigned blocks = div_up_u(total, 256);
    if (ix.occ_layout == OCC_DNA32)
        locate_fill_ssa_kernel<1><<<blocks, 256, 0, st>>>(ov, sv, ix.c_table.ptr, d_L, d_pos_off, npat, total, d_pos);
    else
        locate_fill_ssa_kernel<2><<<blocks, 256, 0, st>>>(ov, sv, ix.c_table.ptr, d_L, d_pos_off, npat, total, d_pos);
    KERNEL_CHECK();
}

// SA[rows[q]] for arbitrary rows (b200sa_sa_lookup)
template <int LAYOUT>
__global__ void __launch_bounds__(256) ssa_rows_kernel(OccView ov, SsaView sv, const u32 *__restrict__ c_dev,
                                                       const u32 *__restrict__ rows, u64 count,
                                                       u32 *__restrict__ out) {
    __shared__ u32 c_sh[256];
    for (u32 i = threadIdx.x; i < 256; i += blockDim.x) c_sh[i] = i < ov.sigma ? c_dev[i] : 0;
    __syncthreads();
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < count) out[t] = ssa_lookup<LAYOUT>(ov, sv, c_sh, rows[t]);
}

__global__ void __launch_bounds__(256) sa_rows_kernel(const u32 *__restrict__ sa, const u32 *__restrict__ rows,
                                                      u64 count, u32 *__restrict__ out) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < count) out[t] = sa[rows[t]];
}

void sa_lookup_rows(const DeviceIndex &ix, const u32 *d_rows, u64 count, u32 *d_out, bool force_sampled,
                    cudaStream_t st) {
    if (!count) return;
    const unsigned blocks = div_up_u(count, 256);
    if (ix.sa.ptr && !force_sampled) {
        sa_rows_kernel<<<blocks, 256, 0, st>>>(ix.sa.ptr, d_rows, count, d_out);
    } else {
        OccView ov = occ_view(ix);
        SsaView sv{ix.ssa_marks.ptr, ix.ssa_vals.ptr};
        if (ix.occ_layout == OCC_DNA32)
            ssa_rows_kernel<1><<<blocks, 256, 0, st>>>(ov, sv, ix.c_table.ptr, d_rows, count, d_out);
        else
            ssa_rows_kernel<2><<<blocks, 256, 0, st>>>(ov, sv, ix.c_table.ptr, d_rows, count, d_out);
    }
    KERNEL_CHECK();
}

// ---- positions of every pattern in ascending order -------------------------------------------
// key = [pattern : high 32 bits | position : low 32 bits]; one stable LSD radix sort of all keys
// (radix_sort.cuh; passes whose digit is the same for every key are skipped) orders the positions
// inside every pattern without touching the CSR offsets.
__global__ void __launch_bounds__(256) sort_keys_make_kernel(const u32 *__restrict__ pos,
                                                             const u64 *__restrict__ pos_off, u64 npat, u64 total,
                                                             u64 *__restrict__ keys) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    u64 lo = 0, hi = npat;
    while (hi - lo > 1) {
        const u64 mid = lo + (hi - lo) / 2;
        if (pos_off[mid] <= t) lo = mid;
        else hi = mid;
    }
    keys[t] = (lo << 32) | (u64)pos[t];
}

__global__ void __launch_bounds__(256) sort_keys_take_kernel(const u64 *__restrict__ keys, u64 total,
                                                             u32 *__restrict__ pos) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < total) pos[t] = (u32)keys[t];
}

void sort_positions(const DeviceIndex &ix, u64 npat, const u64 *d_pos_off, u64 total, u32 *d_pos, cudaStream_t st) {
    if (total < 2) return;
    if (total > 0xFFFFFFFFull || npat > 0xFFFFFFFFull)
        throw std::runtime_error("sort_positions: more than 2^32 - 1 positions or patterns in one batch");
    int qbits = 0;
    while ((1ull << qbits) < npat) ++qbits;
    DevBuf<u64> kA(total, st), kB(total, st);
    DevBuf<u32> vA(total, st), vB(total, st);
    CUDA_CHECK(cudaMemsetAsync(vA.ptr, 0, total * 4, st));
    sort_keys_make_kernel<<<div_up_u(total, 256), 256, 0, st>>>(d_pos, d_pos_off, npat, total, kA.ptr);
    KERNEL_CHECK();
    u64 *kb[2] = {kA.ptr, kB.ptr};
    u32 *vb[2] = {vA.ptr, vB.ptr};
    const auto sorted = rs::Sorter<8>::sort(kb, vb, (u32)total, 32 + qbits, st);
    sort_keys_take_kernel<<<div_up_u(total, 256), 256, 0, st>>>(sorted.keys, total, d_pos);
    KERNEL_CHECK();
    (void)ix;  // (the work buffers are released in stream order)
}

void sort_pairs(u64 *keys[2], u32 *vals[2], u32 n, int key_bits, u64 *&keys_out, u32 *&vals_out, cudaStream_t st) {
    const auto sorted = rs::Sorter<8>::sort(keys, vals, n, key_bits, st);
    keys_out = sorted.keys;
    vals_out = sorted.vals;
}

}  // namespace b200sa
