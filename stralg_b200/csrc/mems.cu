// mems.cu -- matching statistics and super-maximal exact matches (SMEMs) of a pattern batch (sm_100a).
//
// For every end j of a pattern P[0..m): s_j is the smallest s such that P[s..j] occurs in the text (j + 1 when no
// suffix of P[0..j] does), ms[j] = j + 1 - s_j, and [L[j], R[j]) is the SA interval of P[s_j..j] -- (1, 0) when
// ms[j] = 0.  An SMEM is (s_j, ms[j], L[j], R[j]) for every j with ms[j] >= min_len and (j = m - 1 or
// ms[j+1] <= ms[j]): s never decreases, so these are the occurring pieces of P that no other one contains.
//
// One warp per pattern; lane l takes the ends j = m-1-l, m-1-l-32, ..., so the lanes of a warp read the same
// pattern words.  Each end runs the backward recurrence of the exact search (fm_step.cuh) from j and keeps the last
// non-empty interval: the seed entry of the k symbols ending at j when they are letters and the entry is not empty,
// else O steps from j; O steps until the interval is empty or unique; then (TEXTCMP) the symbols before the match
// are compared with the text before its one occurrence s = SA[L]: k symbols agree, the match grows by k and its
// interval is [ISA[s - k], +1).  A code 0 or >= sigma occurs nowhere and ends every match that reaches it.
//
// Two passes: mems_stats_kernel stores ms / L / R per pattern symbol and counts each pattern's SMEMs (the ms of end
// j + 1 sits in the neighbouring lane, or in lane 31 of the previous round); an exclusive scan (scan_u64,
// fm_search.cu) turns the counts into a CSR; mems_emit_kernel writes the SMEMs from the stored arrays, in ascending
// start, without running the recurrence again.
#include "engine.h"
#include "fm_step.cuh"

namespace b200sa {

struct MemsArgs {
    OccView ov;
    CTable5 c5;            // DNA layout: C table
    const u32 *c_dev;      // byte layout: C table (sigma entries)
    TextCmp tc;
    KTable kt;
    int bits;              // bits per packed text symbol
    u32 len;
    const u8 *pat;         // 8-byte aligned, readable up to the next 8-byte boundary after the last pattern
    const u64 *off;
    u32 fixed_len;
    u64 npat;
    u32 min_len;
    u32 *ms, *L, *R;       // per pattern symbol, laid out like `pat`
    u64 *count;            // pass 1: SMEMs per pattern (null: not counted)
    const u64 *smem_off;   // pass 2: exclusive scan of `count`
    u32 *s_start, *s_len, *s_L, *s_R;
};

// ms[j] of one end j of the pattern at `begin`; (L, R) its interval
template <int LAYOUT, bool SC>
__device__ __forceinline__ u32 mems_end(const MemsArgs &A, const u32 *c_sh, u64 begin, int64_t j, u32 &Lout, u32 &Rout) {
    u64 word = 0, word_addr = ~0ull;
    u32 n_pw = 0, n_blk = 0, n_tw = 0;  // (the traffic counters of the shared pieces; not kept here)
    auto P = [&](int64_t idx) -> u32 { return pattern_byte<false>(A.pat, begin + (u64)idx, word, word_addr, n_pw); };
    u32 L = 0, R = A.len, ms = 0;
    int64_t i = j;
    if (A.kt.tab && j + 1 >= (int64_t)A.kt.k) {
        u32 x;
        const bool valid = LAYOUT == 1 ? dna_seed_key<false>(A.pat, begin, j, A.kt.k, word, word_addr, n_pw, x)
                                       : seed_key(P, j, A.kt, x);
        if (valid) {
            const uint2 lr = A.kt.tab[x];
            if (lr.x < lr.y) {  // (an empty entry: the match is shorter than k, found stepwise below)
                L = lr.x;
                R = lr.y;
                ms = (u32)A.kt.k;
                i = j - A.kt.k;
            }
        }
    }
    for (; i >= 0 && !(SC && R - L == 1); --i) {
        const u32 a = P(i);
        if (a == 0 || a >= A.ov.sigma) break;
        u32 nL, nR;
        if (LAYOUT == 1) {
            const uint2 lr = dna_step<false>(A.ov, A.c5, a, L, R, n_blk);
            nL = lr.x;
            nR = lr.y;
        } else {
            const u32 ca = c_sh[a];
            nL = ca + occ_byte(A.ov, a, L);
            nR = ca + occ_byte(A.ov, a, R);
        }
        if (nL >= nR) break;
        L = nL;
        R = nR;
        ++ms;
    }
    // (the loop only stops at a unique interval with symbols left when no step failed)
    if (SC && i >= 0 && R - L == 1) {
        const u32 s = A.tc.sa[L];
        u32 a;
        const u64 k = LAYOUT == 1 ? dna_text_agree<false>(A.pat, begin, i, s, A.tc.packed, word, word_addr, a, n_pw, n_tw)
                                  : text_agree(P, i, s, A.tc.packed, A.bits, a);
        if (k) {
            L = A.tc.isa[s - (u32)k];
            R = L + 1;
            ms += (u32)k;
        }
    }
    if (ms == 0) {
        L = 1;
        R = 0;
    }
    Lout = L;
    Rout = R;
    return ms;
}

template <int LAYOUT, bool SC>
__global__ void __launch_bounds__(256, 4) mems_stats_kernel(MemsArgs A) {
    __shared__ u32 c_sh[256];
    if (LAYOUT != 1) {
        for (u32 k = threadIdx.x; k < 256; k += blockDim.x) c_sh[k] = k < A.ov.sigma ? A.c_dev[k] : 0;
        __syncthreads();
    }
    const u64 q = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= A.npat) return;  // (whole warps)
    const u32 lane = lane_id();
    const u64 begin = A.off ? A.off[q] : q * (u64)A.fixed_len;
    const u64 m = A.off ? A.off[q + 1] - begin : (u64)A.fixed_len;
    u32 carry = 0;  // ms of the lowest end of the previous round (lane 31)
    u64 count = 0;
    for (u64 base = 0; base < m; base += 32) {
        const int64_t j = (int64_t)(m - 1 - base) - (int64_t)lane;
        u32 ms = 0;
        if (j >= 0) {
            u32 L, R;
            ms = mems_end<LAYOUT, SC>(A, c_sh, begin, j, L, R);
            A.ms[begin + (u64)j] = ms;
            A.L[begin + (u64)j] = L;
            A.R[begin + (u64)j] = R;
        }
        u32 next = __shfl_up_sync(0xffffffffu, ms, 1);  // ms[j + 1]
        if (lane == 0) next = carry;
        const bool smem = j >= 0 && ms >= A.min_len && (j == (int64_t)m - 1 || next <= ms);
        count += (u64)__popc(__ballot_sync(0xffffffffu, smem));
        carry = __shfl_sync(0xffffffffu, ms, 31);
    }
    if (A.count && lane == 0) A.count[q] = count;
}

// one warp per pattern, ends in ascending order: the SMEMs of a round leave in lane order at the pattern's offset
__global__ void __launch_bounds__(256) mems_emit_kernel(MemsArgs A) {
    const u64 q = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= A.npat) return;
    const u32 lane = lane_id();
    const u64 begin = A.off ? A.off[q] : q * (u64)A.fixed_len;
    const u64 m = A.off ? A.off[q + 1] - begin : (u64)A.fixed_len;
    u64 at = A.smem_off[q];
    for (u64 base = 0; base < m; base += 32) {
        const u64 j = base + lane;
        u32 ms = 0;
        bool smem = false;
        if (j < m) {
            ms = A.ms[begin + j];
            smem = ms >= A.min_len && (j + 1 == m || A.ms[begin + j + 1] <= ms);
        }
        const u32 bal = __ballot_sync(0xffffffffu, smem);
        if (smem) {
            const u64 o = at + (u64)__popc(bal & ((1u << lane) - 1u));
            A.s_start[o] = (u32)(j + 1 - ms);
            A.s_len[o] = ms;
            A.s_L[o] = A.L[begin + j];
            A.s_R[o] = A.R[begin + j];
        }
        at += (u64)__popc(bal);
    }
}

static MemsArgs mems_args(const DeviceIndex &ix, const u64 *d_off, u32 fixed_len, u64 npat, u32 min_len,
                          const u32 *d_ms, const u32 *d_L, const u32 *d_R) {
    MemsArgs A{};
    A.ov = occ_view(ix);
    for (int i = 0; i < 8; ++i) A.c5.c[i] = ix.c_host[i];
    A.c_dev = ix.c_table.ptr;
    A.tc = TextCmp{ix.sa.ptr, ix.isa.ptr, ix.text_packed.ptr};
    A.kt = KTable{ix.ktable.ptr, ix.ktable_k, ix.occ_layout == OCC_DNA32 ? 0u : ix.sigma - 1};
    A.bits = ix.pk.bits;
    A.len = ix.len;
    A.off = d_off;
    A.fixed_len = fixed_len;
    A.npat = npat;
    A.min_len = min_len;
    A.ms = const_cast<u32 *>(d_ms);
    A.L = const_cast<u32 *>(d_L);
    A.R = const_cast<u32 *>(d_R);
    return A;
}

void mems_stats(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 min_len,
                u32 *d_ms, u32 *d_L, u32 *d_R, u64 *d_count, cudaStream_t st) {
    if (!npat) return;
    MemsArgs A = mems_args(ix, d_off, fixed_len, npat, min_len, d_ms, d_L, d_R);
    A.pat = d_pat;
    A.count = d_count;
    const unsigned blocks = div_up_u(npat * 32, 256);
    const bool tc = A.tc.sa && A.tc.isa && A.tc.packed;
    if (ix.occ_layout == OCC_DNA32) {
        if (tc && ix.pk.bits == 2) mems_stats_kernel<1, true><<<blocks, 256, 0, st>>>(A);
        else mems_stats_kernel<1, false><<<blocks, 256, 0, st>>>(A);
    } else {
        if (tc) mems_stats_kernel<2, true><<<blocks, 256, 0, st>>>(A);
        else mems_stats_kernel<2, false><<<blocks, 256, 0, st>>>(A);
    }
    KERNEL_CHECK();
}

void mems_emit(const DeviceIndex &ix, const u64 *d_off, u32 fixed_len, u64 npat, u32 min_len, const u32 *d_ms,
               const u32 *d_L, const u32 *d_R, const u64 *d_smem_off, u32 *d_start, u32 *d_len, u32 *d_sL, u32 *d_sR,
               cudaStream_t st) {
    if (!npat) return;
    MemsArgs A = mems_args(ix, d_off, fixed_len, npat, min_len, d_ms, d_L, d_R);
    A.smem_off = d_smem_off;
    A.s_start = d_start;
    A.s_len = d_len;
    A.s_L = d_sL;
    A.s_R = d_sR;
    mems_emit_kernel<<<div_up_u(npat * 32, 256), 256, 0, st>>>(A);
    KERNEL_CHECK();
}

}  // namespace b200sa
