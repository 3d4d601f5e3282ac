// sa_build.cu -- suffix-array construction by GPU prefix doubling (sm_100a).
//
// Produces the array the reference's four constructors agree on (stralg/suffix_array.c:32-48,
// sa_is.c:466-509, sa_is_mem.c:471-494, skew.c:388-395): all len = n+1 suffixes of text+sentinel
// in strcmp order, SA[0] = n.  None of the reference's algorithms is ported.  The pipeline:
//
//   pack_text        codes 1..sigma-1 -> (code-1) packed big-endian at 1/2/4/8 bits per symbol,
//                    symbol counts for the C table fused (stralg/remap.c:73-88, bwt.c:35-45)
//   cmer_hist        histogram of all digit-wide symbol groups; every round-0 radix pass's digit
//                    histogram is that histogram up to <= K boundary corrections (round0_bases)
//   make_keys0       key(s) = first K symbols of suffix s; the <= K suffixes that reach the
//                    sentinel inside the window are fed first, shortest first, so that the STABLE
//                    sort leaves them ahead of their padded-equal long neighbours
//   onesweep passes  radix_sort.cuh
//   rank_kernel      bucket heads by key comparison, rank[s] = SA index of the bucket head,
//                    head bitmap for singleton retirement
//   compact          suffixes in non-singleton buckets form the next active set
//   rounds           key = (rank[s], rank[s+h]) for active suffixes only, sort, re-rank, h *= 2
//
// After the last round rank[] is the inverse suffix array (stralg/suffix_array.c:55-62).
#include "engine.h"
#include "radix_sort.cuh"
#include "round0_msd.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <functional>
#include <vector>

namespace b200sa {

// ---------------------------------------------------------------------------------------------
// pack_text: one thread per packed word.  err[0] is set if a code is 0 or >= sigma.
// sym_counts[c] (u64) accumulates the number of text positions holding code c (c >= 1).
// ---------------------------------------------------------------------------------------------
template <int BITS>
__global__ void __launch_bounds__(256) pack_kernel(const u8 *__restrict__ text, u32 n, u32 sigma, u64 nwords,
                                                   u64 *__restrict__ packed,
                                                   unsigned long long *__restrict__ sym_counts,
                                                   int *__restrict__ err) {
    constexpr int CPW = 64 / BITS;
    __shared__ u32 sh_counts[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sh_counts[i] = 0;
    __syncthreads();
    bool bad = false;
    // grid-stride: a block's symbol counts reach the global counters once, not once per 256 words
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += (u64)gridDim.x * blockDim.x) {
        u64 t0 = w * CPW;
        u64 word = 0;
        if (BITS == 2 && t0 + CPW <= n && ((((uintptr_t)(text + t0)) & 31) == 0)) {
            // DNA fast path: 32 codes in one 256-bit load, packed eight at a time without a byte loop
            u64 x[4];
            asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                         : "=l"(x[0]), "=l"(x[1]), "=l"(x[2]), "=l"(x[3]) : "l"(text + t0));
            const u64 ones = 0x0101010101010101ull, high = 0x8080808080808080ull;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const u64 v = x[h];
                // a code is valid when it is in 1..sigma-1: no byte >= 128, none zero, none >= sigma
                const u64 zero = (v - ones) & ~v & high;
                const u64 big = (v | (v + ones * (u64)(0x80u - sigma))) & high;
                if (zero | big) bad = true;
                // symbols = code - 1, first text byte to the most significant end
                const u32 lo32 = (u32)v, hi32 = (u32)(v >> 32);
                u64 y = ((u64)__byte_perm(lo32, 0, 0x0123) << 32) | (u64)__byte_perm(hi32, 0, 0x0123);
                y = (y - ones) & 0x0303030303030303ull;
                y = (y | (y >> 6)) & 0x000F000F000F000Full;
                y = (y | (y >> 12)) & 0x000000FF000000FFull;
                y = (y | (y >> 24)) & 0xFFFFull;
                word |= y << (48 - 16 * h);
            }
#pragma unroll
            for (u32 c = 0; c < 4; ++c) {
                const u64 yy = word ^ (c * 0x5555555555555555ull);
                const u32 cx = (u32)__popcll(~(yy | (yy >> 1)) & 0x5555555555555555ull);
                const u32 tot = __reduce_add_sync(__activemask(), cx);
                if ((threadIdx.x & 31u) == (u32)(__ffs((int)__activemask()) - 1) && tot) atomicAdd(&sh_counts[c + 1], tot);
            }
        } else if (t0 < n) {
            // the CPW text bytes of this word, fetched with the widest loads (one 256-bit load for DNA)
            __align__(32) u8 b[CPW];
            const u8 *src = text + t0;
            if (t0 + CPW <= n && ((((uintptr_t)src) & (CPW < 32 ? CPW - 1 : 31)) == 0)) {
                if (CPW >= 32) {
#pragma unroll
                    for (int h = 0; h < CPW / 32; ++h) {
                        u64 x0, x1, x2, x3;
                        asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                                     : "=l"(x0), "=l"(x1), "=l"(x2), "=l"(x3) : "l"(src + 32 * h));
                        u64 *bw = (u64 *)(b + 32 * h);
                        bw[0] = x0; bw[1] = x1; bw[2] = x2; bw[3] = x3;
                    }
                } else if (CPW == 16) {
                    *(uint4 *)b = ld_stream_u128(src);
                } else {
                    *(u64 *)b = ld_stream_u64((const u64 *)src);
                }
            } else {
#pragma unroll
                for (int q = 0; q < CPW; ++q) b[q] = (t0 + q < n) ? src[q] : (u8)1;
            }
#pragma unroll
            for (int q = 0; q < CPW; ++q) {
                u32 code = b[q];
                u32 sym = 0;
                if (t0 + q < n) {
                    if (code == 0 || code >= sigma) bad = true;
                    sym = (code - 1) & ((1u << BITS) - 1);
                    if (BITS > 2) atomicAdd(&sh_counts[code & 255], 1u);
                }
                word |= (u64)sym << (64 - BITS - q * BITS);
            }
            if (BITS <= 2) {
                // symbol counts straight from the packed word (padding symbols are 0)
                u32 nv = (u32)((u64)n - t0 < (u64)CPW ? (u64)n - t0 : (u64)CPW);
                if (BITS == 1) {
                    u32 c1 = __popcll(word);
                    atomicAdd(&sh_counts[2], c1);
                    atomicAdd(&sh_counts[1], nv - c1);
                } else {
#pragma unroll
                    for (u32 x = 0; x < 4; ++x) {
                        u64 y = word ^ (x * 0x5555555555555555ull);
                        u64 mm = ~(y | (y >> 1)) & 0x5555555555555555ull;
                        u32 cx = __popcll(mm);
                        if (x == 0) cx -= (CPW - nv);
                        if (cx) atomicAdd(&sh_counts[x + 1], cx);
                    }
                }
            }
        }
        packed[w] = word;
    }
    if (bad) *err = 1;
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (sh_counts[i]) atomicAdd(&sym_counts[i], (unsigned long long)sh_counts[i]);
}

// ---------------------------------------------------------------------------------------------
// cmer_hist: H[x] = #{t in [0, n] : first RB bits of the packed stream at symbol t == x}
// ---------------------------------------------------------------------------------------------
template <int RB, int BITS>
__global__ void __launch_bounds__(256) cmer_hist_kernel(const u64 *__restrict__ packed, u32 n, u64 nwords_data,
                                                        u32 *__restrict__ hist) {
    constexpr int BINS = 1 << RB;
    constexpr int CPW = 64 / BITS;
    __shared__ u32 sh[BINS];
    for (int i = threadIdx.x; i < BINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < nwords_data; w += stride) {
        u64 hi = packed[w], lo = packed[w + 1];
        u64 t0 = w * CPW;
#pragma unroll
        for (int q = 0; q < CPW; ++q) {
            if (t0 + q <= n) {
                const int o = q * BITS;
                u64 win = o ? ((hi << o) | (lo >> (64 - o))) : hi;
                atomicAdd(&sh[(u32)(win >> (64 - RB))], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BINS; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// Block p turns H into the exclusive digit offsets of round-0 pass p (p = 0 is the least
// significant digit, i.e. the LAST c symbols of the K-symbol key).
template <int RB>
__global__ void __launch_bounds__(256) round0_bases_kernel(const u32 *__restrict__ H, const u64 *__restrict__ packed,
                                                           u32 n, int K, int bits, u32 *__restrict__ digit_base) {
    constexpr int BINS = 1 << RB;
    constexpr int NT = 256;
    constexpr int DPT = (BINS + NT - 1) / NT;
    __shared__ u32 h[BINS];
    __shared__ u32 warp_tot[NT / 32];
    const int p = blockIdx.x;
    const int c = RB / bits;
    for (int i = threadIdx.x; i < BINS; i += NT) h[i] = H[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        // digit p of suffix s is the c-mer at symbol s + off; suffixes s in [0, n]
        u64 off = (u64)K - (u64)c * (p + 1);
        u64 cut = off < (u64)n + 1 ? off : (u64)n + 1;
        for (u64 t = 0; t < cut; ++t) h[(u32)(window_at(packed, t, bits) >> (64 - RB))]--;
        h[0] += (u32)cut;
    }
    __syncthreads();
    u32 v[DPT];
    u32 sum = 0;
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = threadIdx.x * DPT + q;
        v[q] = d < BINS ? h[d] : 0;
        sum += v[q];
    }
    u32 run = block_exclusive<NT>(sum, warp_tot);
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = threadIdx.x * DPT + q;
        if (d < BINS) digit_base[(size_t)p * BINS + d] = run;
        run += v[q];
    }
}

// ---------------------------------------------------------------------------------------------
// Round-0 key layout (u64):
//   bits [0, K*b)            the first K packed symbols of suffix s (zero padded past the text end)
//   bits [PREV_SHIFT, 64)    code of the PRECEDING symbol (text[s-1], 0 for s == 0), b+1 bits;
//                            above every sorted digit, so it rides along for free and rank0
//                            emits the BWT (stralg/bwt.c:13-20) without a gather
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int prev_shift_for(int bits) { return 64 - (bits + 1); }

// make_keys0: element j -> suffix s (short suffixes first, shortest first).
__global__ void __launch_bounds__(256) make_keys0_kernel(const u64 *__restrict__ packed, u32 n, u32 len, int K,
                                                         int bits, u64 *__restrict__ keys, u32 *__restrict__ vals) {
    const u32 nshort = (u32)K < len ? (u32)K : len;
    const int keybits = K * bits;
    const int pshift = prev_shift_for(bits);
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < len; j += stride) {
        u32 s = j < nshort ? n - (u32)j : (u32)j - nshort;
        u64 key;
        if (s == 0) {
            key = window_at(packed, 0, bits) >> (64 - keybits);
        } else {
            // one window holds the preceding symbol and the K key symbols ((K+1)*b <= 64)
            u64 win = window_at(packed, (u64)s - 1, bits);
            u64 prev_code = (win >> (64 - bits)) + 1;
            key = ((win << bits) >> (64 - keybits)) | (prev_code << pshift);
        }
        keys[j] = key;
        vals[j] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// Lazy ranks.  After round 0 only suffixes in non-singleton buckets ("active") get rank[] written;
// every other entry holds RANK_NONE.  The rank of such a suffix t is its position in the round-0
// order, recovered on demand by a binary search of its K-symbol key in the sorted key array.
// Short suffixes (window reaches the sentinel) stand first inside an equal-key run, shortest
// first, and are singletons; a long singleton stands right after them.
// ---------------------------------------------------------------------------------------------
struct LazyRank {
    const u32 *rank;
    bool sparse;           // rank[t] == RANK_NONE: not materialised (false: rank[] is complete, dense mode)
    const u64 *keys0;      // round-0 sorted keys (LSD round 0); null after the bucketed round 0
    const u32 *bstart;     // bucketed round 0: start of every bucket (2^BB + 1 entries)
    int BB;                // bucketed round 0: leading key bits that select the bucket
    const u32 *sa0;        // suffix array (round-0 order is final at singleton positions)
    const u64 *packed;
    u64 keymask;
    u32 n, len;
    int K, bits;
    int kb;                // bits of a round-0 key: K * bits, or fewer with dense keys
    DenseKey dense;        // bucketed round 0 with dense keys (round0_msd.cuh): nsym != 0
};

// the round-0 key of suffix t, as the bucketed round 0 formed it
__device__ __forceinline__ u64 round0_key_at(const LazyRank &lr, u32 t) {
    if (lr.dense.nsym) return dense_key_at(lr.packed, t, lr.bits, lr.dense);
    return window_at(lr.packed, t, lr.bits) >> (64 - lr.kb);
}

__device__ __forceinline__ u32 lazy_rank_of(const LazyRank &lr, u32 t) {
    {
        const u32 r = lr.rank[t];
        if (!lr.sparse || r != RANK_NONE) return r;
    }
    const int kb = lr.kb;
    const u64 key = round0_key_at(lr, t);
    u32 lo, hi;  // first index with key(index) >= key
    if (lr.keys0) {
        lo = 0;
        hi = lr.len;
        while (lo < hi) {
            u32 mid = lo + (hi - lo) / 2;
            if ((lr.keys0[mid] & lr.keymask) < key) lo = mid + 1;
            else hi = mid;
        }
    } else {
        // the bucket is known from the leading bits; inside it the keys come from the text
        const int rbits = kb - lr.BB;
        const u64 bid = key >> rbits;
        lo = lr.bstart[bid];
        hi = lr.bstart[bid + 1];
        if (hi - lo > 96u && rbits > 0 && rbits <= 32) {
            // the keys of a bucket spread over its remaining bits: two probes around the expected
            // position narrow the search to one or two cache lines of the suffix array
            const u64 rem = key & ((1ull << rbits) - 1ull);
            const u32 g = lo + (u32)((rem * (u64)(hi - lo)) >> rbits);
            const u32 p1 = g > lo + 32u ? g - 32u : lo;
            if (round0_key_at(lr, lr.sa0[p1]) < key) lo = p1 + 1;
            else hi = p1;
            const u32 p2 = g + 32u;
            if (p2 >= lo && p2 < hi) {
                if (round0_key_at(lr, lr.sa0[p2]) < key) lo = p2 + 1;
                else hi = p2;
            }
        }
        while (lo < hi) {
            u32 mid = lo + (hi - lo) / 2;
            u64 km = round0_key_at(lr, lr.sa0[mid]);
            if (km < key) lo = mid + 1;
            else hi = mid;
        }
    }
    // t stands in the run of rows that share its key (short suffixes first; a pair that the text decided holds
    // two long ones): the row that holds it
    while (lo + 1 < lr.len && lr.sa0[lo] != t) ++lo;
    return lo;
}

// make_keys_round: key = (rank[s] << lo_bits) | rank[s + h] for the active suffixes.
// Active suffixes share their first h symbols with another suffix, hence s + h <= n.
//
// After the bucketed round 0 the rank of a retired (singleton) suffix t is the index p of its bucket
// with sa0[p] == t: singleton positions are final, so no key has to be compared -- the VALUE t is
// looked for.  The keys of a bucket spread evenly over its remaining bits, so p lies within a few
// dozen entries of the interpolated index g; eight lanes read one 128-byte segment of the suffix
// array per step (a uint4 each), starting at g's segment and widening to both sides.  One pass over
// a warp's 32 queries = 8 rounds of 4 concurrent group scans, typically one or two steps each.
__device__ __forceinline__ u32 scan_bucket_for(const u32 *__restrict__ sa0, u32 len, u32 t, u32 blo, u32 bhi, u32 g,
                                               u32 gmask, u32 gbase, u32 lane, bool &ok) {
    const u32 seglo = blo >> 5, seghi = (bhi - 1u) >> 5, seg0 = min(max(g >> 5, seglo), seghi);
    const u32 nseg = seghi - seglo + 1u;
    ok = false;
    u32 pos = 0;
    for (u32 k = 0; k < 2u * nseg + 2u; ++k) {
        const u32 dist = (k + 1u) >> 1;
        const bool left = (k & 1u) != 0u;
        if (left ? seg0 < seglo + dist : seg0 + dist > seghi) continue;
        const u32 sg = left ? seg0 - dist : seg0 + dist;
        const u32 e0 = sg * 32u + (lane & 7u) * 4u;
        u32 v[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        if (e0 + 4u <= len) {
            const uint4 x = *(const uint4 *)(sa0 + e0);
            v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (e0 + q < len) v[q] = sa0[e0 + q];
        }
        u32 mine = 0xffffffffu;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (v[q] == t && e0 + q >= blo && e0 + q < bhi) mine = e0 + q;
        const u32 bal = (__ballot_sync(gmask, mine != 0xffffffffu) >> gbase) & 0xffu;
        if (bal) {
            pos = __shfl_sync(gmask, mine, (int)gbase + __ffs((int)bal) - 1);
            ok = true;
            break;
        }
    }
    return pos;
}

__global__ void __launch_bounds__(256) make_keys_round_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp,
                                                              u32 m, LazyRank lr, u64 h, int lo_bits,
                                                              const u8 *__restrict__ cslot,
                                                              const u32 *__restrict__ chainkey,
                                                              u64 *__restrict__ keys, u32 *__restrict__ lazy_count,
                                                              u32 *__restrict__ pv_piv,
                                                              unsigned long long *__restrict__ pv_cnt) {
    const u64 stride = (u64)gridDim.x * blockDim.x;  // a multiple of 32: warps stay together
    const u32 lane = threadIdx.x & 31u, gbase = lane & ~7u, gmask = 0xffu << gbase;
    u32 nlazy = 0;
    for (u64 base = (u64)blockIdx.x * blockDim.x + threadIdx.x - lane; base < m; base += stride) {
        const u64 j = base + lane;
        u32 s = 0, t32 = 0, blo = 0, bhi = 0, g = 0;
        u64 lo = 0;
        bool need = false;
        bool chained = false;
        if (j < m) {
            s = act[j];
            if (cslot && cslot[j]) {  // the group continues: its chain offset, when it reaches at least h
                const u32 ck = chainkey[s];
                if (ck != RANK_NONE) {
                    lo = ck;
                    chained = true;
                }
            }
            const u64 t = (u64)s + h;
            if (!chained && t < lr.len) {
                t32 = (u32)t;
                const u32 rt = lr.rank[t32];
                if (!lr.sparse || rt != RANK_NONE) {
                    lo = rt;
                } else if (lr.keys0) {
                    lo = lazy_rank_of(lr, t32);
                    ++nlazy;
                } else {
                    const int kb = lr.kb, rbits = kb - lr.BB;
                    const u64 key = round0_key_at(lr, t32);
                    const u64 bid = rbits > 0 ? key >> rbits : key;
                    blo = lr.bstart[bid];
                    bhi = lr.bstart[bid + 1];
                    const u64 rem = rbits > 0 ? key & ((1ull << rbits) - 1ull) : 0ull;
                    const u64 size = bhi - blo;
                    g = blo + (u32)(rbits <= 0 ? 0ull : rbits <= 32 ? (rem * size) >> rbits : ((rem >> (rbits - 32)) * size) >> 32);
                    need = true;
                    ++nlazy;
                }
            }
        }
        if (__any_sync(0xffffffffu, need)) {
#pragma unroll 1
            for (int r = 0; r < 8; ++r) {
                const int src = (int)gbase + r;
                const bool nd = __shfl_sync(0xffffffffu, (int)need, src) != 0;
                const u32 qt = __shfl_sync(0xffffffffu, t32, src);
                const u32 qlo = __shfl_sync(0xffffffffu, blo, src), qhi = __shfl_sync(0xffffffffu, bhi, src);
                const u32 qg = __shfl_sync(0xffffffffu, g, src);
                if (nd) {  // uniform over the group of eight
                    bool ok;
                    const u32 pos = scan_bucket_for(lr.sa0, lr.len, qt, qlo, qhi, qg, gmask, gbase, lane, ok);
                    if ((int)lane == src) lo = ok ? (u64)pos : (u64)lazy_rank_of(lr, qt);
                }
                __syncwarp();
            }
        }
        if (j < m) {
            const u32 gj = grp[j];
            keys[j] = ((u64)gj << lo_bits) | lo;
            // pivot path: the first member of a group publishes its second key and clears the group's counters
            if (pv_piv && (j == 0 || grp[j - 1] != gj)) {
                pv_piv[gj >> 1] = (u32)lo;
                pv_cnt[gj >> 1] = 0ull;
            }
        }
    }
    // ranks that had to be recovered: the host moves to complete ranks when they become many
    nlazy = __reduce_add_sync(0xffffffffu, nlazy);
    if (lane == 0 && nlazy) atomicAdd(lazy_count, nlazy);
}

// the same with complete ranks (dense mode): no recovery, no warp-cooperative scans -- a plain gather
__global__ void __launch_bounds__(256) make_keys_dense_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp, u32 m,
                                                              const u32 *__restrict__ rank, u64 h, u32 len, int lo_bits,
                                                              const u8 *__restrict__ cslot,
                                                              const u32 *__restrict__ chainkey, u64 *__restrict__ keys,
                                                              u32 *__restrict__ pv_piv,
                                                              unsigned long long *__restrict__ pv_cnt) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += stride) {
        const u32 s = act[j];
        u64 lo = 0;
        bool chained = false;
        if (cslot && cslot[j]) {
            const u32 ck = chainkey[s];
            if (ck != RANK_NONE) {
                lo = ck;
                chained = true;
            }
        }
        const u64 t = (u64)s + h;
        if (!chained && t < len) lo = rank[t];
        const u32 gj = grp[j];
        keys[j] = ((u64)gj << lo_bits) | lo;
        if (pv_piv && (j == 0 || grp[j - 1] != gj)) {
            pv_piv[gj >> 1] = (u32)lo;
            pv_cnt[gj >> 1] = 0ull;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Chain offsets.  Plain doubling orders a group by the ranks h symbols ahead, h doubling per round:
// two copies of a 6 000-symbol segment stay tied for eight rounds, all of their suffixes sorted again
// in every one of them.  But whether a group G splits at all is visible one symbol ahead: if every
// member's successor lies in ONE group G' ("G continues": all rank[s+1] equal), the members of G are
// ordered exactly like their successors in G' -- and so on along the text, until a group does not
// continue.  d(s) = 1 + d(s+1) while the group of s continues, 1 where it does not, is a property of
// the group (by induction over the chain), the members of G share at least K - 1 + d symbols, and
// ordering G by rank[s + d] is valid and reaches straight to the position where the copies part.
// A group uses its chain offset only when d >= h (the round's doubling offset), so the doubling
// invariant -- groups that stay tied share 2h symbols -- still holds and texts that chains do not
// help (a^n: the one group never "continues", its last member's successor is a singleton) run as
// before.  Three steps: chain_flags (suffix-array order: does the group continue?), chain_keys (text
// order: distance to the end of the chain, rank there), and make_keys_round takes the chain key
// where there is one.
// ---------------------------------------------------------------------------------------------
static constexpr int CF_NT = 256, CF_IPT = 8, CF_TILE = CF_NT * CF_IPT;
static constexpr int CF_STEP = CF_TILE - 512;  // a tile OWNS the groups whose head lies in its first CF_STEP elements
static constexpr u32 CHAIN_CAP = 1u << 16;     // longest offset taken from a chain (longer chains: the cap itself)

// Tiles overlap: tile t loads the list elements [t * CF_STEP, t * CF_STEP + CF_TILE) and decides for the
// groups whose head lies in the first CF_STEP of them, so a group of up to 512 members is seen as a whole by
// exactly one tile wherever it lies (a group cut by a tile border would break every chain that runs through it).
// cslot[] and cont8[] are zeroed by the caller; only "continues" is written.
__global__ void __launch_bounds__(CF_NT) chain_flags_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp, u32 m,
                                                            const u32 *__restrict__ rank, u8 *__restrict__ cslot,
                                                            u8 *__restrict__ cont8, u32 *__restrict__ ncont, u32 tile_mul) {
    __shared__ u32 hq[CF_TILE];    // rank[s + 1] of the group head at this tile-local index
    __shared__ u32 flag[CF_TILE];  // group (by head index): still "continues"
    __shared__ u32 wmax[CF_NT / 32];
    __shared__ u32 bcount;
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    // (tile_mul > 1: a sample of the tiles, evenly spaced)
    const u64 tile_base = (u64)blockIdx.x * tile_mul * CF_STEP;
    const u64 tile_end = min((u64)m, tile_base + CF_TILE);  // one past the last element loaded
    const u64 j0 = tile_base + (u64)tid * CF_IPT;
    if (tid == 0) bcount = 0;
    u32 s[CF_IPT], g[CF_IPT], q1[CF_IPT], hidx[CF_IPT];
    u32 gprev = 0;
    const bool has_prev = j0 > 0 && j0 < m;
    if (has_prev) gprev = grp[j0 - 1];
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q) {
        const u64 j = j0 + q;
        s[q] = j < m ? act[j] : 0u;
        g[q] = j < m ? grp[j] : 0u;
    }
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q) q1[q] = j0 + q < m ? rank[s[q] + 1u] : RANK_NONE;
    // tile-local index + 1 of the latest group head at or before each element (0: none in this thread yet)
    u32 run = 0;
    {
        u32 pg = gprev;
#pragma unroll
        for (int q = 0; q < CF_IPT; ++q) {
            const u64 j = j0 + q;
            const bool head = j < m && (j == 0 || g[q] != pg);
            if (head) run = (u32)(j - tile_base) + 1u;
            hidx[q] = run;
            pg = g[q];
        }
    }
    const u32 ex = warp_inclusive(run, MaxOp());
    if (lane == 31) wmax[warp] = ex;
    u32 pre = warp_exclusive(ex, run, MaxOp(), 0u);
    __syncthreads();
    for (u32 w = 0; w < warp; ++w) pre = max(pre, wmax[w]);
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q)
        if (hidx[q] == 0) hidx[q] = pre;  // 0: the group began before this tile
    // heads publish their successor's rank
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q) {
        const u64 j = j0 + q;
        if (j < m && hidx[q] == (u32)(j - tile_base) + 1u) {
            hq[hidx[q] - 1u] = q1[q];
            flag[hidx[q] - 1u] = q1[q] != RANK_NONE ? 1u : 0u;
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q) {
        const u64 j = j0 + q;
        if (j < m && hidx[q] && q1[q] != hq[hidx[q] - 1u]) flag[hidx[q] - 1u] = 0u;
    }
    // the last group loaded must end inside the loaded range
    if (tile_end > j0 && tile_end - 1 < j0 + CF_IPT) {
        const int q = (int)(tile_end - 1 - j0);
        if (tile_end < m && grp[tile_end] == g[q] && hidx[q]) flag[hidx[q] - 1u] = 0u;
    }
    __syncthreads();
    u32 mine = 0;
#pragma unroll
    for (int q = 0; q < CF_IPT; ++q) {
        const u64 j = j0 + q;
        // owned: the head lies in the first CF_STEP elements of the tile
        if (j < m && hidx[q] && hidx[q] <= (u32)CF_STEP && flag[hidx[q] - 1u]) {
            cslot[j] = 1;
            cont8[s[q]] = 1;
            ++mine;
        }
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if (lane == 0 && mine) atomicAdd(&bcount, mine);
    __syncthreads();
    if (tid == 0 && bcount) atomicAdd(ncont, bcount);
}

// text order: for every position s whose group continues, e = the first position >= s whose group does
// not, d = e - s + 1 (capped); chainkey[s] = rank of suffix s + d when d >= h, RANK_NONE otherwise
static constexpr int CK_NT = 256, CK_BPT = 16, CK_TILE = CK_NT * CK_BPT;

__global__ void __launch_bounds__(CK_NT) chain_keys_kernel(const u8 *__restrict__ cont8, u32 len, LazyRank lr, u64 h,
                                                           u32 *__restrict__ chainkey, u32 *__restrict__ lazy_count) {
    __shared__ u32 RK[CK_TILE];       // rank of suffix e + 1 for chain ends e inside the tile
    __shared__ u32 wmin[CK_NT / 32];
    __shared__ u32 beyond[2];         // first position >= end of tile whose group does not continue; its successor's rank
    __shared__ u8 lastb[CK_NT];       // last byte of every thread's chunk
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 T0 = (u64)blockIdx.x * CK_TILE;
    const u64 p0 = T0 + (u64)tid * CK_BPT;
    // (cont8 is padded with zeros far beyond len: no bounds checks on the loads)
    const uint4 v = *(const uint4 *)(cont8 + p0);
    const u32 w[4] = {v.x, v.y, v.z, v.w};
    u32 bits = 0;  // bit i: the group of position p0 + i continues
#pragma unroll
    for (int i = 0; i < CK_BPT; ++i) bits |= ((w[i >> 2] >> (8 * (i & 3))) & 1u) << i;
    lastb[tid] = (u8)((bits >> (CK_BPT - 1)) & 1u);
    const u32 any = __syncthreads_or((int)bits);
    if (!any) return;  // nothing continues in this tile
    // first position of the chunk (relative to T0) whose bit is clear, or none
    const u32 zeros = ~bits & 0xffffu;
    const u32 NONEPOS = 0xffffffffu;
    u32 firstz = zeros ? tid * CK_BPT + (u32)(__ffs((int)zeros) - 1) : NONEPOS;
    // suffix-min over the threads after this one
    u32 sm = firstz;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_down_sync(0xffffffffu, sm, o);
        if (lane + (u32)o < 32u) sm = min(sm, t);
    }
    if (lane == 0) wmin[warp] = sm;
    u32 after = __shfl_down_sync(0xffffffffu, sm, 1);  // min over the later threads of this warp
    if (lane == 31) after = NONEPOS;
    __syncthreads();
    for (u32 ww = warp + 1; ww < CK_NT / 32; ++ww) after = min(after, wmin[ww]);
    // the chain that runs out of the tile: warp 0 looks for its end (at most CHAIN_CAP positions ahead)
    if (warp == 0) {
        u32 found = NONEPOS;
        if (lastb[CK_NT - 1]) {
            for (u32 it = 0; it < CHAIN_CAP / 256u + 1u && found == NONEPOS; ++it) {
                const u64 at = T0 + CK_TILE + (u64)(it * 32u + lane) * 8u;
                const u64 x = *(const u64 *)(cont8 + at);
                const u64 z = ~x & 0x0101010101010101ull;
                const u32 b = __ballot_sync(0xffffffffu, z != 0);
                if (b) {
                    const int l0 = __ffs((int)b) - 1;
                    const u64 zz = __shfl_sync(0xffffffffu, z, l0);
                    found = (u32)(CK_TILE + (it * 32u + (u32)l0) * 8u + (u32)((__ffsll((long long)zz) - 1) >> 3));
                }
            }
        }
        if (lane == 0) {
            beyond[0] = found;  // relative to T0; NONEPOS: the chain is longer than the cap
            u32 rk = RANK_NONE;
            if (found != NONEPOS && T0 + found + 1 < lr.len) {
                const u32 t = (u32)(T0 + found + 1);
                if (lr.sparse && lr.rank[t] == RANK_NONE) atomicAdd(lazy_count, 1u);
                rk = lazy_rank_of(lr, t);
            }
            beyond[1] = rk;
        }
    }
    // chain ends inside the chunk: position e with a clear bit whose predecessor's bit is set
    {
        const u32 prevbit = tid ? (u32)lastb[tid - 1] : 0u;
        u32 ends = zeros & ((bits << 1) | prevbit);
        u32 nl = 0;
        while (ends) {
            const int i = __ffs((int)ends) - 1;
            ends &= ends - 1;
            const u64 e = p0 + (u64)i;
            u32 rk = RANK_NONE;
            if (e + 1 < lr.len) {
                if (lr.sparse && lr.rank[e + 1] == RANK_NONE) ++nl;
                rk = lazy_rank_of(lr, (u32)(e + 1));
            }
            RK[tid * CK_BPT + i] = rk;
        }
        if (nl) atomicAdd(lazy_count, nl);
    }
    __syncthreads();
    if (!bits) return;
    const u32 bz = beyond[0];
    u32 nextz = after != NONEPOS ? after : bz;  // first clear position after this chunk (relative to T0)
    // walk the chunk backwards
    u32 out[CK_BPT];
#pragma unroll
    for (int i = CK_BPT - 1; i >= 0; --i) {
        const u32 rel = tid * CK_BPT + (u32)i;
        out[i] = RANK_NONE;
        if ((bits >> i) & 1u) {
            u32 d, key;
            if (nextz == NONEPOS || nextz - rel + 1u > CHAIN_CAP) {
                // capped: the target is itself inside the chain (an active suffix, its rank is materialised)
                d = CHAIN_CAP;
                key = lr.rank[T0 + rel + d];
            } else {
                d = nextz - rel + 1u;
                key = nextz < (u32)CK_TILE ? RK[nextz] : beyond[1];
            }
            if ((u64)d >= h) out[i] = key;
        } else {
            nextz = rel;
        }
    }
#pragma unroll
    for (int i = 0; i < CK_BPT; ++i)
        if ((bits >> i) & 1u) chainkey[p0 + i] = out[i];
}

// ---------------------------------------------------------------------------------------------
// rank_kernel: on a sorted (key, suffix) list of m elements.
//   group(key) = key >> gs   (gs >= 64: one group starting at SA index 0 -- round 0)
//   jb = first index of the element's group, jh = first index with the element's full key
//   SA position of element j      = hi + (j - jb)      (hi = group value = SA index of the bucket)
//   new rank of its suffix        = hi + (jh - jb)
// Round 0 (K0 > 0): suffixes whose K-window reaches the sentinel are forced into singleton
// buckets (they were fed first, so they already stand ahead of their padded-equal neighbours);
// ranks are written for active suffixes only (all suffixes when scatter_all), BWT rows come from
// the key's top bits.  Later rounds write SA, rank and BWT rows of every active suffix.
// headbits: bit (j & 7) of byte j >> 3 is set when j starts a new bucket.
// ---------------------------------------------------------------------------------------------
static constexpr int RK_NT = 256;
static constexpr int RK_IPT = 8;
static constexpr int RK_TILE = RK_NT * RK_IPT;

__device__ __forceinline__ u64 group_of(u64 key, int gs) { return gs >= 64 ? 0ull : key >> gs; }

// first index f <= start such that ((keys[f..start] & mask) >> gs) all equal x
// Warp-cooperative (all 32 lanes of one warp call it with the same arguments; the result is uniform).
// The list is sorted, so "key == x" is false ... false true ... true on [0, start]: one step probes
// the 32 positions start - 2^l at once, the following steps split the remaining range 33 ways, so a
// run of a billion equal keys costs seven dependent round trips instead of sixty.
__device__ u32 gallop_first_equal(const u64 *__restrict__ keys, u32 start, u64 x, int gs, u64 mask) {
    const u32 lane = threadIdx.x & 31u;
    // step 1: exponentially spaced probes below `start`
    const u64 off = 1ull << lane;  // 2^lane (lane 31: 2^31)
    bool eq = false;
    if (off <= (u64)start) eq = ((keys[(u64)start - off] & mask) >> gs) == x;
    const u32 eqm = __ballot_sync(0xffffffffu, eq);
    // lanes 0 .. t-1 see equal keys, lane t is the first that does not (or runs below index 0)
    const int t = __ffs((int)~eqm) - 1;  // ~eqm is non-zero unless all 32 probes matched
    u64 good = t > 0 ? (u64)start - (1ull << (t - 1)) : (u64)start;           // known equal
    int64_t bad = (t >= 0 && (1ull << t) <= (u64)start) ? (int64_t)((u64)start - (1ull << t)) : -1;  // known different (or -1)
    if (t < 0) {  // every probe matched (start >= 2^31): the run begins somewhere in [0, start - 2^31]
        good = (u64)start - (1ull << 31);
        bad = -1;
    }
    // step 2: 33-way splits of (bad, good)
    while ((int64_t)good - bad > 1) {
        const u64 span = (u64)((int64_t)good - bad);  // candidates bad+1 .. good-1 are unknown
        const u64 idx = (u64)(bad + 1) + (span - 1) * (u64)lane / 32u;  // lane 0: bad + 1, spread up to good - 1
        const bool e2 = idx < good && ((keys[idx] & mask) >> gs) == x;
        const u32 m2 = __ballot_sync(0xffffffffu, e2);
        if (m2) {
            const int f = __ffs((int)m2) - 1;  // first lane that sees x: the run starts at or before its index
            const u64 gi = (u64)(bad + 1) + (span - 1) * (u64)f / 32u;
            if (f > 0) bad = (int64_t)((u64)(bad + 1) + (span - 1) * (u64)(f - 1) / 32u);
            good = gi;
        } else {
            // no probe below `good` sees x: everything up to the last probe is different
            bad = (int64_t)((u64)(bad + 1) + (span - 1) * 31u / 32u);
        }
    }
    return (u32)good;
}

struct RankArgs {
    const u64 *keys;
    const u32 *vals;
    u32 m;
    int gs;          // group shift (>= 64 in round 0)
    u64 keymask;     // bits that take part in comparisons
    int K0;          // round 0: symbols in the key; 0 in later rounds
    u32 n;
    u32 *rank;
    u32 *newgrp;     // [m] by sorted index: the new rank (= first row of the element's new group)
    int scatter_all; // round 0, dense mode: write every rank, touch nothing else
    u32 *sa_out;     // later rounds
    u8 *headbits;
    u8 *bwt;         // optional
    int prev_shift;  // round 0: where the preceding code sits in the key
    const u64 *packed;
    int bits;
    u32 *primary;
    int always_write;  // later rounds: store every rank (the old identifier of a group need not be its head row)
};

__global__ void __launch_bounds__(RK_NT) rank_kernel(RankArgs a) {
    __shared__ u32 warp_s[RK_NT / 32], warp_b[RK_NT / 32];
    __shared__ u32 carry_s, carry_b;
    const u64 *__restrict__ keys = a.keys;
    const u32 *__restrict__ vals = a.vals;
    const u32 m = a.m, n = a.n;
    const int gs = a.gs, K0 = a.K0;
    const u64 mask = a.keymask;
    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 tile_base = (u64)blockIdx.x * RK_TILE;
    const u64 j0 = tile_base + (u64)tid * RK_IPT;

    u64 k[RK_IPT];
    u32 s[RK_IPT];
    u64 kprev = 0, knext = 0;
    u32 sprev = 0, snext = 0;
    // (lists made by the pivot path start at any element of a buffer: vector loads only where they are aligned)
    if (j0 + RK_IPT <= m && ((((uintptr_t)(keys + j0)) | ((uintptr_t)(vals + j0))) & 15) == 0) {
        const uint4 *kp = (const uint4 *)(keys + j0);
#pragma unroll
        for (int q = 0; q < RK_IPT / 2; ++q) {
            uint4 v = kp[q];
            k[2 * q] = ((u64)v.y << 32) | v.x;
            k[2 * q + 1] = ((u64)v.w << 32) | v.z;
        }
        const uint4 *vp = (const uint4 *)(vals + j0);
#pragma unroll
        for (int q = 0; q < RK_IPT / 4; ++q) {
            uint4 v = vp[q];
            s[4 * q] = v.x; s[4 * q + 1] = v.y; s[4 * q + 2] = v.z; s[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < RK_IPT; ++q) {
            k[q] = j0 + q < m ? keys[j0 + q] : 0;
            s[q] = j0 + q < m ? vals[j0 + q] : 0;
        }
    }
    if (j0 > 0 && j0 < m) {
        kprev = keys[j0 - 1];
        sprev = vals[j0 - 1];
    }
    const bool has_next = j0 + RK_IPT < m;
    if (has_next) {
        knext = keys[j0 + RK_IPT];
        snext = vals[j0 + RK_IPT];
    }

    // ---- flags and thread-local running heads (tile-local index + 1; 0 = none yet) ----
    u32 hs_idx[RK_IPT], hb_idx[RK_IPT];
    u32 run_s = 0, run_b = 0;
    u32 bits = 0;
    {
        u64 pk = kprev;
        u32 ps = sprev;
#pragma unroll
        for (int q = 0; q < RK_IPT; ++q) {
            u64 j = j0 + q;
            bool valid = j < m;
            bool hs = (j == 0) || ((k[q] & mask) != (pk & mask));
            bool hb = (j == 0) || (group_of(k[q] & mask, gs) != group_of(pk & mask, gs));
            if (K0 > 0 && j > 0) {
                bool sh_cur = (u64)s[q] + (u64)K0 > (u64)n;
                bool sh_prev = (u64)ps + (u64)K0 > (u64)n;
                hs = hs || sh_cur || sh_prev;
            }
            if (valid && hs) {
                run_s = (u32)(j - tile_base) + 1;
                bits |= 1u << q;
            }
            if (valid && hb) run_b = (u32)(j - tile_base) + 1;
            hs_idx[q] = run_s;
            hb_idx[q] = run_b;
            pk = k[q];
            ps = s[q];
        }
    }
    // is the element after this thread's last one a bucket head? (end of list counts as one)
    bool next_head = true;
    if (has_next) {
        next_head = (knext & mask) != (k[RK_IPT - 1] & mask);
        if (K0 > 0)
            next_head = next_head || ((u64)snext + (u64)K0 > (u64)n) || ((u64)s[RK_IPT - 1] + (u64)K0 > (u64)n);
    }
    if (!a.scatter_all && j0 < m) a.headbits[j0 >> 3] = (u8)bits;

    // ---- carry-in for the tile (only when its first element does not start a bucket): the first
    // warp looks for the head of the run that reaches into the tile ----
    if (warp == 0) {
        u32 cs = 0, cb = 0;  // global index of the head for the tile's first element
        if (tile_base > 0 && tile_base < m) {  // uniform over the block
            const bool first_is_hs = __shfl_sync(0xffffffffu, (int)(bits & 1u), 0) != 0;
            const bool first_is_hb = __shfl_sync(0xffffffffu, (int)(hb_idx[0] != 0), 0) != 0;
            const u64 k0 = __shfl_sync(0xffffffffu, k[0], 0);
            if (!first_is_hs) {
                u32 f = gallop_first_equal(keys, (u32)tile_base, k0 & mask, 0, mask);
                if (K0 > 0) {
                    // short suffixes stand first inside an equal-key run and are singletons
                    while ((u64)vals[f] + (u64)K0 > (u64)n) ++f;
                }
                cs = f;
            }
            if (!first_is_hb && gs < 64) cb = gallop_first_equal(keys, (u32)tile_base, (k0 & mask) >> gs, gs, mask);
        }
        if (lane == 0) {
            carry_s = cs;
            carry_b = cb;
        }
    }

    // ---- block-wide "last head so far" (max-scan; indices grow with position) ----
    const u32 ex_s = warp_inclusive(run_s, MaxOp()), ex_b = warp_inclusive(run_b, MaxOp());
    if (lane == 31) {
        warp_s[warp] = ex_s;
        warp_b[warp] = ex_b;
    }
    u32 pre_s = warp_exclusive(ex_s, run_s, MaxOp(), 0u), pre_b = warp_exclusive(ex_b, run_b, MaxOp(), 0u);
    __syncthreads();
    for (unsigned w = 0; w < warp; ++w) {
        pre_s = max(pre_s, warp_s[w]);
        pre_b = max(pre_b, warp_b[w]);
    }
    const u32 cs = carry_s, cb = carry_b;

    u64 bwt8 = 0;
#pragma unroll
    for (int q = 0; q < RK_IPT; ++q) {
        u64 j = j0 + q;
        if (j >= m) break;
        u32 ls = hs_idx[q] ? hs_idx[q] : pre_s;
        u32 lb = hb_idx[q] ? hb_idx[q] : pre_b;
        u64 jh = ls ? tile_base + ls - 1 : (u64)cs;
        u64 jb = gs >= 64 ? 0ull : (lb ? tile_base + lb - 1 : (u64)cb);
        u64 hi = group_of(k[q] & mask, gs);
        u32 newrank = (u32)(hi + (jh - jb));
        if (K0 > 0) {
            // round 0
            bool head_here = (bits >> q) & 1u;
            bool head_after = q + 1 < RK_IPT ? (j + 1 >= m || ((bits >> (q + 1)) & 1u)) : next_head;
            bool active = !(head_here && head_after);
            if (a.scatter_all) {
                a.rank[s[q]] = newrank;
            } else {
                if (active) a.rank[s[q]] = newrank;
                a.newgrp[j] = newrank;
                bwt8 |= ((k[q] >> a.prev_shift) & 0xffull) << (8 * q);
                if (s[q] == 0) *a.primary = (u32)j;
            }
        } else {
            u32 pos = (u32)(hi + (j - jb));
            // every member holds the group head as its rank: the members that stay in front keep it
            if (a.always_write || newrank != (u32)hi) a.rank[s[q]] = newrank;
            a.newgrp[j] = newrank;
            a.sa_out[pos] = s[q];
            if (s[q] == 0) {
                *a.primary = pos;
                if (a.bwt) a.bwt[pos] = 0;
            } else if (a.bwt) {
                u64 bitpos = (u64)(s[q] - 1) * a.bits;
                u64 w = a.packed[bitpos >> 6];
                a.bwt[pos] = (u8)(((w >> (64 - a.bits - (unsigned)(bitpos & 63))) & ((1u << a.bits) - 1u)) + 1u);
            }
        }
    }
    if (K0 > 0 && !a.scatter_all && a.bwt && j0 < m) {
        // the BWT buffer is padded to a multiple of 64 rows, so the 8-byte store is always in range
        *(u64 *)(a.bwt + j0) = bwt8;
    }
}

// ---------------------------------------------------------------------------------------------
// Active-set compaction from the head bitmap: element j stays active unless it is a singleton
// (head[j] && (j + 1 == m || head[j + 1])).
// ---------------------------------------------------------------------------------------------
static constexpr int CP_NT = 256;
static constexpr int CP_TILE = CP_NT * 64;

__device__ __forceinline__ u64 active_mask(const u8 *__restrict__ headbits, u64 word, u32 m) {
    // headbits is padded to a multiple of 8 bytes plus one extra word
    const u64 *hb = (const u64 *)headbits;
    u64 base = word * 64;
    if (base >= m) return 0;
    u64 H = hb[word];
    u64 next = hb[word + 1];
    u64 valid = (m - base >= 64) ? ~0ull : ((1ull << (m - base)) - 1ull);
    H &= valid;
    // head of j+1: shift right by one, pull in bit 0 of the next word
    u64 Hn = (H >> 1) | (next << 63);
    // position m (one past the end) counts as a head
    u64 last = m - 1 - base;
    if (m - base <= 64) {
        Hn &= ~(1ull << last);
        Hn |= (1ull << last);
    }
    u64 singleton = H & Hn;
    return (~singleton) & valid;
}

// bits of a plain bitmap (bit per element, padded like headbits)
__device__ __forceinline__ u64 raw_mask(const u8 *__restrict__ bits, u64 word, u32 m) {
    const u64 base = word * 64;
    if (base >= m) return 0;
    const u64 valid = (m - base >= 64) ? ~0ull : ((1ull << (m - base)) - 1ull);
    return ((const u64 *)bits)[word] & valid;
}

// a block takes `sub` consecutive sub-tiles of CP_NT words (long bitmaps: fewer, larger tiles for the scan)
template <bool RAW>
__global__ void __launch_bounds__(CP_NT) count_active_kernel(const u8 *__restrict__ headbits, u32 m, u32 sub,
                                                             u32 *__restrict__ tile_counts) {
    __shared__ u32 wsum[CP_NT / 32];
    u32 c = 0;
    for (u32 q = 0; q < sub; ++q) {
        const u64 word = ((u64)blockIdx.x * sub + q) * CP_NT + threadIdx.x;
        c += __popcll(RAW ? raw_mask(headbits, word, m) : active_mask(headbits, word, m));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane_id() == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
        for (int w = 0; w < CP_NT / 32; ++w) t += wsum[w];
        tile_counts[blockIdx.x] = t;
    }
}

// RAW: `headbits` is the bitmap of the elements to keep (bit per element), not a head bitmap
template <bool RAW>
__global__ void __launch_bounds__(CP_NT) scatter_active_kernel(const u8 *__restrict__ headbits,
                                                               const u32 *__restrict__ vals,
                                                               const u32 *__restrict__ grp_in, u32 m, u32 sub,
                                                               const u32 *__restrict__ tile_offsets,
                                                               u32 *__restrict__ out, u32 *__restrict__ grp_out) {
    __shared__ u32 wsum[CP_NT / 32];
    u32 base = tile_offsets[blockIdx.x];
    const u32 lane = lane_id();
    const u32 lt = lanemask_lt();
    for (u32 q = 0; q < sub; ++q) {
        const u64 word = ((u64)blockIdx.x * sub + q) * CP_NT + threadIdx.x;
        const u64 mask = RAW ? raw_mask(headbits, word, m) : active_mask(headbits, word, m);
        const u32 c = __popcll(mask);
        u32 total;
        const u32 o = base + block_exclusive<CP_NT>(c, wsum, &total);
        base += total;
        __syncthreads();  // wsum is rewritten by the next sub-tile
        if (!__any_sync(0xffffffffu, mask != 0)) continue;  // (most warps of a sparse bitmap)
        // the warp walks its 32 words together: lane l takes element l (then 32 + l) of the word, so the
        // reads of `vals` and the writes of the survivors are coalesced
        const u64 word0 = word - lane;
#pragma unroll 4
        for (int w = 0; w < 32; ++w) {
            const u64 mw = __shfl_sync(0xffffffffu, mask, w);
            const u32 ow = __shfl_sync(0xffffffffu, o, w);
            if (!mw) continue;
            const u64 bw = (word0 + (u64)w) * 64;
            const u32 lo = (u32)mw, hi = (u32)(mw >> 32);
            if ((lo >> lane) & 1u) {
                const u32 at = ow + (u32)__popc(lo & lt);
                out[at] = vals[bw + lane];
                grp_out[at] = grp_in[bw + lane];
            }
            if ((hi >> lane) & 1u) {
                const u32 at = ow + (u32)__popc(lo) + (u32)__popc(hi & lt);
                out[at] = vals[bw + 32 + lane];
                grp_out[at] = grp_in[bw + 32 + lane];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Small groups of a doubling round, ordered where they stand.  The list is grouped, a group's members
// occupy consecutive slots AND consecutive suffix-array rows, and most groups of a text with repeats are
// tiny (two copies of a segment: pairs).  A radix sort of (group, rank) keys moves every element eight
// times to settle an order that each group can find among its own few members.  A tile owns RS_STEP
// consecutive slots and loads RS_HALO more on both sides, so every group of up to RS_GMAX members that
// touches its slots is seen whole (a group that straddles two tiles is ordered by both, identically;
// each writes only the slots it owns): a member's new place is the group's first slot plus the members
// with a smaller key plus the equal ones before it.  Written per owned slot: the suffix now standing
// there, its new group head (= new rank), the bitmaps "starts a group" and "not handled here" (larger
// groups, groups cut by the window: they go through the radix sort as before); per suffix: its row in
// the suffix array and its rank where it changed.
// ---------------------------------------------------------------------------------------------
static constexpr int RS_NT = 256, RS_IPT = 10, RS_WIN = RS_NT * RS_IPT;  // 2560 slots loaded
static constexpr int RS_HALO = 512, RS_STEP = RS_WIN - 2 * RS_HALO;      // 1536 slots owned (24 words of 64)
static constexpr u32 RS_GMAX = 32;

struct SmallArgs {
    const u32 *act, *grp;
    const u64 *keys;
    u32 m;
    int lo_bits;
    u32 *sa, *rank;
    u32 *vals_out, *newgrp_out;
    u64 *headbits64, *notdone64;
    u32 *primary;
    u32 *handled;  // [1] slots handled by this path
    int always_write;  // store every rank (see RankArgs)
};

__global__ void __launch_bounds__(RS_NT) round_small_kernel(SmallArgs a) {
    __shared__ u32 lo_s[RS_WIN];
    __shared__ u32 glast_s[RS_WIN];  // by window index of a group head: last window index of the group
    __shared__ u32 gok_s[RS_WIN];    // by window index of a group head: the group lies inside the window
    __shared__ unsigned long long hw_s[RS_STEP / 64], dw_s[RS_STEP / 64];
    __shared__ u32 wmax[RS_NT / 32];
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 own0 = (u64)blockIdx.x * RS_STEP, own1 = min((u64)a.m, own0 + RS_STEP);
    const u64 w0 = own0 >= (u64)RS_HALO ? own0 - RS_HALO : 0ull, w1 = min((u64)a.m, own0 + RS_STEP + RS_HALO);
    const u32 wn = (u32)(w1 - w0);
    const u32 i0 = tid * RS_IPT;
    const u32 lomask = a.lo_bits >= 32 ? 0xffffffffu : ((1u << a.lo_bits) - 1u);
    u32 s[RS_IPT], g[RS_IPT], lo[RS_IPT], hidx[RS_IPT];
    u32 gprev = 0;
    const bool has_prev = i0 < wn && w0 + i0 > 0;
    if (has_prev) gprev = a.grp[w0 + i0 - 1];
#pragma unroll
    for (int q = 0; q < RS_IPT; ++q) {
        const u32 i = i0 + q;
        s[q] = i < wn ? a.act[w0 + i] : 0u;
        g[q] = i < wn ? a.grp[w0 + i] : 0u;
        lo[q] = i < wn ? (u32)a.keys[w0 + i] & lomask : 0u;
        if (i < wn) {
            lo_s[i] = lo[q];
            glast_s[i] = 0;
            gok_s[i] = 0;
        }
    }
    if (tid < RS_STEP / 64) {
        hw_s[tid] = 0ull;
        dw_s[tid] = 0ull;
    }
    // window index + 1 of the latest group head at or before each element (0: the group began before the window)
    u32 run = 0;
    {
        u32 pg = gprev;
#pragma unroll
        for (int q = 0; q < RS_IPT; ++q) {
            const u32 i = i0 + q;
            const bool head = i < wn && (w0 + i == 0 || g[q] != pg);
            if (head) run = i + 1u;
            hidx[q] = run;
            pg = g[q];
        }
    }
    const u32 ex = warp_inclusive(run, MaxOp());
    if (lane == 31) wmax[warp] = ex;
    u32 pre = warp_exclusive(ex, run, MaxOp(), 0u);
    __syncthreads();
    for (u32 w = 0; w < warp; ++w) pre = max(pre, wmax[w]);
#pragma unroll
    for (int q = 0; q < RS_IPT; ++q)
        if (hidx[q] == 0) hidx[q] = pre;
#pragma unroll
    for (int q = 0; q < RS_IPT; ++q) {
        const u32 i = i0 + q;
        if (i < wn && hidx[q]) {
            if (hidx[q] == i + 1u) gok_s[i] = 1u;
            atomicMax(&glast_s[hidx[q] - 1u], i);
        }
    }
    __syncthreads();
    // the last group loaded must end inside the window
    if (wn > i0 && wn - 1u < i0 + RS_IPT) {
        const int q = (int)(wn - 1u - i0);
        if (w1 < a.m && a.grp[w1] == g[q] && hidx[q]) gok_s[hidx[q] - 1u] = 0u;
    }
    __syncthreads();
#pragma unroll 1
    for (int q = 0; q < RS_IPT; ++q) {
        const u32 i = i0 + q;
        if (i >= wn || !hidx[q]) continue;
        const u32 h = hidx[q] - 1u;
        if (!gok_s[h]) continue;
        const u32 size = glast_s[h] - h + 1u;
        if (size > RS_GMAX) continue;
        u32 smaller = 0, eq_before = 0;
        const u32 mine = lo[q];
        for (u32 k = h; k < h + size; ++k) {
            const u32 lk = lo_s[k];
            smaller += lk < mine ? 1u : 0u;
            eq_before += (lk == mine && k < i) ? 1u : 0u;
        }
        const u64 slot = w0 + h + smaller + eq_before;
        if (slot < own0 || slot >= own1) continue;
        const u32 newrank = g[q] + smaller, row = newrank + eq_before;
        a.vals_out[slot] = s[q];
        a.newgrp_out[slot] = newrank;
        a.sa[row] = s[q];
        if (smaller || a.always_write) a.rank[s[q]] = newrank;  // (members that stay in front keep the group head as their rank)
        if (s[q] == 0) *a.primary = row;
        const u32 bit = (u32)(slot - own0);
        atomicOr(&dw_s[bit >> 6], 1ull << (bit & 63u));
        if (eq_before == 0) atomicOr(&hw_s[bit >> 6], 1ull << (bit & 63u));
    }
    __syncthreads();
    if (tid < RS_STEP / 64) {
        const u64 base = own0 + (u64)tid * 64;
        if (base < a.m) {
            const u64 valid = a.m - base >= 64 ? ~0ull : ((1ull << (a.m - base)) - 1ull);
            const u64 done = dw_s[tid];
            // a slot not handled here counts as a group of its own for the compaction of THIS path's survivors
            a.headbits64[base >> 6] = (u64)hw_s[tid] | ~done;
            a.notdone64[base >> 6] = ~done & valid;
            const u32 c = (u32)__popcll(done);
            if (c) atomicAdd(a.handled, c);
        }
    }
}

// bitmap -> compacted (key, value) pairs in list order (the elements the small-group path left alone)
__global__ void __launch_bounds__(CP_NT) scatter_pairs_kernel(const u8 *__restrict__ bits, const u64 *__restrict__ keys,
                                                              const u32 *__restrict__ vals, u32 m, u32 sub,
                                                              const u32 *__restrict__ tile_offsets,
                                                              u64 *__restrict__ kout, u32 *__restrict__ vout) {
    __shared__ u32 wsum[CP_NT / 32];
    u32 base = tile_offsets[blockIdx.x];
    const u32 lane = lane_id();
    const u32 lt = lanemask_lt();
    for (u32 q = 0; q < sub; ++q) {
        const u64 word = ((u64)blockIdx.x * sub + q) * CP_NT + threadIdx.x;
        const u64 mask = raw_mask(bits, word, m);
        const u32 c = __popcll(mask);
        u32 total;
        const u32 o = base + block_exclusive<CP_NT>(c, wsum, &total);
        base += total;
        __syncthreads();
        if (!__any_sync(0xffffffffu, mask != 0)) continue;
        const u64 word0 = word - lane;
#pragma unroll 4
        for (int w = 0; w < 32; ++w) {
            const u64 mw = __shfl_sync(0xffffffffu, mask, w);
            const u32 ow = __shfl_sync(0xffffffffu, o, w);
            if (!mw) continue;
            const u64 bw = (word0 + (u64)w) * 64;
            const u32 lo = (u32)mw, hi = (u32)(mw >> 32);
            if ((lo >> lane) & 1u) {
                const u32 at = ow + (u32)__popc(lo & lt);
                kout[at] = keys[bw + lane];
                vout[at] = vals[bw + lane];
            }
            if ((hi >> lane) & 1u) {
                const u32 at = ow + (u32)__popc(lo) + (u32)__popc(hi & lt);
                kout[at] = keys[bw + 32 + lane];
                vout[at] = vals[bw + 32 + lane];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Pivot path of a doubling round: large groups that mostly stay together.  On periodic texts (a^n, a
// tiled block, a Fibonacci string) the active list is a few giant groups, and in a round nearly all
// members of a group carry the SAME second key -- the rank of the one group their successors share --
// while a minority (the suffixes whose successor has already been decided) leaves.  Sorting all of them
// by a 64-bit key, eight passes, settles nothing for the majority.  Here every group is split three
// ways around the second key P of its first member:
//     L = {key < P}   E = {key == P}   R = {key > P}
// E keeps its order and slides behind L in one stable compaction (rows head + |L| ..), it stays one
// group; only L and R go through the radix sort, L with the group's head as first key and R with
// head + |L| + |E| -- the row where R starts -- so that rank_kernel places both where they belong.
//
// Ranks are group identifiers: rank[] of a member is ANY row inside its group's row range, the same
// for all members (the head row wherever another kernel writes it); that is all a second key has to
// be.  An E group whose old identifier still lies in its new, smaller range keeps it -- no rank store
// for the majority; otherwise it takes the end of its range that lies away from the cut, so a group
// that keeps losing members on one side (periodic texts: the shorter suffixes, in front) is renamed
// once.
//
// Per-group data lives in two tables indexed by (head row of the group) / 2 -- groups own at least
// two rows, so the index is unique, and every member knows it without looking for the head of its
// group in the list: the pivot key (written by the head's thread when the round keys are made) and
// the counters |E| << 32 | |L| (zeroed there, accumulated by the classification).  Two passes over
// the list: classify (classes, counters, E bitmap, per-tile E counts), apply (rows, identifiers, the
// E part of the NEXT list written in place at the E members' prefix count -- no separate compaction).
// ---------------------------------------------------------------------------------------------
static constexpr int PV_NT = 256, PV_IPT = 8, PV_TILE = PV_NT * PV_IPT;

struct PivotArgs {
    const u32 *act;               // values (suffixes) of the list
    u64 *keys;                    // its round keys: [first row of the group : lo_bits | second key : lo_bits]; R members
                                  // get their first key rewritten
    u32 m;
    int lo_bits;
    u32 *piv;                     // by head row >> 1: the pivot key
    unsigned long long *cnt64;    // by head row >> 1: |E| << 32 | |L|
    u8 *ebits8, *lbits8, *rbits8; // bit per list element: its class
    u32 *tile_e;                  // [tiles + 1] E members per tile (exclusive offsets after the scan)
    u32 *totals;                  // [0] E members (written by the scan), [1] L members (accumulated here)
    u32 *sa, *rank, *primary;
    u32 *out_act, *out_grp;       // where the E part goes in the next list
    u32 *singles;                 // [1] E groups of one member (final; they are taken out of the next list afterwards)
    u32 *dropbits;                // bit per entry of the next list: such a member stands there
    u32 out_base;                 // entry of the next list where this list's E part begins
};

// eight consecutive words of a list (vector loads where the tile is full)
__device__ __forceinline__ void pv_load8(const u32 *__restrict__ p, u64 j0, u32 m, u32 (&v)[PV_IPT]) {
    if (j0 + PV_IPT <= m && ((((uintptr_t)(p + j0)) & 15) == 0)) {
        const uint4 x = *(const uint4 *)(p + j0), y = *(const uint4 *)(p + j0 + 4);
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    } else {
#pragma unroll
        for (int q = 0; q < PV_IPT; ++q) v[q] = j0 + q < m ? p[j0 + q] : 0u;
    }
}
// eight consecutive round keys, split into group (first row) and second key
__device__ __forceinline__ void pv_load8_keys(const u64 *__restrict__ k, u64 j0, u32 m, int lo_bits, u32 lomask,
                                              u32 (&g)[PV_IPT], u32 (&lo)[PV_IPT]) {
    if (j0 + PV_IPT <= m && ((((uintptr_t)(k + j0)) & 15) == 0)) {
#pragma unroll
        for (int q = 0; q < PV_IPT / 2; ++q) {
            const uint4 x = *(const uint4 *)(k + j0 + 2 * q);
            const u64 k0 = ((u64)x.y << 32) | x.x, k1 = ((u64)x.w << 32) | x.z;
            g[2 * q] = (u32)(k0 >> lo_bits);
            lo[2 * q] = x.x & lomask;
            g[2 * q + 1] = (u32)(k1 >> lo_bits);
            lo[2 * q + 1] = x.z & lomask;
        }
    } else {
#pragma unroll
        for (int q = 0; q < PV_IPT; ++q) {
            const u64 kk = j0 + q < m ? k[j0 + q] : 0ull;
            g[q] = (u32)(kk >> lo_bits);
            lo[q] = (u32)kk & lomask;
        }
    }
}

// lists made by the pivot path itself: the first member of every group publishes its second key and clears the
// group's counters (for the round's list the kernels that make the keys do it)
__global__ void __launch_bounds__(PV_NT) pivot_heads_kernel(const u64 *__restrict__ keys, u32 m, int lo_bits,
                                                            u32 *__restrict__ piv, unsigned long long *__restrict__ cnt64) {
    const u64 j0 = ((u64)blockIdx.x * PV_NT + threadIdx.x) * PV_IPT;
    if (j0 >= m) return;
    const u32 lomask = lo_bits >= 32 ? 0xffffffffu : ((1u << lo_bits) - 1u);
    u32 g[PV_IPT], lo[PV_IPT];
    pv_load8_keys(keys, j0, m, lo_bits, lomask, g, lo);
    u32 pg = j0 > 0 ? (u32)(keys[j0 - 1] >> lo_bits) : 0u;
#pragma unroll
    for (int q = 0; q < PV_IPT; ++q) {
        const u64 j = j0 + q;
        if (j < m && (j == 0 || g[q] != pg)) {
            piv[g[q] >> 1] = lo[q];
            cnt64[g[q] >> 1] = 0ull;
        }
        pg = g[q];
    }
}

__global__ void __launch_bounds__(PV_NT) pivot_classify_kernel(PivotArgs a) {
    __shared__ u32 wsum[PV_NT / 32];
    __shared__ u32 blkL, blkE, allL;
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 tile_base = (u64)blockIdx.x * PV_TILE;
    const u64 j0 = tile_base + (u64)tid * PV_IPT;
    const u32 lomask = a.lo_bits >= 32 ? 0xffffffffu : ((1u << a.lo_bits) - 1u);
    u32 g[PV_IPT], lo[PV_IPT];
    pv_load8_keys(a.keys, j0, a.m, a.lo_bits, lomask, g, lo);
    const u32 g0 = (u32)(a.keys[tile_base] >> a.lo_bits);  // the group the tile begins in: its counts are summed over the block first
    if (tid == 0) {
        blkL = 0;
        blkE = 0;
        allL = 0;
    }
    __syncthreads();
    u32 ebyte = 0, lbyte = 0, rbyte = 0;
    u32 cur = 0, nL = 0, nE = 0, P = 0, myL = 0;
    bool have = false, one_run = true;
#pragma unroll
    for (int q = 0; q < PV_IPT; ++q) {
        const u64 j = j0 + q;
        if (j >= a.m) break;
        if (!have || g[q] != cur) {
            if (have) {
                one_run = false;
                if (nL | nE) atomicAdd(&a.cnt64[cur >> 1], ((unsigned long long)nE << 32) | (unsigned long long)nL);
            }
            have = true;
            cur = g[q];
            nL = 0;
            nE = 0;
            P = a.piv[cur >> 1];
        }
        const bool isE = lo[q] == P, isL = lo[q] < P;
        nL += isL ? 1u : 0u;
        myL += isL ? 1u : 0u;
        nE += isE ? 1u : 0u;
        ebyte |= (isE ? 1u : 0u) << q;
        lbyte |= (isL ? 1u : 0u) << q;
        rbyte |= ((isE || isL) ? 0u : 1u) << q;
    }
    // the run a thread ends with: whole warps inside one group add up before they touch a counter
    const u32 cur0 = __shfl_sync(0xffffffffu, cur, 0);
    const bool simple = have && one_run && cur == cur0;
    if (__all_sync(0xffffffffu, simple)) {
        const u32 tl = __reduce_add_sync(0xffffffffu, nL), te = __reduce_add_sync(0xffffffffu, nE);
        if (lane == 0) {
            if (cur0 == g0) {
                if (tl) atomicAdd(&blkL, tl);
                if (te) atomicAdd(&blkE, te);
            } else if (tl | te) {
                atomicAdd(&a.cnt64[cur0 >> 1], ((unsigned long long)te << 32) | (unsigned long long)tl);
            }
        }
    } else if (have && (nL | nE)) {
        if (cur == g0) {
            if (nL) atomicAdd(&blkL, nL);
            if (nE) atomicAdd(&blkE, nE);
        } else {
            atomicAdd(&a.cnt64[cur >> 1], ((unsigned long long)nE << 32) | (unsigned long long)nL);
        }
    }
    if (j0 < a.m) {
        a.ebits8[j0 >> 3] = (u8)ebyte;
        a.lbits8[j0 >> 3] = (u8)lbyte;
        a.rbits8[j0 >> 3] = (u8)rbyte;
    }
    // E members of the tile; L members of the whole list
    const u32 c = __reduce_add_sync(0xffffffffu, (u32)__popc(ebyte));
    const u32 cl = __reduce_add_sync(0xffffffffu, myL);
    if (lane == 0) {
        wsum[warp] = c;
        if (cl) atomicAdd(&allL, cl);
    }
    __syncthreads();
    if (tid == 0) {
        u32 t = 0;
        for (int w = 0; w < PV_NT / 32; ++w) t += wsum[w];
        a.tile_e[blockIdx.x] = t;
        if (blkL | blkE) atomicAdd(&a.cnt64[g0 >> 1], ((unsigned long long)blkE << 32) | (unsigned long long)blkL);
        if (allL) atomicAdd(&a.totals[1], allL);
    }
}

// (the staging arrays are indexed e + e / 32: a thread's eight consecutive E members would otherwise hit four banks)
#define PV_PAD(e) ((e) + ((e) >> 5))
__global__ void __launch_bounds__(PV_NT, 4) pivot_apply_kernel(PivotArgs a) {
    // by tile-local index of a group head (index PV_TILE: the group that began before the tile)
    __shared__ u32 s_id[PV_TILE + 1];   // new identifier of the E group, RANK_NONE: unchanged
    // the tile's E members in list order
    __shared__ u32 sh_s[PV_TILE + PV_TILE / 32], sh_nh[PV_TILE + PV_TILE / 32], sh_rk[PV_TILE + PV_TILE / 32];
    __shared__ u32 sh_drop[PV_TILE / 32];  // E members of the tile that are alone in their group
    __shared__ u32 wmax[PV_NT / 32], wsum[PV_NT / 32];
    __shared__ u32 any_single;
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 tile_base = (u64)blockIdx.x * PV_TILE;
    const u64 j0 = tile_base + (u64)tid * PV_IPT;
    const u32 lomask = a.lo_bits >= 32 ? 0xffffffffu : ((1u << a.lo_bits) - 1u);
    u32 g[PV_IPT], lo[PV_IPT], s[PV_IPT], hidx[PV_IPT];
    pv_load8_keys(a.keys, j0, a.m, a.lo_bits, lomask, g, lo);
    pv_load8(a.act, j0, a.m, s);
    if (tid < PV_TILE / 32) sh_drop[tid] = 0;
    if (tid == 0) any_single = 0;
    const u32 ebyte = j0 < a.m ? (u32)a.ebits8[j0 >> 3] : 0u;
    // tile-local index + 1 of the head of every element's group (0: it began before the tile)
    {
        u32 pg = (j0 > 0 && j0 < a.m) ? (u32)(a.keys[j0 - 1] >> a.lo_bits) : 0u;
        u32 run = 0;
#pragma unroll
        for (int q = 0; q < PV_IPT; ++q) {
            const u64 j = j0 + q;
            const bool head = j < a.m && (j == 0 || g[q] != pg);
            if (head) run = (u32)(j - tile_base) + 1u;
            hidx[q] = run;
            pg = g[q];
        }
        const u32 ex = warp_inclusive(run, MaxOp());
        if (lane == 31) wmax[warp] = ex;
        u32 pre = warp_exclusive(ex, run, MaxOp(), 0u);
        __syncthreads();
        for (u32 w = 0; w < warp; ++w) pre = max(pre, wmax[w]);
#pragma unroll
        for (int q = 0; q < PV_IPT; ++q)
            if (hidx[q] == 0) hidx[q] = pre;
    }
    // E members of the tile before this thread's elements
    u32 ne;  // E members of the tile
    const u32 excl = block_exclusive<PV_NT>((u32)__popc(ebyte), wsum, &ne);
    const u32 tile_off = a.tile_e[blockIdx.x];
    // identifier of an E group: the old one while it lies inside the new range, else the middle of the range (a
    // group that loses members at one end, or at both, keeps it for many rounds)
    auto new_id = [](u32 old, u32 nh, u32 nt) { return (old >= nh && old <= nt) ? RANK_NONE : nh + (nt - nh) / 2u; };
#pragma unroll
    for (int q = 0; q < PV_IPT; ++q) {
        const u64 j = j0 + q;
        if (j < a.m && hidx[q] == (u32)(j - tile_base) + 1u) {
            const unsigned long long c = a.cnt64[g[q] >> 1];
            const u32 nL = (u32)c, nE = (u32)(c >> 32), ix = hidx[q] - 1u;
            s_id[ix] = nE > 1u ? new_id(a.rank[s[q]], g[q] + nL, g[q] + nL + nE - 1u) : RANK_NONE;
        }
    }
    if (tid == 0 && hidx[0] == 0) {  // the group that reaches into the tile
        const unsigned long long c = a.cnt64[g[0] >> 1];
        const u32 nL = (u32)c, nE = (u32)(c >> 32);
        s_id[PV_TILE] = nE > 1u ? new_id(a.rank[s[0]], g[0] + nL, g[0] + nL + nE - 1u) : RANK_NONE;
    }
    __syncthreads();
    {
        u32 cur = 0, nL = 0, nE = 0, P = 0;
        bool have = false;
#pragma unroll
        for (int q = 0; q < PV_IPT; ++q) {
            const u64 j = j0 + q;
            if (j >= a.m) break;
            if (!have || g[q] != cur) {
                have = true;
                cur = g[q];
                const unsigned long long c = a.cnt64[cur >> 1];
                nL = (u32)c;
                nE = (u32)(c >> 32);
                P = a.piv[cur >> 1];
            }
            if ((ebyte >> q) & 1u) {
                const u32 el = excl + (u32)__popc(ebyte & ((1u << q) - 1u));
                const u32 nh = cur + nL;
                sh_s[PV_PAD(el)] = s[q];
                sh_nh[PV_PAD(el)] = nh;
                u32 rk;
                if (nE == 1u) {
                    // alone: final.  (The rows of members that stay in the list are written when they leave it.)
                    rk = nh;
                    a.sa[nh] = s[q];
                    if (s[q] == 0) *a.primary = nh;
                    atomicAdd(a.singles, 1u);
                    atomicOr(&sh_drop[el >> 5], 1u << (el & 31u));
                    any_single = 1;
                } else {
                    rk = s_id[hidx[q] ? hidx[q] - 1u : (u32)PV_TILE];
                }
                sh_rk[PV_PAD(el)] = rk;
            } else if (lo[q] > P) {
                a.keys[j] = ((u64)(cur + nL + nE) << a.lo_bits) | (u64)lo[q];
            }
        }
    }
    __syncthreads();
    // consecutive threads write consecutive entries of the next list
    for (u32 k = tid; k < ne; k += PV_NT) {
        const u32 sv = sh_s[PV_PAD(k)], rk = sh_rk[PV_PAD(k)];
        a.out_act[tile_off + k] = sv;
        a.out_grp[tile_off + k] = sh_nh[PV_PAD(k)];
        if (rk != RANK_NONE) a.rank[sv] = rk;
    }
    if (any_single) {
        for (u32 k = tid; k < ne; k += PV_NT)
            if ((sh_drop[k >> 5] >> (k & 31u)) & 1u) {
                const u32 p = a.out_base + tile_off + k;
                atomicOr(&a.dropbits[p >> 5], 1u << (p & 31u));
            }
    }
}

// drop bitmap -> keep bitmap over the first n entries (one thread per 64 entries)
__global__ void __launch_bounds__(256) pivot_keep_kernel(u64 *__restrict__ bits64, u32 n, u64 nwords) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    const u64 base = w * 64;
    const u64 valid = (u64)n - base >= 64 ? ~0ull : ((1ull << ((u64)n - base)) - 1ull);
    bits64[w] = ~bits64[w] & valid;
}

// ---------------------------------------------------------------------------------------------
// Pairs decided by the text.  After round 0 of a text with long exact repeats nearly every group of
// equal keys is a PAIR {s, s + D}: a position of a copied segment and the same position of its copy.
// All pairs of one segment have the same answer: consecutive pairs (s, s + D), (s + 1, s + 1 + D), ...
// overlap in K - 1 symbols, so the two suffixes of every pair of the run agree up to the end of the
// run's last pair, position e, and are told apart by what follows text[e + K) on the two sides -- ONE
// comparison of a few symbols for thousands of pairs, instead of doubling rounds that find the end
// of the segment by its ranks.  Three passes:
//   pair_partner  (list order)  partner[s] for the two members of every group of exactly two
//   pair_runs     (text order)  the run a pair belongs to ends at the first position whose successor
//                               is not the successor's partner's predecessor; the comparison there
//                               gives 1 (this side is smaller) / 2 (the partner is) / 0 (undecided
//                               within the symbols looked at, or the run is longer than the cap)
//   pair_place    (list order)  decided pairs take their two rows in the right order (the BWT rows
//                               swap with them) and leave the list; their ranks are never materialised
// Everything else -- larger groups, undecided pairs -- goes through the doubling rounds as before.
// ---------------------------------------------------------------------------------------------
static constexpr int PR_NT = 256, PR_BPT = 8, PR_TILE = PR_NT * PR_BPT;
static constexpr u32 PR_CAP = 1u << 16;   // longest run followed beyond a tile (longer runs stay undecided)
static constexpr int PR_CMP_WORDS = 256;  // 64-bit windows compared at the end of a run before giving up (a multiple of 32)

// PQ consecutive list elements per thread: the group heads around them come from three vector loads, and the random
// accesses of a thread's pairs (two at most) are in flight together.
static constexpr int PQ = 4;
// G[k] = grp[j0 - 4 + k] for k in [0, 12) (0xffffffff outside the list; no row has that value: len <= 2^32 - 1),
// A[k] = act[j0 + k] for k in [0, 6)
__device__ __forceinline__ void pair_window(const u32 *__restrict__ act, const u32 *__restrict__ grp, u32 m, u64 j0,
                                            u32 (&G)[12], u32 (&A)[6]) {
    if (j0 >= 4 && j0 + 8 <= m) {
        const uint4 x = *(const uint4 *)(grp + j0 - 4), y = *(const uint4 *)(grp + j0), z = *(const uint4 *)(grp + j0 + 4);
        G[0] = x.x; G[1] = x.y; G[2] = x.z; G[3] = x.w; G[4] = y.x; G[5] = y.y; G[6] = y.z; G[7] = y.w;
        G[8] = z.x; G[9] = z.y; G[10] = z.z; G[11] = z.w;
        const uint4 v = *(const uint4 *)(act + j0);
        A[0] = v.x; A[1] = v.y; A[2] = v.z; A[3] = v.w;
        A[4] = act[j0 + 4];
        A[5] = act[j0 + 5];
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            const int64_t j = (int64_t)j0 - 4 + k;
            G[k] = (j >= 0 && j < (int64_t)m) ? grp[j] : 0xffffffffu;
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) A[k] = j0 + k < m ? act[j0 + k] : 0u;
    }
}
// element q of the thread (list index j0 + q) is the first member of a group of exactly two / exactly three: 2 / 3, else 0
__device__ __forceinline__ u32 pair_head_at(const u32 (&G)[12], int q) {
    const u32 g = G[4 + q];
    if (G[3 + q] == g || G[5 + q] != g) return 0u;
    if (G[6 + q] != g) return 2u;
    return G[7 + q] != g ? 3u : 0u;
}

// partner[s] for the members of groups of two and three.  Two: the member that stands first in the text points to the
// other one (the runs of pair_runs_kernel are made of the first members).  Three: in text order, t0 -> t1 -> t2 -> t0:
// the three comparisons order the group.
__global__ void __launch_bounds__(256) pair_partner_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp, u32 m,
                                                           u32 *__restrict__ partner, u32 *__restrict__ npairs) {
    const u64 j0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * PQ;
    u32 c = 0;
    if (j0 < m) {
        u32 G[12], A[6];
        pair_window(act, grp, m, j0, G, A);
#pragma unroll
        for (int q = 0; q < PQ; ++q) {
            const u32 kind = j0 + q < m ? pair_head_at(G, q) : 0u;
            if (kind == 2u) {
                const u32 s1 = A[q], s2 = A[q + 1];
                partner[min(s1, s2)] = max(s1, s2);
                ++c;
            } else if (kind == 3u) {
                const u32 x = A[q], y = A[q + 1], z = A[q + 2];
                const u32 t0 = min(x, min(y, z)), t2 = max(x, max(y, z)), t1 = x ^ y ^ z ^ t0 ^ t2;
                partner[t0] = t1;
                partner[t1] = t2;
                partner[t2] = t0;
                ++c;
            }
        }
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31u) == 0 && c) atomicAdd(npairs, c);
}

// suffixes u and v (u != v): 1 = u is the smaller one, 2 = v is, 0 = undecided within PR_CMP_WORDS windows.
// Warp-cooperative (all lanes call it with the same arguments, the result is uniform): lane l looks at window
// 32 * step + l, the first lane that sees a difference -- or the end of a suffix -- decides.
__device__ __forceinline__ u32 pair_compare_warp(const u64 *__restrict__ packed, int bits, u32 n, u64 u, u64 v) {
    const u32 lane = threadIdx.x & 31u;
    const u32 spw = 64u / (u32)bits;
#pragma unroll 1
    for (int it = 0; it < PR_CMP_WORDS / 32; ++it) {
        const u64 off = (u64)(it * 32 + (int)lane) * spw;
        const u64 uu = u + off, vv = v + off;
        const u64 ru = uu < n ? n - uu : 0ull, rv = vv < n ? n - vv : 0ull;  // symbols left before the sentinel
        const u64 c = min((u64)spw, min(ru, rv));
        u32 res = 0;
        if (c) {
            const u64 x = window_at(packed, uu, bits), y = window_at(packed, vv, bits);
            const u64 mask = c * bits >= 64 ? ~0ull : ~(~0ull >> (c * bits));
            if ((x ^ y) & mask) res = x > y ? 2u : 1u;  // (big-endian windows: the first differing symbol decides)
        }
        // one suffix ends inside this window (or before it): the sentinel is the smallest symbol
        if (!res && c < spw) res = ru < rv ? 1u : 2u;
        const u32 bal = __ballot_sync(0xffffffffu, res != 0u);
        if (bal) return __shfl_sync(0xffffffffu, res, __ffs((int)bal) - 1);
    }
    return 0u;
}

// partner[] is padded with RANK_NONE far beyond len; ord[] is zeroed by the caller
__global__ void __launch_bounds__(PR_NT) pair_runs_kernel(const u32 *__restrict__ partner, u32 n, const u64 *__restrict__ packed,
                                                          int bits, int K, u8 *__restrict__ ord) {
    __shared__ u8 RES[PR_TILE];        // result of the comparison at the run ends inside the tile
    __shared__ u16 qpos[PR_TILE];      // the run ends inside the tile
    __shared__ u32 qn;
    __shared__ u32 wmin[PR_NT / 32];
    __shared__ u32 beyond[2];          // first position at or after the end of the tile that ends a run; the result there
    __shared__ u8 lastlink[PR_NT];
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u64 T0 = (u64)blockIdx.x * PR_TILE;
    const u64 p0 = T0 + (u64)tid * PR_BPT;
    u32 v[PR_BPT + 1];
    {
        const uint4 a = *(const uint4 *)(partner + p0), b = *(const uint4 *)(partner + p0 + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        v[8] = partner[p0 + 8];
    }
    u32 abits = 0, lbits = 0;  // bit i: position p0 + i is a pair member / its pair is followed by the next position's pair
#pragma unroll
    for (int i = 0; i < PR_BPT; ++i) {
        const bool a = v[i] != RANK_NONE;
        abits |= (a ? 1u : 0u) << i;
        lbits |= ((a && v[i + 1] == v[i] + 1u) ? 1u : 0u) << i;
    }
    lastlink[tid] = (u8)((lbits >> (PR_BPT - 1)) & 1u);
    if (tid == 0) qn = 0;
    if (!__syncthreads_or((int)abits)) return;  // no pair member in this tile
    const u32 NONEPOS = 0xffffffffu;
    const u32 zeros = ~lbits & ((1u << PR_BPT) - 1u);
    const u32 firstz = zeros ? tid * PR_BPT + (u32)(__ffs((int)zeros) - 1) : NONEPOS;
    u32 sm = firstz;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_down_sync(0xffffffffu, sm, o);
        if (lane + (u32)o < 32u) sm = min(sm, t);
    }
    if (lane == 0) wmin[warp] = sm;
    u32 after = __shfl_down_sync(0xffffffffu, sm, 1);  // min over the later threads of this warp
    if (lane == 31) after = NONEPOS;
    // run ends inside the chunk (pair members whose pair is not followed by the next position's pair) are queued
    {
        u32 ends = abits & zeros;
        while (ends) {
            const int i = __ffs((int)ends) - 1;
            ends &= ends - 1;
            qpos[atomicAdd(&qn, 1u)] = (u16)(tid * PR_BPT + (u32)i);
        }
    }
    __syncthreads();
    for (u32 ww = warp + 1; ww < PR_NT / 32; ++ww) after = min(after, wmin[ww]);
    // the run that leaves the tile: warp 0 looks for its end (at most PR_CAP positions ahead, 256 per step)
    if (warp == 0) {
        u32 found = NONEPOS;
        if (lastlink[PR_NT - 1]) {
            for (u32 it = 0; it < PR_CAP / 256u && found == NONEPOS; ++it) {
                const u64 at = T0 + PR_TILE + (u64)it * 256u + (u64)lane * 8u;
                const uint4 a = *(const uint4 *)(partner + at), b = *(const uint4 *)(partner + at + 4);
                const u32 x[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, partner[at + 8]};
                u32 nz = 0;  // bit i: position at + i ends a run
#pragma unroll
                for (int i = 0; i < 8; ++i) nz |= ((x[i] != RANK_NONE && x[i + 1] == x[i] + 1u) ? 0u : 1u) << i;
                const u32 bal = __ballot_sync(0xffffffffu, nz != 0u);
                if (bal) {
                    const int l0 = __ffs((int)bal) - 1;
                    const u32 z0 = __shfl_sync(0xffffffffu, nz, l0);
                    found = (u32)PR_TILE + it * 256u + (u32)l0 * 8u + (u32)(__ffs((int)z0) - 1);
                }
            }
        }
        u32 r = 0;
        if (found != NONEPOS) {  // (uniform over the warp)
            const u64 e = T0 + found;
            const u32 pe = partner[e];
            if (pe != RANK_NONE) r = pair_compare_warp(packed, bits, n, e + (u64)K, (u64)pe + (u64)K);
        }
        if (lane == 0) {
            beyond[0] = found;
            beyond[1] = r;
        }
    }
    // the comparisons at the queued run ends, one warp each
    {
        const u32 nq = qn;
        for (u32 k = warp; k < nq; k += PR_NT / 32) {
            const u32 rel = qpos[k];
            const u64 e = T0 + rel;
            const u32 pe = partner[e];
            const u32 r = pair_compare_warp(packed, bits, n, e + (u64)K, (u64)pe + (u64)K);
            if (lane == 0) RES[rel] = (u8)r;
        }
    }
    __syncthreads();
    if (!abits) return;
    u32 nextz = after != NONEPOS ? after : beyond[0];  // first run end after this chunk (relative to T0)
    u64 out = 0;
#pragma unroll
    for (int i = PR_BPT - 1; i >= 0; --i) {
        const u32 rel = tid * PR_BPT + (u32)i;
        if (!((lbits >> i) & 1u)) nextz = rel;
        if ((abits >> i) & 1u) {
            u32 r = 0;
            if (nextz != NONEPOS && nextz - rel <= PR_CAP) r = nextz < (u32)PR_TILE ? (u32)RES[nextz] : beyond[1];
            out |= (u64)r << (8 * i);
        }
    }
    *(u64 *)(ord + p0) = out;
}

// keep8[j] = 1: the element stays in the list.  The thread that holds the FIRST member of a pair / triple writes the
// bytes of all its members (the others may belong to the next thread's elements: that thread leaves them alone).
__global__ void __launch_bounds__(256) pair_place_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp, u32 m,
                                                         const u8 *__restrict__ ord, u32 *__restrict__ sa, u8 *__restrict__ bwt,
                                                         u32 *__restrict__ actbits, u32 *__restrict__ primary,
                                                         const u8 *__restrict__ keep_in, u8 *__restrict__ keep8,
                                                         u32 *__restrict__ nplaced) {
    // (keep_in: "stays" bytes of a list that has not been compacted yet -- elements it drops stay dropped)
    const u64 j0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * PQ;
    const u32 lane = threadIdx.x & 31u;
    u32 placed = 0;
    u32 cw0 = 0xffffffffu, cw1 = 0xffffffffu, cm0 = 0, cm1 = 0;  // words of the active-row bitmap to clear bits in (two groups at most)
    if (j0 < m) {
        u32 G[12], A[6];
        pair_window(act, grp, m, j0, G, A);
        // the results of the thread's pairs and triples, fetched together
        u32 kind[PQ], o0[PQ], o1[PQ], o2[PQ];
#pragma unroll
        for (int q = 0; q < PQ; ++q) {
            kind[q] = j0 + q < m ? pair_head_at(G, q) : 0u;
            o0[q] = o1[q] = o2[q] = 0;
            if (kind[q] == 2u) {
                o0[q] = ord[min(A[q], A[q + 1])];
            } else if (kind[q] == 3u) {
                o0[q] = ord[A[q]];
                o1[q] = ord[A[q + 1]];
                o2[q] = ord[A[q + 2]];
            }
        }
        int np = 0;
#pragma unroll
        for (int q = 0; q < PQ; ++q) {
            const u64 j = j0 + q;
            if (j >= m) break;
            const u32 g = G[4 + q];
            u32 rows = 0;  // rows that become final (0: none)
            if (kind[q] == 2u) {
                const u32 s1 = A[q], s2 = A[q + 1];
                // the result stands at the member that comes first in the text (1 = that one is the smaller suffix):
                // -> 1: the first list element (s1) is the smaller suffix, 2: the second
                u32 oo = o0[q];
                if (oo && s2 < s1) oo = 3u - oo;
                const u8 k = oo ? 0 : 1;
                keep8[j] = k;
                keep8[j + 1] = k;
                if (oo) {
                    rows = 2;
                    if (oo == 2u) {  // the two rows change places
                        sa[g] = s2;
                        sa[g + 1] = s1;
                        if (bwt) {
                            const u8 b0 = bwt[g], b1 = bwt[g + 1];
                            bwt[g] = b1;
                            bwt[g + 1] = b0;
                        }
                    }
                    if (s1 == 0) *primary = oo == 2u ? g + 1 : g;
                    if (s2 == 0) *primary = oo == 2u ? g : g + 1;
                }
            } else if (kind[q] == 3u) {
                // o_k = result at member k (list order): 1 = it is smaller than the member it points to (the next one in
                // TEXT order, cyclically), 2 = larger.  less(x, y) for every pair follows; the ranks must be 0, 1, 2.
                const u32 x[3] = {A[q], A[q + 1], A[q + 2]};
                const u32 ox[3] = {o0[q], o1[q], o2[q]};
                u32 rk[3] = {0, 0, 0};
                bool ok = ox[0] && ox[1] && ox[2];
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    // the member that x[i] points to: the smallest larger start, or the smallest of all (wrap)
                    int tgt = -1;
#pragma unroll
                    for (int k2 = 0; k2 < 3; ++k2)
                        if (k2 != i && x[k2] > x[i] && (tgt < 0 || x[k2] < x[tgt])) tgt = k2;
                    if (tgt < 0) {
#pragma unroll
                        for (int k2 = 0; k2 < 3; ++k2)
                            if (k2 != i && (tgt < 0 || x[k2] < x[tgt])) tgt = k2;
                    }
                    // ox[i] == 1: x[i] < x[tgt] in suffix order -> tgt gets one more smaller suffix; else x[i] does
                    if (ox[i] == 1u) ++rk[tgt];
                    else ++rk[i];
                }
                ok = ok && rk[0] != rk[1] && rk[0] != rk[2] && rk[1] != rk[2];  // (each in 0..2: a permutation)
                const u8 k = ok ? 0 : 1;
                keep8[j] = k;
                keep8[j + 1] = k;
                keep8[j + 2] = k;
                if (ok) {
                    rows = 3;
                    u8 b[3] = {0, 0, 0};
                    if (bwt) {
                        b[0] = bwt[g];
                        b[1] = bwt[g + 1];
                        b[2] = bwt[g + 2];
                    }
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        sa[g + rk[i]] = x[i];
                        if (bwt) bwt[g + rk[i]] = b[i];
                        if (x[i] == 0) *primary = g + rk[i];
                    }
                }
            } else {
                // the other members of a pair / triple are written by the thread that holds the first one
                const bool same_b = G[3 + q] == g, same_a = G[5 + q] == g;
                const bool second_of_2 = same_b && !same_a && G[2 + q] != g;
                const bool second_of_3 = same_b && same_a && G[2 + q] != g && G[6 + q] != g;
                const bool third_of_3 = same_b && !same_a && G[2 + q] == g && G[1 + q] != g;
                if (!(second_of_2 || second_of_3 || third_of_3)) keep8[j] = keep_in ? keep_in[j] : (u8)1;
            }
            if (rows) {
                placed += rows;
                // the rows are final: no longer "active after round 0"
                const u32 full = (rows == 2u ? 3u : 7u);
                const u32 sh = g & 31u;
                const u32 mask = full << sh;
                if (sh + rows > 32u) atomicAnd(&actbits[(g >> 5) + 1], ~(full >> (32u - sh)));
                if (np == 0) {
                    cw0 = g >> 5;
                    cm0 = mask;
                } else {
                    cw1 = g >> 5;
                    cm1 = mask;
                }
                ++np;
            }
        }
    }
    // rows grow along the list: the lanes of a warp that clear bits of one word do it with one atomic
    {
        const u32 peers = __match_any_sync(0xffffffffu, cw0);
        const u32 all = __reduce_or_sync(peers, cm0);
        if (cw0 != 0xffffffffu && lane == (u32)(__ffs((int)peers) - 1)) atomicAnd(&actbits[cw0], ~all);
    }
    if (__any_sync(0xffffffffu, cw1 != 0xffffffffu)) {
        const u32 peers = __match_any_sync(0xffffffffu, cw1);
        const u32 all = __reduce_or_sync(peers, cm1);
        if (cw1 != 0xffffffffu && lane == (u32)(__ffs((int)peers) - 1)) atomicAnd(&actbits[cw1], ~all);
    }
    placed = __reduce_add_sync(0xffffffffu, placed);
    if (lane == 0 && placed) atomicAdd(nplaced, placed);
}

// groups in a grouped list (positions whose group differs from the one before)
__global__ void __launch_bounds__(256) count_heads_kernel(const u32 *__restrict__ grp, u32 m, u32 *__restrict__ count) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    u32 c = 0;
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += stride) c += (j == 0 || grp[j] != grp[j - 1]) ? 1u : 0u;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31u) == 0 && c) atomicAdd(count, c);
}

// ---------------------------------------------------------------------------------------------
// Host orchestration
// ---------------------------------------------------------------------------------------------
size_t build_workspace_estimate(u32 len, int bits) {
    // packed text + round-0 keys (2 x 8) + one value buffer + ranks + look-back + bitmaps, with slack
    size_t l = len;
    return l * bits / 8 + 16 * l + 4 * l + 4 * l + l / 2 + ((size_t)div_up_u(len, 256 * 12) * 1024 * 8) +
           ((size_t)128 << 20);
}

void pack_text(DeviceIndex &ix, int *d_err) {
    cudaStream_t st = ix.stream;
    const int b = ix.pk.bits, cpw = ix.pk.cpw;
    u64 nwords_data = ((u64)ix.len + cpw - 1) / cpw;  // words holding positions 0..n
    u64 nwords = nwords_data + 4;                      // zero padding for window reads
    ix.packed = ix.arena->get<u64>(nwords);
    unsigned long long *counts = ix.arena->get<unsigned long long>(256);
    CUDA_CHECK(cudaMemsetAsync(counts, 0, 256 * 8, st));
    int tid = ix.timer.begin("pack_text", (double)ix.len * (1.0 + b / 8.0));
    unsigned blocks = std::max(1u, std::min(div_up_u(nwords, 256), 148u * 8u));
    switch (b) {
        case 1: pack_kernel<1><<<blocks, 256, 0, st>>>(ix.text_ptr, ix.n, ix.sigma, nwords, ix.packed, counts, d_err); break;
        case 2: pack_kernel<2><<<blocks, 256, 0, st>>>(ix.text_ptr, ix.n, ix.sigma, nwords, ix.packed, counts, d_err); break;
        case 4: pack_kernel<4><<<blocks, 256, 0, st>>>(ix.text_ptr, ix.n, ix.sigma, nwords, ix.packed, counts, d_err); break;
        default: pack_kernel<8><<<blocks, 256, 0, st>>>(ix.text_ptr, ix.n, ix.sigma, nwords, ix.packed, counts, d_err); break;
    }
    KERNEL_CHECK();
    ix.timer.end(tid);
    unsigned long long hc[256];
    read_back(hc, counts, sizeof hc, st);
    // C table (stralg/bwt.c:35-45): the sentinel is the single occurrence of code 0
    for (int i = 0; i < 256; ++i) ix.sym_counts_host[i] = hc[i];
    ix.sym_counts_host[0] = 1;
    u64 run = 0;
    for (u32 a = 0; a < 256; ++a) {
        ix.c_host[a] = (u32)run;
        if (a < ix.sigma) run += ix.sym_counts_host[a];
    }
    ix.c_table.alloc(ix.sigma > 0 ? ix.sigma : 1, st);
    CUDA_CHECK(cudaMemcpyAsync(ix.c_table.ptr, ix.c_host, (size_t)ix.sigma * 4, cudaMemcpyHostToDevice, st));
}

template <int RB>
static void launch_cmer_hist(const DeviceIndex &ix, u64 nwords_data, u32 *hist, cudaStream_t st) {
    unsigned blocks = div_up_u(nwords_data, 256 * 4);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks == 0) blocks = 1;
    switch (ix.pk.bits) {
        case 1: cmer_hist_kernel<RB, 1><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, hist); break;
        case 2: cmer_hist_kernel<RB, 2><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, hist); break;
        case 4: cmer_hist_kernel<RB, 4><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, hist); break;
        default: cmer_hist_kernel<RB, 8><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, hist); break;
    }
    KERNEL_CHECK();
}

// bitmap -> compacted list of still-active suffixes (in current SA order) and their group heads;
// returns the count.  RAW: the bitmap marks the elements to keep; else it marks bucket heads and an
// element is kept unless it is a singleton.
static u32 compaction_sub(u32 m) { return m > (1u << 26) ? 8u : 1u; }
template <bool RAW>
static u32 count_active(const u8 *bits, u32 m, u32 *tile_counts, u32 *d_total, cudaStream_t st) {
    const u32 sub = compaction_sub(m);
    u32 ntiles = div_up_u(m, (u64)CP_TILE * sub);
    count_active_kernel<RAW><<<ntiles, CP_NT, 0, st>>>(bits, m, sub, tile_counts);
    KERNEL_CHECK();
    scan_sum(tile_counts, ntiles, st, d_total);  // (the count is at most m < 2^32)
    u32 total = 0;
    read_back(&total, d_total, 4, st);
    return total;
}
template <bool RAW>
static void scatter_active(const u8 *bits, const u32 *vals, const u32 *grp_in, u32 m, const u32 *tile_offsets, u32 *out,
                           u32 *grp_out, cudaStream_t st) {
    const u32 sub = compaction_sub(m);
    scatter_active_kernel<RAW><<<div_up_u(m, (u64)CP_TILE * sub), CP_NT, 0, st>>>(bits, vals, grp_in, m, sub, tile_offsets,
                                                                                   out, grp_out);
    KERNEL_CHECK();
}
static void scatter_pairs(const u8 *bits, const u64 *keys, const u32 *vals, u32 m, const u32 *tile_offsets, u64 *kout,
                          u32 *vout, cudaStream_t st) {
    const u32 sub = compaction_sub(m);
    scatter_pairs_kernel<<<div_up_u(m, (u64)CP_TILE * sub), CP_NT, 0, st>>>(bits, keys, vals, m, sub, tile_offsets, kout, vout);
    KERNEL_CHECK();
}

// LSD round 0: rows that are not singletons, from the head bitmap (one thread per 64 rows)
__global__ void __launch_bounds__(256) heads_to_actbits_kernel(const u8 *__restrict__ headbits, u32 m,
                                                               u64 *__restrict__ actbits64, u64 nwords) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < nwords) actbits64[w] = active_mask(headbits, w, m);
}

// BWT rows (stralg/bwt.c:13-20) of the rows that were active after round 0, from the final suffix
// array: the doubling rounds over large active sets do not maintain them (one gather per moved row and
// round); their rows are exactly the rows whose bit is set here.
__device__ __forceinline__ void bwt_fix_row(u64 r, const u32 *__restrict__ sa, const u64 *__restrict__ packed, int bits,
                                            u8 *__restrict__ bwt, u32 *__restrict__ primary) {
    const u32 s = sa[r];
    if (s == 0) {
        bwt[r] = 0;
        *primary = (u32)r;
    } else {
        const u64 bitpos = (u64)(s - 1) * bits;
        const u64 w = packed[bitpos >> 6];
        bwt[r] = (u8)(((w >> (64 - bits - (unsigned)(bitpos & 63))) & ((1u << bits) - 1u)) + 1u);
    }
}

// dense bitmaps (periodic texts: every row): one thread per row
__global__ void __launch_bounds__(256) bwt_fix_rows_kernel(const u32 *__restrict__ actbits, const u32 *__restrict__ sa, u32 len,
                                                           const u64 *__restrict__ packed, int bits, u8 *__restrict__ bwt,
                                                           u32 *__restrict__ primary) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= len || !((actbits[r >> 5] >> (r & 31u)) & 1u)) return;
    bwt_fix_row(r, sa, packed, bits, bwt, primary);
}

// sparse bitmaps (one thread per 32 rows: few rows are left once the pair path has taken its rows out)
__global__ void __launch_bounds__(256) bwt_fix_kernel(const u32 *__restrict__ actbits, const u32 *__restrict__ sa, u32 len,
                                                      const u64 *__restrict__ packed, int bits, u8 *__restrict__ bwt,
                                                      u32 *__restrict__ primary) {
    const u64 wi = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (wi * 32 >= len) return;
    u32 w = actbits[wi];
    while (w) {
        const u32 bit = (u32)__ffs((int)w) - 1u;
        w &= w - 1u;
        const u64 r = wi * 32 + bit;
        if (r >= len) break;
        bwt_fix_row(r, sa, packed, bits, bwt, primary);
    }
}

// ---------------------------------------------------------------------------------------------
// Small groups decided by the text.  After round 0 of a text without long repeats the active set is a
// sprinkle of groups of two to four suffixes that share their K symbols by chance (3 Gbp of random
// ACGT: 8 million suffixes, 0.27 %); a doubling round for them costs gathers with recovered ranks, a
// radix sort and a scatter.  One look at the next 64 bits of text (32 symbols of DNA) orders such a
// group: a member's row is the group's first row plus the members with a smaller extension (plus, among
// equal extensions, the ones listed before it).  Members whose extension is unique are final; members
// that agree on it too (copies of a repeat) stay active as a sub-group.  That also takes the chance
// collisions OUT of the groups of a repeat-rich text -- a group {copy, copy, chance collision} would
// otherwise break every chain that runs through it (chain_flags_kernel) -- so the kernel runs on large
// active sets too, where it skips the pairs (two copies of a repeat agree for thousands of symbols: the
// loads would be wasted).  A group one of whose windows reaches the end of the text is left alone.
// Outputs by list slot (a permutation inside the group's slots): act_out, row_out (the rank to
// materialise: first row of the sub-group = final row of a unique member), keep8 (1: stays active).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) resolve_small_groups_kernel(const u32 *__restrict__ act, const u32 *__restrict__ grp,
                                                                   u32 m, const u64 *__restrict__ packed, int bits, int K,
                                                                   u32 n, int skip_pairs, u32 *__restrict__ sa,
                                                                   u32 *__restrict__ rank, u32 *__restrict__ act_out,
                                                                   u32 *__restrict__ row_out, u8 *__restrict__ bwt,
                                                                   u32 *__restrict__ primary, u8 *__restrict__ keep8,
                                                                   u32 *__restrict__ nresolved) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const u32 g = grp[j], s = act[j];
    // members: list elements j - nl .. j + nr (the list is grouped; a group has at least two members).  The four
    // group heads on either side are fetched at once (independent loads), then counted
    u32 gl[4], gr[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        gl[k] = j >= (u64)k + 1 ? grp[j - k - 1] : ~g;
        gr[k] = j + k + 1 < m ? grp[j + k + 1] : ~g;
    }
    u32 nl = 0, nr = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        nl += (nl == (u32)k && gl[k] == g) ? 1u : 0u;
        nr += (nr == (u32)k && gr[k] == g) ? 1u : 0u;
    }
    const u32 size = nl + nr + 1u;
    bool look = size <= 4u && !(skip_pairs && size == 2u);
    const u32 span = 64u / (u32)bits;
    u64 ext[4];
    for (u32 x = 0; x < size && look; ++x) {
        const u32 t = act[j - nl + x];
        look = (u64)t + (u64)K + span <= (u64)n;
        if (look) ext[x] = window_at(packed, (u64)t + (u64)K, bits);
    }
    if (!look) {  // untouched
        act_out[j] = s;
        row_out[j] = g;
        keep8[j] = 1;
        return;
    }
    u32 smaller = 0, eq_before = 0, eq_total = 0;
    for (u32 x = 0; x < size; ++x) {
        smaller += ext[x] < ext[nl] ? 1u : 0u;
        if (ext[x] == ext[nl]) {
            ++eq_total;
            eq_before += x < nl ? 1u : 0u;
        }
    }
    const u64 slot = j - nl + smaller + eq_before;
    const u32 row = g + smaller + eq_before;
    act_out[slot] = s;
    row_out[slot] = g + smaller;
    keep8[slot] = eq_total > 1u ? 1 : 0;
    if (eq_total == 1u) atomicAdd(nresolved, 1u);
    if (rank) rank[s] = g + smaller;  // (ranks already materialised: LSD round 0)
    sa[row] = s;
    if (s == 0) *primary = row;
    if (bwt) {
        u8 c = 0;
        if (s) {
            const u64 bitpos = (u64)(s - 1) * bits;
            const u64 w = packed[bitpos >> 6];
            c = (u8)(((w >> (64 - bits - (unsigned)(bitpos & 63))) & ((1u << bits) - 1u)) + 1u);
        }
        bwt[row] = c;
    }
}

// how many list elements stand in groups the kernel above would look at (2..4 members; pairs optional)
__global__ void __launch_bounds__(256) count_small_groups_kernel(const u32 *__restrict__ grp, u32 m, int skip_pairs,
                                                                 u32 *__restrict__ count) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool look = false;
    if (j < m) {
        const u32 g = grp[j];
        u32 nl = 0, nr = 0;
        while (nl < 4u && j >= (u64)nl + 1 && grp[j - nl - 1] == g) ++nl;
        while (nr < 4u && j + nr + 1 < m && grp[j + nr + 1] == g) ++nr;
        const u32 size = nl + nr + 1u;
        look = size <= 4u && !(skip_pairs && size == 2u);
    }
    const u32 c = __popc(__ballot_sync(0xffffffffu, look));
    if ((threadIdx.x & 31u) == 0 && c) atomicAdd(count, c);
}

// rank[act[j]] = row[j]; short: [count, (suffix, row) ...]
__global__ void __launch_bounds__(256) scatter_ranks_kernel(const u32 *__restrict__ act, const u32 *__restrict__ row, u32 m,
                                                            const u32 *__restrict__ shorts, u32 *__restrict__ rank) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) rank[act[j]] = row[j];
    if (j == 0 && shorts)
        for (u32 i = 0; i < shorts[0]; ++i) rank[shorts[1 + 2 * i]] = shorts[2 + 2 * i];
}

// rank[act[j]] = row[j] for the elements that leave the list (keep8[j] == 0)
__global__ void __launch_bounds__(256) scatter_ranks_left_kernel(const u32 *__restrict__ act, const u32 *__restrict__ row,
                                                                 const u8 *__restrict__ keep8, u32 m, u32 *__restrict__ rank) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m && !keep8[j]) rank[act[j]] = row[j];
}

// bytes (0 / 1) -> bitmap words, one thread per 64 elements
__global__ void __launch_bounds__(256) bytes_to_bits_kernel(const u8 *__restrict__ b8, u32 m, u64 *__restrict__ bits64,
                                                            u64 nwords) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    u64 v = 0;
    const u64 base = w * 64;
    for (u32 i = 0; i < 64 && base + i < m; ++i) v |= (u64)(b8[base + i] & 1u) << i;
    bits64[w] = v;
}

// environment knobs of the build (DESIGN.md §10), read once at its start
struct BuildKnobs {
    int radix_bits, key_margin;
    bool passes0_set;  // LSD round 0 makes `passes0` passes (clamped), not the number computed from the text
    int passes0;
    int pairs;         // 0: off, 1: on large active sets, 2: on lists of any size (tests)
    bool ext_tiebreak, chain, small_path, pivot;
    bool pivot_force;  // (tests: every round, whatever it finds)
    int bwt_round_frac, chain_min_frac, chain_use_frac, dense_factor;
    u32 pivot_min;
};

static BuildKnobs read_build_knobs() {
    BuildKnobs k;
    k.radix_bits = env_int("B200SA_RADIX_BITS", 8);
    k.key_margin = env_int("B200SA_KEY_MARGIN", 8);
    const char *p0 = getenv("B200SA_PASSES0");
    k.passes0_set = p0 && *p0;
    k.passes0 = k.passes0_set ? atoi(p0) : 0;
    k.pairs = env_int("B200SA_PAIRS", 1);
    k.ext_tiebreak = env_int("B200SA_NO_EXT_TIEBREAK", 0) == 0;
    k.chain = env_int("B200SA_CHAIN", 1) != 0;
    k.small_path = env_int("B200SA_SMALL_PATH", 1) != 0;
    k.pivot = env_int("B200SA_PIVOT", 1) != 0;
    k.pivot_force = env_int("B200SA_PIVOT_FORCE", 0) != 0;
    k.bwt_round_frac = std::max(1, env_int("B200SA_BWT_ROUND_FRAC", 32));
    k.chain_min_frac = std::max(1, env_int("B200SA_CHAIN_MIN_FRAC", 64));
    k.chain_use_frac = std::max(1, env_int("B200SA_CHAIN_USE_FRAC", 2));
    k.dense_factor = std::max(1, env_int("B200SA_DENSE_FACTOR", 12));
    k.pivot_min = (u32)std::max(2, env_int("B200SA_PIVOT_MIN", 1 << 16));
    return k;
}

// what the stages of one build share
struct BuildCtx {
    DeviceIndex &ix;
    const BuildKnobs &kn;
    Arena &ar;
    cudaStream_t st;
    bool want_bwt;
    u32 n, len;
    int b;                   // bits per packed symbol
    int log2len, lo_bits, key_bits;  // doubling rounds: bits of the rank half of a key, bits of a key
    u32 *sa, *d_primary;
    // workspace; actbits: bit per row, active after round 0
    u64 *keysA, *keysB, *lookback;
    u32 *valsV, *rank, *actbits, *hist, *uniform, *ticket, *tile_counts, *d_lazy;
    u8 *headbits;
    u32 *d_total;
    u8 *bwt_rows = nullptr;     // BWT output while the sort writes its rows as it goes
    bool need_bwt_fix = false;  // a path moved rows without writing their BWT rows

    BuildCtx(DeviceIndex &ix_, const BuildKnobs &kn_, bool want_bwt_, u32 *d_primary_)
        : ix(ix_), kn(kn_), ar(*ix_.arena), st(ix_.stream), want_bwt(want_bwt_), n(ix_.n), len(ix_.len), b(ix_.pk.bits),
          sa(ix_.sa.ptr), d_primary(d_primary_) {
        log2len = 0;
        while ((1ull << log2len) < (u64)len) ++log2len;
        lo_bits = std::max(1, log2len);
        key_bits = std::min(64, 2 * lo_bits);
    }
};

// the active list: suffixes whose key is shared with another suffix, in suffix-array order, each with the first row of
// its group; and what round 0 tells the rounds about it
struct ActiveList {
    bool bucketed = false;            // round 0 was the bucket sort (else the LSD passes)
    u32 m = 0;
    u32 *act = nullptr, *grp = nullptr;
    int K = 0;                        // symbols in a round-0 key
    u32 depth0 = 0;                   // symbols every active group shares after round 0 (0: K)
    const u32 *short_rank = nullptr;  // bucketed round 0: ranks of the short suffixes of oversize buckets
    bool bwt_in_sort = true;          // BWT rows ride along with the sort (else: gathered from the final SA)
    u64 *rk_free[2] = {nullptr, nullptr};  // large buffers that are dead after round 0 (round keys go there)
    LazyRank lr{};
};

// bucketed round 0: the list rank[] is scattered from for the suffixes active after it (round0_msd.cu writes no
// ranks); marked: rank[] has been set to "not materialised" (and holds the ranks of decided suffixes)
struct RankSource {
    const u32 *act, *row;
    u32 m;
    bool marked;
};

// the tie-break's permuted list with a "stays" byte per element, when the pair path follows it and one compaction
// serves both (act == nullptr: none); nres elements leave it
struct PendingList {
    u32 *act = nullptr, *row = nullptr;
    u8 *keep = nullptr;
    u32 nres = 0;
};

// rank_kernel's arguments for a doubling round ((group, rank) keys, moved suffixes stored into the SA), or for round 0
// (K0 > 0: keys of K0 symbols under `keymask`, the preceding symbol at `prev_shift`, the SA already in place)
static RankArgs rank_args(const BuildCtx &c, const u64 *keys, const u32 *vals, u32 m, u32 *newgrp, u8 *headbits, u8 *bwt,
                          int always_write, int K0 = 0, u64 keymask = ~0ull, int prev_shift = 0) {
    RankArgs a{};
    a.keys = keys; a.vals = vals; a.m = m; a.gs = K0 ? 64 : c.lo_bits; a.keymask = keymask; a.K0 = K0; a.n = c.n;
    a.rank = c.rank; a.newgrp = newgrp; a.scatter_all = 0; a.sa_out = K0 ? nullptr : c.sa; a.headbits = headbits;
    a.bwt = bwt; a.prev_shift = prev_shift; a.packed = c.ix.packed; a.bits = c.b; a.primary = c.d_primary;
    a.always_write = always_write;
    return a;
}

// One list of a doubling round: radix sort of its (group, rank) keys over the digits that are not uniform, then new
// ranks, the head bitmap and the new group of every element by sorted index (`newgrp`).  (keys, vals) hold the list,
// (keys_other, vals_other) are the other buffer pair; returns the value buffer that holds the sorted list.
template <int RB>
static u32 *sort_and_rank(BuildCtx &c, u64 *keys, u32 *vals, u64 *keys_other, u32 *vals_other, u32 m, u32 *newgrp,
                          u8 *headbits, u8 *bwt, int always_write) {
    u64 *kb[2] = {keys, keys_other};
    u32 *vb[2] = {vals, vals_other};
    const auto sorted = rs::Sorter<RB>::sort(kb, vb, m, c.key_bits, c.hist, c.uniform, c.lookback, c.ticket, c.st,
                                             &c.ix.timer);
    c.ix.stats.passes_elems += (u64)m * sorted.passes;
    int t = c.ix.timer.begin("round_rank", (double)m * 20.0);
    CUDA_CHECK(cudaMemsetAsync(headbits, 0, (((size_t)m + 63) / 64 + 2) * 8, c.st));
    rank_kernel<<<div_up_u(m, RK_TILE), RK_NT, 0, c.st>>>(
        rank_args(c, sorted.keys, sorted.vals, m, newgrp, headbits, bwt, always_write));
    KERNEL_CHECK();
    c.ix.timer.end(t);
    return sorted.vals;
}

// the list elements whose keep byte is set, (act, row) -> (act_out, row_out) in list order; returns their number
static u32 compact_kept(BuildCtx &c, const u8 *keep8, u32 m, const u32 *act, const u32 *row, u32 *act_out, u32 *row_out) {
    const u64 kw = ((u64)m + 63) / 64;
    CUDA_CHECK(cudaMemsetAsync(c.headbits, 0, (kw + 2) * 8, c.st));
    bytes_to_bits_kernel<<<div_up_u(kw, 256), 256, 0, c.st>>>(keep8, m, (u64 *)c.headbits, kw);
    KERNEL_CHECK();
    const u32 m2 = count_active<true>(c.headbits, m, c.tile_counts, c.d_total, c.st);
    if (m2) scatter_active<true>(c.headbits, act, row, m, c.tile_counts, act_out, row_out, c.st);
    return m2;
}

// ---- round 0, preferred: MSD bucket sort of 8-byte elements (round0_msd.cu); false when it does not apply ----
static bool round0_bucketed(BuildCtx &c, ActiveList &L) {
    DeviceIndex &ix = c.ix;
    Round0Msd r0{};
    if (!msd_make_plan(c.len, ix.sigma, c.b, r0.plan, ix.sym_counts_host)) return false;
    Arena::Mark mk = c.ar.mark();
    r0.bufA = c.keysA; r0.bufB = c.keysB; r0.actbits = c.actbits;
    r0.d_primary = c.d_primary;
    if (!round0_msd(ix, c.want_bwt, r0)) {
        c.ar.release_to(mk);
        return false;
    }
    L.bucketed = true;
    L.K = r0.plan.K;
    L.bwt_in_sort = r0.bwt_written;
    L.lr.keys0 = nullptr; L.lr.bstart = r0.bucket_start; L.lr.BB = r0.plan.BB; L.lr.K = L.K;
    L.lr.kb = r0.plan.KB; L.lr.dense = r0.plan.dense;
    ix.stats.dense_keys = r0.plan.dense.nsym;
    L.lr.keymask = (L.K * c.b >= 64) ? ~0ull : ((1ull << (L.K * c.b)) - 1ull);
    ix.stats.k0 = L.K;
    ix.stats.radix_bits = r0.plan.D[0];
    ix.stats.passes0 = r0.plan.nlevels;
    ix.stats.round0_mode = 1;
    ix.stats.bucket_bits = r0.plan.BB;
    ix.stats.passes_elems = (u64)c.len * r0.plan.nlevels;
    ix.stats.shallow_buckets = r0.shallow_buckets;
    ix.stats.shallow_elems = r0.shallow_buckets ? r0.shallow_elems : 0;
    L.depth0 = r0.depth0;
    L.short_rank = r0.short_rank;
    // the active rows, in row order, with their group heads
    int t = ix.timer.begin("compact0", (double)c.len * 0.125);
    L.m = count_active<true>((const u8 *)c.actbits, c.len, c.tile_counts, c.d_total, c.st);
    if (L.m) {
        L.grp = c.ar.get<u32>(L.m);
        scatter_active<true>((const u8 *)c.actbits, c.sa, r0.grow, c.len, c.tile_counts, L.act, L.grp, c.st);
    }
    ix.timer.end(t);
    L.rk_free[0] = c.keysA;
    L.rk_free[1] = c.keysB;
    return true;
}

// ---- round 0, general: LSD radix passes over (u64 key, u32 suffix) pairs ----
template <int RB>
static void round0_lsd(BuildCtx &c, ActiveList &L) {
    typedef rs::Sorter<RB> S;
    constexpr int BINS = 1 << RB;
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 len = c.len;
    const int b = c.b;
    const int spd = RB / b;  // symbols per digit
    const int pshift = prev_shift_for(b);
    const int maxP = pshift / RB;  // the preceding-symbol field sits above the sorted digits
    double eff = std::log2((double)(ix.sigma > 2 ? ix.sigma - 1 : 1));
    if (eff < 0.5) eff = 0.5;
    int P0 = c.kn.passes0_set ? c.kn.passes0 : (int)std::ceil((c.log2len + c.kn.key_margin) / (spd * eff));
    P0 = std::max(1, std::min(P0, maxP));
    L.K = spd * P0;
    const u64 keymask0 = (L.K * b >= 64) ? ~0ull : ((1ull << (L.K * b)) - 1ull);
    ix.stats.k0 = L.K;
    ix.stats.radix_bits = RB;
    ix.stats.passes0 = P0;
    ix.stats.passes_elems = (u64)len * P0;
    u32 *bases0 = c.ar.get<u32>((size_t)P0 * BINS);

    u64 nwords_data = ((u64)len + ix.pk.cpw - 1) / ix.pk.cpw;
    int t = ix.timer.begin("cmer_hist", (double)len * b / 8.0);
    CUDA_CHECK(cudaMemsetAsync(c.hist, 0, (size_t)BINS * 4, st));
    launch_cmer_hist<RB>(ix, nwords_data, c.hist, st);
    round0_bases_kernel<RB><<<P0, 256, 0, st>>>(c.hist, ix.packed, c.n, L.K, b, bases0);
    KERNEL_CHECK();
    ix.timer.end(t);

    // the value ping-pong is arranged so that the last pass writes straight into the SA output
    u64 *kin = c.keysA, *kout = c.keysB;
    u32 *vin = (P0 % 2) ? c.valsV : c.sa;
    u32 *vout = (P0 % 2) ? c.sa : c.valsV;
    t = ix.timer.begin("make_keys0", (double)len * 12.0);
    make_keys0_kernel<<<div_up_u(len, 256 * 4), 256, 0, st>>>(ix.packed, c.n, len, L.K, b, kin, vin);
    KERNEL_CHECK();
    ix.timer.end(t);
    for (int p = 0; p < P0; ++p) {
        t = ix.timer.begin("radix_pass0", (double)len * 24.0);
        S::pass(kin, vin, kout, vout, len, p * RB, RB, bases0 + (size_t)p * BINS, c.lookback, c.ticket, st);
        ix.timer.end(t);
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    const u64 *keys0 = kin;  // vin == sa
    u32 *newgrp0 = (u32 *)kout;  // (the other key buffer is free: new ranks by sorted index)

    t = ix.timer.begin("rank0", (double)len * 16.0);
    CUDA_CHECK(cudaMemsetAsync(c.headbits, 0, (((size_t)len + 63) / 64 + 2) * 8, st));
    CUDA_CHECK(cudaMemsetAsync(c.rank, 0xff, (size_t)len * 4, st));  // nothing materialised yet
    rank_kernel<<<div_up_u(len, RK_TILE), RK_NT, 0, st>>>(
        rank_args(c, keys0, c.sa, len, newgrp0, c.headbits, c.want_bwt ? ix.bwt.ptr : nullptr, 0, L.K, keymask0, pshift));
    KERNEL_CHECK();
    ix.timer.end(t);

    t = ix.timer.begin("compact0", (double)len * 0.125);
    L.m = count_active<false>(c.headbits, len, c.tile_counts, c.d_total, st);
    if (L.m) {
        L.grp = c.ar.get<u32>(L.m);
        scatter_active<false>(c.headbits, c.sa, newgrp0, len, c.tile_counts, L.act, L.grp, st);  // valsV is free once the sort is done
        const size_t act_words = ((size_t)len + 63) / 64;
        heads_to_actbits_kernel<<<div_up_u(act_words, 256), 256, 0, st>>>(c.headbits, len, (u64 *)c.actbits, act_words);
        KERNEL_CHECK();
    }
    ix.timer.end(t);
    L.lr.keys0 = keys0; L.lr.keymask = keymask0; L.lr.K = L.K; L.lr.kb = L.K * b;
    L.rk_free[0] = kout;  // (keys0 stays: lazy ranks are looked up in it)
}

// the pair path takes the list after round 0
static bool pair_path_applies(const BuildCtx &c, const ActiveList &L) {
    return L.bucketed && c.kn.pairs && ((u64)L.m * 64 >= (u64)c.len || c.kn.pairs == 2);
}

// ---- groups of two to four equal keys are ordered by the next 64 bits of text (pairs only while the active set is
// small: in a large one they are copies of repeats) ----
static void text_tiebreak(BuildCtx &c, ActiveList &L, RankSource &rsrc, PendingList &pend) {
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = L.m;
    int t = ix.timer.begin("resolve_small", (double)m * 40.0);
    u32 *d_nres = c.ar.get<u32>(2);
    CUDA_CHECK(cudaMemsetAsync(d_nres, 0, 8, st));
    const int skip_pairs = (u64)m * 64 > (u64)c.len ? 1 : 0;
    // (when most suffixes are active the groups are usually giant -- periodic texts: a cheap look first)
    u32 nsmall = 1;
    if ((u64)m * 2 > (u64)c.len) {
        count_small_groups_kernel<<<div_up_u(m, 256), 256, 0, st>>>(L.grp, m, skip_pairs, d_nres + 1);
        KERNEL_CHECK();
        read_back(&nsmall, d_nres + 1, 4, st);
        if ((u64)nsmall * 64 < (u64)m) nsmall = 0;  // (a trip over the whole list for a sprinkle of small groups: the rounds take them)
    }
    if (nsmall) {
        // the permuted list goes into a buffer that is dead until the rounds write their keys (both m <= len words)
        u8 *keep8 = c.ar.get<u8>((size_t)m + 64);
        u32 *act_p = (u32 *)L.rk_free[0], *row_p = act_p + (((size_t)m + 3) & ~(size_t)3);  // (vector stores: 16-byte aligned)
        resolve_small_groups_kernel<<<div_up_u(m, 256), 256, 0, st>>>(L.act, L.grp, m, ix.packed, c.b, L.K, c.n, skip_pairs,
                                                                      c.sa, L.bucketed ? nullptr : c.rank, act_p, row_p,
                                                                      c.bwt_rows, c.d_primary, keep8, d_nres);
        KERNEL_CHECK();
        u32 nres = 0;
        read_back(&nres, d_nres, 4, st);
        ix.stats.resolved_small = nres;
        // (the permuted list replaces the old one even when nothing was decided: sub-groups may have formed)
        rsrc.act = act_p;
        rsrc.row = row_p;
        // the list the rounds start from goes back into the buffers of the old one (dead now); the rank source stays
        // where it is until the ranks have been scattered
        if (nres && L.bucketed && nres < m) {
            // the suffixes decided here are final but their rows still count as "active after round 0": when rounds
            // follow, their ranks are materialised now (the pair path below may replace the list the other ranks
            // are scattered from)
            CUDA_CHECK(cudaMemsetAsync(c.rank, 0xff, (size_t)c.len * 4, st));
            scatter_ranks_left_kernel<<<div_up_u(m, 256), 256, 0, st>>>(act_p, row_p, keep8, m, c.rank);
            KERNEL_CHECK();
            rsrc.marked = true;
        }
        if (nres && nres < m && pair_path_applies(c, L)) {
            pend.act = act_p; pend.row = row_p; pend.keep = keep8; pend.nres = nres;
        } else if (nres) {
            L.m = compact_kept(c, keep8, m, act_p, row_p, L.act, L.grp);
        } else {
            CUDA_CHECK(cudaMemcpyAsync(L.act, act_p, (size_t)m * 4, cudaMemcpyDeviceToDevice, st));
            CUDA_CHECK(cudaMemcpyAsync(L.grp, row_p, (size_t)m * 4, cudaMemcpyDeviceToDevice, st));
        }
    }
    ix.timer.end(t);
}

// ---- pairs of a text with long exact repeats: decided by one comparison per copied segment (pair_runs_kernel).  It
// also finishes the compaction the tie-break left pending ----
static void pair_path(BuildCtx &c, ActiveList &L, RankSource &rsrc, const PendingList &pend) {
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = L.m, len = c.len;
    // (the list the pair path reads: the permuted one when the tie-break left its compaction to this path)
    const u32 *pl_act = pend.act ? pend.act : L.act, *pl_grp = pend.act ? pend.row : L.grp;
    bool placed = false;
    int t = ix.timer.begin("pair_partner", (double)m * 16.0 + (double)len * 4.0);
    const size_t pt_entries = (size_t)len + PR_CAP + 2 * PR_TILE + 16;
    const size_t pt_padded = (pt_entries + 127) & ~(size_t)127;
    const size_t ord_bytes = (((size_t)len + PR_TILE) / PR_TILE + 1) * PR_TILE;
    // (in the round-key buffer that is free now when the text is long enough for the padding to fit, else carved)
    u32 *partner = pt_padded * 4 + ord_bytes <= ((size_t)len + 2) * 8 ? (u32 *)L.rk_free[1]
                                                                    : (u32 *)c.ar.get<u8>(pt_padded * 4 + ord_bytes);
    u8 *ord = (u8 *)(partner + pt_padded);
    u32 *d_pr = c.ar.get<u32>(2);
    CUDA_CHECK(cudaMemsetAsync(partner, 0xff, pt_entries * 4, st));
    CUDA_CHECK(cudaMemsetAsync(d_pr, 0, 8, st));
    pair_partner_kernel<<<div_up_u(m, 256 * PQ), 256, 0, st>>>(pl_act, pl_grp, m, partner, d_pr);
    KERNEL_CHECK();
    u32 npairs = 0;
    read_back(&npairs, d_pr, 4, st);
    ix.timer.end(t);
    if (npairs && ((u64)npairs * 8 >= (u64)m || c.kn.pairs == 2)) {  // (two members each: at least a quarter of the list)
        t = ix.timer.begin("pair_runs", (double)len * 5.0);
        CUDA_CHECK(cudaMemsetAsync(ord, 0, ord_bytes, st));
        pair_runs_kernel<<<div_up_u(len, PR_TILE), PR_NT, 0, st>>>(partner, c.n, ix.packed, c.b, L.K, ord);
        KERNEL_CHECK();
        ix.timer.end(t);
        t = ix.timer.begin("pair_place", (double)m * 14.0);
        u8 *keep8 = c.ar.get<u8>((size_t)m + 64);
        pair_place_kernel<<<div_up_u(m, 256 * PQ), 256, 0, st>>>(pl_act, pl_grp, m, ord, c.sa, c.bwt_rows, c.actbits,
                                                                c.d_primary, pend.keep, keep8, d_pr + 1);
        KERNEL_CHECK();
        u32 nplaced = 0;
        read_back(&nplaced, d_pr + 1, 4, st);
        ix.stats.pair_placed = nplaced;
        ix.timer.end(t);
        t = ix.timer.begin("pair_compact", (double)m * 10.0);
        if (nplaced) {
            // the rest of the list (its ranks are the only ones that are needed: only suffixes that stay active get
            // one).  From the tie-break's permuted list it goes straight into the list's own buffers; else through
            // the buffer that held the list round 0 left
            u32 *tmpA = (u32 *)L.rk_free[0], *tmpB = tmpA + m;
            const u32 m2 = pend.act ? compact_kept(c, keep8, m, pend.act, pend.row, L.act, L.grp)
                                    : compact_kept(c, keep8, m, L.act, L.grp, tmpA, tmpB);
            if (m2 != m - nplaced - pend.nres)
                throw std::runtime_error("pair path: list accounting is inconsistent (internal error)");
            if (m2 && !pend.act) {
                CUDA_CHECK(cudaMemcpyAsync(L.act, tmpA, (size_t)m2 * 4, cudaMemcpyDeviceToDevice, st));
                CUDA_CHECK(cudaMemcpyAsync(L.grp, tmpB, (size_t)m2 * 4, cudaMemcpyDeviceToDevice, st));
            }
            L.m = m2;
            rsrc.act = L.act;
            rsrc.row = L.grp;
            rsrc.m = m2;
            placed = true;
        }
        ix.timer.end(t);
    }
    if (pend.act && !placed) {
        // the pair path placed nothing: the tie-break's own compaction after all
        t = ix.timer.begin("resolve_small", (double)m * 16.0);
        L.m = compact_kept(c, pend.keep, m, pend.act, pend.row, L.act, L.grp);
        ix.timer.end(t);
    }
}

// ---- bucketed round 0: ranks of the suffixes that were active after it (first row of their group, or their final
// row where the text decided); everything else is marked "not materialised" first.  A text without repeats never gets
// here: its few chance collisions are all decided above.  (LSD round 0: rank_kernel wrote the ranks, the tie-break
// kept them up to date.) ----
static void scatter_round0_ranks(BuildCtx &c, const ActiveList &L, const RankSource &rsrc) {
    int t = c.ix.timer.begin("rank_scatter", (double)rsrc.m * 12.0 + (double)c.len * 4.0);
    if (!rsrc.marked) CUDA_CHECK(cudaMemsetAsync(c.rank, 0xff, (size_t)c.len * 4, c.st));
    scatter_ranks_kernel<<<div_up_u(rsrc.m, 256), 256, 0, c.st>>>(rsrc.act, rsrc.row, rsrc.m, L.short_rank, c.rank);
    KERNEL_CHECK();
    c.ix.timer.end(t);
}

// complete ranks ("dense"): ranks of retired suffixes are no longer recovered on demand
static void go_dense(BuildCtx &c, LazyRank &lr) {
    int t = c.ix.timer.begin("rank0_fill", (double)c.len * 16.0);
    fill_singleton_ranks(c.ix, c.actbits, c.rank);
    c.ix.timer.end(t);
    lr.sparse = false;
}

// the list and the buffers of the doubling rounds
struct RoundState {
    u32 m;
    u32 *act, *grp, *act2, *grp2;  // the list and the buffers of the next one
    u64 *rkA, *rkB;                // round keys and the other key buffer of the sort
    u64 h;                         // symbols every active group shares
    u32 bwt_small;                 // active sets up to this size maintain their BWT rows in the rounds
    // One region serves the chain arrays (live from chain_flags to make_keys) and the outputs of the small-group path
    // (live from there to the end of the round).
    size_t cont_bytes;
    u8 *cont8, *cslot, *notdone, *headB;
    u32 *chainkey, *d_ncont, *d_handled, *d_nheads;
    // three list-sized buffers of the split paths; `r0` changes places with the list when the pivot path has
    // assembled the next one there (every list buffer holds m_init words) -- from then on the region holds a
    // list and the chain arrays, which share it, are not used any more
    u32 *r0, *newgrpT, *bvals;
    // pivot path: per-group tables by (head row) / 2, E bitmap, per-tile counts
    u8 *ebits8, *rbits8;
    u32 *pv_tile_e, *pv_piv;
    u32 *d_pvtot;
    unsigned long long *pv_cnt;
    bool chain_on, small_on, pivot_on;
    bool prefer_pivot;            // large groups or small ones?  (decides which of the two split paths a round tries first)
    bool ids_are_heads = true;    // rank[] of an active suffix is the first row of its group (until the pivot path runs)
    int small_pause = 0, small_fails = 0;  // rounds the small-group path sits out after finding almost nothing
    int pivot_pause = 0, pivot_fails = 0;  // the same for the pivot path
};

// ---- chain offsets (see chain_flags_kernel): tried while the active set is a noticeable part of the text, dropped for
// good once a round finds few groups that continue.  True when this round's keys use them ----
static bool chain_offsets(BuildCtx &c, RoundState &R, const LazyRank &lr) {
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = R.m;
    if (!R.chain_on || R.h > (u64)CHAIN_CAP || (u64)m * (u64)c.kn.chain_min_frac < (u64)c.len) return false;
    int t = ix.timer.begin("chain_flags", (double)m * 13.0 + (double)c.len);
    CUDA_CHECK(cudaMemsetAsync(R.cont8, 0, R.cont_bytes, st));
    CUDA_CHECK(cudaMemsetAsync(R.cslot, 0, m, st));
    CUDA_CHECK(cudaMemsetAsync(R.d_ncont, 0, 4, st));
    const u32 cf_tiles = div_up_u(m, CF_STEP);
    u32 ncont = 0;
    bool worth = true;
    if (cf_tiles > 16384) {
        // a sample of 2 048 tiles first: a list whose groups do not continue (diverged copies, periodic
        // texts) is not worth the full pass (what the sample marks is what the full pass would mark)
        const u32 mul = cf_tiles / 2048;
        chain_flags_kernel<<<2048, CF_NT, 0, st>>>(R.act, R.grp, m, c.rank, R.cslot, R.cont8, R.d_ncont, mul);
        KERNEL_CHECK();
        read_back(&ncont, R.d_ncont, 4, st);
        worth = (u64)ncont * (u64)c.kn.chain_use_frac * 2 >= (u64)2048 * CF_STEP;
        CUDA_CHECK(cudaMemsetAsync(R.d_ncont, 0, 4, st));
        ncont = 0;
    }
    if (worth) {
        chain_flags_kernel<<<cf_tiles, CF_NT, 0, st>>>(R.act, R.grp, m, c.rank, R.cslot, R.cont8, R.d_ncont, 1);
        KERNEL_CHECK();
        read_back(&ncont, R.d_ncont, 4, st);
    }
    ix.timer.end(t);
    // worth it when most groups continue (copies of long segments); texts whose groups are large and
    // shallow (many diverged copies) gain nothing from it
    if ((u64)ncont * (u64)c.kn.chain_use_frac < (u64)m) {
        R.chain_on = false;
        return false;
    }
    t = ix.timer.begin("chain_keys", (double)c.len + (double)ncont * 4.0);
    chain_keys_kernel<<<div_up_u(c.len, CK_TILE), CK_NT, 0, st>>>(R.cont8, c.len, lr, R.h, R.chainkey, c.d_lazy);
    KERNEL_CHECK();
    ix.timer.end(t);
    ix.stats.chain_rounds++;
    ix.stats.chain_elems += ncont;
    return true;
}

// ---- large groups that mostly stay together: split around a pivot key (pivot_classify_kernel).  The E part of
// every group goes straight into the next list; its L members and its R members, each compacted into a list of their
// own, are split again the same way (a group whose members carry two or three distinct second keys -- a Fibonacci
// string -- never reaches the radix sort); lists that are small, or whose groups scatter, are sorted.  True when the
// round was done this way: the next list is in (R.act, R.grp2), `m2` long ----
template <int RB>
static bool pivot_round(BuildCtx &c, RoundState &R, u32 &m2) {
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = R.m;
    const bool pivot_force = c.kn.pivot_force;
    const u32 pivot_sub_min = std::max(2u, c.kn.pivot_min / 16u);  // lists of the pivot path that are split again
    PivotArgs base{};
    base.lo_bits = c.lo_bits; base.piv = R.pv_piv; base.cnt64 = R.pv_cnt; base.ebits8 = R.ebits8; base.lbits8 = R.notdone;
    base.rbits8 = R.rbits8; base.tile_e = R.pv_tile_e; base.totals = R.d_pvtot; base.sa = c.sa; base.rank = c.rank;
    base.primary = c.d_primary; base.singles = R.d_nheads;
    u32 out_n = 0;           // entries of the next list (r0 / grp2) written so far
    u64 pv_e = 0, pv_sorted = 0;
    auto classify = [&](u64 *kx, const u32 *vx, u32 n, bool publish, u32 &ne, u32 &nl) {
        PivotArgs pv = base;
        pv.keys = kx; pv.act = vx; pv.m = n;
        const u32 ntl = div_up_u(n, PV_TILE);
        const u64 kw = ((u64)n + 63) / 64;
        CUDA_CHECK(cudaMemsetAsync(R.ebits8 + kw * 8, 0, 16, st));
        CUDA_CHECK(cudaMemsetAsync(R.notdone + kw * 8, 0, 16, st));
        CUDA_CHECK(cudaMemsetAsync(R.rbits8 + kw * 8, 0, 16, st));
        CUDA_CHECK(cudaMemsetAsync(R.d_pvtot, 0, 8, st));
        if (publish) {
            pivot_heads_kernel<<<div_up_u(n, PV_TILE), PV_NT, 0, st>>>(kx, n, c.lo_bits, R.pv_piv, R.pv_cnt);
            KERNEL_CHECK();
        }
        pivot_classify_kernel<<<ntl, PV_NT, 0, st>>>(pv);
        KERNEL_CHECK();
        scan_sum(R.pv_tile_e, ntl, st, R.d_pvtot);
        u32 tot[2] = {0, 0};
        read_back(tot, R.d_pvtot, 8, st);
        ne = tot[0];
        nl = tot[1];
    };
    // radix sort of one list, new ranks, survivors appended to the next list
    auto sort_list = [&](u64 *kx, u32 *vx, u32 n, u64 *ky, u32 *vy, u32 *ng) {
        const u32 *sorted = sort_and_rank<RB>(c, kx, vx, ky, vy, n, ng, R.headB, nullptr, 1);
        int tt = ix.timer.begin("compact", (double)n * 4.0);
        const u32 mB = count_active<false>(R.headB, n, c.tile_counts, c.d_total, st);
        if (mB) scatter_active<false>(R.headB, sorted, ng, n, c.tile_counts, R.r0 + out_n, R.grp2 + out_n, st);
        out_n += mB;
        pv_sorted += n;
        ix.timer.end(tt);
    };
    // one list: keys / values in (kx, vx); (ky, vy) = the other buffer pair over the same index range;
    // ng = as many free words (new ranks by sorted index)
    std::function<void(int, u64 *, u32 *, u32, u64 *, u32 *, u32 *, u32, u32)> process;
    process = [&](int level, u64 *kx, u32 *vx, u32 n, u64 *ky, u32 *vy, u32 *ng, u32 ne, u32 nl) {
        // (level 0 arrives classified)
        bool go = level == 0;
        if (level > 0 && level < 8 && n >= pivot_sub_min) {
            int tt = ix.timer.begin("pivot_classify", (double)n * 16.0);
            classify(kx, vx, n, true, ne, nl);
            ix.timer.end(tt);
            go = (u64)ne * 3 >= (u64)n || pivot_force;
        }
        if (!go) {
            sort_list(kx, vx, n, ky, vy, ng);
            return;
        }
        int tt = ix.timer.begin("pivot_apply", (double)n * 24.0);
        PivotArgs pv = base;
        pv.keys = kx; pv.act = vx; pv.m = n;
        pv.out_act = R.r0 + out_n; pv.out_grp = R.grp2 + out_n; pv.out_base = out_n; pv.dropbits = (u32 *)c.headbits;
        pivot_apply_kernel<<<div_up_u(n, PV_TILE), PV_NT, 0, st>>>(pv);
        KERNEL_CHECK();
        ix.timer.end(tt);
        out_n += ne;
        pv_e += ne;
        const u32 nr = n - ne - nl;
        if (nl | nr) {
            tt = ix.timer.begin("compact_big", (double)n * 0.25 + (double)(nl + nr) * 24.0);
            if (nl) {
                const u32 cnt = count_active<true>(R.notdone, n, c.tile_counts, c.d_total, st);
                if (cnt != nl) throw std::runtime_error("pivot path: L members miscounted (internal error)");
                scatter_pairs(R.notdone, kx, vx, n, c.tile_counts, ky, vy, st);
            }
            if (nr) {
                const u32 cnt = count_active<true>(R.rbits8, n, c.tile_counts, c.d_total, st);
                if (cnt != nr) throw std::runtime_error("pivot path: R members miscounted (internal error)");
                scatter_pairs(R.rbits8, kx, vx, n, c.tile_counts, ky + nl, vy + nl, st);
            }
            ix.timer.end(tt);
            if (nl) process(level + 1, ky, vy, nl, kx, vx, ng, 0, 0);
            if (nr) process(level + 1, ky + nl, vy + nl, nr, kx + nl, vx + nl, ng + nl, 0, 0);
        }
    };
    int t = ix.timer.begin("pivot_classify", (double)m * 16.0);
    u32 n_e = 0, n_l = 0;
    classify(R.rkA, R.act, m, false, n_e, n_l);
    ix.timer.end(t);
    if ((u64)n_e * 3 < (u64)m && !pivot_force) {
        // the groups scatter: nothing was changed, the round goes on as usual; back off 2, 4, 8 ... rounds
        R.pivot_pause = 2 << std::min(R.pivot_fails, 4);
        ++R.pivot_fails;
        return false;
    }
    R.ids_are_heads = false;
    R.chain_on = false;
    R.pivot_fails = 0;
    CUDA_CHECK(cudaMemsetAsync(R.d_nheads, 0, 4, st));
    CUDA_CHECK(cudaMemsetAsync(c.headbits, 0, (((size_t)m + 63) / 64 + 2) * 8, st));  // (no entry of the next list is dropped)
    // (the old list is dead once its L and R members have been copied out: its value buffer is the
    // scratch of the deeper levels; the old group heads are dead already, the keys carry them)
    process(0, R.rkA, R.act, m, R.rkB, R.bvals, R.grp, n_e, n_l);
    ix.stats.sorted_total -= (u64)m - pv_sorted;
    ix.stats.pivot_rounds++;
    ix.stats.pivot_elems += pv_e;
    if (c.bwt_rows) c.need_bwt_fix = true;  // (this path does not write BWT rows)
    // E groups of one member are final: out of the list (rare; through two buffers that are free now)
    u32 n_single = 0;
    read_back(&n_single, R.d_nheads, 4, st);
    m2 = out_n;
    if (n_single) {
        // the survivors are copied to the old list's buffers (free now), which stay the list
        t = ix.timer.begin("compact", (double)out_n * 16.0);
        const u64 kw = ((u64)out_n + 63) / 64;
        pivot_keep_kernel<<<div_up_u(kw, 256), 256, 0, st>>>((u64 *)c.headbits, out_n, kw);
        KERNEL_CHECK();
        m2 = count_active<true>(c.headbits, out_n, c.tile_counts, c.d_total, st);
        if (m2 != out_n - n_single) throw std::runtime_error("pivot path: single-member groups miscounted (internal error)");
        if (m2) scatter_active<true>(c.headbits, R.r0, R.grp2, out_n, c.tile_counts, R.act, R.newgrpT, st);
        std::swap(R.grp2, R.newgrpT);
        ix.timer.end(t);
    } else {
        std::swap(R.act, R.r0);
    }
    return true;
}

// ---- groups of up to RS_GMAX members are ordered where they stand (round_small_kernel); returns how many list
// elements it placed ----
static u32 small_groups_round(BuildCtx &c, RoundState &R) {
    if (R.small_pause > 0) {
        --R.small_pause;
        return 0;
    }
    if (!R.small_on) return 0;
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = R.m;
    int t = ix.timer.begin("round_small", (double)m * 28.0);
    const u64 kw = ((u64)m + 63) / 64;
    CUDA_CHECK(cudaMemsetAsync(c.headbits + kw * 8, 0, 16, st));
    CUDA_CHECK(cudaMemsetAsync(R.notdone + kw * 8, 0, 16, st));
    CUDA_CHECK(cudaMemsetAsync(R.d_handled, 0, 4, st));
    SmallArgs sm{};
    sm.act = R.act; sm.grp = R.grp; sm.keys = R.rkA; sm.m = m; sm.lo_bits = c.lo_bits; sm.sa = c.sa; sm.rank = c.rank;
    sm.vals_out = R.r0; sm.newgrp_out = R.newgrpT; sm.headbits64 = (u64 *)c.headbits; sm.notdone64 = (u64 *)R.notdone;
    sm.primary = c.d_primary; sm.handled = R.d_handled; sm.always_write = R.ids_are_heads ? 0 : 1;
    round_small_kernel<<<div_up_u(m, RS_STEP), RS_NT, 0, st>>>(sm);
    KERNEL_CHECK();
    u32 handled = 0;
    read_back(&handled, R.d_handled, 4, st);
    ix.timer.end(t);
    ix.stats.small_path_elems += handled;
    if ((u64)handled * 32 < (u64)m) {  // (periodic texts: a few giant groups) -- back off 3, 6, 12 ... rounds
        R.small_pause = 3 << std::min(R.small_fails, 4);
        ++R.small_fails;
        R.prefer_pivot = true;  // (large groups: the pivot path is the one to try)
    }
    if (handled && c.bwt_rows) c.need_bwt_fix = true;  // (this path does not write BWT rows)
    return handled;
}

// ---- everything the small-group path left: radix sort of (group, rank) keys, new ranks from the sorted list; then
// the next active set, the survivors of both paths one after the other (groups stay contiguous).  Returns its
// length ----
template <int RB>
static u32 sort_round(BuildCtx &c, RoundState &R, u32 handled) {
    DeviceIndex &ix = c.ix; const cudaStream_t st = c.st;
    const u32 m = R.m, mb = m - handled;
    u64 *bk = R.rkA, *k_other = R.rkB;  // keys / values of the elements that go through the sort
    u32 *bv = R.act;
    if (handled && mb) {
        int t = ix.timer.begin("compact_big", (double)m * 0.125 + (double)mb * 24.0);
        const u32 cnt = count_active<true>(R.notdone, m, c.tile_counts, c.d_total, st);
        if (cnt != mb) throw std::runtime_error("split paths: slot accounting is inconsistent (internal error)");
        scatter_pairs(R.notdone, R.rkA, R.act, m, c.tile_counts, R.rkB, R.bvals, st);
        ix.timer.end(t);
        bk = R.rkB; bv = R.bvals; k_other = R.rkA;
    }
    u8 *hb_big = handled ? R.headB : c.headbits;
    const u32 *sorted_vals = nullptr;
    if (mb) {
        // BWT rows of moved suffixes: one gather per element and round -- kept in the rounds while the
        // active set is small, otherwise one pass over the rows of round 0's active set at the end
        u8 *bwt = m <= R.bwt_small ? c.bwt_rows : nullptr;
        if (c.bwt_rows && !bwt) c.need_bwt_fix = true;
        // (newgrp: the old heads are dead, the keys carry them)
        sorted_vals = sort_and_rank<RB>(c, bk, bv, k_other, R.act2, mb, R.grp, hb_big, bwt, R.ids_are_heads ? 0 : 1);
    }
    int t = ix.timer.begin("compact", (double)m * 4.0);
    // (`act` was read for the last time by the sort or by the compaction of its part; the survivors go to the value
    // buffer the sort left free)
    u32 *dst = sorted_vals == R.act ? R.act2 : R.act;
    u32 mA = 0, mB = 0;
    if (handled) {
        mA = count_active<false>(c.headbits, m, c.tile_counts, c.d_total, st);
        if (mA) scatter_active<false>(c.headbits, R.r0, R.newgrpT, m, c.tile_counts, dst, R.grp2, st);
    }
    if (mb) {
        mB = count_active<false>(hb_big, mb, c.tile_counts, c.d_total, st);
        if (mB) scatter_active<false>(hb_big, sorted_vals, R.grp, mb, c.tile_counts, dst + mA, R.grp2 + mA, st);
    }
    if (dst == R.act2) std::swap(R.act, R.act2);
    ix.timer.end(t);
    return mA + mB;
}

// ---- doubling rounds over the active set ----
template <int RB>
static void doubling_rounds(BuildCtx &c, ActiveList &L) {
    DeviceIndex &ix = c.ix;
    Arena &ar = c.ar;
    const cudaStream_t st = c.st;
    const u32 len = c.len;
    LazyRank &lr = L.lr;
    const u32 m = L.m;
    // complete ranks ("dense") from the start when most suffixes are active; otherwise ranks of
    // retired suffixes are recovered on demand, until a round needs many of them
    if ((u64)m * 2 > (u64)len) {
        go_dense(c, lr);
        if (!L.bucketed) L.rk_free[1] = const_cast<u64 *>(lr.keys0);  // the sorted round-0 keys are dead now
    }
    RoundState R;
    R.m = m; R.act = L.act; R.grp = L.grp;
    R.rkA = L.rk_free[0] ? L.rk_free[0] : ar.get<u64>(m);
    R.rkB = L.rk_free[1] ? L.rk_free[1] : ar.get<u64>(m);
    R.act2 = ar.get<u32>(m); R.grp2 = ar.get<u32>(m);
    R.h = L.depth0 ? (u64)L.depth0 : (u64)L.K;
    R.bwt_small = std::max(1u, len / (u32)c.kn.bwt_round_frac);
    R.chain_on = c.kn.chain && (u64)m * (u64)c.kn.chain_min_frac >= (u64)len;
    R.small_on = c.kn.small_path; R.pivot_on = c.kn.pivot;
    R.cont_bytes = ((size_t)len + 2 * (size_t)CHAIN_CAP + 8192 + 511) & ~(size_t)511;
    const size_t m_init = m;
    const size_t third = (m_init * 4 + 64 + 511) & ~(size_t)511;
    size_t chain_bytes = R.chain_on ? R.cont_bytes + (size_t)len * 4 + ((m_init + 511) & ~(size_t)511) : 0;
    size_t split_bytes = (R.small_on || R.pivot_on) ? 3 * third : 0;
    // the optional paths are dropped, the larger first, rather than running the device out of memory
    const size_t mem_margin = (size_t)2 << 30;
    if (split_bytes > chain_bytes && !ar.can_fit(split_bytes, mem_margin)) {
        split_bytes = 0;
        R.small_on = R.pivot_on = false;
    }
    if (chain_bytes && !ar.can_fit(std::max(chain_bytes, split_bytes), mem_margin)) {
        chain_bytes = 0;
        R.chain_on = false;
        if (split_bytes && !ar.can_fit(split_bytes, mem_margin)) {
            split_bytes = 0;
            R.small_on = R.pivot_on = false;
        }
    }
    u8 *region = ar.get<u8>(std::max<size_t>(std::max(chain_bytes, split_bytes), 512));
    R.cont8 = region; R.cslot = region + R.cont_bytes + (size_t)len * 4; R.chainkey = (u32 *)(region + R.cont_bytes);
    R.r0 = (u32 *)region; R.newgrpT = (u32 *)(region + third); R.bvals = (u32 *)(region + 2 * third);
    R.d_ncont = ar.get<u32>(4); R.d_handled = R.d_ncont + 1; R.d_nheads = R.d_ncont + 2;
    const size_t bm_bytes = ((m_init + 63) / 64 + 2) * 8;
    R.notdone = ar.get<u8>(bm_bytes); R.headB = ar.get<u8>(bm_bytes);
    const size_t pv_entries = (size_t)len / 2 + 2;
    if (R.pivot_on && !ar.can_fit(pv_entries * 12 + 2 * bm_bytes, mem_margin)) R.pivot_on = false;
    R.ebits8 = R.pivot_on ? ar.get<u8>(bm_bytes) : nullptr;
    R.pv_tile_e = R.pivot_on ? ar.get<u32>((size_t)div_up_u(m_init, PV_TILE) + 2) : nullptr;
    R.rbits8 = R.pivot_on ? ar.get<u8>(bm_bytes) : nullptr;
    R.d_pvtot = ar.get<u32>(2);
    R.pv_cnt = R.pivot_on ? ar.get<unsigned long long>(pv_entries) : nullptr;
    R.pv_piv = R.pivot_on ? ar.get<u32>(pv_entries) : nullptr;
    R.prefer_pivot = c.kn.pivot_force;
    if (R.pivot_on && !c.kn.pivot_force && m >= c.kn.pivot_min) {
        CUDA_CHECK(cudaMemsetAsync(R.d_nheads, 0, 4, st));
        count_heads_kernel<<<std::max(1u, std::min(div_up_u(m, 256 * 8), 148u * 8u)), 256, 0, st>>>(R.grp, m, R.d_nheads);
        KERNEL_CHECK();
        u32 nheads = 0;
        read_back(&nheads, R.d_nheads, 4, st);
        R.prefer_pivot = (u64)nheads * 64 <= (u64)m;
    }
    while (R.m > 0) {
        ix.stats.rounds++;
        ix.stats.sorted_total += R.m;
        CUDA_CHECK(cudaMemsetAsync(c.d_lazy, 0, 4, st));
        const bool use_chain = chain_offsets(c, R, lr);
        int t = ix.timer.begin("round_keys", (double)R.m * 16.0);
        const bool try_pivot = R.pivot_on && R.prefer_pivot && R.pivot_pause == 0 && R.m >= c.kn.pivot_min;
        const unsigned kgrid = std::max(1u, std::min(div_up_u(R.m, 256 * 4), 148u * 16u));
        if (lr.sparse)
            make_keys_round_kernel<<<kgrid, 256, 0, st>>>(R.act, R.grp, R.m, lr, R.h, c.lo_bits, use_chain ? R.cslot : nullptr,
                                                          R.chainkey, R.rkA, c.d_lazy, try_pivot ? R.pv_piv : nullptr, R.pv_cnt);
        else
            make_keys_dense_kernel<<<kgrid, 256, 0, st>>>(R.act, R.grp, R.m, c.rank, R.h, len, c.lo_bits,
                                                          use_chain ? R.cslot : nullptr, R.chainkey, R.rkA,
                                                          try_pivot ? R.pv_piv : nullptr, R.pv_cnt);
        KERNEL_CHECK();
        ix.timer.end(t);

        u32 m2 = 0;
        bool pivoted = false;
        if (try_pivot) pivoted = pivot_round<RB>(c, R, m2);
        else if (R.pivot_pause > 0) --R.pivot_pause;
        if (!pivoted) m2 = sort_round<RB>(c, R, small_groups_round(c, R));

        u32 nlazy = 0;
        read_back(&nlazy, c.d_lazy, 4, st);
        ix.stats.lazy_lookups += nlazy;
        std::swap(R.grp, R.grp2);
        R.m = m2;
        R.h *= 2;
        if (R.h > (u64)len * 2 + 2 && R.m > 0)
            throw std::runtime_error("prefix doubling failed to converge (internal error)");
        // a lookup costs several random accesses, completing the ranks one random store per suffix
        if (R.m > 0 && lr.sparse && (u64)nlazy * (u64)c.kn.dense_factor > (u64)len) go_dense(c, lr);
    }
}

// ---- BWT rows the rounds did not maintain, from the final SA ----
static void bwt_fix(BuildCtx &c, u32 m_round0) {
    int t = c.ix.timer.begin("bwt_fix", (double)c.len * 0.125);
    // rows still marked: those round 0 left active minus the ones the pair path made final
    const u64 marked = (u64)m_round0 - (u64)c.ix.stats.pair_placed;
    if (marked * 8 > (u64)c.len)
        bwt_fix_rows_kernel<<<div_up_u(c.len, 256), 256, 0, c.st>>>(c.actbits, c.sa, c.len, c.ix.packed, c.b, c.ix.bwt.ptr,
                                                                    c.d_primary);
    else
        bwt_fix_kernel<<<div_up_u(div_up_u(c.len, 32), 256), 256, 0, c.st>>>(c.actbits, c.sa, c.len, c.ix.packed, c.b,
                                                                            c.ix.bwt.ptr, c.d_primary);
    KERNEL_CHECK();
    c.ix.timer.end(t);
}

template <int RB>
static void build_sa_impl(DeviceIndex &ix, const BuildKnobs &kn, bool want_bwt) {
    typedef rs::Sorter<RB> S;
    constexpr int BINS = 1 << RB;
    cudaStream_t st = ix.stream;
    const u32 len = ix.len;
    ix.stats = BuildStats{};
    ix.stats.sorted_total = len;

    // ---- outputs (stream-ordered allocations that outlive the build) ----
    ix.sa.alloc_output(len, st);
    size_t bwt_bytes = (((size_t)len + 63) / 64 + 1) * 64;
    if (want_bwt) {
        ix.bwt.alloc_output(bwt_bytes, st);
        CUDA_CHECK(cudaMemsetAsync(ix.bwt.ptr + (bwt_bytes - 128), 0, 128, st));
    }
    DevBuf<u32> d_primary(1, st);

    // ---- workspace ----
    BuildCtx c(ix, kn, want_bwt, d_primary.ptr);
    Arena &ar = c.ar;
    // + 2: the bulk copies of round0_msd.cu read whole 16-byte units
    c.keysA = ar.get<u64>((size_t)len + 2); c.keysB = ar.get<u64>((size_t)len + 2);
    c.valsV = ar.get<u32>(len);
    c.rank = ar.get<u32>(len);
    c.actbits = (u32 *)ar.get<u64>(((size_t)len + 63) / 64 + 2);
    c.lookback = ar.get<u64>(S::lookback_words(len));
    c.hist = ar.get<u32>((size_t)8 * BINS); c.uniform = ar.get<u32>(8); c.ticket = ar.get<u32>(1);
    c.headbits = ar.get<u8>((((size_t)len + 63) / 64 + 2) * 8);
    c.tile_counts = ar.get<u32>(div_up_u(len, CP_TILE) + 1);
    c.d_total = ar.get<u32>(1);
    c.d_lazy = ar.get<u32>(1);

    ActiveList L;
    L.act = c.valsV;
    L.lr.rank = c.rank; L.lr.sparse = true; L.lr.sa0 = c.sa; L.lr.packed = ix.packed; L.lr.n = c.n; L.lr.len = len;
    L.lr.bits = c.b;
    if (!round0_bucketed(c, L)) round0_lsd<RB>(c, L);
    const u32 m_round0 = L.m;  // rows round 0 left active (their bits are set in `actbits`)
    c.bwt_rows = (want_bwt && L.bwt_in_sort) ? ix.bwt.ptr : nullptr;

    RankSource rsrc{L.act, L.grp, L.m, false};
    PendingList pend;
    // (a large active set that the pair path takes next: that path orders groups of two and three -- a chance collision
    // next to a pair included -- by the text itself; the tie-break would only add a trip over the list)
    const bool pairs_first = L.bucketed && kn.pairs == 1 && (u64)L.m * 64 >= (u64)len;
    if (L.m && c.b <= 8 && !pairs_first && kn.ext_tiebreak) text_tiebreak(c, L, rsrc, pend);
    if (L.m && c.b <= 8 && pair_path_applies(c, L)) pair_path(c, L, rsrc, pend);
    if (L.m && L.bucketed) scatter_round0_ranks(c, L, rsrc);
    if (L.m) doubling_rounds<RB>(c, L);
    if (c.need_bwt_fix) bwt_fix(c, m_round0);
    read_back(&ix.primary, d_primary.ptr, 4, st);
    if (want_bwt && !L.bwt_in_sort) gather_bwt(ix);  // the element had no room for the preceding symbol
}

void build_suffix_array(DeviceIndex &ix, bool want_bwt) {
    const BuildKnobs kn = read_build_knobs();
    // the digit must hold a whole number of packed symbols
    if (kn.radix_bits == 10 && (10 % ix.pk.bits) == 0) build_sa_impl<10>(ix, kn, want_bwt);
    else build_sa_impl<8>(ix, kn, want_bwt);
}

// inverse suffix array on request (stralg/suffix_array.c:55-62): isa[sa[r]] = r
__global__ void __launch_bounds__(256) inverse_kernel(const u32 *__restrict__ sa, u32 len, u32 *__restrict__ isa) {
    u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < len) isa[sa[r]] = (u32)r;
}

void build_inverse(DeviceIndex &ix) {
    ix.isa.alloc_output(ix.len, ix.stream);
    int t = ix.timer.begin("inverse", (double)ix.len * 8.0);
    inverse_kernel<<<div_up_u(ix.len, 256), 256, 0, ix.stream>>>(ix.sa.ptr, ix.len, ix.isa.ptr);
    KERNEL_CHECK();
    ix.timer.end(t);
}

}  // namespace b200sa
