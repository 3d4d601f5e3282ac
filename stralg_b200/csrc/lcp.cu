// lcp.cu -- LCP array from SA (sm_100a), the values of stralg/suffix_array.c:64-85 (compute_lcp):
//     lcp[0] = 0,  lcp[r] = |longest common prefix of suffixes sa[r-1] and sa[r]|.
//
// Kasai's loop is sequential in text order; here it is reorganised as the permuted LCP array
// (Karkkainen, Manzini, Puglisi, CPM 2009):  Phi[sa[r]] = sa[r-1],  PLCP[i] = lcp(i, Phi[i]).
// If T[i-1] == T[Phi[i]-1] ("reducible") then PLCP[i] = PLCP[i-1] - 1, i.e. v[i] = PLCP[i] + i
// is constant along reducible runs.  Only irreducible positions are compared symbol by symbol
// (64 packed bits per step); comparisons still running after a few words are finished by a
// whole thread block each, so periodic texts (one comparison of length ~n) stay parallel.
//
//   phi_kernel            Phi scatter                                 (suffix_array.c:55-62 analogue)
//   plcp_irreducible      v[i] at irreducible i, marker elsewhere, long pairs queued
//   plcp_long             block-cooperative finish of queued pairs
//   plcp tile_last/scan/fill   "copy last defined value" scan -> v[i] everywhere
//   lcp_gather            lcp[r] = v[sa[r]] - sa[r]
#include "engine.h"
#include "round0_msd.cuh"  // window_at
#include "scan.cuh"

namespace b200sa {

static constexpr u32 UNDEF = 0xFFFFFFFFu;

__device__ __forceinline__ u64 lcp_window(const u64 *__restrict__ packed, u64 sym_index, int bits) {
    u64 bitpos = sym_index * (u64)bits;
    u64 wi = bitpos >> 6;
    unsigned o = (unsigned)(bitpos & 63);
    u64 hi = packed[wi];
    if (o == 0) return hi;
    return (hi << o) | (packed[wi + 1] >> (64 - o));
}

__global__ void __launch_bounds__(256) phi_kernel(const u32 *__restrict__ sa, u32 len, u32 *__restrict__ phi) {
    u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= len) return;
    u32 s = sa[r];
    phi[s] = r ? sa[r - 1] : UNDEF;
}

struct LongPair {
    u32 i, matched;
};

static constexpr int T1_WORDS = 4;  // words compared by the per-position thread before queueing

__global__ void __launch_bounds__(256) plcp_irreducible_kernel(const u64 *__restrict__ packed, int bits, u32 n,
                                                               const u32 *__restrict__ phi, u32 *__restrict__ v,
                                                               LongPair *__restrict__ queue,
                                                               unsigned long long *__restrict__ queue_count,
                                                               u64 queue_cap) {
    u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx > n) return;
    const u32 i = (u32)idx;
    const u32 j = phi[i];
    const int cpw = 64 / bits;
    if (j == UNDEF) {  // the first suffix in SA order (the sentinel suffix): lcp[0] = 0
        v[i] = i;
        return;
    }
    bool reducible = i > 0 && j > 0 && sym_at(packed, i - 1, bits) == sym_at(packed, j - 1, bits);
    if (reducible) {
        v[i] = UNDEF;
        return;
    }
    // the shorter suffix ends first and its sentinel matches nothing
    const u32 maxl = n - (i > j ? i : j);
    u32 l = 0;
    bool done = maxl == 0;
#pragma unroll 1
    for (int w = 0; w < T1_WORDS && !done; ++w) {
        u64 x = lcp_window(packed, (u64)i + l, bits) ^ lcp_window(packed, (u64)j + l, bits);
        if (x) {
            l += (u32)(__clzll((long long)x) / bits);
            done = true;
        } else {
            l += cpw;
        }
        if (l >= maxl) done = true;
    }
    if (!done) {
        unsigned long long slot = atomicAdd(queue_count, 1ull);
        if (slot < queue_cap) {
            queue[slot].i = i;
            queue[slot].matched = l;
            v[i] = i;  // placeholder (defined); plcp_long_kernel writes the final value
            return;
        }
        // queue full (cannot happen within the 2 n log n bound, kept for safety): finish here
        while (l < maxl) {
            u64 x = lcp_window(packed, (u64)i + l, bits) ^ lcp_window(packed, (u64)j + l, bits);
            if (x) {
                l += (u32)(__clzll((long long)x) / bits);
                break;
            }
            l += cpw;
        }
    }
    v[i] = (l < maxl ? l : maxl) + i;
}

__global__ void __launch_bounds__(256) plcp_long_kernel(const u64 *__restrict__ packed, int bits, u32 n,
                                                        const u32 *__restrict__ phi, u32 *__restrict__ v,
                                                        const LongPair *__restrict__ queue,
                                                        const unsigned long long *__restrict__ queue_count,
                                                        u64 queue_cap) {
    __shared__ u32 wmin[8];
    __shared__ u32 result;
    const int cpw = 64 / bits;
    const u64 count = *queue_count < queue_cap ? *queue_count : queue_cap;
    for (u64 q = blockIdx.x; q < count; q += gridDim.x) {
        const u32 i = queue[q].i;
        const u32 j = phi[i];
        const u32 maxl = n - (i > j ? i : j);
        u64 l0 = queue[q].matched;
        u32 found = UNDEF;
        while (true) {
            u64 off = l0 + (u64)threadIdx.x * cpw;
            u32 cand = UNDEF;
            if (off >= maxl) {
                cand = maxl;
            } else {
                u64 x = lcp_window(packed, (u64)i + off, bits) ^ lcp_window(packed, (u64)j + off, bits);
                if (x) {
                    u64 p = off + (u64)(__clzll((long long)x) / bits);
                    cand = p < maxl ? (u32)p : maxl;
                } else if (off + cpw >= maxl) {
                    cand = maxl;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
            if (lane_id() == 0) wmin[threadIdx.x >> 5] = cand;
            __syncthreads();
            if (threadIdx.x == 0) {
                u32 m = UNDEF;
                for (int w = 0; w < 8; ++w) m = min(m, wmin[w]);
                result = m;
            }
            __syncthreads();
            found = result;
            __syncthreads();
            if (found != UNDEF) break;
            l0 += (u64)blockDim.x * cpw;
        }
        if (threadIdx.x == 0) v[i] = found + i;
    }
}

// ---- "last defined value" scan over v[0..count) ------------------------------------------------
static constexpr int FL_NT = 256, FL_IPT = 8, FL_TILE = FL_NT * FL_IPT;

__device__ __forceinline__ u32 pick(u32 left, u32 right) { return right != UNDEF ? right : left; }
struct PickOp {
    __device__ __forceinline__ u32 operator()(u32 left, u32 right) const { return pick(left, right); }
};

__global__ void __launch_bounds__(FL_NT) plcp_tile_last_kernel(const u32 *__restrict__ v, u64 count,
                                                               u32 *__restrict__ tile_last) {
    __shared__ u32 wl[FL_NT / 32];
    u64 base = (u64)blockIdx.x * FL_TILE + (u64)threadIdx.x * FL_IPT;
    u32 last = UNDEF;
#pragma unroll
    for (int q = 0; q < FL_IPT; ++q)
        if (base + q < count) last = pick(last, v[base + q]);
    last = warp_inclusive(last, PickOp());
    if (lane_id() == 31) wl[threadIdx.x >> 5] = last;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 m = UNDEF;
        for (int w = 0; w < FL_NT / 32; ++w) m = pick(m, wl[w]);
        tile_last[blockIdx.x] = m;
    }
}

// exclusive "last defined" scan over the tile aggregates, in place (single block)
__global__ void __launch_bounds__(1024) plcp_scan_tiles_kernel(u32 *__restrict__ tile_last, u32 ntiles) {
    cta_exclusive_scan(
        ntiles, [=](u32 i) { return tile_last[i]; }, [=](u32 i, u32 e) { tile_last[i] = e; }, PickOp(), UNDEF);
}

__global__ void __launch_bounds__(FL_NT) plcp_fill_kernel(u32 *__restrict__ v, u64 count,
                                                          const u32 *__restrict__ tile_carry) {
    __shared__ u32 wl[FL_NT / 32];
    u64 base = (u64)blockIdx.x * FL_TILE + (u64)threadIdx.x * FL_IPT;
    u32 x[FL_IPT];
    u32 last = UNDEF;
#pragma unroll
    for (int q = 0; q < FL_IPT; ++q) {
        x[q] = base + q < count ? v[base + q] : UNDEF;
        last = pick(last, x[q]);
    }
    const u32 incl = warp_inclusive(last, PickOp());
    if (lane_id() == 31) wl[threadIdx.x >> 5] = incl;
    const u32 excl = warp_exclusive(incl, last, PickOp(), UNDEF);
    __syncthreads();
    u32 pre = tile_carry[blockIdx.x];
    for (unsigned w = 0; w < (threadIdx.x >> 5); ++w) pre = pick(pre, wl[w]);
    u32 run = pick(pre, excl);
#pragma unroll
    for (int q = 0; q < FL_IPT; ++q) {
        run = pick(run, x[q]);
        if (base + q < count && x[q] == UNDEF) v[base + q] = run;
    }
}

__global__ void __launch_bounds__(256) lcp_gather_kernel(const u32 *__restrict__ sa, const u32 *__restrict__ v,
                                                         u32 len, u32 *__restrict__ lcp) {
    u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= len) return;
    u32 s = sa[r];
    lcp[r] = r ? v[s] - s : 0u;
}

// ---------------------------------------------------------------------------------------------
// Direct path for texts without long repeats: row r compares the suffixes SA[r-1] and SA[r] on the
// packed text, 64 bits per step (two random word pairs per row instead of the Phi scatter, the
// PLCP pass and the final gather).  A comparison still running after DIRECT_CAP symbols raises
// `overflow`; the caller then runs the Phi / PLCP pipeline, whose cost does not depend on the
// LCP values.  The unique sentinel ends every comparison (stralg/suffix_array.c:73-84): the
// common prefix cannot pass the end of the shorter suffix.
// ---------------------------------------------------------------------------------------------
static constexpr u32 DIRECT_CAP = 4096;

__global__ void __launch_bounds__(256) lcp_direct_kernel(const u64 *__restrict__ packed, int bits, u32 n,
                                                         const u32 *__restrict__ sa, u32 len,
                                                         u32 *__restrict__ lcp, int *__restrict__ overflow) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= len) return;
    if (r == 0) {
        lcp[0] = 0;
        return;
    }
    const u32 a = sa[r - 1], b = sa[r];
    const u32 lim = n - max(a, b);  // symbols the shorter suffix has before the sentinel
    const u32 spw = 64u / (u32)bits;
    u32 l = 0;
    while (l < lim) {
        const u64 x = window_at(packed, (u64)a + l, bits) ^ window_at(packed, (u64)b + l, bits);
        if (x) {
            l += (u32)__clzll((long long)x) / (u32)bits;
            break;
        }
        l += spw;
        if (l >= DIRECT_CAP) {
            *overflow = 1;
            break;
        }
    }
    lcp[r] = min(l, lim);
}

void build_lcp(DeviceIndex &ix) {
    cudaStream_t st = ix.stream;
    const u32 len = ix.len, n = ix.n;
    const int bits = ix.pk.bits;
    Arena &ar = *ix.arena;
    // texts that needed few doubling rounds have no long repeats to speak of: try the direct path
    static const bool no_direct = getenv("B200SA_LCP_NO_DIRECT") != nullptr;
    if (!no_direct && ix.stats.rounds <= 3) {
        ix.lcp.alloc_output(len, st);
        int *d_over = ar.get<int>(1);
        CUDA_CHECK(cudaMemsetAsync(d_over, 0, 4, st));
        int t = ix.timer.begin("lcp_direct", (double)len * 12.0);
        lcp_direct_kernel<<<div_up_u(len, 256), 256, 0, st>>>(ix.packed, bits, n, ix.sa.ptr, len, ix.lcp.ptr, d_over);
        KERNEL_CHECK();
        ix.timer.end(t);
        int over = 0;
        CUDA_CHECK(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        if (!over) return;
    }
    u32 *phi = ar.get<u32>(len), *v = ar.get<u32>(len);
    int t = ix.timer.begin("lcp_phi", (double)len * 8.0);
    phi_kernel<<<div_up_u(len, 256), 256, 0, st>>>(ix.sa.ptr, len, phi);
    KERNEL_CHECK();
    ix.timer.end(t);

    // every queued pair consumed T1_WORDS full words first, and irreducible LCPs sum to at most
    // 2 n log2 n symbols, which bounds the queue; len entries is a safe (and simple) capacity
    const u64 qcap = (u64)len / 2 + 1024;
    LongPair *queue = ar.get<LongPair>(qcap);
    unsigned long long *qcount = ar.get<unsigned long long>(1);
    CUDA_CHECK(cudaMemsetAsync(qcount, 0, 8, st));
    t = ix.timer.begin("lcp_irreducible", (double)len * 8.0);
    plcp_irreducible_kernel<<<div_up_u((u64)n + 1, 256), 256, 0, st>>>(ix.packed, bits, n, phi, v,
                                                                       queue, qcount, qcap);
    KERNEL_CHECK();
    plcp_long_kernel<<<148 * 4, 256, 0, st>>>(ix.packed, bits, n, phi, v, queue, qcount, qcap);
    KERNEL_CHECK();
    ix.timer.end(t);

    t = ix.timer.begin("lcp_fill", (double)len * 8.0);
    u32 ntiles = div_up_u(len, FL_TILE);
    u32 *tile_last = ar.get<u32>(ntiles);
    plcp_tile_last_kernel<<<ntiles, FL_NT, 0, st>>>(v, len, tile_last);
    KERNEL_CHECK();
    plcp_scan_tiles_kernel<<<1, 1024, 0, st>>>(tile_last, ntiles);
    KERNEL_CHECK();
    plcp_fill_kernel<<<ntiles, FL_NT, 0, st>>>(v, len, tile_last);
    KERNEL_CHECK();
    ix.timer.end(t);

    if (!ix.lcp.ptr) ix.lcp.alloc_output(len, st);
    t = ix.timer.begin("lcp_gather", (double)len * 12.0);
    lcp_gather_kernel<<<div_up_u(len, 256), 256, 0, st>>>(ix.sa.ptr, v, len, ix.lcp.ptr);
    KERNEL_CHECK();
    ix.timer.end(t);
}

}  // namespace b200sa
