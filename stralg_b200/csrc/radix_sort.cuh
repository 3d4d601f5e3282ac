// radix_sort.cuh -- stable LSD radix sort of (u64 key, u32 value) pairs for sm_100a.
//
// One kernel per digit ("onesweep"): every CTA takes the next tile from an atomic ticket, ranks
// its keys per warp with match.any + per-warp shared-memory histograms, publishes its per-digit
// counts and resolves the counts of all earlier tiles with a decoupled look-back, reorders the
// tile in shared memory and writes digit runs out coalesced.  Global digit offsets come from a
// histogram computed once for all passes (hist_kernel, or the c-mer histogram of sa_build.cu
// for round 0).  Replaces the byte-wise CPU radix passes of stralg/skew.c:53-99 and the bucket
// scatters of stralg/sa_is.c:203-263; none of that code is reused.
#pragma once
#include "scan.cuh"

namespace b200sa {
namespace rs {

static constexpr u64 LB_VALUE_MASK = (1ull << 62) - 1;
static constexpr u64 LB_AGGREGATE = 1ull << 62;
static constexpr u64 LB_PREFIX = 1ull << 63;

// ---------------------------------------------------------------------------------------------
// Histogram of every digit of every pass in one read of the keys.
// hist layout: [npass][BINS] u32.  Pass p covers bits [begin_bit + p*RB, min(.., end_bit)).
// ---------------------------------------------------------------------------------------------
template <int RB>
__global__ void __launch_bounds__(512) hist_kernel(const u64 *__restrict__ keys, u32 n, int begin_bit,
                                                   int end_bit, int npass, u32 *__restrict__ hist) {
    constexpr int BINS = 1 << RB;
    extern __shared__ u32 sh_hist[];
    for (int i = threadIdx.x; i < npass * BINS; i += blockDim.x) sh_hist[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    // four keys in flight per thread before the first shared atomic
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 4 * stride) {
        u64 kk[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) kk[q] = i + q * stride < n ? ld_stream_u64(keys + i + q * stride) : 0ull;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (i + q * stride >= n) break;
            u64 k = kk[q] >> begin_bit;
            int bits_left = end_bit - begin_bit;
#pragma unroll 1
            for (int p = 0; p < npass; ++p) {
                u32 mask = bits_left >= RB ? (u32)(BINS - 1) : ((1u << bits_left) - 1u);
                // (same-address shared atomics of a warp are combined by the hardware: a warp-uniform fast path
                // with a shuffle and a vote per digit measured 2.4x SLOWER on periodic texts)
                atomicAdd(&sh_hist[p * BINS + ((u32)k & mask)], 1u);
                k >>= RB;
                bits_left -= RB;
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npass * BINS; i += blockDim.x) {
        u32 v = sh_hist[i];
        if (v) atomicAdd(&hist[i], v);
    }
}

// In-place exclusive scan of each pass's histogram; uniform[p] = 1 when one bin holds all n keys
// (that pass is the identity permutation and is skipped by the host).
template <int RB>
__global__ void __launch_bounds__(256) scan_hist_kernel(u32 *__restrict__ hist, u32 n, u32 *__restrict__ uniform) {
    constexpr int BINS = 1 << RB;
    constexpr int NT = 256;
    constexpr int DPT = (BINS + NT - 1) / NT;
    __shared__ u32 warp_tot[NT / 32];
    __shared__ u32 any_full;
    u32 *h = hist + (size_t)blockIdx.x * BINS;
    if (threadIdx.x == 0) any_full = 0;
    __syncthreads();
    u32 v[DPT];
    u32 sum = 0;
    bool full = false;
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = threadIdx.x * DPT + q;
        v[q] = d < BINS ? h[d] : 0;
        full |= (v[q] == n);
        sum += v[q];
    }
    if (full) any_full = 1;
    u32 run = block_exclusive<NT>(sum, warp_tot);
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = threadIdx.x * DPT + q;
        if (d < BINS) h[d] = run;
        run += v[q];
    }
    if (threadIdx.x == 0) uniform[blockIdx.x] = any_full;
}

// ---------------------------------------------------------------------------------------------
// One onesweep pass.
// ---------------------------------------------------------------------------------------------
template <int RB, int NT, int IPT>
struct PassCfg {
    static constexpr int BINS = 1 << RB;
    static constexpr int TILE = NT * IPT;
    static constexpr int WARPS = NT / 32;
    static constexpr int DPT = (BINS + NT - 1) / NT;  // digits owned per thread
    static constexpr int RBATCH = IPT % 6 == 0 ? 6 : 4;  // items ranked per match/atomic/shuffle batch
    static constexpr size_t SMEM = (size_t)TILE * 8 + (size_t)TILE * 4 + (size_t)WARPS * BINS * 4 +
                                   (size_t)BINS * 4 * 2 + 64 * 4;
};

template <int RB, int NT, int IPT>
__global__ void __launch_bounds__(NT, (NT <= 256 ? 4 : (NT <= 384 ? 2 : 2))) onesweep_pass_kernel(const u64 *__restrict__ kin, const u32 *__restrict__ vin,
                                                           u64 *__restrict__ kout, u32 *__restrict__ vout, u32 n,
                                                           int shift, u32 digit_mask,
                                                           const u32 *__restrict__ digit_base,
                                                           u64 *__restrict__ lookback, u32 *__restrict__ ticket) {
    typedef PassCfg<RB, NT, IPT> Cfg;
    constexpr int BINS = Cfg::BINS, TILE = Cfg::TILE, WARPS = Cfg::WARPS, DPT = Cfg::DPT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 *keys_s = (u64 *)smem_raw;
    u32 *vals_s = (u32 *)(keys_s + TILE);
    u32 *warp_hist = (u32 *)(vals_s + TILE);       // [WARPS][BINS]
    u32 *tile_start = (u32 *)(warp_hist + WARPS * BINS);  // [BINS]
    u32 *adj = tile_start + BINS;                  // [BINS]
    u32 *misc = adj + BINS;                        // [64]: warp totals, tile id

    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) misc[63] = atomicAdd(ticket, 1u);
    // zero this warp's histogram row
    {
        u32 *row32 = warp_hist + warp * BINS;
        for (int i = lane; i < BINS; i += 32) row32[i] = 0;
    }
    __syncthreads();
    const u32 tile = misc[63];
    const u64 base = (u64)tile * TILE;
    const u32 nvalid = (u32)((u64)n - base < (u64)TILE ? (u64)n - base : (u64)TILE);
    const u64 wbase = base + (u64)warp * (32 * IPT) + lane;

    // ---- load keys (warp-contiguous, coalesced) ----
    u64 k[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        u64 idx = wbase + (u64)j * 32;
        k[j] = idx < n ? ld_stream_u64(kin + idx) : ~0ull;
    }
    // ---- per-warp stable ranking ----
    // Batches of RBATCH items keep several match / shared-atomic / shuffle chains in flight.
    // The shared atomics of one warp retire in program order (and __syncwarp orders them between
    // lanes), so an earlier item always receives the smaller offset: the ranking is stable.
    u32 *myhist = warp_hist + warp * BINS;
    u32 pos[IPT];
    const unsigned lt = lanemask_lt();
    constexpr int RBATCH = Cfg::RBATCH;
#pragma unroll
    for (int j0 = 0; j0 < IPT; j0 += RBATCH) {
        unsigned peers[RBATCH];
        u32 dg[RBATCH], before[RBATCH];
#pragma unroll
        for (int b = 0; b < RBATCH; ++b) {
            dg[b] = (u32)(k[j0 + b] >> shift) & digit_mask;
            peers[b] = __match_any_sync(0xffffffffu, dg[b]);
        }
#pragma unroll
        for (int b = 0; b < RBATCH; ++b) {
            before[b] = 0;
            if ((peers[b] & lt) == 0) before[b] = atomicAdd(&myhist[dg[b]], (u32)__popc(peers[b]));
            __syncwarp();
        }
#pragma unroll
        for (int b = 0; b < RBATCH; ++b) {
            int leader = __ffs(peers[b]) - 1;
            before[b] = __shfl_sync(0xffffffffu, before[b], leader);
            pos[j0 + b] = before[b] + __popc(peers[b] & lt);
        }
    }
    // values: issued now, consumed after the digit scan (their latency hides behind it)
    u32 v[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        u64 idx = wbase + (u64)j * 32;
        v[j] = idx < n ? ld_stream_u32(vin + idx) : 0u;
    }
    __syncthreads();

    // ---- per digit: exclusive scan over warps, tile totals ----
    u32 cnt[DPT];
    u32 tsum = 0;
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = tid * DPT + q;
        u32 run = 0;
        if (d < BINS) {
#pragma unroll
            for (int w = 0; w < WARPS; ++w) {
                u32 c = warp_hist[w * BINS + d];
                warp_hist[w * BINS + d] = run;
                run += c;
            }
            // publish this tile's count right away so later tiles can make progress
            u64 flag = tile == 0 ? LB_PREFIX : LB_AGGREGATE;
            st_relaxed_u64(lookback + (size_t)tile * BINS + d, flag | run);
        }
        cnt[q] = run;
        tsum += run;
    }
    // block exclusive scan of the tile's digit counts -> tile_start[]
    {
        u32 run = block_exclusive<NT>(tsum, misc);
#pragma unroll
        for (int q = 0; q < DPT; ++q) {
            int d = tid * DPT + q;
            if (d < BINS) tile_start[d] = run;
            run += cnt[q];
        }
    }
    __syncthreads();

    // ---- move keys to their tile-local sorted slot ----
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        u32 d = (u32)(k[j] >> shift) & digit_mask;
        u32 p = pos[j] + tile_start[d] + warp_hist[warp * BINS + d];
        keys_s[p] = k[j];
        vals_s[p] = v[j];
    }
    // ---- decoupled look-back: exclusive count of each digit over all earlier tiles ----
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
        int d = tid * DPT + q;
        if (d < BINS) {
            u32 excl = 0;
            if (tile > 0) {
                // LB_UNROLL predecessors are fetched per step so their L2 latencies overlap
                constexpr int LB_UNROLL = 8;
                int t = (int)tile - 1;
                bool done = false;
                while (!done) {
                    u64 sv[LB_UNROLL];
#pragma unroll
                    for (int u = 0; u < LB_UNROLL; ++u)
                        sv[u] = t - u >= 0 ? ld_relaxed_u64(lookback + (size_t)(t - u) * BINS + d) : LB_PREFIX;
#pragma unroll
                    for (int u = 0; u < LB_UNROLL; ++u) {
                        if (done) break;
                        u64 sx = sv[u];
                        while ((sx >> 62) == 0) sx = ld_relaxed_u64(lookback + (size_t)(t - u) * BINS + d);
                        excl += (u32)(sx & LB_VALUE_MASK);
                        if (sx & LB_PREFIX) done = true;
                    }
                    t -= LB_UNROLL;
                }
                st_relaxed_u64(lookback + (size_t)tile * BINS + d, LB_PREFIX | (u64)(excl + cnt[q]));
            }
            adj[d] = digit_base[d] + excl - tile_start[d];
        }
    }
    __syncthreads();

    // ---- write out: consecutive threads write consecutive slots of a digit run ----
    for (u32 i = tid; i < nvalid; i += NT) {
        u64 key = keys_s[i];
        u32 d = (u32)(key >> shift) & digit_mask;
        u32 g = i + adj[d];
        kout[g] = key;
        vout[g] = vals_s[i];
    }
}

// ---------------------------------------------------------------------------------------------
// Host driver.
// ---------------------------------------------------------------------------------------------
struct SortPlan {
    int radix_bits;
    int begin_bit, end_bit;
    int npass;
};

template <int RB>
struct Sorter {
    static constexpr int BINS = 1 << RB;
    // pass-kernel shape
    static constexpr int PASS_NT = 256, PASS_IPT = 12;
    typedef PassCfg<RB, PASS_NT, PASS_IPT> Cfg;

    static size_t lookback_words(u32 n) { return (size_t)div_up_u(n, Cfg::TILE) * BINS; }

    static void configure() {
        static PerDeviceOnce once;
        if (once.first())
            CUDA_CHECK(cudaFuncSetAttribute(hist_kernel<RB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            8 * BINS * 4));
    }

    // Generic all-pass histogram over existing keys.  hist must hold npass*BINS u32.
    static void histogram(const u64 *keys, u32 n, int begin_bit, int end_bit, int npass, u32 *hist,
                          cudaStream_t st) {
        configure();
        CUDA_CHECK(cudaMemsetAsync(hist, 0, (size_t)npass * BINS * 4, st));
        if (n == 0) return;
        unsigned blocks = div_up_u(n, 512 * 16);
        if (blocks > 148 * 4) blocks = 148 * 4;
        hist_kernel<RB><<<blocks, 512, (size_t)npass * BINS * 4, st>>>(keys, n, begin_bit, end_bit, npass, hist);
        KERNEL_CHECK();
    }

    static void scan(u32 *hist, u32 n, int npass, u32 *uniform, cudaStream_t st) {
        scan_hist_kernel<RB><<<npass, 256, 0, st>>>(hist, n, uniform);
        KERNEL_CHECK();
    }

    // One pass; digit_base = the scanned histogram row of this pass.
    static void pass(const u64 *kin, const u32 *vin, u64 *kout, u32 *vout, u32 n, int shift, int bits,
                     const u32 *digit_base, u64 *lookback, u32 *ticket, cudaStream_t st) {
        u32 mask = bits >= RB ? (u32)(BINS - 1) : ((1u << bits) - 1u);
        static PerDeviceOnce once;
        if (once.first())
            CUDA_CHECK(cudaFuncSetAttribute(onesweep_pass_kernel<RB, PASS_NT, PASS_IPT>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
        unsigned tiles = div_up_u(n, Cfg::TILE);
        CUDA_CHECK(cudaMemsetAsync(lookback, 0, (size_t)tiles * BINS * 8, st));
        CUDA_CHECK(cudaMemsetAsync(ticket, 0, 4, st));
        onesweep_pass_kernel<RB, PASS_NT, PASS_IPT><<<tiles, PASS_NT, Cfg::SMEM, st>>>(kin, vin, kout, vout, n, shift, mask,
                                                                                     digit_base, lookback, ticket);
        KERNEL_CHECK();
    }

    struct Sorted {
        u64 *keys;   // the buffer pair that holds the sorted pairs
        u32 *vals;
        int passes;  // passes run (the others had one digit for every key)
    };

    // Stable sort of (keys[0], vals[0]) on the low key_bits (<= 64) bits of the keys; (keys[1], vals[1]) is the
    // other buffer pair.  One histogram of every digit, then one pass per digit that is not the same for every
    // key.  Work buffers: hist 8 * BINS words, uniform 8 words, lookback lookback_words(n), ticket 1 word.
    // With a timer: stages "round_hist" (histogram, scan and the read-back of the uniform flags) and "radix_pass".
    static Sorted sort(u64 *keys[2], u32 *vals[2], u32 n, int key_bits, u32 *hist, u32 *uniform, u64 *lookback,
                       u32 *ticket, cudaStream_t st, StageTimer *timer = nullptr) {
        if (key_bits <= 0 || n < 2) return Sorted{keys[0], vals[0], 0};
        const int npass = (key_bits + RB - 1) / RB;
        u32 huniform[8];
        int t = timer ? timer->begin("round_hist", (double)n * 8.0) : -1;
        histogram(keys[0], n, 0, key_bits, npass, hist, st);
        scan(hist, n, npass, uniform, st);
        read_back(huniform, uniform, (size_t)npass * 4, st);
        if (timer) timer->end(t);
        int in = 0, passes = 0;
        for (int p = 0; p < npass; ++p) {
            if (huniform[p]) continue;
            const int bits_here = key_bits - p * RB < RB ? key_bits - p * RB : RB;
            t = timer ? timer->begin("radix_pass", (double)n * 24.0) : -1;
            pass(keys[in], vals[in], keys[in ^ 1], vals[in ^ 1], n, p * RB, bits_here, hist + (size_t)p * BINS,
                 lookback, ticket, st);
            if (timer) timer->end(t);
            in ^= 1;
            ++passes;
        }
        return Sorted{keys[in], vals[in], passes};
    }

    // the same with work buffers of its own, from the library's pool
    static Sorted sort(u64 *keys[2], u32 *vals[2], u32 n, int key_bits, cudaStream_t st) {
        DevBuf<u64> lookback(lookback_words(n), st);
        DevBuf<u32> hist((size_t)8 * BINS, st), uniform(8, st), ticket(1, st);
        return sort(keys, vals, n, key_bits, hist.ptr, uniform.ptr, lookback.ptr, ticket.ptr, st);
    }
};

}  // namespace rs
}  // namespace b200sa
