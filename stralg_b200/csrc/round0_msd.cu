// round0_msd.cu -- the initial K-symbol sort of suffix-array construction as an MSD bucket sort
// (sm_100a).  Replaces, for round 0 only, the LSD passes of radix_sort.cuh: every suffix is one
// 8-byte element
//
//      [ rest of the key : KB - D1 bits | preceding symbol : pb bits | suffix start : 32 bits ]
//
// that is partitioned by the leading digits of its K-symbol key (1..3 levels, <= 1024 bins each,
// a digit that has been consumed is implied by the bucket and dropped), until buckets fit one
// SM's shared memory, where they are ordered by the remaining key bits.  MSD partitioning needs
// no stability, so ranking inside a tile is ONE shared-memory atomicAdd per element (2.7 SM
// cycles per warp on B200 against 62 for match.any, tools/ubench.cu) and tiles reserve their
// output ranges with global atomics instead of a look-back chain.  The last kernel emits, per
// bucket, what round 0 of prefix doubling needs (stralg/sa_is.c:295-336 "naming" is the
// reference's counterpart): SA order, BWT rows (stralg/bwt.c:13-20), and for suffixes whose
// K-symbol key is shared: the rank of their group, the valid bit and a slot in the active list.
//
// Suffixes whose K-window reaches the sentinel ("short", at most K of them) are padded with the
// smallest symbol; among equal padded keys they precede every long suffix, shortest first, which
// is strcmp order on NUL-terminated strings (stralg/suffix_array.c:26-30).
//
// The key is the K raw symbol fields of the packed text, or, for alphabets that leave most codes of
// a symbol field unused (DNA with N, amino acids), the base-nsym number the K symbols spell (DenseKey,
// round0_msd.cuh): any monotone, injective map of K-symbol prefixes serves, and only the level-1
// kernels that read the text know which one is in use.
#include "round0_msd.cuh"
#include "scan.cuh"

#include <vector>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace b200sa {

static constexpr int MSD_MAXBINS = 1024;           // digits of up to 10 bits
static constexpr int P_MAXBINS = MSD_MAXBINS;
// partition kernels
static constexpr int P_NT = 512;
static constexpr int P_IPT = 8;
static constexpr int P_TILE = P_NT * P_IPT;  // 4096 elements
// local sort
static constexpr int L3_NT = 512;
static constexpr int L3_TSZ = 1792;                // a tile owns the buckets that START in its span
static constexpr int L3_MAXB = 3328;               // largest bucket the fast path accepts
static constexpr int L3_CAP = L3_TSZ + L3_MAXB;    // 5120 elements of a tile in shared memory
static constexpr int L3_IPT = L3_CAP / L3_NT;      // 10
static constexpr int L3_CTAS = 3;                  // resident CTAs per SM
static constexpr int L3_CROWD = 64;                // more elements than this in one sub-bin -> robust kernel
static constexpr int L3_MASKW = 160;               // words of segment-start bits (>= L3_CAP / 32, a multiple of 32)
static_assert(L3_CAP % L3_NT == 0 && L3_MASKW * 32 >= L3_CAP && L3_MASKW % 32 == 0, "local-sort geometry");
static constexpr int RB_N = 8192;                  // robust kernel: bitonic network size

static unsigned sm_count(int device) {
    static int cached[64] = {0};
    int &c = cached[device & 63];
    if (!c) CUDA_CHECK(cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, device));
    return (unsigned)c;
}

// ---------------------------------------------------------------------------------------------
// Planning
// ---------------------------------------------------------------------------------------------
static int bit_length_u64(u64 v) {
    int l = 0;
    while (v) { ++l; v >>= 1; }
    return l;
}
static u64 pow_u64(u64 x, int k) {
    u64 r = 1;
    for (int i = 0; i < k; ++i) r *= x;
    return r;
}

// Dense keys (see DenseKey): digits are not tied to symbol boundaries, a partly used top digit is
// accounted for when the bucket bits are chosen.
static bool msd_make_plan_dense(u32 len, u32 nsym, int b, MsdPlan &pl, const u64 *sym_counts) {
    const int dmax = std::max(4, std::min(10, env_int("B200SA_MSD_DMAX", 10)));
    const int target = std::max(1, env_int("B200SA_MSD_AVG", 3000));
    int log2len = 0;
    while ((1ull << log2len) < (u64)len) ++log2len;
    // bits a symbol really carries: the order-0 entropy of the text when the letter counts are known (a rare
    // letter -- N in DNA -- takes a digit value but adds next to nothing), else that of equally likely letters
    double eff = std::log2((double)nsym);
    if (sym_counts) {
        double tot = 0.0, H = 0.0;
        for (u32 a = 1; a <= nsym; ++a) tot += (double)sym_counts[a];
        for (u32 a = 1; a <= nsym && tot > 0.0; ++a)
            if (sym_counts[a]) {
                const double p = (double)sym_counts[a] / tot;
                H -= p * std::log2(p);
            }
        if (tot > 0.0) eff = std::min(eff, std::max(0.25, H));
    }
    const int margin = env_int("B200SA_KEY_MARGIN", 8);
    const int k_wanted = std::max(1, (int)std::ceil((log2len + margin) / eff));
    int best_K = 0;
    for (int pb = b; pb >= 0; pb -= b) {
        int K = std::min(k_wanted, 128 / b - (pb ? 1 : 0));  // a 128-bit window holds prev + K symbols
        const int kf = env_int("B200SA_MSD_K", 0);
        if (kf > 0) K = std::min(K, kf);
        for (; K >= 1; --K) {
            const u64 span = pow_u64(nsym, K);            // keys are 0 .. span - 1
            const int KB = bit_length_u64(span - 1);
            if (KB > 42) continue;
            // bucket bits: until an average USED bucket holds <= target suffixes
            int BB = 1;
            auto used = [&](int bb) { return bb >= KB ? span : ((span - 1) >> (KB - bb)) + 1; };
            while ((u64)len / used(BB) > (u64)target && BB + 1 <= 3 * dmax && BB + 1 <= KB) ++BB;
            const int forced = env_int("B200SA_MSD_BB", 0);
            if (forced > 0) BB = std::max(1, std::min(std::min(3 * dmax, KB), forced));
            const int nl = (BB + dmax - 1) / dmax;
            int D[3] = {0, 0, 0};
            // (a wide first digit leaves the element's 32 - pb bits to a deeper key)
            D[0] = std::min(dmax, BB);
            for (int i = 1; i < nl; ++i) D[i] = (BB - D[0]) / (nl - 1) + (i - 1 < (BB - D[0]) % (nl - 1) ? 1 : 0);
            if (KB - D[0] > 32 - pb) continue;            // 32 + pb + (KB - D1) <= 64
            if (KB - BB > 32) continue;
            if (K <= best_K) break;                       // (the variant that carries the preceding symbol reached as deep)
            best_K = K;
            pl.nlevels = nl;
            for (int i = 0; i < 3; ++i) pl.D[i] = D[i];
            pl.BB = BB;
            pl.dmax = dmax;
            pl.K = K;
            pl.KB = KB;
            pl.pb = pb;
            pl.R = KB - BB;
            pl.dense.nsym = nsym;
            int Klo = 0;
            while (Klo < K && pow_u64(nsym, Klo + 1) <= 0xffffffffull) ++Klo;
            pl.dense.Klo = (u32)Klo;
            pl.dense.Khi = (u32)(K - Klo);
            pl.dense.powlo = (u32)pow_u64(nsym, Klo);
            pl.dense.ptop = pow_u64(nsym, K - 1);
            break;
        }
        // (carrying the preceding symbol saves the BWT gather: worth a key that is a few bits short of the wish)
        if (best_K >= k_wanted || best_K * eff >= log2len + margin / 2) break;
    }
    return best_K > 0;
}

bool msd_make_plan(u32 len, u32 sigma, int bits, MsdPlan &pl, const u64 *sym_counts) {
    const char *mode = getenv("B200SA_ROUND0");
    if (mode && !strcmp(mode, "lsd")) return false;
    const int b = bits;
    pl.dense = DenseKey{0, 0, 0, 0, 0};
    {
        // alphabets that use less than 9/10 of the codes of their symbol width: dense keys
        const u32 nsym = sigma > 1 ? sigma - 1 : 1;
        const int dk = env_int("B200SA_DENSE_KEYS", -1);
        const bool sparse_alphabet = b >= 2 && nsym >= 2 && (u64)nsym * 10 <= (9ull << b);
        if (dk != 0 && b >= 2 && nsym >= 2 && (sparse_alphabet || dk > 0) && msd_make_plan_dense(len, nsym, b, pl, sym_counts)) return true;
        pl.dense = DenseKey{0, 0, 0, 0, 0};
    }
    // Bucket bits: whole symbols (a digit never splits a symbol: with alphabets that do not fill
    // their b bits the leading bits of a symbol carry no information), until an average bucket
    // holds <= `target` suffixes.  At most 10 bits per level.
    int dmax = (b == 4 || b == 8) ? 8 : 10;
    dmax = env_int("B200SA_MSD_DMAX", dmax);
    dmax = std::max(b, std::min(10, dmax / b * b));
    const int target = std::max(1, env_int("B200SA_MSD_AVG", 3000));
    int BB = b;
    while (((u64)len >> BB) > (u64)target && BB + b <= 3 * dmax) BB += b;
    int forced = env_int("B200SA_MSD_BB", 0);
    if (forced > 0) BB = std::max(b, std::min(3 * dmax, forced / b * b));
    const int nl = (BB + dmax - 1) / dmax;
    const int syms = BB / b;
    for (int i = 0; i < 3; ++i) pl.D[i] = 0;
    for (int i = 0; i < nl; ++i) pl.D[i] = b * (syms / nl + (i < syms % nl ? 1 : 0));
    pl.nlevels = nl;
    pl.BB = BB;
    pl.dmax = dmax;

    int log2len = 0;
    while ((1ull << log2len) < (u64)len) ++log2len;
    double eff = std::log2((double)(sigma > 2 ? sigma - 1 : 1));
    if (eff < 0.5) eff = 0.5;
    const int margin = env_int("B200SA_KEY_MARGIN", 8);
    const int k_wanted = std::max(1, (int)std::ceil((log2len + margin) / eff));
    const int k_min = (BB + b - 1) / b;
    auto kcap = [&](int pb) {
        int by_elem = (32 - pb + pl.D[0]) / b;      // 32 + pb + (KB - D1) <= 64
        int by_window = 64 / b - (pb ? 1 : 0);      // one 64-bit window holds prev + K symbols
        return std::min(by_elem, by_window);
    };
    int kc = std::min(k_wanted, kcap(b)), kn = std::min(k_wanted, kcap(0));
    int K, pb;
    if (kc >= k_wanted || kn <= kc) {
        K = kc;
        pb = b;
    } else {
        K = kn;
        pb = 0;
    }
    int kf = env_int("B200SA_MSD_K", 0);
    if (kf > 0) K = std::min(kf, kcap(pb));
    if (K < k_min) {
        K = k_min;
        if (K > kcap(pb)) return false;
    }
    pl.K = K;
    pl.KB = K * b;
    pl.pb = pb;
    pl.R = pl.KB - BB;
    return pl.R >= 0 && pl.R <= 32;
}

// ---------------------------------------------------------------------------------------------
// Level-1 histogram straight from the packed text: hist[x] = #{t in [0, n] : first D key bits of
// suffix t == x}
// ---------------------------------------------------------------------------------------------
template <int BITS, bool DENSE = false>
__global__ void __launch_bounds__(256) msd_hist_text_kernel(const u64 *__restrict__ packed, u32 n, u64 nwords_data,
                                                            int D, u32 *__restrict__ hist, DenseKey dk = DenseKey{0, 0, 0, 0, 0},
                                                            int dshift = 0) {
    constexpr int CPW = 64 / BITS;
    __shared__ u32 sh[MSD_MAXBINS];
    const int bins = 1 << D;
    for (int i = threadIdx.x; i < bins; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < nwords_data; w += stride) {
        u64 hi = packed[w], lo = packed[w + 1];
        const u64 lo2 = DENSE ? packed[w + 2] : 0ull;
        u64 t0 = w * CPW;
        if (DENSE) {
            // the keys of the word's CPW consecutive suffixes: the first one in full, the others by sliding
            const u32 K = dk.Khi + dk.Klo;
            u64 key = dense_key_of<BITS>(hi, lo, dk);
#pragma unroll
            for (int q = 0; q < CPW; ++q) {
                if (q) key = dense_key_slide(key, sym_at192<BITS>(hi, lo, lo2, (u32)(q - 1) * BITS),
                                             sym_at192<BITS>(hi, lo, lo2, ((u32)(q - 1) + K) * BITS), dk);
                if (t0 + q <= n) atomicAdd(&sh[(u32)(key >> dshift)], 1u);
            }
            continue;
        }
#pragma unroll
        for (int q = 0; q < CPW; ++q) {
            if (t0 + q <= n) {
                const int o = q * BITS;
                u64 win = o ? ((hi << o) | (lo >> (64 - o))) : hi;
                atomicAdd(&sh[(u32)(win >> (64 - D))], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// One CTA per parent bucket: child_start[p*B + d] = parent_start[p] + exclusive scan of the
// parent's digit counts; the counts are replaced by the same values (they become the write
// cursors of the partition kernel).  blockDim.x = min(B, 1024) rounded up to a warp; a thread
// owns B / blockDim.x consecutive digits.
__global__ void __launch_bounds__(1024) msd_scan_children_kernel(u32 *__restrict__ hist,
                                                                 const u32 *__restrict__ parent_start, int D,
                                                                 u32 nparents, u32 len, u32 *__restrict__ child_start,
                                                                 u32 *__restrict__ maxbucket) {
    __shared__ u32 wsum[32];
    __shared__ u32 wmax[32];
    const u32 B = 1u << D;
    const u32 p = blockIdx.x, tid = threadIdx.x;
    const unsigned lane = tid & 31u, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const u32 per = B > blockDim.x ? B / blockDim.x : 1u;  // 1 or 2
    const u32 d0 = tid * per;
    const size_t at = (size_t)p * B + d0;
    u32 c0 = d0 < B ? hist[at] : 0u;
    u32 c1 = (per > 1 && d0 + 1 < B) ? hist[at + 1] : 0u;
    u32 mx = max(c0, c1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) wmax[warp] = mx;
    // (a block of fewer than 1024 threads leaves the last words of wsum unwritten: they only reach the
    // prefixes of warps that do not exist)
    const u32 excl = block_exclusive<1024>(c0 + c1, wsum);
    if (d0 < B) {
        u32 st = (parent_start ? parent_start[p] : 0u) + excl;
        child_start[at] = st;
        hist[at] = st;
        if (per > 1 && d0 + 1 < B) {
            child_start[at + 1] = st + c0;
            hist[at + 1] = st + c0;
        }
    }
    if (tid == 0) {
        if (maxbucket) {
            u32 m = 0;
            for (unsigned w = 0; w < nwarps; ++w) m = max(m, wmax[w]);
            atomicMax(maxbucket, m);
        }
        if (p == nparents - 1) child_start[(size_t)nparents * B] = len;
    }
}

// ---------------------------------------------------------------------------------------------
// Tiles of a partition level >= 2: a tile never straddles two parent buckets.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) msd_tile_offsets_kernel(const u32 *__restrict__ pstart, u32 nparents,
                                                                u32 *__restrict__ tile_off, u32 *__restrict__ d_ntiles) {
    const u32 ntiles = cta_exclusive_scan(
        nparents, [=](u32 p) { return (pstart[p + 1] - pstart[p] + (P_TILE - 1)) / P_TILE; },
        [=](u32 p, u32 e) { tile_off[p] = e; }, SumOp(), 0u);
    if (threadIdx.x == 0) {
        tile_off[nparents] = ntiles;
        *d_ntiles = ntiles;
    }
}

// one warp per parent: desc = {first element, count, parent, 0}
__global__ void __launch_bounds__(256) msd_tile_desc_kernel(const u32 *__restrict__ pstart, u32 nparents,
                                                            const u32 *__restrict__ tile_off, uint4 *__restrict__ desc) {
    u32 p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= nparents) return;
    const u32 s0 = pstart[p], c = pstart[p + 1] - s0;
    const u32 nt = (c + (P_TILE - 1)) / P_TILE, t0 = tile_off[p];
    for (u32 k = threadIdx.x & 31u; k < nt; k += 32) {
        u32 off = k * P_TILE;
        desc[t0 + k] = make_uint4(s0 + off, min((u32)P_TILE, c - off), p, 0u);
    }
}

// digit histogram of one level >= 2 (per parent), from the elements the previous level wrote.
// A CTA takes a CONTIGUOUS range of tiles: consecutive tiles mostly share their parent, so the
// shared-memory counts are added to the parent's global row only when the parent changes (a few
// million global atomics for the whole level instead of one per tile and digit).
__global__ void __launch_bounds__(P_NT) msd_hist_elems_kernel(const u64 *__restrict__ in, const uint4 *__restrict__ desc,
                                                              const u32 *__restrict__ d_ntiles, int D, int dshift,
                                                              u32 *__restrict__ hist) {
    const u32 ntiles = *d_ntiles;
    const u32 per = (ntiles + gridDim.x - 1) / gridDim.x;
    const u32 t0 = blockIdx.x * per, t1 = min(ntiles, t0 + per);
    if (t0 >= t1) return;
    __shared__ u32 sh[P_MAXBINS];
    const u32 B = 1u << D;
    for (u32 i = threadIdx.x; i < B; i += P_NT) sh[i] = 0;
    __syncthreads();
    u32 parent = desc[t0].z;
    uint4 ds = desc[t0];
    for (u32 t = t0; t < t1; ++t) {
        const uint4 nx = t + 1 < t1 ? desc[t + 1] : ds;
        if (ds.z != parent) {  // uniform over the CTA
            __syncthreads();
            u32 *h = hist + (size_t)parent * B;
            for (u32 i = threadIdx.x; i < B; i += P_NT) {
                if (sh[i]) atomicAdd(&h[i], sh[i]);
                sh[i] = 0;
            }
            __syncthreads();
            parent = ds.z;
        }
        const u64 *src = in + ds.x;
        // four loads in flight per thread before the first shared atomic
        for (u32 i = threadIdx.x; i < ds.y; i += 4 * P_NT) {
            u64 e[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) e[q] = i + q * P_NT < ds.y ? ld_stream_u64(src + i + q * P_NT) : 0ull;
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (i + q * P_NT < ds.y) atomicAdd(&sh[(u32)(e[q] >> dshift) & (B - 1)], 1u);
        }
        ds = nx;
    }
    __syncthreads();
    u32 *h = hist + (size_t)parent * B;
    for (u32 i = threadIdx.x; i < B; i += P_NT)
        if (sh[i]) atomicAdd(&h[i], sh[i]);
}

// ---------------------------------------------------------------------------------------------
// Partition of a level >= 2: a tile of <= P_TILE elements written by the previous level is split
// by the digit at element bit `dshift`.  Persistent CTAs (two per SM): while a tile is being
// ranked, grouped and written out, the TMA engine copies the CTA's NEXT tile into the other half
// of a shared-memory double buffer (cp.async.bulk + mbarrier), so no warp waits on HBM latency.
// ---------------------------------------------------------------------------------------------
struct PartArgs {
    const u64 *in;
    u64 *out;
    int D;
    int dshift;       // digit = (e >> dshift) & (B - 1)
    u32 *cursor;      // [nparents << D] next free slot of every child bucket
    const uint4 *desc;
    const u32 *d_ntiles;
};

static constexpr int P_INB = P_TILE + 2;  // landing buffer: the copy starts at a 16-byte boundary
static constexpr size_t P_SMEM = (size_t)P_INB * 8 * 2 + (size_t)P_TILE * 8 + (size_t)P_MAXBINS * 4 * 2 + 32 * 4 + 2 * 8;

__global__ void __launch_bounds__(P_NT, 2) msd_partition_kernel(PartArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 *inb = (u64 *)smem_raw;                   // [2][P_INB] landing buffers
    u64 *buf = inb + 2 * P_INB;                   // [P_TILE] elements grouped by digit
    u32 *hist = (u32 *)(buf + P_TILE);            // [MAXBINS] counts, then tile-local offsets
    u32 *gofs = hist + P_MAXBINS;                 // [MAXBINS] global slot of the digit's run minus its tile offset
    u32 *wsum = gofs + P_MAXBINS;                 // [32]
    u64 *mbar = (u64 *)(wsum + 32);               // [2]

    const u32 tid = threadIdx.x;
    const u32 B = 1u << a.D;
    const u32 ntiles = *a.d_ntiles;
    if (blockIdx.x >= ntiles) return;

    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        mbar_init_fence();
    }
    __syncthreads();

    // thread 0 owns the copies: tile -> landing buffer (from the 16-byte boundary at or below its start)
    auto issue = [&](u32 tile, u32 stage) {
        const uint4 ds = a.desc[tile];
        const u32 a0 = ds.x & ~1u;
        const u32 bytes = ((ds.x - a0 + ds.y + 1u) & ~1u) * 8u;
        mbar_arrive_expect_tx(&mbar[stage], bytes);
        bulk_copy_g2s(inb + stage * P_INB, a.in + a0, bytes, &mbar[stage]);
    };
    if (tid == 0) issue(blockIdx.x, 0);

    u32 it = 0;
    uint4 ds_next = a.desc[blockIdx.x];
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const u32 stage = it & 1u;
        const uint4 ds = ds_next;
        if (tile + gridDim.x < ntiles) ds_next = a.desc[tile + gridDim.x];
        const u32 count = ds.y, parent = ds.z;
        const u64 *in = inb + stage * P_INB + (ds.x & 1u);
        // the other landing buffer was last read before the barrier that ended the previous iteration
        if (tid == 0 && tile + gridDim.x < ntiles) issue(tile + gridDim.x, stage ^ 1u);
        for (u32 i = tid; i < B; i += P_NT) hist[i] = 0;
        __syncthreads();
        mbar_wait_parity(&mbar[stage], (it >> 1) & 1u);

        // ---- digits and slots inside the tile's digit groups (arbitrary order: MSD) ----
        u32 dsl[P_IPT];
#pragma unroll
        for (int j = 0; j < P_IPT; ++j) {
            const u32 i = (u32)j * P_NT + tid;
            dsl[j] = 0;
            if (i < count) {
                const u32 d = (u32)(in[i] >> a.dshift) & (B - 1);
                dsl[j] = d | (atomicAdd(&hist[d], 1u) << 10);
            }
        }
        __syncthreads();

        // ---- exclusive scan of the digit counts; reserve the runs in the child buckets ----
        {
            constexpr int DPT = P_MAXBINS / P_NT;
            const u32 d0 = tid * DPT;
            u32 c[DPT], g[DPT];
            u32 sum = 0;
#pragma unroll
            for (int q = 0; q < DPT; ++q) {
                c[q] = d0 + q < B ? hist[d0 + q] : 0u;
                sum += c[q];
            }
#pragma unroll
            for (int q = 0; q < DPT; ++q) {
                g[q] = 0;
                if (c[q]) g[q] = atomicAdd(&a.cursor[(size_t)parent * B + d0 + q], c[q]);
            }
            u32 run = block_exclusive<P_NT>(sum, wsum);
#pragma unroll
            for (int q = 0; q < DPT; ++q) {
                if (d0 + q < B) {
                    hist[d0 + q] = run;
                    gofs[d0 + q] = g[q] - run;
                }
                run += c[q];
            }
        }
        __syncthreads();

        // ---- group the tile by digit in shared memory ----
#pragma unroll
        for (int j = 0; j < P_IPT; ++j) {
            const u32 i = (u32)j * P_NT + tid;
            if (i < count) buf[hist[dsl[j] & 1023u] + (dsl[j] >> 10)] = in[i];
        }
        __syncthreads();

        // ---- consecutive threads write consecutive slots of a digit run ----
#pragma unroll 4
        for (u32 i = tid; i < count; i += P_NT) {
            const u64 v = buf[i];
            a.out[gofs[(u32)(v >> a.dshift) & (B - 1)] + i] = v;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Level-1 partition straight from the packed text.  A tile is T1_TILE consecutive suffix starts;
// its slice of the packed text (<= 8 KB) is staged in shared memory once, and a thread forms
// T1_IPT CONSECUTIVE elements from one 128-bit window by shifting, instead of two global loads
// per element.  Elements are not kept in registers across the digit scan: they are formed again
// from the staged text when the tile is grouped by digit.
// ---------------------------------------------------------------------------------------------
static constexpr int T1_NT = 512;
static constexpr int T1_IPT = 16;
static constexpr int T1_TILE = T1_NT * T1_IPT;     // 8192 suffix starts
static constexpr int T1_STAGE_MAX = T1_TILE * 8 / 64 + 5;
static constexpr size_t T1_SMEM = (size_t)T1_TILE * 8 + (size_t)MSD_MAXBINS * 4 * 2 + (size_t)T1_STAGE_MAX * 8 + 32 * 4;

struct Text1Args {
    const u64 *packed;
    u64 nwords;       // words readable in `packed` (data + zero padding)
    u64 *out;
    u32 len;
    int bits, KB, pb;
    int D, dshift;    // digit = key >> dshift
    u64 restmask;     // rest = key & restmask
    int rest_shift;   // 32 + pb
    u32 *cursor;      // [1 << D] next free slot of every level-1 bucket
    DenseKey dense;   // nsym != 0: the key is the base-nsym number of the K symbols (KB bits), digit = key >> dshift
};

// 128-bit window (H:L) of the staged text starting at bit `off`
__device__ __forceinline__ void stage_window(const u64 *st, u32 off, u64 &H, u64 &L) {
    const u32 w = off >> 6, o = off & 63u;
    const u64 w0 = st[w], w1 = st[w + 1], w2 = st[w + 2];
    H = o ? (w0 << o) | (w1 >> (64 - o)) : w0;
    L = o ? (w1 << o) | (w2 >> (64 - o)) : w1;
}

// 192-bit window (H:L:M) for the dense keys, whose K symbols may take more than one word
__device__ __forceinline__ void stage_window3(const u64 *st, u32 off, u64 &H, u64 &L, u64 &M) {
    const u32 w = off >> 6, o = off & 63u;
    const u64 w0 = st[w], w1 = st[w + 1], w2 = st[w + 2], w3 = st[w + 3];
    H = o ? (w0 << o) | (w1 >> (64 - o)) : w0;
    L = o ? (w1 << o) | (w2 >> (64 - o)) : w1;
    M = o ? (w2 << o) | (w3 >> (64 - o)) : w2;
}
// the 128 bits that start at the key's first symbol, from the window of position q of a group of eight
template <int BITS, u32 LEAD>
__device__ __forceinline__ u64 dense_key_q(u64 H, u64 L, u64 M, int sh, const DenseKey &dk) {
    u64 a = sh ? (H << sh) | (L >> (64 - sh)) : H;
    u64 b = sh ? (L << sh) | (M >> (64 - sh)) : L;
    if (LEAD) {
        a = (a << LEAD) | (b >> (64 - LEAD));
        b <<= LEAD;
    }
    return dense_key_of<BITS>(a, b, dk);
}

// BITS = symbol width, HAS_PREV = the preceding symbol is carried in the element (pb == BITS):
// compile-time so that every per-symbol shift is an immediate.  DENSE = the key is a.dense's
// base-nsym number of the K symbols.
template <int BITS, bool HAS_PREV, bool DENSE>
__global__ void __launch_bounds__(T1_NT, 2) msd_partition_text_kernel(Text1Args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 *buf = (u64 *)smem_raw;                   // [T1_TILE] elements grouped by digit
    u64 *stage = buf + T1_TILE;                   // [T1_STAGE_MAX] packed text of the tile (one word of lead-in)
    u32 *hist = (u32 *)(stage + T1_STAGE_MAX);    // [MAXBINS] counts, then tile-local offsets
    u32 *gofs = hist + MSD_MAXBINS;               // [MAXBINS] global slot of the digit's run minus its tile offset
    u32 *wsum = gofs + MSD_MAXBINS;               // [32]
    static_assert(T1_TILE <= (1 << 14) && MSD_MAXBINS <= (1 << 10), "tile-local low word: 14 bits of position, 10 of digit");

    constexpr int b = BITS;
    constexpr u32 lead = HAS_PREV ? (u32)BITS : 0u;
    const u32 tid = threadIdx.x;
    const u32 B = 1u << a.D;
    const u64 begin = (u64)blockIdx.x * T1_TILE;
    const u32 count = (u32)min((u64)T1_TILE, (u64)a.len - begin);

    // ---- stage the tile's text: word k of `stage` is packed[begin*b/64 - 1 + k] ----
    {
        constexpr u32 nstage = (u32)(T1_TILE / 64) * b + 5;
        const u64 w0 = begin * (u64)b / 64;
        for (u32 k = tid; k < nstage; k += T1_NT) {
            const u64 w = w0 + k;  // index + 1
            stage[k] = (w >= 1 && w - 1 < a.nwords) ? a.packed[w - 1] : 0ull;
        }
        for (u32 i = tid; i < B; i += T1_NT) hist[i] = 0;
    }
    __syncthreads();

    // bit offset (inside `stage`) of the window of the thread's first position: it starts at the
    // preceding symbol when that symbol is carried in the element, else at the position itself
    const u32 i0 = tid * T1_IPT;
    const u32 off0 = 64u + i0 * (u32)b - lead;
    const int kshift = 64 - a.KB;
    const int dsh = 32 - a.D;                           // digit = leading D bits of the key
    const u32 restmask = (u32)a.restmask;               // KB - D <= 32 bits

    // ---- digits and slots inside the tile's digit groups (arbitrary order: MSD) ----
    u64 dkey = 0;
    const u32 dK = a.dense.Khi + a.dense.Klo;
    u32 ds[T1_IPT];
#pragma unroll
    for (int g = 0; g < T1_IPT / 8; ++g) {
        u64 H, L, M = 0;
        if (DENSE) stage_window3(stage, off0 + (u32)(8 * g * b), H, L, M);
        else stage_window(stage, off0 + (u32)(8 * g * b), H, L);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int j = 8 * g + q;
            const int sh = q * b;
            const u64 win = sh ? (H << sh) | (L >> (64 - sh)) : H;
            const u32 khi = (u32)((win << lead) >> 32);  // leading 32 bits of the key
            if (DENSE) {  // the first key of the group of eight in full, the others by sliding
                if (q == 0) dkey = dense_key_q<BITS, lead>(H, L, M, 0, a.dense);
                else dkey = dense_key_slide(dkey, sym_at192<BITS>(H, L, M, lead + (u32)(q - 1) * BITS),
                                            sym_at192<BITS>(H, L, M, lead + ((u32)(q - 1) + dK) * BITS), a.dense);
            }
            ds[j] = 0;
            if (i0 + j < count) {
                const u32 d = DENSE ? (u32)(dkey >> a.dshift) : khi >> dsh;
                const u32 slot = atomicAdd(&hist[d], 1u);
                ds[j] = d | (slot << 10);
            }
        }
    }
    __syncthreads();

    // ---- exclusive scan of the digit counts; reserve the runs in the level-1 buckets ----
    u32 gsub[MSD_MAXBINS / T1_NT], gres[MSD_MAXBINS / T1_NT];
    {
        constexpr int DPT = MSD_MAXBINS / T1_NT;
        const u32 d0 = tid * DPT;
        u32 c[DPT], g[DPT];
        u32 sum = 0;
#pragma unroll
        for (int q = 0; q < DPT; ++q) {
            c[q] = d0 + q < B ? hist[d0 + q] : 0u;
            sum += c[q];
        }
#pragma unroll
        for (int q = 0; q < DPT; ++q) {
            g[q] = 0;
            if (c[q]) g[q] = atomicAdd(&a.cursor[d0 + q], c[q]);
        }
        u32 run = block_exclusive<T1_NT>(sum, wsum);
#pragma unroll
        for (int q = 0; q < DPT; ++q) {
            if (d0 + q < B) hist[d0 + q] = run;
            gsub[q] = run;
            gres[q] = g[q];
            run += c[q];
        }
    }
    __syncthreads();

    // ---- form the elements (again from the staged text) and group the tile by digit.  An
    // element is two 32-bit words: [rest of key | preceding symbol] and the suffix start ----
#pragma unroll
    for (int g = 0; g < T1_IPT / 8; ++g) {
        u64 H, L, M = 0;
        if (DENSE) stage_window3(stage, off0 + (u32)(8 * g * b), H, L, M);
        else stage_window(stage, off0 + (u32)(8 * g * b), H, L);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int j = 8 * g + q;
            if (DENSE) {
                if (q == 0) dkey = dense_key_q<BITS, lead>(H, L, M, 0, a.dense);
                else dkey = dense_key_slide(dkey, sym_at192<BITS>(H, L, M, lead + (u32)(q - 1) * BITS),
                                            sym_at192<BITS>(H, L, M, lead + ((u32)(q - 1) + dK) * BITS), a.dense);
            }
            if (i0 + j < count) {
                const int sh = q * b;
                const u64 win = sh ? (H << sh) | (L >> (64 - sh)) : H;
                const u32 rest = (DENSE ? (u32)dkey : (u32)((win << lead) >> kshift)) & restmask;
                const u32 hiw = HAS_PREV ? (rest << b) | (u32)(win >> (64 - b)) : rest;
                const u32 d = ds[j] & 1023u;
                const u32 pos = hist[d] + (ds[j] >> 10);
                // in shared memory the low word is [digit : 10 | position in the tile : 14]; the
                // write-out turns it into the suffix start
                buf[pos] = ((u64)hiw << 32) | (u64)((d << 14) | (i0 + (u32)j));
            }
        }
    }
    // the reserved global slots are first needed now: the round trip of the reservation (a global
    // atomic per digit) ran behind the grouping above
    {
        const u32 d0 = tid * (MSD_MAXBINS / T1_NT);
#pragma unroll
        for (int q = 0; q < MSD_MAXBINS / T1_NT; ++q)
            if (d0 + q < B) gofs[d0 + q] = gres[q] - gsub[q];
    }
    __syncthreads();

    // ---- consecutive threads write consecutive slots of a digit run ----
    const u32 begin32 = (u32)begin;
#pragma unroll 4
    for (u32 i = tid; i < count; i += T1_NT) {
        const u64 v = buf[i];
        const u32 lo = (u32)v;
        a.out[gofs[lo >> 14] + i] = (v & 0xffffffff00000000ull) | (u64)(begin32 + (lo & 16383u));
    }
}

// ---------------------------------------------------------------------------------------------
// Local-sort tiles: tile t owns the buckets whose first element lies in [t*TSZ, (t+1)*TSZ).
// tile_first[t] = smallest bucket b with bstart[b] >= t*TSZ  (b in [0, nb]; bstart[nb] = len)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) msd_tile_first_kernel(const u32 *__restrict__ bstart, u64 nb, u32 ntiles,
                                                             u32 *__restrict__ tile_first) {
    u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (b > nb) return;
    const u32 s = bstart[b];
    u32 lo = b == 0 ? 0u : bstart[b - 1] / L3_TSZ + 1u;
    u32 hi = b == nb ? ntiles : s / L3_TSZ;
    if (hi > ntiles) hi = ntiles;
    for (u32 t = lo; t <= hi; ++t) tile_first[t] = (u32)b;
}

struct L3Args {
    const u64 *in;
    const u32 *bstart;
    const u32 *tile_first;
    u32 n;
    int K, pb, R;
    u32 *sa;
    u8 *bwt;           // may be null
    u32 *short_rank;   // [1 + 2 * 32]: count, then (suffix, row) of the short suffixes of oversize buckets
    u32 *grow;         // [len] by ROW: first row of the group, for the rows of suffixes whose key is shared
    u32 *actbits;      // bit per row: the suffix in this row shares its key with another one ("active")
    u32 *primary;
    u32 *flagged, *nflagged;   // tiles the fast kernel declined (a crowded bin)
    u32 *big, *nbig;           // tiles that hold a bucket too large for one SM (msd_bigtile_kernel)
    u32 ntiles;
    int par_shift;     // bucket >> par_shift = its level-1 parent (0 with a single level)
};

__device__ __forceinline__ u32 seg_index(const u32 *segmask, const u32 *segpre, u32 i) {
    // number of segment starts at positions <= i, minus one
    return segpre[i >> 5] + (u32)__popc(segmask[i >> 5] & (0xffffffffu >> (31u - (i & 31u)))) - 1u;
}

// segment-start bitmap, per-word prefix counts and (offset, count) of every non-empty bucket
__device__ __forceinline__ void l3_segments(const u32 *__restrict__ bstart, u32 b0, u32 b1, u32 E0, u32 M, u32 *segmask,
                                            u32 *segpre, uint2 *segtab, int NT) {
    const u32 tid = threadIdx.x;
    for (u32 i = tid; i < (u32)L3_MASKW + 1; i += NT) segmask[i] = 0;
    __syncthreads();
    for (u32 b = b0 + tid; b < b1; b += NT) {
        u32 s0 = bstart[b], s1 = bstart[b + 1];
        if (s1 > s0) atomicOr(&segmask[(s0 - E0) >> 5], 1u << ((s0 - E0) & 31u));
    }
    __syncthreads();
    if (tid < 32) {
        constexpr int WPL = L3_MASKW / 32;  // words per lane
        u32 loc[WPL];
        u32 sum = 0;
#pragma unroll
        for (int q = 0; q < WPL; ++q) {
            loc[q] = (u32)__popc(segmask[tid * WPL + q]);
            sum += loc[q];
        }
        u32 run = warp_inclusive(sum, SumOp()) - sum;
#pragma unroll
        for (int q = 0; q < WPL; ++q) {
            segpre[tid * WPL + q] = run;
            run += loc[q];
        }
    }
    __syncthreads();
    for (u32 b = b0 + tid; b < b1; b += NT) {
        u32 s0 = bstart[b], s1 = bstart[b + 1];
        if (s1 > s0) {
            u32 i0 = s0 - E0;
            segtab[seg_index(segmask, segpre, i0)] = make_uint2(i0, s1 - s0);
        }
    }
    (void)M;
}

__device__ __forceinline__ bool is_short_suffix(u32 s, int K, u32 n) { return (u64)s + (u64)K > (u64)n; }

// emits one sorted position: SA, BWT row, and for members of a group of equal long keys the
// group rank, the valid bit and a slot in the active list (warp-aggregated append)
// emits one sorted position: SA, BWT row, and for members of a group of equal long keys the group
// head (by suffix and by row) and the row's bit in the active bitmap.  `sbits` = the tile's slice of
// that bitmap in shared memory, bit (g - gbase) (fast kernel); null: straight to global memory.
__device__ __forceinline__ void l3_emit(const L3Args &a, u32 g, u64 e, bool active, u32 group_head, u32 *sbits = nullptr,
                                        u32 gbase = 0) {
    const u32 s = (u32)e;
    a.sa[g] = s;
    u32 bw = ((u32)(e >> 32) & ((1u << a.pb) - 1u)) + 1u;
    if (s == 0) {  // (one element of the whole text: the row of the sentinel)
        bw = 0;
        *a.primary = g;
    }
    if (a.bwt) a.bwt[g] = (u8)bw;
    if (active) {
        a.grow[g] = group_head;  // (rank[s] is written from the compacted list of active rows, sa_build.cu)
        if (sbits) atomicOr(&sbits[(g - gbase) >> 5], 1u << ((g - gbase) & 31u));
        else atomicOr(&a.actbits[g >> 5], 1u << (g & 31u));
    }
}

static constexpr int L3_CNTN = L3_CAP + 16;        // counters per tile (the blocked scan reads a little past bin M)
static constexpr int L3_PAD = L3_CROWD;             // guard elements on both sides of X (the ordering window never exceeds it)
static constexpr int L3_ABW = L3_MASKW + 2;         // words of the tile's slice of the active bitmap (any alignment)
static constexpr int L3_WLW = L3_MASKW;             // words of per-32-position window bounds
static constexpr size_t L3_SMEM = (size_t)(L3_CAP + 2 * L3_PAD) * 8 + (size_t)L3_CNTN * 4 + (size_t)L3_CNTN * 2 +
                                  (size_t)(L3_MASKW + 1) * 4 * 2 + 64 * 4 + 8 * 4 + (size_t)L3_ABW * 4 + (size_t)L3_WLW * 4;

// sum of the four bytes of x
__device__ __forceinline__ u32 bytesum(u32 x) { return __dp4a(x, 0x01010101u, 0u); }

// Persistent CTAs (two per SM).  While a tile is being ordered and written out, thread 0 walks
// tile_first -> bucket_start for the CTA's NEXT tile and asks the TMA engine to pull that tile's
// elements into L2 (cp.async.bulk.prefetch), so the chain of dependent loads is off every
// warp's critical path and the next tile's first pass reads L2, not HBM.
__global__ void __launch_bounds__(L3_NT, L3_CTAS) msd_local_sort_kernel(L3Args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // elements grouped by bin, as two word arrays (neighbouring high words sit in neighbouring banks):
    u32 *Xhi = (u32 *)smem_raw + L3_PAD;              // [-PAD, CAP + PAD) [rest of key | preceding symbol], guards around
    u32 *Xlo = Xhi + L3_CAP + L3_PAD;                 // [0, CAP + PAD) suffix starts
    u32 *cnt = Xlo + L3_CAP + L3_PAD;                 // [L3_CNTN] four byte-wide sub-bin counts per position
    u16 *pre = (u16 *)(cnt + L3_CNTN);                // [L3_CNTN] exclusive prefix of the per-position totals
    u32 *segmask = (u32 *)(pre + L3_CNTN);            // [MASKW + 1]
    u32 *segpre = segmask + (L3_MASKW + 1);           // [MASKW + 1]
    u32 *misc = segpre + (L3_MASKW + 1);              // [64]
    u32 *nxt = misc + 64;                             // [8] next tile: index, b0, b1, E0, M
    u32 *abits = nxt + 8;                             // [L3_ABW] active bits of the tile's rows, global word alignment
    u32 *wloc = abits + L3_ABW;                       // [L3_WLW] per 32 positions of the grouped tile: the largest (sub-bin
                                                      // occupancy - 1) of an element standing there = the window pass 3 needs
    uint2 *segtab = (uint2 *)Xhi;                     // aliases the element arrays until the elements are scattered
    u16 *queue = pre;                                 // positions with an equal key within reach (pass 3 -> top of the next iteration;
                                                      // `pre` is free between pass 2 and the next tile's scan)
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u32 remmask = a.R >= 32 ? ~0u : ((1u << a.R) - 1u);
    const u32 remsh = a.R > 0 ? 32u - (u32)a.R : 0u;  // R == 0: every key of a bucket is equal, rem == 0

    // thread 0: publish the CTA's next non-empty tile at or after `t` and start its prefetch
    auto advance = [&](u32 t) {
        u32 b0 = 0, b1 = 0, E0 = 0, M = 0;
        for (; t < a.ntiles; t += gridDim.x) {
            b0 = a.tile_first[t];
            b1 = a.tile_first[t + 1];
            if (b0 == b1) continue;
            E0 = a.bstart[b0];
            M = a.bstart[b1] - E0;
            if (M > (u32)L3_CAP) {  // holds an oversize bucket: left to msd_bigtile_kernel
                a.big[atomicAdd(a.nbig, 1u)] = t;
                continue;
            }
            if (M) break;
        }
        nxt[0] = t; nxt[1] = b0; nxt[2] = b1; nxt[3] = E0; nxt[4] = M;
        if (t < a.ntiles) {
            const u32 a0 = E0 & ~1u;
            const u32 bytes = ((E0 - a0 + M + 1u) & ~1u) * 8u;
            bulk_prefetch_l2(a.in + a0, bytes);
        }
    };
    if (tid == 0) advance(blockIdx.x);

    // the counters of the first tile (later tiles: zeroed again right after their last use)
    for (u32 i = tid; i < (u32)L3_CNTN; i += L3_NT) cnt[i] = 0;
    // left guards: the smallest key, never "larger than" an element (pass 3)
    if (tid < (u32)L3_PAD) Xhi[-(int)tid - 1] = 0u;
    if (tid == 0) {
        misc[32] = 0;  // largest slot seen in the tile
        misc[35] = 0;  // positions queued for the tie-break pass
        misc[36] = 0;  // ... of a tile that spans two level-1 parents (bucket boundaries are checked)
        misc[37] = 0;  // this tile defers its tie-breaks
        misc[38] = 0;  // tie-breaks done in place in this tile
    }
    for (u32 i = tid; i < (u32)L3_ABW; i += L3_NT) abits[i] = 0;
    for (u32 i = tid; i < (u32)L3_WLW; i += L3_NT) wloc[i] = 0;
    u32 prevE0 = 0, prevM = 0;   // rows of the previous tile whose active bits still sit in `abits`

    while (true) {
        __syncthreads();  // `nxt` is published, the counters are zero, the previous tile has left X
        const u32 qn = misc[35];
        if (qn) {  // (uniform) positions of the previous tile whose tie-break was deferred
            const u32 qE0 = prevE0, qM = prevM;
            const bool qseg = misc[36] != 0u;
            const u32 pbm = (1u << a.pb) - 1u;
            for (u32 k = tid; k < qn; k += L3_NT) {
                const u32 p = queue[k];
                const u32 hp = Xhi[p], kp = hp >> a.pb;
                const u32 Wl = wloc[p >> 5];
                const u32 se = Xlo[p];
                const bool e_short = is_short_suffix(se, a.K, a.n);
                // position among the other keys (as in pass 3), then the final order among equal keys: short suffixes
                // first, shortest (largest start) first; then the long ones in position order, which form an active group
                u32 r = p, longs_before = 0;
                bool active = false, lv = true, rv = true;
                for (u32 d = 1; d <= Wl; ++d) {
                    lv = lv && p >= d;
                    rv = rv && p + d < qM;
                    if (qseg) {
                        const u32 xl = p - d + 1u, xr = p + d;  // a bucket starts here: the neighbour is beyond it
                        if (lv && ((segmask[xl >> 5] >> (xl & 31u)) & 1u)) lv = false;
                        if (rv && ((segmask[xr >> 5] >> (xr & 31u)) & 1u)) rv = false;
                    }
                    if (lv) {
                        const u32 ko = Xhi[p - d] >> a.pb;
                        r -= ko > kp ? 1u : 0u;
                        if (ko == kp) {
                            const u32 so = Xlo[p - d];
                            const bool o_short = is_short_suffix(so, a.K, a.n);
                            // the left neighbour belongs AFTER this element
                            if (o_short ? (e_short && so < se) : e_short) --r;
                            if (!o_short && !e_short) { active = true; ++longs_before; }
                        }
                    }
                    if (rv) {
                        const u32 ko = Xhi[p + d] >> a.pb;
                        r += ko < kp ? 1u : 0u;
                        if (ko == kp) {
                            const u32 so = Xlo[p + d];
                            const bool o_short = is_short_suffix(so, a.K, a.n);
                            // the right neighbour belongs BEFORE this element
                            if (o_short ? (!e_short || so > se) : false) ++r;
                            if (!o_short && !e_short) active = true;
                        }
                    }
                }
                l3_emit(a, qE0 + r, ((u64)hp << 32) | (u64)se, active, qE0 + r - longs_before, abits, qE0 & ~31u);
            }
            (void)pbm;
            __syncthreads();  // the active bits of these rows are in `abits`; `wloc`, the queue, the segment bitmap have been read
        }
        if (tid == 0) {
            // equal keys in the tile just finished: more than a sixteenth of it -> the next tile defers its tie-breaks
            misc[37] = (qn + misc[38]) * 16u > prevM ? 1u : 0u;
            misc[38] = 0;
            if (qn) misc[35] = 0;
        }
        if (tid < (u32)L3_WLW) wloc[tid] = 0;  // (written by pass 2, behind the barriers of pass 1)
        if (prevM) {
            // the previous tile's slice of the active bitmap: interior words are owned by the tile, the
            // first and the last one may be shared with its neighbours
            const u32 w0 = prevE0 >> 5, nw = ((prevE0 & 31u) + prevM + 31u) >> 5;
            for (u32 i = tid; i < nw; i += L3_NT) {
                const u32 v = abits[i];
                abits[i] = 0;
                if (i == 0 || i + 1 == nw) {
                    if (v) atomicOr(&a.actbits[w0 + i], v);
                } else {
                    a.actbits[w0 + i] = v;
                }
            }
            prevM = 0;
        }
        const u32 t = nxt[0], b0 = nxt[1], b1 = nxt[2], E0 = nxt[3], M = nxt[4];
        if (t >= a.ntiles) break;
        const u64 *src = a.in + E0;
        // bucket boundaries need a look only in tiles that span two level-1 parents (pass 3)
        const bool segcheck = (b0 >> a.par_shift) != ((b1 - 1u) >> a.par_shift);
        if (tid == 0) misc[36] = segcheck ? 1u : 0u;  // (read by the deferred tie-break pass at the top of the next iteration)
        // Common case: a handful of buckets under one parent -- every thread keeps their
        // (start, size) in registers and nothing about segments goes through shared memory.
        const bool few = (b1 - b0 <= 4u) && !segcheck;
        u32 e1 = M, e2 = M, e3 = M, e4 = M;  // tile-local starts of buckets b0+1 .. b0+4 (M: none)
        if (few) {
            const u32 nbk = b1 - b0;
            if (nbk > 1u) e1 = a.bstart[b0 + 1] - E0;
            if (nbk > 2u) e2 = a.bstart[b0 + 2] - E0;
            if (nbk > 3u) e3 = a.bstart[b0 + 3] - E0;
        } else {
            l3_segments(a.bstart, b0, b1, E0, M, segmask, segpre, segtab, L3_NT);
            __syncthreads();
        }
        (void)e4;

        // ---- pass 1: sub-bin = expected sorted position of the element inside its bucket at a
        // quarter of a position's resolution; the four sub-bins of a position are byte counters
        // of one word (a crowded sub-bin declines the tile before a byte can overflow) ----
        u32 meta[L3_IPT];
        u32 myslot = 0;
        // all loads of the pass are issued before the first shared-memory atomic (the high word of
        // an element is all this pass needs)
        const u32 *src_hi = (const u32 *)src + 1;
#pragma unroll
        for (int j = 0; j < L3_IPT; ++j) {
            const u32 i = (u32)j * L3_NT + tid;
            meta[j] = i < M ? src_hi[2 * i] : 0u;
        }
#pragma unroll
        for (int j = 0; j < L3_IPT; ++j) {
            const u32 i = (u32)j * L3_NT + tid;
            if ((u32)j * L3_NT >= M) break;
            if (i < M) {
                const u32 hi = meta[j];
                uint2 sg;
                if (few) {
                    sg.x = i >= e3 ? e3 : i >= e2 ? e2 : i >= e1 ? e1 : 0u;
                    sg.y = (i >= e3 ? M : i >= e2 ? e3 : i >= e1 ? e2 : e1) - sg.x;
                } else {
                    sg = segtab[seg_index(segmask, segpre, i)];
                }
                const u32 rem = (hi >> a.pb) & remmask;
                // (rem * 4 * size) >> R as one high multiply (rem < 2^R, R <= 32)
                const u32 fb = __umulhi(rem << remsh, sg.y * 4u);
                const u32 word = sg.x + (fb >> 2), sub8 = (fb & 3u) * 8u;
                const u32 slot = (atomicAdd(&cnt[word], 1u << sub8) >> sub8) & 255u;
                myslot = max(myslot, slot);
                meta[j] = word | (sub8 << 13) | (slot << 18);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) myslot = max(myslot, __shfl_xor_sync(0xffffffffu, myslot, o));
        if (lane == 0 && myslot) atomicMax(&misc[32], myslot);
        __syncthreads();
        // W = largest sub-bin occupancy of the tile minus one: how far an element can stand from
        // its sorted position once the tile is grouped by sub-bin
        const u32 W = misc[32];
        const bool crowded = W >= (u32)L3_CROWD;

        if (!crowded) {
            // ---- exclusive scan of the per-position totals (thread owns L3_IPT consecutive positions) ----
            {
                const u32 base = tid * L3_IPT;
                const bool mine = base <= M;  // positions past M are empty (and were not zeroed)
                u32 v[L3_IPT];
                u32 sum = 0;
#pragma unroll
                for (int q = 0; q < L3_IPT; ++q) {
                    v[q] = mine ? bytesum(cnt[base + q]) : 0u;
                    sum += v[q];
                }
                u32 run = block_exclusive<L3_NT>(sum, misc);
                if (mine) {
#pragma unroll
                    for (int q = 0; q < L3_IPT; ++q) {
                        pre[base + q] = (u16)run;
                        run += v[q];
                    }
                }
            }
            __syncthreads();

            // ---- pass 2: elements go to their sub-bin (any order inside it) ----
#pragma unroll
            for (int j = 0; j < L3_IPT; ++j) {
                const u32 i = (u32)j * L3_NT + tid;
                if ((u32)j * L3_NT >= M) break;
                if (i < M) {
                    const u32 word = meta[j] & 8191u, sub8 = (meta[j] >> 13) & 31u, slot = meta[j] >> 18;
                    const u32 cw = cnt[word];
                    const u32 below = bytesum(cw & ((1u << sub8) - 1u));
                    const u64 e = src[i];
                    const u32 at = (u32)pre[word] + below + slot;
                    Xhi[at] = (u32)(e >> 32);
                    Xlo[at] = (u32)e;
                    // an element is at most (occupancy of its sub-bin - 1) positions away from its place
                    const u32 need = ((cw >> sub8) & 255u) - 1u;
                    if (need) atomicMax(&wloc[at >> 5], need);
                }
            }
            // right guards: the largest key, never "smaller than" an element
            if (tid < W) Xhi[M + tid] = ~0u;
        }
        __syncthreads();

        // the counters were last read above: zero them for the CTA's next tile
        for (u32 i = tid; i < min((u32)L3_CNTN, M + 16u); i += L3_NT) cnt[i] = 0;
        if (tid == 0) {
            misc[32] = 0;
            if (crowded) a.flagged[atomicAdd(a.nflagged, 1u)] = t;
            advance(t + gridDim.x);
        }
        if (crowded) continue;
        prevE0 = E0;
        prevM = M;

        // ---- pass 3, one thread per POSITION of the grouped tile.  Sub-bins are contiguous and
        // ordered by key, so the sorted position of the element at p is p minus the larger keys
        // among the W positions to its left plus the smaller keys among the W to its right
        // (elements outside its sub-bin contribute nothing).  No per-element loop bounds: W is
        // uniform over a warp (Wl <= W).  The high word of an element is [rest of key | preceding
        // symbol]; its bits above `pb` order the elements of all buckets under one level-1
        // parent, so bucket boundaries need a check only in tiles that span two parents
        // (always with a single level).  Equal keys (a short suffix next to its padded twin, or
        // long suffixes that stay active) are rare and take the tie-break path. ----
        const u32 pbmask = (1u << a.pb) - 1u;
        const bool defer = misc[37] != 0u;  // (set behind the barrier of pass 1)
        for (u32 p = tid; p < M; p += L3_NT) {
            const u32 hp = Xhi[p];
            // the window the 32 positions of this warp need (uniform over the warp): the tile-wide bound W is set by
            // one or two crowded sub-bins, and by every pair of equal keys on a text with repeats
            const u32 Wl = wloc[p >> 5];
            u32 r = p;
            bool eq = false;
            if (!segcheck) {
                // keys compared as raw high words: a > (b | mask) <=> (a >> pb) > (b >> pb), and
                // a < (b & ~mask) likewise; the guards on both sides of X make bounds checks unnecessary
                const u32 hp_hi = hp | pbmask, hp_lo = hp & ~pbmask;
                u32 near = 0xffffffffu;  // smallest difference to a neighbour's word: <= pbmask means an equal key
#define L3_STEP(D)                                                        \
    {                                                                     \
        const u32 hl = Xhi[(int)p - (D)], hr = Xhi[p + (D)];              \
        r -= hl > hp_hi ? 1u : 0u;                                        \
        r += hr < hp_lo ? 1u : 0u;                                        \
        near = min(near, min(hl ^ hp, hr ^ hp));                          \
    }
                // (Wl is uniform over the warp and small: straight-line steps with constant offsets, no loop control)
                if (Wl >= 1u) L3_STEP(1)
                if (Wl >= 2u) L3_STEP(2)
                if (Wl >= 3u) L3_STEP(3)
                if (Wl >= 4u) L3_STEP(4)
                for (u32 d = 5; d <= Wl; ++d) L3_STEP((int)d)
#undef L3_STEP
                eq = near <= pbmask;
            } else {
                const u32 kp = hp >> a.pb;
                bool lv = true, rv = true;
                for (u32 d = 1; d <= Wl; ++d) {
                    lv = lv && p >= d;
                    rv = rv && p + d < M;
                    const u32 xl = p - d + 1u, xr = p + d;  // a bucket starts here: the neighbour is beyond it
                    if (lv && ((segmask[xl >> 5] >> (xl & 31u)) & 1u)) lv = false;
                    if (rv && ((segmask[xr >> 5] >> (xr & 31u)) & 1u)) rv = false;
                    if (lv) {
                        const u32 ko = Xhi[p - d] >> a.pb;
                        r -= ko > kp ? 1u : 0u;
                        eq = eq || ko == kp;
                    }
                    if (rv) {
                        const u32 ko = Xhi[p + d] >> a.pb;
                        r += ko < kp ? 1u : 0u;
                        eq = eq || ko == kp;
                    }
                }
            }
            const u32 kp = hp >> a.pb;
            const u64 e = ((u64)hp << 32) | (u64)Xlo[p];
            bool active = false;
            u32 head = r;
            if (eq) {
                if (defer) {
                    // the CTA's tiles are full of equal keys (a text with repeats): the tie-break runs in a pass of its
                    // own at the top of the next iteration, where every lane has such an element -- here it would make
                    // every warp walk both paths
                    queue[atomicAdd(&misc[35], 1u)] = (u16)p;
                    continue;
                }
                atomicAdd(&misc[38], 1u);
                // final order among equal keys: short suffixes first, shortest (largest start)
                // first; then the long ones in position order, which form an active group
                const u32 se = (u32)e;
                const bool e_short = is_short_suffix(se, a.K, a.n);
                u32 longs_before = 0;
                bool lv = true, rv = true;
                for (u32 d = 1; d <= Wl; ++d) {
                    lv = lv && p >= d;
                    rv = rv && p + d < M;
                    if (segcheck) {
                        const u32 xl = p - d + 1u, xr = p + d;
                        if (lv && ((segmask[xl >> 5] >> (xl & 31u)) & 1u)) lv = false;
                        if (rv && ((segmask[xr >> 5] >> (xr & 31u)) & 1u)) rv = false;
                    }
                    if (lv && (Xhi[p - d] >> a.pb) == kp) {
                        const u32 so = Xlo[p - d];
                        const bool o_short = is_short_suffix(so, a.K, a.n);
                        // the left neighbour belongs AFTER this element
                        if (o_short ? (e_short && so < se) : e_short) --r;
                        if (!o_short && !e_short) { active = true; ++longs_before; }
                    }
                    if (rv && (Xhi[p + d] >> a.pb) == kp) {
                        const u32 so = Xlo[p + d];
                        const bool o_short = is_short_suffix(so, a.K, a.n);
                        // the right neighbour belongs BEFORE this element
                        if (o_short ? (!e_short || so > se) : false) ++r;
                        if (!o_short && !e_short) active = true;
                    }
                }
                head = r - longs_before;
            }
            l3_emit(a, E0 + r, e, active, E0 + head, abits, E0 & ~31u);
        }
    }
}

// Robust variant for the tiles the fast kernel declined: bitonic sort of (composite key, element)
// pairs.  composite = [segment : 13 | remaining key : 32 | long : 1 | n - s for short suffixes : 8]
template <int RBN>
static constexpr size_t rb_smem() {
    return (size_t)RBN * 8 * 2 + (size_t)(L3_MASKW + 1) * 4 * 2 + (size_t)(RBN / 32 + 1) * 4 + 64;
}
static constexpr size_t RB_SMEM = rb_smem<RB_N>();
static constexpr int RB_N_SMALL = 4096;            // most declined tiles fit half the network: three CTAs per SM

// orders the buckets [b0, b1) (M = their elements, <= min(L3_CAP, RBN)) and emits them; all threads of the CTA
template <int RBN>
__device__ void robust_sort_range(const L3Args &a, u32 b0, u32 b1, unsigned char *smem_raw) {
    u64 *SK = (u64 *)smem_raw;            // [RBN]
    u64 *XV = SK + RBN;                   // [RBN]
    u32 *segmask = (u32 *)(XV + RBN);
    u32 *segpre = segmask + (L3_MASKW + 1);
    u32 *headbits = segpre + (L3_MASKW + 1);  // [RBN / 32 + 1] bit i: position i starts a run of equal composites
    uint2 *segtab = (uint2 *)XV;          // only while the composites are formed
    const u32 tid = threadIdx.x;
    const u32 E0 = a.bstart[b0], E1 = a.bstart[b1];
    const u32 M = E1 - E0;
    l3_segments(a.bstart, b0, b1, E0, M, segmask, segpre, segtab, L3_NT);
    __syncthreads();
    const int eshift = 32 + a.pb;
    const u64 remmask = a.R >= 64 ? ~0ull : ((1ull << a.R) - 1ull);
    u32 N = 32;
    while (N < M) N <<= 1;
    for (u32 i = tid; i < N; i += L3_NT) {
        u64 sk = ~0ull;
        if (i < M) {
            const u64 e = a.in[E0 + i];
            const u32 s = (u32)e;
            const u64 seg = seg_index(segmask, segpre, i);
            const u64 rem = (e >> eshift) & remmask;
            const bool sh = is_short_suffix(s, a.K, a.n);
            sk = (seg << 41) | (rem << 9) | (sh ? (u64)(a.n - s) : 256ull);
        }
        SK[i] = sk;
    }
    __syncthreads();
    for (u32 i = tid; i < N; i += L3_NT) XV[i] = i < M ? a.in[E0 + i] : 0ull;
    __syncthreads();
    for (u32 k = 2; k <= N; k <<= 1) {
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            for (u32 i = tid; i < N; i += L3_NT) {
                const u32 x = i ^ j;
                if (x > i) {
                    const bool asc = (i & k) == 0;
                    const u64 ka = SK[i], kb = SK[x];
                    if ((ka > kb) == asc && ka != kb) {
                        SK[i] = kb;
                        SK[x] = ka;
                        const u64 va = XV[i];
                        XV[i] = XV[x];
                        XV[x] = va;
                    }
                }
            }
            __syncthreads();
        }
    }
    // run heads as a bitmap (a group of equal long keys may hold thousands of members: no walk back element by element)
    for (u32 i = tid; i < ((M + 31u) & ~31u); i += L3_NT) {
        const bool hd = i < M && (i == 0 || SK[i - 1] != SK[i]);
        const u32 bal = __ballot_sync(0xffffffffu, hd);
        if ((tid & 31u) == 0) headbits[i >> 5] = bal;
    }
    __syncthreads();
    for (u32 i = tid; i < M; i += L3_NT) {
        const u64 sk = SK[i];
        const bool is_long = ((sk >> 8) & 1ull) != 0;
        bool active = false;
        u32 h = i;
        if (is_long) {
            const bool head_here = (headbits[i >> 5] >> (i & 31u)) & 1u;
            const bool next_same = i + 1 < M && !((headbits[(i + 1) >> 5] >> ((i + 1) & 31u)) & 1u);
            active = !head_here || next_same;
            u32 w = i >> 5;
            u32 m = headbits[w] & (0xffffffffu >> (31u - (i & 31u)));
            while (!m) m = headbits[--w];  // (bit 0 of word 0 is always set)
            h = w * 32u + 31u - (u32)__clz(m);
        }
        l3_emit(a, E0 + i, XV[i], active, E0 + h);
    }
}

// Two launches over the list of declined tiles: tiles of up to RB_N_SMALL elements with the half-size network (three
// CTAs per SM), the others with the full one; a CTA whose tile belongs to the other launch leaves at once.
template <int RBN, int CTAS>
__global__ void __launch_bounds__(L3_NT, CTAS) msd_local_sort_robust_kernel(L3Args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (blockIdx.x >= *a.nflagged) return;
    const u32 t = a.flagged[blockIdx.x];
    const u32 b0 = a.tile_first[t], b1 = a.tile_first[t + 1];
    const u32 M = a.bstart[b1] - a.bstart[b0];
    if ((M <= (u32)RB_N_SMALL) != (RBN == RB_N_SMALL)) return;
    robust_sort_range<RBN>(a, b0, b1, smem_raw);
}

// ---------------------------------------------------------------------------------------------
// Oversize buckets.  A bucket that one SM cannot order in shared memory (more than L3_MAXB
// suffixes share its BB leading key bits: poly-A, tandem and interspersed repeats of a genome) is
// not sorted at all in round 0: it is emitted as ONE group of suffixes that are known to share
// d0 = BB / bits symbols -- rank = first row of the bucket, every member active -- and the doubling
// rounds, which then start at h = d0 instead of K, order it together with the groups of equal
// K-symbol keys.  The at most d0 - 1 suffixes shorter than d0 symbols (their key is padded with the
// smallest symbol) stand first in their bucket, shortest first (strcmp order,
// stralg/suffix_array.c:26-30); they are final after round 0 and are moved there by
// msd_fix_shorts_kernel.  The other buckets of a tile that holds an oversize bucket are ordered by
// the bitonic network of the robust kernel, in batches that fit shared memory.
// ---------------------------------------------------------------------------------------------
struct OverArgs {
    uint4 *list;         // {first row, suffixes, bucket, short suffixes in it} per oversize bucket
    u32 *count;
    const u32 *shortb;   // [32] bucket of suffix n - j for j < d0, 0xffffffff beyond
    u32 d0;
    u32 *fix, *nfix;     // short suffixes met in oversize buckets: {row, suffix, first row of the bucket, -}
};

__global__ void msd_short_buckets_kernel(const u64 *__restrict__ packed, u32 n, int bits, int BB, u32 d0,
                                         u32 *__restrict__ shortb, DenseKey dk, int R) {
    const u32 j = threadIdx.x;
    u32 v = 0xffffffffu;
    if (j < d0 && j <= n) {
        v = dk.nsym ? (u32)(dense_key_at(packed, (u64)(n - j), bits, dk) >> R)
                    : (u32)(window_at(packed, (u64)(n - j), bits) >> (64 - BB));
    }
    shortb[j] = v;
}
// Dense keys: the members of bucket x hold the keys [x << R, (x + 1) << R) (below `span` = nsym^K); they share the
// leading base-nsym digits the two ends of that range share.  depth = the minimum over the oversize buckets.
__global__ void __launch_bounds__(256) msd_dense_depth_kernel(const u32 *__restrict__ bstart, u64 nb, u32 maxb, int R,
                                                              u32 nsym, u32 K, u64 span, u32 *__restrict__ depth) {
    const u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb || bstart[b + 1] - bstart[b] <= maxb) return;
    u64 lo = b << R, hi = ((b + 1) << R) - 1;
    if (hi >= span) hi = span - 1;
    u32 j = 0;  // trailing digits dropped until the two ends agree
    while (lo != hi && j < K) {
        lo /= nsym;
        hi /= nsym;
        ++j;
    }
    atomicMin(depth, K - j);
}

// out[0] = buckets with more than maxb suffixes, out[1] = suffixes in them
__global__ void __launch_bounds__(256) msd_count_oversize_kernel(const u32 *__restrict__ bstart, u64 nb, u32 maxb,
                                                                 unsigned long long *__restrict__ out) {
    const u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 c = 0;
    if (b < nb) {
        c = bstart[b + 1] - bstart[b];
        if (c <= maxb) c = 0;
    }
    const unsigned m = __ballot_sync(0xffffffffu, c != 0);
    if (!m) return;
    unsigned long long sum = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31u) == 0) {
        atomicAdd(&out[0], (unsigned long long)__popc(m));
        atomicAdd(&out[1], sum);
    }
}

__global__ void __launch_bounds__(L3_NT, 1) msd_bigtile_kernel(L3Args a, OverArgs o) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (blockIdx.x >= *a.nbig) return;
    const u32 t = a.big[blockIdx.x];
    const u32 b0 = a.tile_first[t], b1 = a.tile_first[t + 1];
    u32 bb = b0;
    while (bb < b1) {  // uniform over the CTA
        const u32 s0 = a.bstart[bb], c = a.bstart[bb + 1] - s0;
        if (c == 0) {
            ++bb;
            continue;
        }
        if (c > (u32)L3_MAXB) {
            if (threadIdx.x == 0) {
                u32 k = 0;
                for (u32 j = 0; j < 32; ++j) k += o.shortb[j] == bb ? 1u : 0u;
                o.list[atomicAdd(o.count, 1u)] = make_uint4(s0, c, bb, k);
            }
            ++bb;
            continue;
        }
        u32 be = bb + 1, M = c;
        while (be < b1) {
            const u32 c2 = a.bstart[be + 1] - a.bstart[be];
            if (c2 > (u32)L3_MAXB || M + c2 > (u32)L3_CAP) break;
            M += c2;
            ++be;
        }
        robust_sort_range<RB_N>(a, bb, be, smem_raw);
        __syncthreads();
        bb = be;
    }
}

__global__ void __launch_bounds__(256) msd_emit_shallow_kernel(L3Args a, OverArgs o) {
    const u32 nov = *o.count;
    constexpr u32 CH = 256 * 8;  // suffixes per chunk
    for (u32 i = 0; i < nov; ++i) {
        const uint4 en = o.list[i];
        const u32 nch = (en.y + CH - 1) / CH;
        // a bucket of a few chunks is taken by one CTA, a large one is spread over the grid
        u32 c0 = blockIdx.x, cstep = gridDim.x;
        if (nch <= 32) {
            if (i % gridDim.x != blockIdx.x) continue;
            c0 = 0;
            cstep = 1;
        }
        for (u32 ch = c0; ch < nch; ch += cstep) {
#pragma unroll 2
            for (u32 q = 0; q < 8; ++q) {
                const u32 j = ch * CH + q * 256 + threadIdx.x;
                if (j < en.y) {
                    const u32 g = en.x + j;
                    const u64 e = ld_stream_u64(a.in + g);
                    const u32 s = (u32)e;
                    const bool sh = (u64)s + (u64)o.d0 > (u64)a.n;
                    if (sh) {
                        const u32 slot = atomicAdd(o.nfix, 1u);
                        if (slot < 32) {
                            o.fix[4 * slot] = g;
                            o.fix[4 * slot + 1] = s;
                            o.fix[4 * slot + 2] = en.x;
                        }
                    }
                    l3_emit(a, g, e, !sh, en.x + en.w);
                }
            }
        }
    }
}

// one thread: the (at most d0 - 1) short suffixes of the oversize buckets swap places with whatever
// stands in the first rows of their bucket
__global__ void msd_fix_shorts_kernel(L3Args a, OverArgs o) {
    const u32 nf = min(*o.nfix, 32u);
    u32 pos[32], sv[32], st[32], tgt[32];
    for (u32 i = 0; i < nf; ++i) {
        pos[i] = o.fix[4 * i];
        sv[i] = o.fix[4 * i + 1];
        st[i] = o.fix[4 * i + 2];
    }
    for (u32 i = 0; i < nf; ++i) {
        u32 c = 0;
        for (u32 j = 0; j < nf; ++j) c += (st[j] == st[i] && sv[j] > sv[i]) ? 1u : 0u;
        tgt[i] = st[i] + c;  // shortest (largest start) first
    }
    a.short_rank[0] = nf;
    for (u32 i = 0; i < nf; ++i) {
        const u32 p = pos[i], q = tgt[i];
        if (p != q) {
            const u32 x = a.sa[q];
            a.sa[q] = sv[i];
            a.sa[p] = x;
            if (a.bwt) {
                const u8 xb = a.bwt[q];
                a.bwt[q] = a.bwt[p];
                a.bwt[p] = xb;
            }
            if (x == 0) *a.primary = p;
            // the active bit and the group head are kept by ROW: they move with the suffix
            const bool x_active = (a.actbits[q >> 5] >> (q & 31u)) & 1u;  // (x may be another short suffix)
            if (x_active) {
                a.actbits[p >> 5] |= 1u << (p & 31u);
                a.grow[p] = a.grow[q];
            } else {
                a.actbits[p >> 5] &= ~(1u << (p & 31u));
            }
            a.actbits[q >> 5] &= ~(1u << (q & 31u));
            for (u32 j = 0; j < nf; ++j)
                if (j != i && pos[j] == q) pos[j] = p;
            pos[i] = q;
        }
        // its rank is materialised by the caller (nothing can look for it inside the unsorted bucket)
        a.short_rank[1 + 2 * i] = sv[i];
        a.short_rank[2 + 2 * i] = q;
        if (sv[i] == 0) *a.primary = q;
    }
}

// ---------------------------------------------------------------------------------------------
// rows whose active bit is clear hold suffixes that are final: their rank is their row
__global__ void __launch_bounds__(256) fill_singleton_ranks_kernel(const u32 *__restrict__ sa, u32 len,
                                                                   const u32 *__restrict__ actbits, u32 *__restrict__ rank) {
    u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= len) return;
    if (!((actbits[g >> 5] >> (g & 31u)) & 1u)) rank[sa[g]] = (u32)g;
}

void fill_singleton_ranks(const DeviceIndex &ix, const u32 *actbits, u32 *rank) {
    fill_singleton_ranks_kernel<<<div_up_u(ix.len, 256), 256, 0, ix.stream>>>(ix.sa.ptr, ix.len, actbits, rank);
    KERNEL_CHECK();
}

// ---------------------------------------------------------------------------------------------
// Host orchestration
// ---------------------------------------------------------------------------------------------
template <int BITS>
static void launch_hist_text(const DeviceIndex &ix, u64 nwords_data, int D, u32 *hist, cudaStream_t st,
                             const MsdPlan &pl) {
    unsigned blocks = div_up_u(nwords_data, 256 * 4);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks == 0) blocks = 1;
    if (pl.dense.nsym)
        msd_hist_text_kernel<BITS, true><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, D, hist, pl.dense, pl.KB - D);
    else
        msd_hist_text_kernel<BITS><<<blocks, 256, 0, st>>>(ix.packed, ix.n, nwords_data, D, hist);
    KERNEL_CHECK();
}

template <int BITS, bool HAS_PREV, bool DENSE>
static void launch_part_text(const Text1Args &ta, int device, cudaStream_t st) {
    static PerDeviceOnce once;
    if (once.first(device))
        CUDA_CHECK(cudaFuncSetAttribute(msd_partition_text_kernel<BITS, HAS_PREV, DENSE>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T1_SMEM));
    msd_partition_text_kernel<BITS, HAS_PREV, DENSE><<<div_up_u(ta.len, T1_TILE), T1_NT, T1_SMEM, st>>>(ta);
}

bool round0_msd(DeviceIndex &ix, bool want_bwt, Round0Msd &r) {
    cudaStream_t st = ix.stream;
    Arena &ar = *ix.arena;
    MsdPlan &pl = r.plan;  // a partition level may be added below
    const u32 n = ix.n, len = ix.len;
    const int b = ix.pk.bits;

    static PerDeviceOnce once;
    if (once.first(ix.device)) {
        CUDA_CHECK(cudaFuncSetAttribute(msd_partition_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P_SMEM));
        CUDA_CHECK(cudaFuncSetAttribute(msd_local_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L3_SMEM));
        CUDA_CHECK(cudaFuncSetAttribute(msd_local_sort_robust_kernel<RB_N, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RB_SMEM));
        CUDA_CHECK(cudaFuncSetAttribute(msd_local_sort_robust_kernel<RB_N_SMALL, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rb_smem<RB_N_SMALL>()));
        CUDA_CHECK(cudaFuncSetAttribute(msd_bigtile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RB_SMEM));
    }

    // ---- tables (those of a level are carved when the level is reached: one may be added) ----
    u64 nb[3] = {0, 0, 0};  // buckets after level l
    u32 *start[3] = {nullptr, nullptr, nullptr}, *cursor[3] = {nullptr, nullptr, nullptr};
    auto level_tables = [&](int l) {
        nb[l] = (l ? nb[l - 1] : 1ull) << pl.D[l];
        start[l] = ar.get<u32>(nb[l] + 1);
        cursor[l] = ar.get<u32>(nb[l]);
        CUDA_CHECK(cudaMemsetAsync(cursor[l], 0, nb[l] * 4, st));
    };
    // 0: max final bucket, 1: tiles of the current level, 4: declined tiles, 5: big tiles,
    // 6: oversize buckets, 7: short suffixes met in them
    u32 *d_misc = ar.get<u32>(8);
    CUDA_CHECK(cudaMemsetAsync(d_misc, 0, 8 * 4, st));
    unsigned long long *d_over = ar.get<unsigned long long>(2);
    r.shallow_buckets = 0;
    r.shallow_elems = 0;
    r.depth0 = (u32)pl.K;
    r.levels_added = 0;

    // Once the bucket sizes of the last planned level are known (before that level moves anything): do
    // the buckets fit one SM?
    //   * all do: go on (uniform texts);
    //   * buckets that do not hold more than 1/64 of the text and the key has bits left: one more
    //     partition level (texts with a skewed k-mer spectrum, e.g. real genomes, where the planned
    //     average says little about the common k-mers);
    //   * what is still too large afterwards is emitted unsorted as shallow groups (see OverArgs) --
    //     unless that is more than 1/8 of the text (periodic texts: every bucket), where the caller's
    //     LSD path, whose keys are K symbols deep instead of BB / bits, is the better start.
    enum { GO, MORE, FALLBACK };
    u32 dense_d0 = 0;
    auto decide = [&](const u32 *final_start, u64 nbuckets) -> int {
        u32 maxbucket = 0;
        read_back(&maxbucket, d_misc, 4, st);
        if (env_int("B200SA_DEBUG_PLAN", 0))
            fprintf(stderr, "[b200sa] round-0 plan: levels %d D %d/%d/%d BB %d K %d KB %d pb %d R %d dense %u (%u+%u, powlo %u) max bucket %u\n",
                    pl.nlevels, pl.D[0], pl.D[1], pl.D[2], pl.BB, pl.K, pl.KB, pl.pb, pl.R, pl.dense.nsym, pl.dense.Khi,
                    pl.dense.Klo, pl.dense.powlo, maxbucket);
        if (maxbucket <= (u32)L3_MAXB) return GO;
        if (env_int("B200SA_MSD_NO_OVERSIZE", 0)) return FALLBACK;
        CUDA_CHECK(cudaMemsetAsync(d_over, 0, 16, st));
        msd_count_oversize_kernel<<<div_up_u(nbuckets, 256), 256, 0, st>>>(final_start, nbuckets, (u32)L3_MAXB, d_over);
        KERNEL_CHECK();
        unsigned long long h[2];
        read_back(h, d_over, 16, st);
        if (env_int("B200SA_DEBUG_PLAN", 0)) fprintf(stderr, "[b200sa] oversize buckets: %llu with %llu suffixes\n", h[0], h[1]);
        const int more_frac = std::max(1, env_int("B200SA_MSD_MORE_FRAC", 64));
        const int bbmax = env_int("B200SA_MSD_BBMAX", 26);
        const int bq = pl.dense.nsym ? 1 : b;  // (dense keys: digits are not tied to symbol boundaries)
        int room = std::min(std::min(pl.dmax, pl.R), bbmax - pl.BB) / bq * bq;
        if (h[1] > (unsigned long long)len / (unsigned)more_frac && pl.nlevels < 3 && room >= bq) {
            pl.D[pl.nlevels++] = room;
            pl.BB += room;
            pl.R -= room;
            ++r.levels_added;
            CUDA_CHECK(cudaMemsetAsync(d_misc, 0, 4, st));
            return MORE;
        }
        const int frac = std::max(1, env_int("B200SA_MSD_OVER_FRAC", 8));
        if (h[1] > (unsigned long long)len / (unsigned)frac) return FALLBACK;
        if (pl.dense.nsym) {
            // what the members of an oversize bucket of dense keys are known to share
            CUDA_CHECK(cudaMemsetAsync(d_misc + 2, 0xff, 4, st));
            msd_dense_depth_kernel<<<div_up_u(nbuckets, 256), 256, 0, st>>>(final_start, nbuckets, (u32)L3_MAXB, pl.R, pl.dense.nsym,
                                                                           (u32)pl.K, pow_u64(pl.dense.nsym, pl.K), d_misc + 2);
            KERNEL_CHECK();
            read_back(&dense_d0, d_misc + 2, 4, st);
            if (env_int("B200SA_DEBUG_PLAN", 0)) fprintf(stderr, "[b200sa] dense keys: oversize buckets share %u symbols\n", dense_d0);
            // (a bucket that straddles a change of a leading symbol shares little: rare)
            if (dense_d0 < (u32)std::max(2, pl.K / 4) || dense_d0 > 32) return FALLBACK;
        }
        r.shallow_elems = h[1];  // (an upper bound: such a bucket is still sorted when its whole tile fits)
        return GO;
    };

    const u32 ntl3 = div_up_u(len, L3_TSZ);
    u32 *tile_first = ar.get<u32>((size_t)ntl3 + 2);
    u32 *flagged = ar.get<u32>((size_t)ntl3 + 1);
    u32 *bigtiles = ar.get<u32>((size_t)ntl3 + 1);
    // no row is active
    CUDA_CHECK(cudaMemsetAsync(r.actbits, 0, (((size_t)len + 31) / 32 + 2) * 4, st));
    r.short_rank = ar.get<u32>(1 + 2 * 32);
    CUDA_CHECK(cudaMemsetAsync(r.short_rank, 0, 4, st));

    // ---- level 1: from the text ----
    level_tables(0);
    const u64 nwords_data = ((u64)len + ix.pk.cpw - 1) / ix.pk.cpw;
    int t = ix.timer.begin("msd_hist1", (double)len * b / 8.0);
    switch (b) {
        case 1: launch_hist_text<1>(ix, nwords_data, pl.D[0], cursor[0], st, pl); break;
        case 2: launch_hist_text<2>(ix, nwords_data, pl.D[0], cursor[0], st, pl); break;
        case 4: launch_hist_text<4>(ix, nwords_data, pl.D[0], cursor[0], st, pl); break;
        default: launch_hist_text<8>(ix, nwords_data, pl.D[0], cursor[0], st, pl); break;
    }
    if (pl.dense.nsym && !env_int("B200SA_MSD_BB", 0)) {
        // Dense keys spread evenly when the letters are equally likely.  The level-1 histogram tells how far the text
        // is from that (a rare letter -- N in DNA --, skewed amino-acid frequencies): with H1 bits of entropy in its
        // D1 leading key bits, a key bit carries h = (H1 - log2 fill) / D1 bits (fill: the used part of the top
        // digit's range), and BB bucket bits give about fill * 2^(h * BB) buckets of equal weight.  More bucket bits
        // are planned when that is fewer than the suffixes need.
        std::vector<u32> h1((size_t)nb[0]);
        read_back(h1.data(), cursor[0], (size_t)nb[0] * 4, st);
        double H1 = 0.0;
        for (u32 c : h1)
            if (c) {
                const double p = (double)c / (double)len;
                H1 -= p * std::log2(p);
            }
        const double lfill = std::log2((double)pow_u64(pl.dense.nsym, pl.K)) - (double)pl.KB;  // <= 0
        const double h = std::min(1.0, std::max(0.05, (H1 - lfill) / (double)pl.D[0]));
        const double want = std::log2(std::max(2.0, (double)len / 2000.0));
        int BBn = (int)std::ceil((want - lfill) / h);
        BBn = std::min(BBn, std::min(pl.D[0] + 2 * pl.dmax, pl.KB));
        {
            // (never more than one bucket per 64 suffixes: a text of one letter has no entropy to plan with, and its
            // tables must not outgrow it)
            int log2len = 0;
            while ((1ull << log2len) < (u64)len) ++log2len;
            BBn = std::min(BBn, std::max(pl.BB, log2len - 6));
        }
        if (BBn > pl.BB) {
            const int rem = BBn - pl.D[0], nl2 = (rem + pl.dmax - 1) / pl.dmax;
            for (int i = 0; i < nl2; ++i) pl.D[1 + i] = rem / nl2 + (i < rem % nl2 ? 1 : 0);
            for (int i = 1 + nl2; i < 3; ++i) pl.D[i] = 0;
            pl.nlevels = 1 + nl2;
            pl.BB = BBn;
            pl.R = pl.KB - BBn;
        }
        if (env_int("B200SA_DEBUG_PLAN", 0))
            fprintf(stderr, "[b200sa] dense keys: level-1 entropy %.2f of %d bits, %.3f per key bit -> %d bucket bits\n", H1, pl.D[0], h, pl.BB);
    }
    {
        unsigned bd = std::min(1024u, std::max(32u, (unsigned)nb[0]));
        msd_scan_children_kernel<<<1, bd, 0, st>>>(cursor[0], nullptr, pl.D[0], 1, len, start[0],
                                                   pl.nlevels == 1 ? d_misc : nullptr);
        KERNEL_CHECK();
    }
    ix.timer.end(t);
    if (pl.nlevels == 1 && decide(start[0], nb[0]) == FALLBACK) return false;

    {
        Text1Args ta{};
        ta.packed = ix.packed;
        ta.nwords = nwords_data + 4;  // pack_text pads with 4 zero words
        ta.out = r.bufA;
        ta.len = len; ta.bits = b; ta.KB = pl.KB; ta.pb = pl.pb;
        ta.D = pl.D[0];
        ta.dshift = pl.KB - pl.D[0];
        ta.restmask = ta.dshift >= 64 ? ~0ull : ((1ull << ta.dshift) - 1ull);
        ta.rest_shift = 32 + pl.pb;
        ta.cursor = cursor[0];
        t = ix.timer.begin("msd_part1", (double)len * (8.0 + b / 8.0));
        ta.dense = pl.dense;
        const int dev = ix.device;
        const bool prev = pl.pb != 0;
        if (pl.dense.nsym) {  // (dense keys: 2, 4 or 8 bits per symbol)
            switch (b) {
                case 2: prev ? launch_part_text<2, true, true>(ta, dev, st) : launch_part_text<2, false, true>(ta, dev, st); break;
                case 4: prev ? launch_part_text<4, true, true>(ta, dev, st) : launch_part_text<4, false, true>(ta, dev, st); break;
                default: prev ? launch_part_text<8, true, true>(ta, dev, st) : launch_part_text<8, false, true>(ta, dev, st); break;
            }
        } else {
            switch (b) {
                case 1: prev ? launch_part_text<1, true, false>(ta, dev, st) : launch_part_text<1, false, false>(ta, dev, st); break;
                case 2: prev ? launch_part_text<2, true, false>(ta, dev, st) : launch_part_text<2, false, false>(ta, dev, st); break;
                case 4: prev ? launch_part_text<4, true, false>(ta, dev, st) : launch_part_text<4, false, false>(ta, dev, st); break;
                default: prev ? launch_part_text<8, true, false>(ta, dev, st) : launch_part_text<8, false, false>(ta, dev, st); break;
            }
        }
        KERNEL_CHECK();
        ix.timer.end(t);
    }
    PartArgs pa{};
    u64 *cur = r.bufA, *other = r.bufB;
    int consumed = pl.D[0];
    for (int l = 1; l < pl.nlevels; ++l) {
        level_tables(l);
        const u32 nparents = (u32)nb[l - 1];
        const int dshift = 32 + pl.pb + (pl.KB - consumed - pl.D[l]);
        // tiles of this level (a tile never straddles two parents)
        const size_t desc_cap = (size_t)div_up_u(len, P_TILE) + nparents + 1;
        uint4 *desc = ar.get<uint4>(desc_cap);
        u32 *tile_off = ar.get<u32>((size_t)nparents + 2);
        t = ix.timer.begin("msd_hist", (double)len * 8.0);
        msd_tile_offsets_kernel<<<1, 1024, 0, st>>>(start[l - 1], nparents, tile_off, d_misc + 1);
        KERNEL_CHECK();
        msd_tile_desc_kernel<<<div_up_u(nparents, 8), 256, 0, st>>>(start[l - 1], nparents, tile_off, desc);
        KERNEL_CHECK();
        const unsigned grid = (unsigned)std::min<size_t>(desc_cap, 0x7fffffffu);
        msd_hist_elems_kernel<<<std::min(grid, 4u * sm_count(ix.device)), P_NT, 0, st>>>(cur, desc, d_misc + 1, pl.D[l], dshift, cursor[l]);
        KERNEL_CHECK();
        {
            unsigned bd = std::min(1024u, std::max(32u, 1u << pl.D[l]));
            msd_scan_children_kernel<<<nparents, bd, 0, st>>>(cursor[l], start[l - 1], pl.D[l], nparents, len, start[l],
                                                              l == pl.nlevels - 1 ? d_misc : nullptr);
            KERNEL_CHECK();
        }
        ix.timer.end(t);
        // (MORE extends pl.nlevels: the loop then runs one more level after this one)
        if (l == pl.nlevels - 1 && decide(start[l], nb[l]) == FALLBACK) return false;
        pa.in = cur; pa.out = other;
        pa.D = pl.D[l];
        pa.dshift = dshift;
        pa.cursor = cursor[l];
        pa.desc = desc; pa.d_ntiles = d_misc + 1;
        t = ix.timer.begin("msd_part", (double)len * 16.0);
        msd_partition_kernel<<<std::min(grid, 2u * sm_count(ix.device)), P_NT, P_SMEM, st>>>(pa);
        KERNEL_CHECK();
        ix.timer.end(t);
        std::swap(cur, other);
        consumed += pl.D[l];
    }

    // ---- in-SM sort of every bucket, outputs of round 0 ----
    const int last = pl.nlevels - 1;
    t = ix.timer.begin("msd_local_sort", (double)len * (8.0 + 4.0 + (want_bwt && pl.pb ? 1.0 : 0.0)));
    msd_tile_first_kernel<<<div_up_u(nb[last] + 1, 256), 256, 0, st>>>(start[last], nb[last], ntl3, tile_first);
    KERNEL_CHECK();
    L3Args la{};
    la.in = cur; la.bstart = start[last]; la.tile_first = tile_first; la.n = n;
    la.K = pl.K; la.pb = pl.pb; la.R = pl.R;
    la.par_shift = pl.BB - pl.D[0];
    la.sa = ix.sa.ptr;
    la.bwt = (want_bwt && pl.pb) ? ix.bwt.ptr : nullptr;
    la.short_rank = r.short_rank; la.actbits = r.actbits;
    la.grow = (u32 *)other;  // the ping-pong buffer the elements do NOT sit in is free
    la.primary = r.d_primary;
    la.flagged = flagged; la.nflagged = d_misc + 4;
    la.big = bigtiles; la.nbig = d_misc + 5;
    la.ntiles = ntl3;
    msd_local_sort_kernel<<<std::min(ntl3, (unsigned)L3_CTAS * sm_count(ix.device)), L3_NT, L3_SMEM, st>>>(la);
    KERNEL_CHECK();
    u32 hmisc[8];
    read_back(hmisc, d_misc, sizeof hmisc, st);
    if (hmisc[4]) {
        msd_local_sort_robust_kernel<RB_N_SMALL, 3><<<hmisc[4], L3_NT, rb_smem<RB_N_SMALL>(), st>>>(la);
        KERNEL_CHECK();
        msd_local_sort_robust_kernel<RB_N, 1><<<hmisc[4], L3_NT, RB_SMEM, st>>>(la);
        KERNEL_CHECK();
        read_back(hmisc, d_misc, sizeof hmisc, st);
    }
    ix.timer.end(t);
    if (hmisc[5]) {
        // tiles with an oversize bucket: their other buckets are ordered by the bitonic network, the
        // oversize ones are emitted as shallow groups
        t = ix.timer.begin("msd_oversize", (double)r.shallow_elems * (8.0 + 4.0 + 4.0 + 4.0));
        OverArgs oa{};
        oa.list = ar.get<uint4>((size_t)len / (size_t)L3_MAXB + 2);
        oa.count = d_misc + 6;
        u32 *shortb = ar.get<u32>(32);
        oa.shortb = shortb;
        oa.d0 = pl.dense.nsym ? dense_d0 : (u32)(pl.BB / b);
        oa.fix = ar.get<u32>(4 * 32);
        oa.nfix = d_misc + 7;
        msd_short_buckets_kernel<<<1, 32, 0, st>>>(ix.packed, n, b, pl.BB, oa.d0, shortb, pl.dense, pl.R);
        KERNEL_CHECK();
        msd_bigtile_kernel<<<hmisc[5], L3_NT, RB_SMEM, st>>>(la, oa);
        KERNEL_CHECK();
        msd_emit_shallow_kernel<<<8u * sm_count(ix.device), 256, 0, st>>>(la, oa);
        KERNEL_CHECK();
        msd_fix_shorts_kernel<<<1, 1, 0, st>>>(la, oa);
        KERNEL_CHECK();
        read_back(hmisc, d_misc, sizeof hmisc, st);
        r.shallow_buckets = hmisc[6];
        if (hmisc[6]) r.depth0 = oa.d0;
        ix.timer.end(t);
    }

    r.bucket_start = start[last];
    r.grow = la.grow;
    r.bwt_written = la.bwt != nullptr;
    return true;
}

}  // namespace b200sa
