// walk.cuh -- the host side of the depth-first FM-index walks (approx.cu, hamming.cu, levenshtein.cu): launches sized
// by their frame stacks, and the arguments and shared passes of the two searches on an index pair.
#pragma once
#include "engine.h"
#include "fm_step.cuh"

#include <algorithm>

namespace b200sa {

// Work units per launch: the frame stacks of one launch stay under ~1 GiB (at least 1024 units a launch).
inline u64 walk_units_per_launch(u64 units, u64 bytes_per_unit) {
    return std::min(std::max<u64>(1024, ((u64)1 << 30) / bytes_per_unit), units);
}

// a walk kernel of each layout and pass: [DNA layout ? 0 : 1][emitting pass]
template <class Args>
using WalkKernels = void (*const[2][2])(Args);

// Runs units [0, units) of a walk, `chunk` units a launch (A.first, A.count), threads_per_unit threads a unit in
// blocks of `block`.
template <class Args>
void run_walk(WalkKernels<Args> &kernels, const DeviceIndex &ix, bool emit, Args &A, u64 units, u64 chunk,
              u32 threads_per_unit, u32 block, cudaStream_t st) {
    void (*const kernel)(Args) = kernels[ix.occ_layout == OCC_DNA32 ? 0 : 1][emit ? 1 : 0];
    for (u64 first = 0; first < units; first += chunk) {
        A.first = first;
        A.count = std::min(chunk, units - first);
        kernel<<<div_up_u(A.count * threads_per_unit, block), block, 0, st>>>(A);
        KERNEL_CHECK();
    }
}

// ---- the k-mismatch and edit-distance searches on an index pair ------------------------------------------------
struct PairArgs {
    OccView fv, bv;        // F (the text) and B (the reversed text)
    CTable5 c5;            // DNA layout: C table (both indices)
    const u32 *c_dev;      // byte layout: C table (sigma entries)
    u32 len, k;
    const u8 *pat;
    const u64 *off;
    u32 fixed_len;
    u64 first, count;      // work units [first, first + count) run in this launch; unit u = (u / (k + 1), u % (k + 1))
    uint4 *stack;          // count * frames per unit frames (hamming.cu, levenshtein.cu: their layout)
    u32 *stack_w;          // edit distance: the fifth word of each frame (null for k-mismatch)
    // counting pass
    u64 *unit_count;       // (raw) hits per unit
    // emitting pass
    const u64 *unit_off;   // exclusive scan of unit_count
    u64 *key;              // per (raw) hit: the sort key, [pattern | L] or [pattern | L | length offset]
    u32 *val, *R, *d;      // per (raw) hit: its index, R and its distance
};

extern WalkKernels<PairArgs> hamming_walk_kernels, levenshtein_walk_kernels;

// The emitting walk of one piece and the stable radix sort of its hits on key_bits + ceil(log2 npat) key bits
// (hamming.cu): R and d are indexed by the sorted hit indices `val`.
struct PairHits {
    DevBuf<u64> kA, kB;
    DevBuf<u32> vA, vB, R, d;
    u64 *key = nullptr;  // the sorted keys and hit indices: kA / vA or kB / vB
    u32 *val = nullptr;
};
PairHits pair_sorted_hits(PairSearch s, const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat,
                          const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m, u32 k, const u64 *d_unit_off, u64 hits,
                          int key_bits, cudaStream_t st);

}  // namespace b200sa
