// approx.cu -- batched approximate (edit distance <= d) backward search (sm_100a).
//
// Reference: rec_approx_matching / init_bwt_approx_iter, stralg/bwt.c:226-382.  The reference
// walks, per pattern, a depth-first tree of (L, R, i, matched length, edits left) nodes from the
// last pattern symbol to the first.  Children of a node, in order: for every letter a = 1..sigma-1
// a match/substitution step 'M' (cost 0 when a == pattern[i], else 1) to (C[a]+O(a,L), C[a]+O(a,R),
// i-1); one insertion step 'I' (same interval, i-1, cost 1); for every letter a deletion step 'D'
// (narrowed interval, same i, cost 1).  The first level has no deletions and no D-table test
// (bwt.c:349-377).  A node with edits_left < D[i] is abandoned (bwt.c:237-240), empty intervals
// are not entered, and i < 0 is a hit: (L, R, matched length, operations of the path).
//
// Here a group of 16 lanes owns one pattern and runs that walk with an explicit stack of 16-byte
// frames in HBM (frame f of pattern t at [f * patterns + t]); the children of a node are evaluated
// by the lanes side by side and taken in exactly the reference's order, so the hits of a pattern
// come out in the reference's report order.  Conditions that make the reference return immediately from a
// child (edits_left < D, empty interval) are tested BEFORE the O lookups of that child -- they
// have no side effects, so the hit list is unchanged.  The walk runs twice: a counting pass
// (hits and CIGAR bytes per pattern), an exclusive scan, and an emitting pass that
// writes every hit at its final offset -- no atomics, deterministic output.
//
// Records index (records.cu): letter 1 is the separator between records.  Its match / substitution
// and deletion children are not viable, so no walk crosses a record boundary; child numbering, and
// so the report order, is that of the plain walk.  The flag is off for a plain index.
//
// D table (bwt.c:319-337): forward over the pattern with the O table of the REVERSED text (a
// second index), restarting the interval whenever it empties; D[i] = restarts so far.
#include "engine.h"
#include "occ.cuh"
#include "scan.cuh"

#include <algorithm>

namespace b200sa {

struct ApproxArgs {
    OccView ov;
    const u32 *c_dev;
    u32 len, sigma;
    const u8 *pat;
    const u64 *off;
    u32 fixed_len;
    u64 first, count;      // patterns [first, first + count) of the batch run in this launch
    const u8 *dtab;        // D value per pattern symbol (same offsets as `pat`), or null
    int max_edits;
    bool no_sep;           // records index: letter 1 is the record separator and is never consumed
    uint4 *stack;          // count * max_depth frames
    u32 max_depth;
    // counting pass
    u32 *hit_count;        // per pattern
    u64 *ops_count;        // per pattern: bytes of CIGAR text (NULs included)
    // emitting pass
    const u64 *hit_off;    // per pattern (exclusive scan of hit_count), [npat] = total
    const u64 *ops_off;    // per pattern (exclusive scan of ops_count)
    u32 *out_L, *out_R, *out_mlen;
    u64 *out_ops_off;      // per hit: start of its CIGAR in out_ops
    char *out_ops;         // CIGAR strings (NUL-terminated), one per hit
};

// frame: x = L, y = R, z = (i + 1) | edits_left << 16 | op << 24, w = cursor | matched length << 16
__device__ __forceinline__ uint4 make_frame(u32 L, u32 R, int i, int left, u32 op, u32 cursor, u32 mlen) {
    return make_uint4(L, R, (u32)(i + 1) | ((u32)left << 16) | (op << 24), cursor | (mlen << 16));
}

template <int LAYOUT>
__device__ __forceinline__ u32 occ_sym(const OccView &ov, u32 a, u32 i) {
    return LAYOUT == 1 ? occ_dna(ov, a, i) : occ_byte(ov, a, i);
}

// One GROUP of 16 lanes owns one pattern (two patterns per warp).  The node state is uniform over
// the group; lane j evaluates child j of the current node (its edit cost, the D-table test and the
// two O lookups), a ballot gives the viable children, and they are taken in the reference's order:
//   * a child with i < 0 is a hit;
//   * a child with no edits left can only continue by exact matching (every other step costs an
//     edit): its whole subtree is the chain pattern[i], pattern[i-1], ... which is run inline,
//     without touching the stack, and ends in at most one hit;
//   * any other child is entered: the current node is parked in the stack with the index of its
//     next child, and re-evaluated when the walk comes back to it.
// sigma - 1 <= 7 letters fit one evaluation (2 (sigma-1) + 1 <= 15 children); larger alphabets take
// their children 16 at a time.
static constexpr int AG = 16;  // lanes per pattern

template <int LAYOUT, bool EMIT>
__global__ void __launch_bounds__(128, 8) approx_walk_kernel(ApproxArgs A) {
    __shared__ u32 c_sh[256];
    for (u32 k = threadIdx.x; k < 256; k += blockDim.x) c_sh[k] = k < A.sigma ? A.c_dev[k] : 0;
    __syncthreads();
    const u64 t = ((u64)blockIdx.x * blockDim.x + threadIdx.x) / AG;  // group = pattern of this launch
    if (t >= A.count) return;
    const u32 gl = threadIdx.x & (AG - 1);                  // lane inside the group
    const u32 gshift = (threadIdx.x & 31u) & ~(u32)(AG - 1);  // first warp lane of the group
    const u32 gmask = 0xffffu << gshift;
    const u64 q = A.first + t;
    const u64 begin = A.off ? A.off[q] : q * (u64)A.fixed_len;
    const u32 m = A.off ? (u32)(A.off[q + 1] - begin) : A.fixed_len;
    const u8 *p = A.pat + begin;
    const u8 *dt = A.dtab ? A.dtab + begin : nullptr;
    const u32 nsym = A.sigma - 1;  // letters 1..nsym
    uint4 *stk = A.stack + t;
    const u64 lanes = A.count;

    u32 nhits = 0;
    u64 nops = 0;
    u64 hit_at = 0, ops_at = 0;
    if (EMIT) {
        hit_at = A.hit_off[q];
        ops_at = A.ops_off[q];
    }
    if (m == 0 || nsym == 0) {
        if (!EMIT && gl == 0) {
            A.hit_count[q] = 0;
            A.ops_count[q] = 0;
        }
        return;
    }

    // the root: whole range, all symbols left, all edits left
    u32 L = 0, R = A.len, cursor = 0, mlen = 0, op = 0;
    int i = (int)m - 1, left = A.max_edits;
    u32 depth = 0;  // frames below the current one
    while (true) {
        const u32 nchildren = depth == 0 ? nsym + 1 : 2 * nsym + 1;
        if (cursor >= nchildren) {
            if (depth == 0) break;
            --depth;
            const uint4 f = stk[(u64)depth * lanes];
            L = f.x; R = f.y;
            i = (int)(f.z & 0xffffu) - 1;
            left = (int)((f.z >> 16) & 0xffu);
            op = (f.z >> 24) & 3u;
            cursor = f.w & 0xffffu;
            mlen = f.w >> 16;
            continue;
        }
        // ---- lane gl evaluates child cb + gl ----
        const u32 cb = cursor & ~(u32)(AG - 1);
        const u32 cidx = cb + gl;
        u32 a, cop;
        int ci, cleft;
        if (cidx < nsym) {  // match / substitution
            a = cidx + 1;
            cop = 0;
            ci = i - 1;
            cleft = left - (a == (u32)p[i] ? 0 : 1);
        } else if (cidx == nsym) {  // insertion: the pattern symbol is skipped
            a = 0;
            cop = 1;
            ci = i - 1;
            cleft = left - 1;
        } else {  // deletion: a text symbol is skipped
            a = cidx - nsym;
            cop = 2;
            ci = i;
            cleft = left - 1;
        }
        // (on a records index a match / substitution or deletion of the separator would run into the next record)
        bool viable = cidx >= cursor && cidx < nchildren && cleft >= 0 && !(A.no_sep && a == 1);
        if (viable) {
            const int need = (ci >= 0 && dt) ? (int)dt[ci] : 0;
            viable = cleft >= need;
        }
        u32 cL = L, cR = R;
        if (viable && a) {
            const u32 ca = c_sh[a];
            cL = ca + occ_sym<LAYOUT>(A.ov, a, L);
            cR = ca + occ_sym<LAYOUT>(A.ov, a, R);
            viable = cL < cR;
        }
        u32 vmask = (__ballot_sync(gmask, viable) >> gshift) & 0xffffu;
        // Children that still have edits left must be entered; every viable child ahead of the first
        // of them is a hit (i < 0) or a zero-edit chain.  The chains of those children run side by side,
        // lane j walking pattern[i], pattern[i-1], ... for child j; the children behind the first one to
        // enter are looked at again when the walk returns to this node.
        const u32 dmask = (__ballot_sync(gmask, viable && ci >= 0 && cleft > 0) >> gshift) & 0xffffu;
        const u32 first_enter = dmask ? (u32)__ffs((int)dmask) - 1u : (u32)AG;
        u32 chain = 0;  // exact steps taken below this lane's child (no edits left)
        bool lane_hit = viable && gl < first_enter && ci < 0;
        if (viable && gl < first_enter && ci >= 0) {  // cleft == 0 here
            lane_hit = true;
            while (ci >= 0) {
                const u32 x = p[ci];
                if ((dt && dt[ci] > 0) || x == 0 || x > nsym) {
                    lane_hit = false;
                    break;
                }
                const u32 ca = c_sh[x];
                const u32 nl = ca + occ_sym<LAYOUT>(A.ov, x, cL), nr = ca + occ_sym<LAYOUT>(A.ov, x, cR);
                if (nl >= nr) {
                    lane_hit = false;
                    break;
                }
                cL = nl; cR = nr;
                --ci;
                ++chain;
            }
        }
        __syncwarp(gmask);
        u32 hmask = (__ballot_sync(gmask, lane_hit) >> gshift) & 0xffffu;
        // hits of the children ahead of the first one to enter, in child order
        while (hmask) {
            const int j = __ffs((int)hmask) - 1;
            hmask &= hmask - 1u;
            const int src = (int)gshift + j;
            const u32 bL = __shfl_sync(gmask, cL, src), bR = __shfl_sync(gmask, cR, src);
            const u32 bop = __shfl_sync(gmask, cop, src);
            const u32 bchain = __shfl_sync(gmask, chain, src);
            const u32 bm = mlen + (bop != 1 ? 1u : 0u) + bchain;
            {
                // The path in pattern order (= reversed): the chain's matches, the child's step, the
                // current node's own step, then the parked frames from the top down to frame 1;
                // run-length encoded into the CIGAR text of cigar.c:17-31 (sprintf("%d%c")).
                const u32 plen = depth + 1 + bchain;
                auto path_op = [&](u32 k) -> u32 {
                    if (k < bchain) return 0u;
                    k -= bchain;
                    return k == 0 ? bop : k == 1 ? op : ((stk[(u64)(depth + 1 - k) * lanes].z >> 24) & 3u);
                };
                char *w = EMIT ? A.out_ops + ops_at + nops : nullptr;
                u32 bytes = 0;
                for (u32 k = 0; k < plen;) {
                    const u32 o = path_op(k);
                    u32 run = (o == 0 && k < bchain) ? bchain - k : 1u;
                    while (k + run < plen && path_op(k + run) == o) ++run;
                    const u32 digits = run >= 10000u ? 5u : run >= 1000u ? 4u : run >= 100u ? 3u : run >= 10u ? 2u : 1u;
                    if (EMIT && gl == 0) {
                        u32 v = run;
                        for (u32 dgt = digits; dgt-- > 0;) {
                            w[bytes + dgt] = (char)('0' + v % 10u);
                            v /= 10u;
                        }
                        w[bytes + digits] = o == 0 ? 'M' : o == 1 ? 'I' : 'D';
                    }
                    bytes += digits + 1u;
                    k += run;
                }
                if (EMIT && gl == 0) {
                    w[bytes] = '\0';
                    const u64 h = hit_at + nhits;
                    A.out_L[h] = bL;
                    A.out_R[h] = bR;
                    A.out_mlen[h] = bm;
                    A.out_ops_off[h] = ops_at + nops;
                }
                ++nhits;
                nops += bytes + 1u;
            }
        }
        if (first_enter < (u32)AG) {
            // enter that child: park the current node with the index of its next child
            const int src = (int)(gshift + first_enter);
            const u32 bL = __shfl_sync(gmask, cL, src), bR = __shfl_sync(gmask, cR, src);
            const int bi = __shfl_sync(gmask, ci, src), bleft = __shfl_sync(gmask, cleft, src);
            const u32 bop = __shfl_sync(gmask, cop, src);
            if (gl == 0) stk[(u64)depth * lanes] = make_frame(L, R, i, left, op, cb + first_enter + 1u, mlen);
            __syncwarp(gmask);
            ++depth;
            mlen += bop != 1 ? 1u : 0u;
            L = bL; R = bR; i = bi; left = bleft; op = bop; cursor = 0;
        } else {
            cursor = cb + AG;
        }
    }
    if (!EMIT && gl == 0) {
        A.hit_count[q] = nhits;
        A.ops_count[q] = nops;
    }
}

// D table: one lane per pattern, forward over the pattern with the reversed text's O table
template <int LAYOUT>
__global__ void __launch_bounds__(256) approx_dtable_kernel(OccView rov, const u32 *__restrict__ c_dev, u32 len,
                                                            const u8 *__restrict__ pat, const u64 *__restrict__ off,
                                                            u32 fixed_len, u64 npat, u8 *__restrict__ dtab) {
    __shared__ u32 c_sh[256];
    for (u32 k = threadIdx.x; k < 256; k += blockDim.x) c_sh[k] = k < rov.sigma ? c_dev[k] : 0;
    __syncthreads();
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npat) return;
    const u64 begin = off ? off[q] : q * (u64)fixed_len;
    const u32 m = off ? (u32)(off[q + 1] - begin) : fixed_len;
    u32 L = 0, R = len, need = 0;
    for (u32 k = 0; k < m; ++k) {
        const u32 a = pat[begin + k];
        if (a == 0 || a >= rov.sigma) {
            L = 1;
            R = 0;
        } else {
            const u32 ca = c_sh[a];
            const u32 nl = ca + occ_sym<LAYOUT>(rov, a, L), nr = ca + occ_sym<LAYOUT>(rov, a, R);
            L = nl;
            R = nr;
        }
        if (L >= R) {
            ++need;
            L = 0;
            R = len;
        }
        dtab[begin + k] = (u8)(need > 255u ? 255u : need);
    }
}

void approx_dtable(const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u8 *d_dtab,
                   cudaStream_t st) {
    if (!npat) return;
    OccView rov = occ_view(rev);
    const unsigned blocks = div_up_u(npat, 256);
    if (rev.occ_layout == OCC_DNA32)
        approx_dtable_kernel<1><<<blocks, 256, 0, st>>>(rov, rev.c_table.ptr, rev.len, d_pat, d_off, fixed_len, npat, d_dtab);
    else
        approx_dtable_kernel<2><<<blocks, 256, 0, st>>>(rov, rev.c_table.ptr, rev.len, d_pat, d_off, fixed_len, npat, d_dtab);
    KERNEL_CHECK();
}

// exclusive scans of the per-pattern counts (one CTA; the batch is scanned in 1024-wide steps)
__global__ void __launch_bounds__(1024) approx_scan_kernel(const u32 *__restrict__ hit_count,
                                                           const u64 *__restrict__ ops_count, u64 npat,
                                                           u64 *__restrict__ hit_off, u64 *__restrict__ ops_off) {
    __shared__ u64 wsum[32][2];
    __shared__ u64 carry[2];
    if (threadIdx.x == 0) carry[0] = carry[1] = 0;
    __syncthreads();
    for (u64 base = 0; base < npat; base += 1024) {
        const u64 k = base + threadIdx.x;
        const u64 v0 = k < npat ? (u64)hit_count[k] : 0, v1 = k < npat ? ops_count[k] : 0;
        const u64 i0 = warp_inclusive(v0, SumOp()), i1 = warp_inclusive(v1, SumOp());
        if (lane_id() == 31) {
            wsum[threadIdx.x >> 5][0] = i0;
            wsum[threadIdx.x >> 5][1] = i1;
        }
        __syncthreads();
        u64 b0 = 0, b1 = 0;
        for (unsigned w = 0; w < (threadIdx.x >> 5); ++w) {
            b0 += wsum[w][0];
            b1 += wsum[w][1];
        }
        const u64 e0 = carry[0] + b0 + i0 - v0, e1 = carry[1] + b1 + i1 - v1;
        if (k < npat) {
            hit_off[k] = e0;
            ops_off[k] = e1;
        }
        __syncthreads();
        if (threadIdx.x == 1023) {
            carry[0] = e0 + v0;
            carry[1] = e1 + v1;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        hit_off[npat] = carry[0];
        ops_off[npat] = carry[1];
    }
}

static void launch_walk(const DeviceIndex &ix, ApproxArgs &A, bool emit, u64 npat, u32 max_m, cudaStream_t st) {
    // lanes per launch: the frame stacks of one launch stay under ~1 GiB
    const u64 frame_bytes = (u64)A.max_depth * 16;
    u64 chunk = std::max<u64>(1024, ((u64)1 << 30) / frame_bytes);
    chunk = std::min(chunk, npat);
    DevBuf<uint4> stack((size_t)chunk * A.max_depth, st);
    A.stack = stack.ptr;
    for (u64 first = 0; first < npat; first += chunk) {
        A.first = first;
        A.count = std::min(chunk, npat - first);
        const unsigned blocks = div_up_u(A.count * AG, 128);
        if (ix.occ_layout == OCC_DNA32) {
            if (emit) approx_walk_kernel<1, true><<<blocks, 128, 0, st>>>(A);
            else approx_walk_kernel<1, false><<<blocks, 128, 0, st>>>(A);
        } else {
            if (emit) approx_walk_kernel<2, true><<<blocks, 128, 0, st>>>(A);
            else approx_walk_kernel<2, false><<<blocks, 128, 0, st>>>(A);
        }
        KERNEL_CHECK();
    }
    (void)max_m;
}

// Counting pass + scan.  d_hit_off / d_ops_off: npat + 1 entries each.  Returns (hits, ops).
void approx_count(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m,
                  const u8 *d_dtab, int max_edits, u64 *d_hit_off, u64 *d_ops_off, u64 *hits, u64 *ops,
                  cudaStream_t st) {
    *hits = *ops = 0;
    if (!npat) {
        CUDA_CHECK(cudaMemsetAsync(d_hit_off, 0, 8, st));
        CUDA_CHECK(cudaMemsetAsync(d_ops_off, 0, 8, st));
        return;
    }
    DevBuf<u32> hit_count(npat, st);
    DevBuf<u64> ops_count(npat, st);
    ApproxArgs A{};
    A.ov = occ_view(ix);
    A.c_dev = ix.c_table.ptr;
    A.len = ix.len;
    A.sigma = ix.sigma;
    A.pat = d_pat; A.off = d_off; A.fixed_len = fixed_len;
    A.dtab = d_dtab;
    A.max_edits = max_edits;
    A.no_sep = ix.nrec > 0;
    A.max_depth = max_m + (u32)max_edits + 2;
    A.hit_count = hit_count.ptr;
    A.ops_count = ops_count.ptr;
    launch_walk(ix, A, false, npat, max_m, st);
    approx_scan_kernel<<<1, 1024, 0, st>>>(hit_count.ptr, ops_count.ptr, npat, d_hit_off, d_ops_off);
    KERNEL_CHECK();
    u64 h[2] = {0, 0};
    CUDA_CHECK(cudaMemcpyAsync(&h[0], d_hit_off + npat, 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaMemcpyAsync(&h[1], d_ops_off + npat, 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    *hits = h[0];
    *ops = h[1];
}

void approx_emit(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m,
                 const u8 *d_dtab, int max_edits, const u64 *d_hit_off, const u64 *d_ops_off, u32 *d_L, u32 *d_R,
                 u32 *d_mlen, u64 *d_hit_ops_off, char *d_ops, cudaStream_t st) {
    if (!npat) return;
    ApproxArgs A{};
    A.ov = occ_view(ix);
    A.c_dev = ix.c_table.ptr;
    A.len = ix.len;
    A.sigma = ix.sigma;
    A.pat = d_pat; A.off = d_off; A.fixed_len = fixed_len;
    A.dtab = d_dtab;
    A.max_edits = max_edits;
    A.no_sep = ix.nrec > 0;
    A.max_depth = max_m + (u32)max_edits + 2;
    A.hit_off = d_hit_off;
    A.ops_off = d_ops_off;
    A.out_L = d_L; A.out_R = d_R; A.out_mlen = d_mlen;
    A.out_ops_off = d_hit_ops_off;
    A.out_ops = d_ops;
    launch_walk(ix, A, true, npat, max_m, st);
}

}  // namespace b200sa
