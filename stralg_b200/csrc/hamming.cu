// hamming.cu -- batched k-mismatch search on a bidirectional FM index (sm_100a).
//
// The hits of a pattern P[0..m) are the distinct strings Q of length m over the letters that occur in the text with
// Hamming(P, Q) <= k, each as (its SA interval [L, R) on the index of the text, Hamming(P, Q)).
//
// Search scheme (Lam et al. 2009; Kucherov, Salikhov & Tsur 2016): P is split into k + 1 parts P_0 .. P_k, left to
// right, of floor(m / (k + 1)) or one more symbols, the longer parts first.  Search i matches P_i exactly, extends to
// the right through P_{i+1} .. P_k with any mismatches up to k in all, then to the left through P_{i-1} .. P_0 with
// at least one mismatch in each of those parts.  A string Q at distance <= k agrees with P on at least one part; let
// i* be the first: search i* finds Q, a search j < i* needs P_j exact where Q differs, and a search j > i* needs a
// mismatch in P_{i*} where Q has none -- so every hit is found by exactly one search and nothing is deduplicated.
// Search i needs its left parts to be non-empty, so only searches i <= m run when m <= k.
//
// The two indices: F (the text) and B (the reversed text) hold a string as intervals of the same width; a right
// extension is a step on B, a left extension a step on F, and each also moves the start on the other index
// (fm_step.cuh, bidirectional steps).  Search i takes steps s = 0 .. m - 1: steps s < nright = m - start(P_i) are the
// positions start(P_i) + s to the right, the others the positions m - 1 - s to the left.
//
// One thread walks one work unit, a (pattern, search) pair, depth first.  At a node it evaluates the children of all
// letters (DNA layout: from the one or two 32-byte blocks of one step) and prunes a child whose interval is empty or
// whose mismatches plus the left parts still owing one exceed k.  A child that completes the pattern is a hit; a
// child with no mismatch left can only continue by exact steps, run inline without the stack (a chain); the first
// other child is entered, and the node is parked in a stack of 16-byte frames in HBM (frame f of unit t at
// [f * units + t]) only when a later child may still be viable.  The walk runs twice: a counting pass (hits per
// unit), an exclusive scan (scan_u64), and an emitting pass that writes every hit at its final offset with the key
// [pattern | L]; one stable radix sort of the keys (sort_pairs, locate.cu) puts every pattern's hits in ascending L,
// and R and d follow through the permutation.  The edit-distance search (levenshtein.cu) runs the same count pass and
// emitting walk with its sort (pair_count, pair_sorted_hits, below).
#include "walk.cuh"

namespace b200sa {

// frame: x = x, y = y, z = w, w = step | mismatches << 16 | part flag << 20 | next letter << 21
template <int LAYOUT, bool EMIT>
__global__ void __launch_bounds__(256) hamming_walk_kernel(PairArgs A) {
    __shared__ u32 c_sh[256];
    if (LAYOUT != 1) {
        for (u32 j = threadIdx.x; j < 256; j += blockDim.x) c_sh[j] = j < A.fv.sigma ? A.c_dev[j] : 0;
        __syncthreads();
    }
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= A.count) return;
    const u64 u = A.first + t;
    const u32 k = A.k;
    const u64 q = u / (k + 1);
    const u32 i = (u32)(u - q * (k + 1));
    const u64 begin = A.off ? A.off[q] : q * (u64)A.fixed_len;
    const u32 m = A.off ? (u32)(A.off[q + 1] - begin) : A.fixed_len;
    const u8 *p = A.pat + begin;
    const u32 nsym = A.fv.sigma - 1;  // letters 1..nsym
    u64 nh = 0;
    const u64 at = EMIT ? A.unit_off[u] : 0;
    auto hit = [&](u32 L, u32 w, u32 dist) {
        if (EMIT) {
            const u64 h = at + nh;
            A.key[h] = q << 32 | L;
            A.val[h] = (u32)h;
            A.R[h] = L + w;
            A.d[h] = dist;
        }
        ++nh;
    };
    auto index_of = [&](bool right) { return step_index(A.fv, A.bv, right); };
    if (m && i <= m && nsym) {
        const u32 qs = m / (k + 1), r = m % (k + 1);
        const u32 st = part_start(i, qs, r), size_i = part_start(i + 1, qs, r) - st;
        const u32 nright = m - st;
        // (x, y) of a node after step s: the step after it runs on the other index when s + 1 == nright, and after
        // the last step (s + 1 == m) x is the start on F either way
        auto turn = [&](u32 s1, u32 &x, u32 &y) {
            if (s1 == nright) {
                const u32 tmp = x;
                x = y;
                y = tmp;
            }
        };
        // exact steps from step s0 on; one hit at the end when none empties the interval
        auto chain = [&](u32 s0, u32 x, u32 y, u32 w, u32 dist) {
            for (u32 s = s0; s < m; ++s) {
                const bool right = s < nright;
                const u32 a = p[right ? st + s : m - 1 - s];
                if (a == 0 || a > nsym) return;
                const OccView ov = index_of(right);
                u32 nx, nw, ny = 0;
                // (to the left the walk never turns again: y is not needed)
                if (LAYOUT == 1 && !right) {
                    u32 n_blk = 0;
                    const uint2 lr = dna_step<false>(ov, A.c5, a, x, x + w, n_blk);
                    nx = lr.x;
                    nw = lr.y - lr.x;
                } else {
                    bidi_child<LAYOUT>(ov, A.c5, c_sh, a, x, w, y, right, nx, nw, ny);
                }
                if (!nw) return;
                turn(s + 1, nx, ny);
                x = nx;
                y = ny;
                w = nw;
            }
            hit(x, w, dist);
        };

        uint4 *stk = A.stack + t;
        const u64 lanes = A.count;
        // the node: next step s, mismatches e, whether the current left part has one (flag), and its intervals
        u32 s = 0, e = 0, flag = 0, x = 0, y = 0, w = A.len, cursor = 1, depth = 0;
        while (true) {
            if (cursor > nsym) {
                if (depth == 0) break;
                --depth;
                const uint4 f = stk[(u64)depth * lanes];
                x = f.x;
                y = f.y;
                w = f.z;
                s = f.w & 0xffffu;
                e = (f.w >> 16) & 15u;
                flag = (f.w >> 20) & 1u;
                cursor = f.w >> 21;
                continue;
            }
            const bool right = s < nright;
            const u32 pos = right ? st + s : m - 1 - s;
            const u32 pc = p[pos];
            u32 pj = 0;
            bool completes = false;
            if (!right) {
                pj = part_of(pos, qs, r);
                completes = pos == part_start(pj, qs, r);
            }
            // may a child of this step with `cost` (0: the pattern's letter, 1: another) still lead to a hit?  To
            // the right: P_i is exact, then e + the i left parts' mismatches <= k.  To the left: the parts below the
            // current one and the current one (until it has a mismatch) each still owe one; a part that ends
            // without one is dead.
            auto allowed = [&](u32 cost) -> bool {
                if (right) return s < size_i ? cost == 0 : e + cost + i <= k;
                const u32 f = flag | cost;
                return completes ? (f && e + cost + pj <= k) : e + cost + pj + (f ^ 1u) <= k;
            };
            const bool ok_match = allowed(0), ok_miss = allowed(1);
            const OccView ov = index_of(right);
            // a viable child: a hit, a chain, or (true) the child to enter, left in (ex, ey, ew, ee)
            u32 ex = 0, ey = 0, ew = 0, ee = 0;
            auto take = [&](u32 a, u32 cx, u32 cw, u32 cy) -> bool {
                const u32 ce = e + (a != pc ? 1u : 0u);
                turn(s + 1, cx, cy);
                if (s + 1 == m) {
                    hit(cx, cw, ce);
                    return false;
                }
                if (ce == k) {  // (then no part owes a mismatch any more: the rest is exact)
                    chain(s + 1, cx, cy, cw, ce);
                    return false;
                }
                ex = cx;
                ey = cy;
                ew = cw;
                ee = ce;
                return true;
            };
            u32 enter = 0;
            bool more = false;  // a child after the entered one may be viable
            if (LAYOUT == 1) {
                const BiChildren ch = dna_bidi_children(ov, A.c5, x, w, y);
                u32 vmask = 0;
#pragma unroll
                for (u32 a = 1; a <= 4; ++a)
                    if (a >= cursor && a <= nsym && ch.w[a - 1] && (a == pc ? ok_match : ok_miss)) vmask |= 1u << a;
                while (vmask) {
                    const u32 a = (u32)__ffs((int)vmask) - 1u;
                    vmask &= vmask - 1u;
                    if (take(a, pick4(ch.x, a), pick4(ch.w, a), pick4(ch.y, a))) {
                        enter = a;
                        more = vmask != 0;
                        break;
                    }
                }
            } else if (ok_match || ok_miss) {
                u32 run = byte_bidi_run(ov, x, w, y, cursor);
                for (u32 a = cursor; a <= nsym; ++a) {
                    u32 cx, cw, cy;
                    byte_bidi_child(ov, c_sh, a, x, w, run, cx, cw, cy);
                    if (!cw || !(a == pc ? ok_match : ok_miss)) continue;
                    if (take(a, cx, cw, cy)) {
                        enter = a;
                        more = (ok_miss && a < nsym) || (ok_match && pc > a && pc <= nsym);
                        break;
                    }
                }
            }
            if (!enter) {
                cursor = nsym + 1;  // every child taken: back to the parked node
                continue;
            }
            if (more) {
                stk[(u64)depth * lanes] = make_uint4(x, y, w, s | e << 16 | flag << 20 | (enter + 1) << 21);
                ++depth;
            }
            flag = (right || completes) ? 0u : (flag | (enter != pc ? 1u : 0u));
            x = ex;
            y = ey;
            w = ew;
            e = ee;
            ++s;
            cursor = 1;
        }
    }
    if (!EMIT) A.unit_count[u] = nh;
}

// [pattern | L] keys and hit indices sorted: L, and R and d through the permutation
__global__ void __launch_bounds__(256) hamming_take_kernel(const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                           const u32 *__restrict__ R, const u32 *__restrict__ d,
                                                           u64 hits, u32 *__restrict__ out_L, u32 *__restrict__ out_R,
                                                           u32 *__restrict__ out_d) {
    const u64 h = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= hits) return;
    const u32 j = val[h];
    out_L[h] = (u32)key[h];
    out_R[h] = R[j];
    out_d[h] = d[j];
}

// pattern q's hits start where its search 0 does
__global__ void __launch_bounds__(256) hamming_pattern_off_kernel(const u64 *__restrict__ unit_off, u64 npat, u32 k,
                                                                  u64 *__restrict__ pat_off) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q <= npat) pat_off[q] = unit_off[q * (k + 1)];
}

WalkKernels<PairArgs> hamming_walk_kernels = {{hamming_walk_kernel<1, false>, hamming_walk_kernel<1, true>},
                                               {hamming_walk_kernel<2, false>, hamming_walk_kernel<2, true>}};

// ---- the passes both searches on an index pair share (levenshtein.cu runs them too) -----------------------------
static PairArgs pair_args(const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off,
                          u32 fixed_len, u32 k) {
    PairArgs A{};
    A.fv = occ_view(ix);
    A.bv = occ_view(rev);
    for (int j = 0; j < 8; ++j) A.c5.c[j] = ix.c_host[j];
    A.c_dev = ix.c_table.ptr;
    A.len = ix.len;
    A.k = k;
    A.pat = d_pat;
    A.off = d_off;
    A.fixed_len = fixed_len;
    return A;
}

// A k-mismatch walk parks at most one 16-byte frame per step; an edit-distance walk one 20-byte frame per right node
// depth (|Q_R| <= |P_>i| + k) and one per left node depth (|Q_L| <= |P_<i| + k).
static void pair_walk(PairSearch s, const DeviceIndex &ix, PairArgs &A, bool emit, u64 units, u32 max_m,
                      cudaStream_t st) {
    const bool lev = s == PairSearch::LEVENSHTEIN;
    const u64 frames = lev ? (u64)max_m + 2 * A.k + 2 : std::max<u32>(max_m, 1);
    const u64 chunk = walk_units_per_launch(units, frames * (lev ? 20 : 16));
    DevBuf<uint4> stack((size_t)(chunk * frames), st);
    DevBuf<u32> stack_w(lev ? (size_t)(chunk * frames) : 0, st);
    A.stack = stack.ptr;
    A.stack_w = stack_w.ptr;
    run_walk(lev ? levenshtein_walk_kernels : hamming_walk_kernels, ix, emit, A, units, chunk, 1, 256, st);
}

u64 pair_count(PairSearch s, const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off,
               u32 fixed_len, u64 npat, u32 max_m, u32 k, u64 *d_unit_off, cudaStream_t st) {
    const u64 units = npat * (k + 1);
    if (!units) {
        CUDA_CHECK(cudaMemsetAsync(d_unit_off, 0, 8, st));
        return 0;
    }
    PairArgs A = pair_args(ix, rev, d_pat, d_off, fixed_len, k);
    A.unit_count = d_unit_off;
    pair_walk(s, ix, A, false, units, max_m, st);
    scan_u64(d_unit_off, units, st);
    u64 hits = 0;
    read_back(&hits, d_unit_off + units, 8, st);
    return hits;
}

PairHits pair_sorted_hits(PairSearch s, const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat,
                          const u64 *d_off, u32 fixed_len, u64 npat, u32 max_m, u32 k, const u64 *d_unit_off, u64 hits,
                          int key_bits, cudaStream_t st) {
    PairHits H;
    H.kA.alloc(hits, st);
    H.kB.alloc(hits, st);
    H.vA.alloc(hits, st);
    H.vB.alloc(hits, st);
    H.R.alloc(hits, st);
    H.d.alloc(hits, st);
    PairArgs A = pair_args(ix, rev, d_pat, d_off, fixed_len, k);
    A.unit_off = d_unit_off;
    A.key = H.kA.ptr;
    A.val = H.vA.ptr;
    A.R = H.R.ptr;
    A.d = H.d.ptr;
    pair_walk(s, ix, A, true, npat * (k + 1), max_m, st);
    int qbits = 0;
    while ((1ull << qbits) < npat) ++qbits;
    u64 *kb[2] = {H.kA.ptr, H.kB.ptr};
    u32 *vb[2] = {H.vA.ptr, H.vB.ptr};
    sort_pairs(kb, vb, (u32)hits, key_bits + qbits, H.key, H.val, st);
    return H;
}

void hamming_emit(const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off, u32 fixed_len,
                  u64 npat, u32 max_m, u32 k, const u64 *d_unit_off, u64 hits, u64 *d_pat_off, u32 *d_L, u32 *d_R,
                  u32 *d_d, cudaStream_t st) {
    if (!npat) return;
    hamming_pattern_off_kernel<<<div_up_u(npat + 1, 256), 256, 0, st>>>(d_unit_off, npat, k, d_pat_off);
    KERNEL_CHECK();
    if (!hits) return;
    if (hits > 0xFFFFFFFFull || npat > 0xFFFFFFFFull)
        throw std::runtime_error("hamming_emit: more than 2^32 - 1 hits or patterns in one piece");
    const PairHits H = pair_sorted_hits(PairSearch::HAMMING, ix, rev, d_pat, d_off, fixed_len, npat, max_m, k,
                                        d_unit_off, hits, 32, st);
    hamming_take_kernel<<<div_up_u(hits, 256), 256, 0, st>>>(H.key, H.val, H.R.ptr, H.d.ptr, hits, d_L, d_R, d_d);
    KERNEL_CHECK();
}

}  // namespace b200sa
