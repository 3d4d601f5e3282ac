// levenshtein.cu -- batched edit-distance search on a bidirectional FM index (sm_100a).
//
// The hits of a pattern P[0..m) are the distinct non-empty strings Q over the letters that occur in the text with
// ED(P, Q) <= k (unit-cost Levenshtein distance), each as (its SA interval [L, R) on the index of the text, |Q|,
// ED(P, Q)).
//
// Search scheme: P is split into k + 1 parts P_0 .. P_k as in the k-mismatch search (part_start, fm_step.cuh; parts
// are empty when m <= k).  Fix an optimal alignment of P with Q and charge each substitution or deleted pattern symbol
// to the part of its pattern symbol, each inserted text symbol to the part of the next pattern symbol (the last part
// when none follows).  Some part P_i has no charge, so Q = Q_L P_i Q_R with ED(P, Q) = ED(P_<i, Q_L) + ED(P_>i, Q_R).
// Search i matches P_i exactly (right steps), then extends to the right letter by letter keeping the DP column of
// P_>i against Q_R; at every node whose column reaches the end of P_>i with eR <= k it starts a left walk that keeps
// the DP column of reverse(P_<i) against reverse(Q_L) within the budget k - eR and reports every node whose column
// reaches the end of P_<i.  The nodes are strings, not edit paths, but a string can be found by several searches
// (and by one search where P_i occurs twice in it), each time with a distance >= ED(P, Q) and once (by the search of
// an uncharged part) with ED(P, Q) itself: the raw hits are sorted by [pattern | L | |Q| - (m - k)] and each run
// of equal keys becomes one hit with the smallest distance of the run.
//
// A DP column is kept as its band of 2k + 1 cells around the diagonal -- after t text symbols, cell b holds the
// distance to the pattern prefix of t + b - k symbols -- saturated at k + 1, 3 bits a cell: 27 bits at k = 4.
//
// One thread walks one (pattern, search) unit depth first, as in hamming.cu: a right step is a step on B and a left
// step a step on F (fm_step.cuh, bidirectional steps); at the turn x and y swap, and the left walk keeps no y.  A node
// is parked in a stack of 20-byte frames in HBM (frame f of unit t at [f * units + t]) only when a later child may
// still be viable.  Passes: a counting walk (raw hits per unit), scan_u64, an emitting walk that writes each raw hit
// at its final offset, one stable radix sort of the keys (sort_pairs) -- these as in hamming.cu (pair_count,
// pair_sorted_hits) -- a head flag per key run and its scan, and one pass that writes each run's hit with its minimum
// distance at its merged offset; per-pattern offsets come from a binary search over the merged hits' patterns.
#include "walk.cuh"

namespace b200sa {

__device__ __forceinline__ u32 band_cell(u32 band, u32 b) { return (band >> (3 * b)) & 7u; }

// the column after no text symbol: cell b is the prefix of b - k symbols of a pattern string of n symbols
__device__ __forceinline__ u32 band_init(u32 n, u32 k) {
    u32 band = 0;
#pragma unroll
    for (u32 b = 0; b < 9; ++b)
        if (b <= 2 * k) {
            const u32 v = (b < k || b - k > n) ? k + 1 : min(b - k, k + 1);
            band |= v << (3 * b);
        }
    return band;
}

// the distance to the whole pattern string (n symbols) after t text symbols, k + 1 when outside the band
__device__ __forceinline__ u32 band_end(u32 band, u32 n, u32 t, u32 k) {
    const u32 b = n + k - t;  // (wraps above 2k when t > n + k)
    return b <= 2 * k ? band_cell(band, b) : k + 1;
}

// The column after text symbol c (a letter) from the column after t symbols.  sy[b] is the pattern string's symbol
// at t + b - k (0 where there is none): the one the diagonal move into new cell b compares with c.  mn gets the
// smallest cell of the new column.
__device__ __forceinline__ u32 band_step(u32 band, const u32 (&sy)[9], u32 c, u32 t, u32 n, u32 k, u32 &mn) {
    const u32 sat = k + 1;
    u32 out = 0, prev = sat, lo = sat;
#pragma unroll
    for (u32 b = 0; b < 9; ++b)
        if (b <= 2 * k) {
            const u32 j = t + 1 + b - k;  // pattern prefix of the new cell (wraps when negative)
            u32 v = sat;
            if (t + 1 + b >= k && j <= n) {
                const u32 up = b < 2 * k ? band_cell(band, b + 1) + 1 : sat;  // c against nothing
                const u32 diag = j >= 1 ? band_cell(band, b) + (sy[b] != c ? 1u : 0u) : sat;
                v = min(min(up, diag), min(prev + 1, sat));  // prev + 1: a pattern symbol against nothing
            }
            out |= v << (3 * b);
            prev = v;
            lo = min(lo, v);
        }
    mn = lo;
    return out;
}

// frame: (x, y or |Q_R|, w, band) in stack, t | cursor << 17 | left << 26 | eR << 27 in stack_w; raw hit key:
// pattern << 36 | L << 4 | (|Q| + k - m)
template <int LAYOUT, bool EMIT>
__global__ void __launch_bounds__(256) levenshtein_walk_kernel(PairArgs A) {
    __shared__ u32 c_sh[256];
    if (LAYOUT != 1) {
        for (u32 j = threadIdx.x; j < 256; j += blockDim.x) c_sh[j] = j < A.fv.sigma ? A.c_dev[j] : 0;
        __syncthreads();
    }
    const u64 t0 = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t0 >= A.count) return;
    const u64 u = A.first + t0;
    const u32 k = A.k;
    const u64 q = u / (k + 1);
    const u32 i = (u32)(u - q * (k + 1));
    const u64 begin = A.off ? A.off[q] : q * (u64)A.fixed_len;
    const u32 m = A.off ? (u32)(A.off[q + 1] - begin) : A.fixed_len;
    const u8 *p = A.pat + begin;
    const u32 nsym = A.fv.sigma - 1;  // letters 1..nsym
    u64 nh = 0;
    const u64 at = EMIT ? A.unit_off[u] : 0;
    auto hit = [&](u32 L, u32 w, u32 qlen, u32 dist) {
        if (EMIT) {
            const u64 h = at + nh;
            A.key[h] = q << 36 | (u64)L << 4 | (qlen + k - m);
            A.val[h] = (u32)h;
            A.R[h] = L + w;
            A.d[h] = dist;
        }
        ++nh;
    };
    if (m && nsym) {
        const u32 qs = m / (k + 1), r = m % (k + 1);
        const u32 st = part_start(i, qs, r), en = part_start(i + 1, qs, r);
        const u32 size_i = en - st, nR = m - en, nL = st;
        // P_i exactly, by right steps (on B) from the root
        u32 x = 0, y = 0, w = A.len;
        const OccView bv = step_index(A.fv, A.bv, true);
        for (u32 s = 0; s < size_i && w; ++s) {
            const u32 a = p[st + s];
            if (a == 0 || a > nsym) {
                w = 0;
                break;
            }
            u32 cx, cw, cy;
            bidi_child<LAYOUT>(bv, A.c5, c_sh, a, x, w, y, true, cx, cw, cy);
            x = cx;
            w = cw;
            y = cy;
        }
        uint4 *stk = A.stack + t0;
        u32 *stkw = A.stack_w + t0;
        const u64 lanes = A.count;
        // the node: its side (left walk or not), text symbols t on that side, DP band, intervals (to the left, y is
        // |Q_R|), eR (left walk: the distance of P_>i to Q_R) and the next child (cursor; 0 on the right: the left
        // walk of the node, still to start)
        u32 left = 0, t = 0, band = band_init(nR, k), eR = 0, cursor = w ? 0 : nsym + 1, depth = 0;
        while (true) {
            if (cursor > nsym) {
                if (depth == 0) break;
                --depth;
                const uint4 f = stk[(u64)depth * lanes];
                const u32 fw = stkw[(u64)depth * lanes];
                x = f.x;
                y = f.y;
                w = f.z;
                band = f.w;
                t = fw & 0x1ffffu;
                cursor = (fw >> 17) & 0x1ffu;
                left = (fw >> 26) & 1u;
                eR = fw >> 27;
                continue;
            }
            const u32 n = left ? nL : nR;
            if (!left && cursor == 0) {
                cursor = 1;
                const u32 e = band_end(band, nR, t, k);
                if (e <= k) {
                    if (t < nR + k) {  // the node's own children may follow
                        stk[(u64)depth * lanes] = make_uint4(x, y, w, band);
                        stkw[(u64)depth * lanes] = t | 1u << 17;
                        ++depth;
                    }
                    // the left walk starts on F at X = P_i Q_R
                    x = y;
                    y = t;
                    eR = e;
                    left = 1;
                    t = 0;
                    band = band_init(nL, k);
                    if (size_i + y && nL <= k - eR) hit(x, w, size_i + y, eR + nL);
                    continue;
                }
            }
            const u32 budget = k - eR;  // (eR = 0 on the right)
            u32 sy[9];
#pragma unroll
            for (u32 b = 0; b < 9; ++b) {
                const u32 j = t + b - k;  // (wraps when negative)
                sy[b] = (b <= 2 * k && t + b >= k && j < n) ? p[left ? nL - 1 - j : en + j] : 0u;
            }
            // the child to enter: (ex, ew, ey) and its band
            u32 ex = 0, ew = 0, ey = 0, eb = 0, enter = 0;
            bool more = false;  // a later child may be viable
            if (LAYOUT == 1) {
                const BiChildren ch = dna_bidi_children(step_index(A.fv, A.bv, !left), A.c5, x, w, y);
                u32 vmask = 0;
#pragma unroll
                for (u32 a = 1; a <= 4; ++a) {
                    u32 mn;
                    band_step(band, sy, a, t, n, k, mn);
                    if (a >= cursor && a <= nsym && ch.w[a - 1] && mn <= budget) vmask |= 1u << a;
                }
                if (vmask) {
                    enter = (u32)__ffs((int)vmask) - 1u;
                    more = (vmask & (vmask - 1u)) != 0;
                    ex = pick4(ch.x, enter);
                    ew = pick4(ch.w, enter);
                    ey = pick4(ch.y, enter);
                }
            } else {
                // a letter that is none of sy[] gives the band of c = 0; only when that band is viable can every
                // letter be
                u32 mn0;
                band_step(band, sy, 0, t, n, k, mn0);
                const OccView ov = step_index(A.fv, A.bv, !left);
                u32 run = byte_bidi_run(ov, x, w, y, left ? 1u : cursor);
                for (u32 a = cursor; a <= nsym; ++a) {
                    u32 cx, cw, cy, mn;
                    byte_bidi_child(ov, c_sh, a, x, w, run, cx, cw, cy);
                    if (!cw) continue;
                    band_step(band, sy, a, t, n, k, mn);
                    if (mn > budget) continue;
                    enter = a;
                    ex = cx;
                    ew = cw;
                    ey = cy;
                    more = mn0 <= budget && a < nsym;
#pragma unroll
                    for (u32 b = 0; b < 9; ++b) more = more || (sy[b] > a && sy[b] <= nsym);
                    break;
                }
            }
            if (!enter) {
                cursor = nsym + 1;  // every child taken: back to the parked node
                continue;
            }
            u32 mn;
            eb = band_step(band, sy, enter, t, n, k, mn);
            if (more) {
                stk[(u64)depth * lanes] = make_uint4(x, y, w, band);
                stkw[(u64)depth * lanes] = t | (enter + 1) << 17 | left << 26 | eR << 27;
                ++depth;
            }
            ++t;
            band = eb;
            w = ew;
            if (left) {
                x = ex;  // (y keeps |Q_R|)
                const u32 e = band_end(band, nL, t, k);
                if (e <= budget) hit(x, w, size_i + y + t, eR + e);
                cursor = 1;
            } else {
                x = ex;
                y = ey;
                cursor = 0;
            }
        }
    }
    if (!EMIT) A.unit_count[u] = nh;
}

// flag[h] = 1 where a run of equal keys starts in the sorted raw hits
__global__ void __launch_bounds__(256) levenshtein_head_kernel(const u64 *__restrict__ key, u64 hits,
                                                               u64 *__restrict__ flag) {
    const u64 h = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (h < hits) flag[h] = (h == 0 || key[h] != key[h - 1]) ? 1u : 0u;
}

// one hit per run, at the run's merged offset (the scan of the flags): L and |Q| from the key, R from the run's first
// raw hit (every raw hit of a run has the same interval), d the minimum over the run
__global__ void __launch_bounds__(256) levenshtein_merge_kernel(const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                                const u32 *__restrict__ R, const u32 *__restrict__ d,
                                                                u64 hits, const u64 *__restrict__ merged_at,
                                                                const u64 *__restrict__ off, u32 fixed_len, u32 k,
                                                                u32 *__restrict__ out_q, u32 *__restrict__ out_L,
                                                                u32 *__restrict__ out_R, u32 *__restrict__ out_len,
                                                                u32 *__restrict__ out_d) {
    const u64 h = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= hits) return;
    const u64 kh = key[h];
    if (h && key[h - 1] == kh) return;
    u32 dm = d[val[h]];
    for (u64 g = h + 1; g < hits && key[g] == kh; ++g) dm = min(dm, d[val[g]]);
    const u64 o = merged_at[h];
    const u64 q = kh >> 36;
    const u32 m = off ? (u32)(off[q + 1] - off[q]) : fixed_len;
    out_q[o] = (u32)q;
    out_L[o] = (u32)(kh >> 4);
    out_R[o] = R[val[h]];
    out_len[o] = (u32)(kh & 15u) + m - k;
    out_d[o] = dm;
}

// pat_off[q] = the merged hits of the patterns before q (out_q is ascending)
__global__ void __launch_bounds__(256) levenshtein_pattern_off_kernel(const u32 *__restrict__ hit_q, u64 merged,
                                                                      u64 npat, u64 *__restrict__ pat_off) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q > npat) return;
    u64 lo = 0, hi = merged;
    while (lo < hi) {
        const u64 mid = (lo + hi) / 2;
        if (hit_q[mid] < q) lo = mid + 1;
        else hi = mid;
    }
    pat_off[q] = lo;
}

WalkKernels<PairArgs> levenshtein_walk_kernels = {
    {levenshtein_walk_kernel<1, false>, levenshtein_walk_kernel<1, true>},
    {levenshtein_walk_kernel<2, false>, levenshtein_walk_kernel<2, true>}};

u64 levenshtein_emit(const DeviceIndex &ix, const DeviceIndex &rev, const u8 *d_pat, const u64 *d_off, u32 fixed_len,
                     u64 npat, u32 max_m, u32 k, const u64 *d_unit_off, u64 raw_hits, u64 *d_pat_off, u32 *d_L,
                     u32 *d_R, u32 *d_len, u32 *d_d, cudaStream_t st) {
    if (!npat) return 0;
    u64 merged = 0;
    if (raw_hits) {
        if (raw_hits > 0xFFFFFFFFull || npat > ((u64)1 << 28))
            throw std::runtime_error("levenshtein_emit: more than 2^32 - 1 raw hits or 2^28 patterns in one piece");
        const u64 hits = raw_hits;
        DevBuf<u64> flag(hits + 1, st);
        DevBuf<u32> hq(hits, st);
        const PairHits H = pair_sorted_hits(PairSearch::LEVENSHTEIN, ix, rev, d_pat, d_off, fixed_len, npat, max_m, k,
                                            d_unit_off, hits, 36, st);
        levenshtein_head_kernel<<<div_up_u(hits, 256), 256, 0, st>>>(H.key, hits, flag.ptr);
        KERNEL_CHECK();
        scan_u64(flag.ptr, hits, st);
        levenshtein_merge_kernel<<<div_up_u(hits, 256), 256, 0, st>>>(H.key, H.val, H.R.ptr, H.d.ptr, hits, flag.ptr,
                                                                       d_off, fixed_len, k, hq.ptr, d_L, d_R, d_len, d_d);
        KERNEL_CHECK();
        read_back(&merged, flag.ptr + hits, 8, st);
        levenshtein_pattern_off_kernel<<<div_up_u(npat + 1, 256), 256, 0, st>>>(hq.ptr, merged, npat, d_pat_off);
        KERNEL_CHECK();
    } else {
        CUDA_CHECK(cudaMemsetAsync(d_pat_off, 0, (npat + 1) * 8, st));
    }
    return merged;
}

}  // namespace b200sa
