// fm_search.cu -- batched FM-index backward exact search and locate (sm_100a).
//
// One lane per pattern runs the recurrence of stralg/bwt.c:164-199:
//     L = 0, R = len;  a pattern longer than len gives (L, R) = (1, 0);
//     for i = m-1 .. 0 while L < R:  L = C(a) + O(a, L),  R = C(a) + O(a, R)
// and locate expands [L, R) into SA[L..R) in suffix-array order (bwt.c:201-217).
// O(a, i) is one 32-byte block fetch + popcount (occ.cuh).  The two fetches of a step are
// independent, so every lane keeps two sector loads in flight; occupancy hides the rest.
// A pattern symbol outside 1..sigma-1 (the reference asserts, bwt.c:189-190) yields the empty
// interval (1, 0).  An empty pattern yields (0, len) (the reference underflows, bwt.c:185).
#include "engine.h"
#include "fm_step.cuh"
#include "scan.cuh"

#include <algorithm>
#include <cstdlib>

namespace b200sa {

// Any alphabet (byte-wide O blocks).  SC: once a single candidate row is left, the remaining symbols are compared
// with the packed text at SA[L] instead of one O lookup each (the recurrence would walk ISA[s-1], ISA[s-2], ... as
// long as the symbols agree); on a difference the failing step is replayed with the O table so that (L, R) is the
// pair the reference's loop ends with (bwt.c:186-198).
template <int LAYOUT, bool SC = false, bool AL = false>
__global__ void __launch_bounds__(256) fm_search_kernel(OccView ov, CTable5 c5, const u32 *__restrict__ c_dev,
                                                        u32 len, const u8 *__restrict__ pat,
                                                        const u64 *__restrict__ off, u32 fixed_len, u64 npat,
                                                        u32 *__restrict__ outL, u32 *__restrict__ outR,
                                                        TextCmp tc = TextCmp{nullptr, nullptr, nullptr}, int bits = 0,
                                                        KTable kt = KTable{nullptr, 0, 0}) {
    __shared__ u32 c_sh[256];
    if (LAYOUT != 1) {
        for (u32 i = threadIdx.x; i < 256; i += blockDim.x) c_sh[i] = i < ov.sigma ? c_dev[i] : 0;
        __syncthreads();
    }
    u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npat) return;
    u64 begin = off ? off[q] : q * (u64)fixed_len;
    u64 m = off ? off[q + 1] - begin : (u64)fixed_len;
    // AL: the pattern buffer is 8-byte aligned and readable up to the next 8-byte boundary (as for the DNA path): symbols
    // come from an aligned word fetched once per eight of them instead of a byte load each -- the lanes of a warp read
    // different patterns, so byte loads cost a sector apiece
    u64 pword = 0, pword_addr = ~0ull;
    auto P = [&](int64_t idx) -> u32 {
        const u64 addr = begin + (u64)idx;
        if (AL) {
            if ((addr & ~7ull) != pword_addr) {
                pword_addr = addr & ~7ull;
                pword = *(const u64 *)(pat + pword_addr);
            }
            return (u32)(pword >> (8 * (addr & 7))) & 0xffu;
        }
        return pat[addr];
    };
    u32 L = 0, R = len;
    if (m > (u64)len) {
        L = 1;
        R = 0;
    }
    int64_t i = (int64_t)m - 1;
    if (LAYOUT == 2 && kt.tab && m >= (u64)kt.k && L < R) {
        // the last k symbols select the interval the first k steps would reach (an entry with L >= R is the pair at
        // the step that emptied the interval); a byte outside 1..nsym takes the stepwise path
        u32 x;
        if (seed_key(P, i, kt, x)) {
            const uint2 lr = kt.tab[x];
            L = lr.x;
            R = lr.y;
            i -= kt.k;
        }
    }
    for (; i >= 0 && L < R && !(SC && R - L == 1); --i) {
        u32 a = P(i);
        if (a == 0 || a >= ov.sigma) {
            L = 1;
            R = 0;
            break;
        }
        u32 oL, oR, ca;
        if (LAYOUT == 1) {
            oL = occ_dna(ov, a, L);
            oR = occ_dna(ov, a, R);
            ca = c5.c[a];
        } else {
            oL = occ_byte(ov, a, L);
            oR = occ_byte(ov, a, R);
            ca = c_sh[a];
        }
        L = ca + oL;
        R = ca + oR;
    }
    if (SC && LAYOUT == 2 && i >= 0 && R - L == 1) {
        const u32 s = tc.sa[L];
        const u64 rem = (u64)i + 1;
        u32 a;
        const u64 k = text_agree(P, i, s, tc.packed, bits, a);
        if (k == rem) {
            L = tc.isa[s - (u32)rem];
            R = L + 1;
        } else if (a == 0 || a >= ov.sigma) {
            L = 1;
            R = 0;
        } else {
            // the step that fails: BWT[Lk] != a, so both ranks coincide and the interval is empty
            const u32 Lk = k ? tc.isa[s - (u32)k] : L;
            L = c_sh[a] + occ_byte(ov, a, Lk);
            R = c_sh[a] + occ_byte(ov, a, Lk + 1);
        }
    }
    outL[q] = L;
    outR[q] = R;
}

// ---------------------------------------------------------------------------------------------
// DNA32 fast path.  Per backward step a lane issues ONE 256-bit load per distinct block (dna_step),
// and pattern symbols come from an aligned 8-byte word fetched once per 8 steps.
// Requires the pattern buffer to be 8-byte aligned and readable up to the next 8-byte boundary
// (true for cudaMalloc / torch allocations; the host entry point pads its staging buffer).
// ---------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) ktable_build_kernel(OccView ov, CTable5 c5, u32 len, int k, u64 entries,
                                                           uint2 *__restrict__ tab) {
    const u64 x64 = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x64 >= entries) return;
    const u32 x = (u32)x64;  // (k <= 16: a k-mer is at most 32 bits)
    u32 L = 0, R = len;
    for (int j = 0; j < k && L < R; ++j) {
        const u32 a = ((x >> (2 * (k - 1 - j))) & 3u) + 1u;
        if (a >= ov.sigma) {  // a letter the text does not have (the reference asserts, bwt.c:189-190)
            L = 1;
            R = 0;
            break;
        }
        const u32 oL = occ_dna(ov, a, L), oR = occ_dna(ov, a, R);
        L = c5.c[a] + oL;
        R = c5.c[a] + oR;
    }
    tab[x] = make_uint2(L, R);
}

// STATS: count the memory operations of the batch (b200sa_search_traffic, a measurement aid):
// stats[0] 32-byte O-block loads, [1] 8-byte pattern words, [2] 8-byte text words, [3] 4-byte SA/ISA loads.
// one pattern: pat[begin .. begin + m), readable in aligned 8-byte words; (L, R) = the interval of bwt.c:171-198
template <bool SC, bool STATS>
__device__ __forceinline__ void fm_search_dna_one(const OccView &ov, const CTable5 &c5, const TextCmp &tc, const KTable &kt,
                                                  u32 len, const u8 *__restrict__ pat, u64 begin, u64 m, u32 &Lout, u32 &Rout,
                                                  u32 &n_blk, u32 &n_pw, u32 &n_tw, u32 &n_sa) {
    u32 L = 0, R = len;
    if (m > (u64)len) {
        L = 1;
        R = 0;
    }
    u64 word = 0;
    u64 word_addr = ~0ull;
    int64_t i = (int64_t)m - 1;
    if (kt.tab && m >= (u64)kt.k && L < R) {
        // the last k symbols select the interval the first k steps would reach
        u32 x;
        if (dna_seed_key<STATS>(pat, begin, i, kt.k, word, word_addr, n_pw, x)) {
            // (a byte outside 1..4 takes the stepwise path: it answers (1, 0) where it is reached)
            const uint2 lr = kt.tab[x];
            if (STATS) n_sa += 2;  // one 8-byte table entry
            L = lr.x;
            R = lr.y;
            i -= kt.k;
        }
    }
    // O steps until the pattern is used up, the interval is empty, or (SC) a single candidate is left:
    // the lanes of a warp reach that point after different numbers of steps, and run the comparison
    // below together, once
    for (; i >= 0 && L < R && !(SC && R - L == 1); --i) {
        const u32 a = pattern_byte<STATS>(pat, begin + (u64)i, word, word_addr, n_pw);
        if (a - 1u > 3u || a >= ov.sigma) {
            L = 1;
            R = 0;
            break;
        }
        const uint2 lr = dna_step<STATS>(ov, c5, a, L, R, n_blk);
        L = lr.x;
        R = lr.y;
    }
    if (SC && i >= 0 && R - L == 1) {
        const u32 s = tc.sa[L];
        if (STATS) ++n_sa;
        const u64 rem = (u64)i + 1;
        u32 a;
        const u64 k = dna_text_agree<STATS>(pat, begin, i, s, tc.packed, word, word_addr, a, n_pw, n_tw);
        if (k == rem) {
            L = tc.isa[s - (u32)rem];
            R = L + 1;
            if (STATS) ++n_sa;
        } else if (a - 1u > 3u || a >= ov.sigma) {
            L = 1;
            R = 0;
        } else {
            // the step that fails: BWT[Lk] != a, so both ranks coincide and the interval is empty
            const u32 Lk = k ? tc.isa[s - (u32)k] : L;
            BlockRegs kb = load_dna_block(ov.blocks, Lk >> 6);
            BlockRegs kb2 = kb;
            if (((Lk + 1) >> 6) != (Lk >> 6)) kb2 = load_dna_block(ov.blocks, (Lk + 1) >> 6);
            if (STATS) {
                n_sa += k ? 1u : 0u;
                n_blk += 1u + ((((Lk + 1) >> 6) != (Lk >> 6)) ? 1u : 0u);
            }
            L = c5.c[a] + rank_in_block(kb, a, Lk, ov.primary);
            R = c5.c[a] + rank_in_block(kb2, a, Lk + 1, ov.primary);
        }
    }
    Lout = L;
    Rout = R;
}

template <bool SC, bool STATS>
__global__ void __launch_bounds__(256) fm_search_dna_kernel(OccView ov, CTable5 c5, TextCmp tc, KTable kt, u32 len,
                                                            const u8 *__restrict__ pat,
                                                            const u64 *__restrict__ off, u32 fixed_len, u64 npat,
                                                            u32 *__restrict__ outL, u32 *__restrict__ outR,
                                                            unsigned long long *__restrict__ stats) {
    u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npat) return;
    u32 n_blk = 0, n_pw = 0, n_tw = 0, n_sa = 0;
    u64 begin = off ? off[q] : q * (u64)fixed_len;
    u64 m = off ? off[q + 1] - begin : (u64)fixed_len;
    u32 L, R;
    fm_search_dna_one<SC, STATS>(ov, c5, tc, kt, len, pat, begin, m, L, R, n_blk, n_pw, n_tw, n_sa);
    outL[q] = L;
    outR[q] = R;
    if (STATS) {
        atomicAdd(&stats[0], (unsigned long long)n_blk);
        atomicAdd(&stats[1], (unsigned long long)n_pw);
        atomicAdd(&stats[2], (unsigned long long)n_tw);
        atomicAdd(&stats[3], (unsigned long long)n_sa);
    }
}

// ---------------------------------------------------------------------------------------------
// One pattern at a time (the drop-in's init_bwt_exact_match_iter): a one-warp kernel that stays resident
// while requests keep coming.  The host writes a request into a slot of mapped pinned memory -- 32 words
// of 8 bytes, each [tag : 16 | 6 bytes of payload], word 0 = [tag | length | -], so that one coalesced
// read of the slot tells the warp whether a complete request with the expected tag stands there -- the
// warp unpacks the pattern into shared memory, lane 0 runs the search of the batch kernel, and (L, R) go
// back as two tagged words the host spins on.  No launch, no stream synchronisation per pattern; the
// kernel leaves after `idle_limit` polls without a request (or when told to), so a device-wide
// synchronisation elsewhere in the process waits a few milliseconds at most.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 ld_sys_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_sys_u64(u64 *p, u64 v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <bool SC>
__global__ void __launch_bounds__(32) fm_mailbox_server_kernel(OccView ov, CTable5 c5, TextCmp tc, KTable kt, u32 len, u64 *slot,
                                                               u32 tag, u32 idle_limit) {
    __shared__ __align__(16) u8 spat[32 * 6 + 32];
    const u32 lane = threadIdx.x;
    u64 *req = slot, *resp = slot + 32, *ctl = slot + 40;  // ctl[0]: alive (set by the host, cleared here), ctl[1]: quit
    u32 idle = 0;
    for (;;) {
        const u32 expect = (tag + 1u) & 0xffffu;
        // the whole slot in one coalesced, uncached read (ld.cv: "fetch again"; a system-scope load per lane would be
        // 32 separate trips to host memory)
        u64 w;
        asm volatile("ld.global.cv.u64 %0, [%1];" : "=l"(w) : "l"(req + lane) : "memory");
        const u64 w0 = __shfl_sync(0xffffffffu, w, 0);
        if ((u32)(w0 >> 48) != expect) {
            ++idle;
            bool quit = idle > idle_limit;
            if ((idle & 15u) == 0u) quit = quit || __shfl_sync(0xffffffffu, lane == 0 ? ld_sys_u64(ctl + 1) : 0ull, 0) != 0ull;
            if (quit) break;
            continue;
        }
        const u32 m = (u32)(w0 >> 32) & 0xffffu;
        const u32 nw = 1u + (m + 5u) / 6u;
        // (a word that still carries an older tag: the request is being written, look again)
        if (!__all_sync(0xffffffffu, lane >= nw || (u32)(w >> 48) == expect)) continue;
        if (lane >= 1u && lane < nw) {
#pragma unroll
            for (int b = 0; b < 6; ++b) spat[(lane - 1u) * 6u + (u32)b] = (u8)(w >> (8 * b));
        }
        __syncwarp();
        if (lane < 16u) spat[m + lane] = 0;  // the search reads whole aligned words
        __syncwarp();
        if (lane == 0) {
            u32 L, R, c0 = 0, c1 = 0, c2 = 0, c3 = 0;
            u64 t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            fm_search_dna_one<SC, false>(ov, c5, tc, kt, len, spat, 0, (u64)m, L, R, c0, c1, c2, c3);
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            st_sys_u64(resp + 2, t1 - t0);  // (nanoseconds inside the search: B200SA_MAIL_DEBUG)
            st_sys_u64(resp, (u64)L | ((u64)expect << 48));
            st_sys_u64(resp + 1, (u64)R | ((u64)expect << 48));
            __threadfence_system();
        }
        tag = expect;
        idle = 0;
    }
    if (lane == 0) {
        __threadfence_system();
        st_sys_u64(ctl, 0ull);
    }
}

void fm_mailbox_server_launch(const DeviceIndex &ix, void *d_slot, u32 tag, u32 idle_limit, cudaStream_t st) {
    OccView ov = occ_view(ix);
    CTable5 c5;
    for (int i = 0; i < 8; ++i) c5.c[i] = ix.c_host[i];
    TextCmp tc{ix.sa.ptr, ix.isa.ptr, ix.text_packed.ptr};
    KTable kt{ix.ktable.ptr, ix.ktable_k};
    const bool sc = tc.sa && tc.isa && tc.packed && ix.pk.bits == 2;
    if (sc) fm_mailbox_server_kernel<true><<<1, 32, 0, st>>>(ov, c5, tc, kt, ix.len, (u64 *)d_slot, tag, idle_limit);
    else fm_mailbox_server_kernel<false><<<1, 32, 0, st>>>(ov, c5, tc, kt, ix.len, (u64 *)d_slot, tag, idle_limit);
    KERNEL_CHECK();
}

// ---------------------------------------------------------------------------------------------
// Packed reads (VERDICT r1 item 3).  A read of m bases is m 2-bit symbols (code - 1), four to a
// byte, the FIRST base in the two most significant bits of its byte (the order of the packed text,
// sa_build.cu pack_kernel<2>, so that pattern and text fields compare with one XOR); read q starts
// at byte q * stride.  A quarter of the bytes over PCIe and through the kernel, and the text
// comparison of the unique-interval shortcut takes up to 32 symbols per step.  Same recurrence,
// same (L, R) -- including the interval at the step that emptied it -- as fm_search_dna_kernel.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 bswap64(u64 v) {
    return ((u64)__byte_perm((u32)v, 0, 0x0123) << 32) | (u64)__byte_perm((u32)(v >> 32), 0, 0x0123);
}

// the `nbits` (2..64, even) bits of a big-endian bit stream that END just before bit `endbit`
// (endbit >= nbits), right-aligned.  SWAP: the stream is stored as bytes (reads), else as u64 words (text)
template <bool SWAP>
__device__ __forceinline__ u64 bits_ending(const u64 *__restrict__ words, u64 endbit, u32 nbits, u64 &c_idx, u64 &c_word,
                                           u32 &loads) {
    const u64 last = endbit - 1;           // last bit wanted
    const u64 wi = last >> 6;
    if (wi != c_idx) {
        c_idx = wi;
        c_word = SWAP ? bswap64(words[wi]) : words[wi];
        ++loads;
    }
    const u32 used = (u32)(last & 63u) + 1u;  // bits of word wi up to and including `last`
    u64 v = c_word >> (64u - used);
    if (used < nbits) {                        // the field starts in the previous word
        const u64 prev = SWAP ? bswap64(words[wi - 1]) : words[wi - 1];
        ++loads;
        v |= prev << used;
        // going on downwards, the previous word is the next current one
        c_idx = wi - 1;
        c_word = prev;
    }
    return nbits >= 64 ? v : (v & ((1ull << nbits) - 1ull));
}

template <bool SC, bool STATS>
__global__ void __launch_bounds__(256, 1) fm_search_dna_packed_kernel(OccView ov, CTable5 c5, TextCmp tc, KTable kt, u32 len,
                                                                      const u64 *__restrict__ pw, u32 m, u32 stride,
                                                                      u64 npat, u32 *__restrict__ outL,
                                                                      u32 *__restrict__ outR,
                                                                      unsigned long long *__restrict__ stats) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npat) return;
    u32 n_blk = 0, n_pw = 0, n_tw = 0, n_sa = 0;
    const u64 bitbase = q * (u64)stride * 8ull;  // bit offset of base 0 of the read
    u32 L = 0, R = len;
    if (m > len) {
        L = 1;
        R = 0;
    }
    u64 p_idx = ~0ull, p_word = 0;
    int64_t i = (int64_t)m - 1;
    if (kt.tab && m >= (u32)kt.k && L < R) {
        // the last k bases, the last one most significant (the order the recurrence consumes them)
        const u64 w = bits_ending<true>(pw, bitbase + 2ull * m, 2u * (u32)kt.k, p_idx, p_word, n_pw);
        u32 r = __brev((u32)w) >> (32 - 2 * kt.k);                // pairs reversed, bits inside a pair swapped
        r = ((r & 0x55555555u) << 1) | ((r >> 1) & 0x55555555u);
        const uint2 lr = kt.tab[r];
        if (STATS) n_sa += 2;
        L = lr.x;
        R = lr.y;
        i -= kt.k;
    }
    for (; i >= 0 && L < R && !(SC && R - L == 1); --i) {
        const u32 a = (u32)bits_ending<true>(pw, bitbase + 2ull * (u64)i + 2ull, 2u, p_idx, p_word, n_pw) + 1u;
        if (a >= ov.sigma) {
            L = 1;
            R = 0;
            break;
        }
        const u32 bL = L >> 6, bR = R >> 6;
        BlockRegs kL = load_dna_block(ov.blocks, bL);
        BlockRegs kR = kL;
        if (bR != bL) kR = load_dna_block(ov.blocks, bR);
        if (STATS) n_blk += bR != bL ? 2u : 1u;
        const u32 ca = c5.c[a];
        L = ca + rank_in_block(kL, a, L, ov.primary);
        R = ca + rank_in_block(kR, a, R, ov.primary);
    }
    if (SC && i >= 0 && R - L == 1) {
        // one candidate suffix s = SA[L]: the remaining bases pattern[0..i] must equal text[s-1-i .. s-1]
        const u32 s = tc.sa[L];
        if (STATS) ++n_sa;
        const u32 rem = (u32)i + 1u;
        u32 k = 0;  // bases matched so far, from pattern[i] / text[s-1] downwards
        u64 t_idx = ~0ull, t_word = 0;
        bool mismatch = false;
        while (k < rem) {
            const u32 c = min(32u, min(rem - k, s - k));  // bases compared in this step
            if (c == 0) {  // the text is used up: the next base meets the sentinel
                mismatch = true;
                break;
            }
            const u64 P = bits_ending<true>(pw, bitbase + 2ull * (u64)(i - k) + 2ull, 2u * c, p_idx, p_word, n_pw);
            const u64 T = bits_ending<false>(tc.packed, 2ull * (u64)(s - k), 2u * c, t_idx, t_word, n_tw);
            const u64 d = P ^ T;
            if (d) {
                k += (u32)((__ffsll((long long)d) - 1) >> 1);
                mismatch = true;
                break;
            }
            k += c;
        }
        if (!mismatch) {
            L = tc.isa[s - rem];
            R = L + 1;
            if (STATS) ++n_sa;
        } else {
            const u32 a = (u32)bits_ending<true>(pw, bitbase + 2ull * (u64)(i - k) + 2ull, 2u, p_idx, p_word, n_pw) + 1u;
            if (a >= ov.sigma) {
                L = 1;
                R = 0;
            } else {
                // the step that fails: BWT[Lk] != a, so both ranks coincide and the interval is empty
                const u32 Lk = k ? tc.isa[s - k] : L;
                BlockRegs kb = load_dna_block(ov.blocks, Lk >> 6);
                BlockRegs kb2 = kb;
                if (((Lk + 1) >> 6) != (Lk >> 6)) kb2 = load_dna_block(ov.blocks, (Lk + 1) >> 6);
                if (STATS) {
                    n_sa += k ? 1u : 0u;
                    n_blk += 1u + ((((Lk + 1) >> 6) != (Lk >> 6)) ? 1u : 0u);
                }
                L = c5.c[a] + rank_in_block(kb, a, Lk, ov.primary);
                R = c5.c[a] + rank_in_block(kb2, a, Lk + 1, ov.primary);
            }
        }
    }
    outL[q] = L;
    outR[q] = R;
    if (STATS) {
        atomicAdd(&stats[0], (unsigned long long)n_blk);
        atomicAdd(&stats[1], (unsigned long long)n_pw);
        atomicAdd(&stats[2], (unsigned long long)n_tw);
        atomicAdd(&stats[3], (unsigned long long)n_sa);
    }
}

// codes 1..4 (one byte per base, read q at q * m) -> packed reads (read q at q * stride bytes)
__global__ void __launch_bounds__(256) pack_reads_kernel(const u8 *__restrict__ codes, u32 m, u32 stride, u64 npat,
                                                         u8 *__restrict__ out, int *__restrict__ err) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per output byte
    if (t >= npat * (u64)stride) return;
    const u64 q = t / stride;
    const u32 j0 = (u32)(t % stride) * 4u;
    u32 v = 0;
#pragma unroll
    for (u32 x = 0; x < 4; ++x) {
        u32 sym = 0;
        if (j0 + x < m) {
            const u32 c = codes[q * (u64)m + j0 + x];
            if (c - 1u > 3u) *err = 1;
            sym = (c - 1u) & 3u;
        }
        v |= sym << (6u - 2u * x);
    }
    out[t] = (u8)v;
}

void pack_reads(const u8 *d_codes, u32 m, u32 stride, u64 npat, u8 *d_out, int *d_err, cudaStream_t st) {
    if (!npat) return;
    pack_reads_kernel<<<div_up_u(npat * (u64)stride, 256), 256, 0, st>>>(d_codes, m, stride, npat, d_out, d_err);
    KERNEL_CHECK();
}

void fm_search_packed(const DeviceIndex &ix, const u8 *d_packed, u32 m, u32 stride, u64 npat, u32 *d_L, u32 *d_R,
                      cudaStream_t st, unsigned long long *d_stats) {
    if (!npat) return;
    OccView ov = occ_view(ix);
    CTable5 c5;
    for (int i = 0; i < 8; ++i) c5.c[i] = ix.c_host[i];
    const unsigned blocks = div_up_u(npat, 256);
    TextCmp tc{ix.sa.ptr, ix.isa.ptr, ix.text_packed.ptr};
    KTable kt{ix.ktable.ptr, ix.ktable_k};
    const bool sc = tc.sa && tc.isa && tc.packed && ix.pk.bits == 2;
    const u64 *pw = (const u64 *)d_packed;
    if (d_stats) {
        if (sc) fm_search_dna_packed_kernel<true, true><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, pw, m, stride, npat, d_L, d_R, d_stats);
        else fm_search_dna_packed_kernel<false, true><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, pw, m, stride, npat, d_L, d_R, d_stats);
    } else if (sc) {
        fm_search_dna_packed_kernel<true, false><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, pw, m, stride, npat, d_L, d_R, nullptr);
    } else {
        fm_search_dna_packed_kernel<false, false><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, pw, m, stride, npat, d_L, d_R, nullptr);
    }
    KERNEL_CHECK();
}

void fm_search(const DeviceIndex &ix, const u8 *d_pat, const u64 *d_off, u32 fixed_len, u64 npat, u32 *d_L,
               u32 *d_R, cudaStream_t st, unsigned long long *d_stats) {
    if (!npat) return;
    OccView ov = occ_view(ix);
    CTable5 c5;
    for (int i = 0; i < 8; ++i) c5.c[i] = ix.c_host[i];
    unsigned blocks = div_up_u(npat, 256);
    static const bool force_generic = getenv("B200SA_SEARCH_GENERIC") != nullptr;
    if (ix.occ_layout == OCC_DNA32 && (((uintptr_t)d_pat) & 7) == 0 && !force_generic)
    {
        TextCmp tc{ix.sa.ptr, ix.isa.ptr, ix.text_packed.ptr};
        KTable kt{ix.ktable.ptr, ix.ktable_k};
        const bool sc = tc.sa && tc.isa && tc.packed && ix.pk.bits == 2;
        if (d_stats) {
            if (sc) fm_search_dna_kernel<true, true><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R, d_stats);
            else fm_search_dna_kernel<false, true><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R, d_stats);
        } else if (sc) {
            fm_search_dna_kernel<true, false><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R, nullptr);
        } else {
            fm_search_dna_kernel<false, false><<<blocks, 256, 0, st>>>(ov, c5, tc, kt, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R, nullptr);
        }
    }
    else if (ix.occ_layout == OCC_DNA32)
        fm_search_kernel<1><<<blocks, 256, 0, st>>>(ov, c5, ix.c_table.ptr, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R);
    else {
        TextCmp tc{ix.sa.ptr, ix.isa.ptr, ix.text_packed.ptr};
        KTable kt{ix.ktable.ptr, ix.ktable_k, ix.sigma - 1};
        const bool al = (((uintptr_t)d_pat) & 7) == 0 && !force_generic;
        const bool sc2 = tc.sa && tc.isa && tc.packed;
#define LAUNCH_GEN(SC_, AL_) fm_search_kernel<2, SC_, AL_><<<blocks, 256, 0, st>>>(ov, c5, ix.c_table.ptr, ix.len, d_pat, d_off, fixed_len, npat, d_L, d_R, tc, ix.pk.bits, kt)
        if (sc2 && al) LAUNCH_GEN(true, true);
        else if (sc2) LAUNCH_GEN(true, false);
        else if (al) LAUNCH_GEN(false, true);
        else LAUNCH_GEN(false, false);
#undef LAUNCH_GEN
    }
    KERNEL_CHECK();
}

// The largest k whose table (8 bytes per k-mer) stays under a budget of bytes per text symbol: three for a lean
// index (k = 15, 8.6 GB, at 3 Gbp; 13 at 256 Mi; 9 at 1 Mi), twelve -- and k up to 16 -- for an index that keeps the
// suffix array, its inverse and the packed text for the unique-interval shortcut anyway (8.25 bytes per symbol):
// k = 16, 34 GB, at 3 Gbp.  Once the search kernel had become DRAM-bound every extra symbol of k paid (3 Gbp, 10^8
// reads of 100 bp, byte kernel: k = 12: 23.6 ms, 13: 20.5, 14: 17.7, 15: 15.7; packed kernel: 15: 13.5, 16: 11.5) --
// each one removes random O-block fetches from every read.
// the same over any alphabet: entry x = the k symbols as a base-nsym number, first processed symbol most significant
__global__ void __launch_bounds__(256) ktable_build_generic_kernel(OccView ov, const u32 *__restrict__ c_dev, u32 len, int k,
                                                                   u32 nsym, u32 ptop, u64 entries, uint2 *__restrict__ tab) {
    const u64 x64 = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x64 >= entries) return;
    u32 x = (u32)x64, pw = ptop;  // ptop = nsym^(k-1); entries < 2^32
    u32 L = 0, R = len;
    for (int j = 0; j < k && L < R; ++j) {
        const u32 a = x / pw + 1u;
        x %= pw;
        pw /= nsym;
        const u32 ca = c_dev[a];
        L = ca + occ_byte(ov, a, L);
        R = ca + occ_byte(ov, a, R);
    }
    tab[x64] = make_uint2(L, R);
}

static void build_ktable_generic(DeviceIndex &ix) {
    const u32 nsym = ix.sigma - 1;
    if (nsym < 2) return;
    const bool rich = ix.text_packed.ptr && ix.isa.ptr && ix.sa.ptr;
    const u64 budget = (rich ? 12ull : 3ull) * (u64)ix.len / 8;  // entries
    int k = 0;
    u64 entries = 1;
    while (k < 16 && entries * nsym <= budget && entries * nsym <= 2 * (u64)ix.len && entries * nsym < (1ull << 32)) {
        entries *= nsym;
        ++k;
    }
    if (const char *e = getenv("B200SA_KTABLE_K")) {
        const int want = std::max(1, std::min(16, atoi(e)));
        while (k > want) {
            entries /= nsym;
            --k;
        }
    }
    if (k < 2) return;
    ix.ktable.alloc(entries, ix.stream);
    ix.ktable_k = k;
    OccView ov = occ_view(ix);
    int t = ix.timer.begin("ktable", (double)entries * 8.0);
    ktable_build_generic_kernel<<<div_up_u(entries, 256), 256, 0, ix.stream>>>(ov, ix.c_table.ptr, ix.len, k, nsym,
                                                                             (u32)(entries / nsym), entries, ix.ktable.ptr);
    KERNEL_CHECK();
    ix.timer.end(t);
}

void build_ktable(DeviceIndex &ix) {
    if (ix.occ_layout == OCC_BYTE) {
        build_ktable_generic(ix);
        return;
    }
    if (ix.occ_layout != OCC_DNA32) return;
    const bool rich = ix.text_packed.ptr && ix.isa.ptr && ix.sa.ptr;
    int k = rich ? 16 : 15;
    while (k > 0 && (8ull << (2 * k)) > (rich ? 12ull : 3ull) * (u64)ix.len) --k;
    if (const char *e = getenv("B200SA_KTABLE_K")) {
        // (an explicit request may go one symbol further: k = 16 is a 34 GB table, 11 bytes per symbol at 3 Gbp)
        k = std::max(4, std::min(16, atoi(e)));
        while (k > 0 && (1ull << (2 * k)) > 2 * (u64)ix.len) --k;
    }
    if (k < 4) return;
    u64 entries = 1ull << (2 * k);
    // (a table that does not fit next to what the device already holds: one symbol less)
    for (;; --k, entries >>= 2) {
        size_t free_b = 0, total_b = 0;
        if (k <= 12 || cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || free_b > entries * 8 + ((size_t)4 << 30)) break;
    }
    ix.ktable.alloc(entries, ix.stream);
    ix.ktable_k = k;
    OccView ov = occ_view(ix);
    CTable5 c5;
    for (int i = 0; i < 8; ++i) c5.c[i] = ix.c_host[i];
    int t = ix.timer.begin("ktable", (double)entries * 8.0);
    ktable_build_kernel<<<div_up_u(entries, 256), 256, 0, ix.stream>>>(ov, c5, ix.len, k, entries, ix.ktable.ptr);
    KERNEL_CHECK();
    ix.timer.end(t);
}

// ---- locate -----------------------------------------------------------------------------------
static constexpr int LC_NT = 1024;

__global__ void __launch_bounds__(LC_NT) locate_count_kernel(const u32 *__restrict__ L, const u32 *__restrict__ R,
                                                             u64 npat, u64 *__restrict__ pos_off,
                                                             u64 *__restrict__ tile_tot) {
    __shared__ u64 wsum[32];
    u64 q = (u64)blockIdx.x * LC_NT + threadIdx.x;
    u64 v = 0;
    if (q < npat) {
        u32 l = L[q], r = R[q];
        v = r > l ? (u64)(r - l) : 0;
    }
    u64 total;
    const u64 excl = block_exclusive<LC_NT>(v, wsum, &total);
    if (q < npat) pos_off[q] = excl;
    if (threadIdx.x == 0) tile_tot[blockIdx.x] = total;
}

void scan_u64(u64 *d_vals, u64 count, cudaStream_t st) { scan_sum(d_vals, count, st, d_vals + count); }

__global__ void __launch_bounds__(LC_NT) locate_add_kernel(u64 *__restrict__ pos_off, u64 npat,
                                                           const u64 *__restrict__ tile_prefix,
                                                           const u64 *__restrict__ total) {
    u64 q = (u64)blockIdx.x * LC_NT + threadIdx.x;
    if (q < npat) pos_off[q] += tile_prefix[blockIdx.x];
    if (q == npat - 1) pos_off[npat] = *total;
}

u64 fm_locate_count(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, u64 *d_pos_off,
                    cudaStream_t st) {
    if (!npat) {
        CUDA_CHECK(cudaMemsetAsync(d_pos_off, 0, 8, st));
        return 0;
    }
    unsigned tiles = div_up_u(npat, LC_NT);
    DevBuf<u64> tile_tot(tiles, st), total(1, st);
    locate_count_kernel<<<tiles, LC_NT, 0, st>>>(d_L, d_R, npat, d_pos_off, tile_tot.ptr);
    KERNEL_CHECK();
    scan_sum(tile_tot.ptr, (u64)tiles, st, total.ptr);
    locate_add_kernel<<<tiles, LC_NT, 0, st>>>(d_pos_off, npat, tile_tot.ptr, total.ptr);
    KERNEL_CHECK();
    u64 h = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h, total.ptr, 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    return h;
}

// one thread per output position; the owning pattern is found by binary search in pos_off
__global__ void __launch_bounds__(256) locate_fill_kernel(const u32 *__restrict__ sa, const u32 *__restrict__ L,
                                                          const u64 *__restrict__ pos_off, u64 npat, u64 total,
                                                          u32 *__restrict__ pos) {
    u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    // largest q with pos_off[q] <= t
    u64 lo = 0, hi = npat;  // pos_off[npat] = total > t
    while (hi - lo > 1) {
        u64 mid = lo + (hi - lo) / 2;
        if (pos_off[mid] <= t) lo = mid;
        else hi = mid;
    }
    pos[t] = sa[(u64)L[lo] + (t - pos_off[lo])];
}

void fm_locate_fill(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, const u64 *d_pos_off,
                    u64 total, u32 *d_pos, cudaStream_t st) {
    (void)d_R;
    if (!total) return;
    locate_fill_kernel<<<div_up_u(total, 256), 256, 0, st>>>(ix.sa.ptr, d_L, d_pos_off, npat, total, d_pos);
    KERNEL_CHECK();
}

}  // namespace b200sa
