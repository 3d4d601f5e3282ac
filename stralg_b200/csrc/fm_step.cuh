// fm_step.cuh -- device pieces of the backward search recurrence that the exact search (fm_search.cu) and the
// matching statistics (mems.cu) both run: the k-mer seed key, one O step of the DNA layout, and the comparison of
// pattern symbols with the packed text that finishes a unique interval; and the bidirectional steps (the children of
// all letters, the exact child of one letter, the byte layout's running start) and the pattern split of the
// k-mismatch and edit-distance searches (hamming.cu, levenshtein.cu).
#pragma once
#include "occ.cuh"

namespace b200sa {

struct CTable5 {
    u32 c[8];
};

// Pointers for the unique-interval shortcut (B200SA_BUILD_TEXTCMP); all null when it is off.
struct TextCmp {
    const u32 *sa;
    const u32 *isa;
    const u64 *packed;  // symbols of `bits` bits (code - 1), big-endian inside each word (sa_build.cu pack_kernel)
};

// k-mer seed table (B200SA_BUILD_KTABLE): tab[x] = the (L, R) the recurrence reaches on the k-mer whose symbols, in
// the order the recurrence consumes them (last pattern symbol first), are the digits of x, most significant first:
// base 4 for the DNA layout (nsym = 0), base nsym otherwise.  An entry with L >= R is the interval at the step that
// emptied it, i.e. the final answer of every pattern ending in that k-mer.
struct KTable {
    const uint2 *tab;
    int k;
    u32 nsym;
};

// ---- DNA layout (OCC_DNA32) ---------------------------------------------------------------------
struct BlockRegs {
    u32 c0, c1, c2, c3;
    u64 w0, w1;
};

__device__ __forceinline__ BlockRegs load_dna_block(const u8 *blocks, u32 b) {
    u64 a, bb, c, d;
    const u8 *p = blocks + (size_t)b * 32;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(a), "=l"(bb), "=l"(c), "=l"(d) : "l"(p));
    BlockRegs r;
    r.c0 = (u32)a; r.c1 = (u32)(a >> 32); r.c2 = (u32)bb; r.c3 = (u32)(bb >> 32);
    r.w0 = c; r.w1 = d;
    return r;
}

__device__ __forceinline__ u32 rank_in_block(const BlockRegs &blk, u32 a, u32 i, u32 primary) {
    u32 base = a == 1 ? blk.c0 : a == 2 ? blk.c1 : a == 3 ? blk.c2 : blk.c3;
    u32 c = base + dna_match_count(blk.w0, blk.w1, a - 1, i & 63u);
    if (a == 1) {
        u32 start = i & ~63u;
        if (primary >= start && primary < i) c -= 1;  // the sentinel row is stored as value 0
    }
    return c;
}

// One backward step by letter a (1..4) from [L, R): ONE 256-bit load per distinct block (the L and R rows share a
// block once the interval is narrower than 64 rows, i.e. after ~log4(len) steps on random DNA).
template <bool STATS>
__device__ __forceinline__ uint2 dna_step(const OccView &ov, const CTable5 &c5, u32 a, u32 L, u32 R, u32 &n_blk) {
    const u32 bL = L >> 6, bR = R >> 6;
    BlockRegs kL = load_dna_block(ov.blocks, bL);
    BlockRegs kR = kL;
    if (bR != bL) kR = load_dna_block(ov.blocks, bR);
    if (STATS) n_blk += bR != bL ? 2u : 1u;
    const u32 ca = c5.c[a];
    return make_uint2(ca + rank_in_block(kL, a, L, ov.primary), ca + rank_in_block(kR, a, R, ov.primary));
}

// Pattern symbol at byte address `addr` through a one-word cache of aligned 8-byte words (the pattern buffer is
// 8-byte aligned and readable up to the next 8-byte boundary).
template <bool STATS>
__device__ __forceinline__ u32 pattern_byte(const u8 *__restrict__ pat, u64 addr, u64 &word, u64 &word_addr, u32 &n_pw) {
    if ((addr & ~7ull) != word_addr) {
        word_addr = addr & ~7ull;
        word = *(const u64 *)(pat + word_addr);
        if (STATS) ++n_pw;
    }
    return (u32)(word >> (8 * (addr & 7))) & 0xffu;
}

// Seed key of the DNA table: the k symbols pattern[i], pattern[i-1], ..., pattern[i-k+1] (i >= k-1) as a 2k-bit
// number, pattern[i] most significant.  False when one of them is outside 1..4.
template <bool STATS>
__device__ __forceinline__ bool dna_seed_key(const u8 *__restrict__ pat, u64 begin, int64_t i, int k, u64 &word,
                                             u64 &word_addr, u32 &n_pw, u32 &x) {
    x = 0;
    bool valid = true;
    for (int j = 0; j < k; ++j) {
        const u32 a = pattern_byte<STATS>(pat, begin + (u64)i - (u64)j, word, word_addr, n_pw);
        valid = valid && (a - 1u <= 3u);
        x = (x << 2) | ((a - 1u) & 3u);
    }
    return valid;
}

// One candidate suffix s = SA[L] is left after the pattern symbols above i were consumed.  The recurrence would now
// consume pattern[i], pattern[i-1], ... one O lookup each, moving to ISA[s-1], ISA[s-2], ... as long as they equal
// text[s-1], text[s-2], ...; compare them against the 2-bit packed text instead.  Returns k, the number of symbols
// that agree (k <= i + 1, k <= s); when k < i + 1, `a` is pattern[i-k], the symbol that stopped the run.
template <bool STATS>
__device__ __forceinline__ u64 dna_text_agree(const u8 *__restrict__ pat, u64 begin, int64_t i, u32 s,
                                              const u64 *__restrict__ packed, u64 &word, u64 &word_addr, u32 &a,
                                              u32 &n_pw, u32 &n_tw) {
    const u64 rem = (u64)i + 1;
    u64 k = 0;
    u64 tw = 0, tw_idx = ~0ull;
    a = 0;
    // Eight symbols per step while at least eight are left on both sides: the pattern bytes
    // pattern[i-k-7 .. i-k] (an unaligned 8-byte window, byte-swapped so that pattern[i-k]
    // comes first) are packed to 16 bits and compared with the 16 bits of packed text that
    // hold text[s-1-k-7 .. s-1-k]; the first difference, in the order the recurrence would
    // meet the symbols, ends the run.  The scalar loop below takes over from there (it finds
    // the failing symbol at once, or finishes a tail shorter than eight).
    {
        const u64 ones = 0x0101010101010101ull;
        u64 plo = 0, phi = 0, pbase = ~0ull;  // aligned pattern words at pbase and pbase + 8
        while (rem - k >= 8 && (u64)s - k >= 8) {
            const u64 first = begin + (u64)i - k - 7;  // address of pattern[i-k-7]
            const u64 base8 = first & ~7ull;
            const u32 sh = (u32)(first & 7u) * 8u;
            if (base8 != pbase) {
                phi = (pbase != ~0ull && base8 + 8 == pbase) ? plo : (sh ? *(const u64 *)(pat + base8 + 8) : 0ull);
                plo = *(const u64 *)(pat + base8);
                if (STATS) n_pw += (pbase != ~0ull && base8 + 8 == pbase) ? 1u : (sh ? 2u : 1u);
                pbase = base8;
            }
            const u64 P = sh ? (plo >> sh) | (phi << (64u - sh)) : plo;  // byte j = pattern[i-k-7+j]
            const u64 v = P - ones;
            if (v & 0xFCFCFCFCFCFCFCFCull) break;  // a byte outside 1..4: the scalar loop decides
            // byte-swap (pattern[i-k] to the low end), then squeeze the 2-bit symbols together
            u64 y = ((u64)__byte_perm((u32)v, 0, 0x0123) << 32) | (u64)__byte_perm((u32)(v >> 32), 0, 0x0123);
            y &= 0x0303030303030303ull;
            y = (y | (y >> 6)) & 0x000F000F000F000Full;
            y = (y | (y >> 12)) & 0x000000FF000000FFull;
            y = (y | (y >> 24)) & 0xFFFFull;  // bits 2j..2j+1 = pattern[i-k-j] - 1
            // text[s-1-k-j] for j = 0..7 in the same order: position t = s-1-k sits lowest
            const u64 t = (u64)s - 1 - k;
            const u64 w = t >> 5;
            const u32 tsh = 62u - 2u * (u32)(t & 31u);
            if (w != tw_idx) {
                tw_idx = w;
                tw = packed[w];
                if (STATS) ++n_tw;
            }
            u64 T = tw >> tsh;
            if ((t & 31u) < 7u) {  // the field runs into the previous word
                const u64 prev = packed[w - 1];
                if (STATS) ++n_tw;
                T |= prev << (64u - tsh);
                // going on downwards, the previous word is the next current one
                tw_idx = w - 1;
                tw = prev;
            }
            const u32 d = (u32)((T ^ y) & 0xFFFFull);
            if (d) {
                k += (u64)((__ffs((int)d) - 1) >> 1);
                break;
            }
            k += 8;
        }
        // hand the pattern word the scalar loop will ask for first over to its one-word cache
        if (pbase != ~0ull && k < rem) {
            const u64 need = (begin + (u64)i - k) & ~7ull;
            if (need == pbase) {
                word_addr = need;
                word = plo;
            }
        }
    }
    while (k < rem) {
        a = pattern_byte<STATS>(pat, begin + (u64)i - k, word, word_addr, n_pw);
        if (k >= (u64)s) break;  // suffix 0 is preceded by the sentinel only
        u64 t = (u64)s - 1 - k;
        if ((t >> 5) != tw_idx) {
            tw_idx = t >> 5;
            tw = packed[tw_idx];
            if (STATS) ++n_tw;
        }
        u32 sym = (u32)(tw >> (62 - 2 * (t & 31))) & 3u;
        if (a - 1u != sym) break;
        ++k;
    }
    return k;
}

// ---- any alphabet (OCC_BYTE); `P(idx)` gives pattern[idx] --------------------------------------------
// Seed key: pattern[i], ..., pattern[i-k+1] as a base-nsym number, pattern[i] most significant; false when one
// of them is outside 1..nsym.
template <class Pat>
__device__ __forceinline__ bool seed_key(Pat &&P, int64_t i, const KTable &kt, u32 &x) {
    x = 0;
    bool valid = true;
    for (int j = 0; j < kt.k; ++j) {
        const u32 a = P(i - j);
        valid = valid && (a - 1u < kt.nsym);
        x = x * kt.nsym + (a - 1u);
    }
    return valid;
}

// dna_text_agree for a packed text of `bits` (1, 2, 4 or 8) bits per symbol, one symbol per step.
template <class Pat>
__device__ __forceinline__ u64 text_agree(Pat &&P, int64_t i, u32 s, const u64 *__restrict__ packed, int bits, u32 &a) {
    const u64 rem = (u64)i + 1;
    const u32 mask = (1u << bits) - 1u;
    const u32 lg = bits == 8 ? 3u : bits == 4 ? 4u : bits == 2 ? 5u : 6u;  // log2 of the symbols per word
    u64 k = 0, tw = 0, tw_idx = ~0ull;
    a = 0;
    while (k < rem) {
        a = P(i - (int64_t)k);
        if (k >= (u64)s) break;  // suffix 0 is preceded by the sentinel only
        const u64 t = (u64)s - 1 - k;
        if ((t >> lg) != tw_idx) {
            tw_idx = t >> lg;
            tw = packed[tw_idx];
        }
        const u32 sym = (u32)(tw >> (64u - (u32)bits - (u32)(t & ((1u << lg) - 1u)) * (u32)bits)) & mask;
        if (a - 1u != sym) break;
        ++k;
    }
    return k;
}

// ---- bidirectional steps (hamming.cu, levenshtein.cu) -------------------------------------------------
// A string X is held on two indices, F over the text T and B over reverse(T): [x, x + w) on the index a step runs
// on, [y, y + w) on the other.  Extending X to the left (aX) is a step on F, extending it to the right (Xa) a step
// on B; for both
//   x_a = C[a] + O(a, x),   w_a = O(a, x + w) - O(a, x),   y_a = y + [x <= primary < x + w] + sum_{b < a} w_b
// since on the other index the one-letter extensions of X sit side by side in letter order, after the one row that
// ends in the sentinel when X starts the text (its row on the stepped index is `primary`).  Both indices have the
// same C table.
__device__ __forceinline__ u32 bidi_sentinel(const OccView &ov, u32 x, u32 w) { return ov.primary - x < w ? 1u : 0u; }

struct BiChildren {
    u32 x[4], w[4], y[4];  // the child of letter a at [a - 1]
};

// v[a - 1] for a letter a in 1..4
__device__ __forceinline__ u32 pick4(const u32 (&v)[4], u32 a) {
    return a == 1 ? v[0] : a == 2 ? v[1] : a == 3 ? v[2] : v[3];
}

// DNA layout: the children of all four letters from the one or two blocks that dna_step loads
__device__ __forceinline__ BiChildren dna_bidi_children(const OccView &ov, const CTable5 &c5, u32 x, u32 w, u32 y) {
    const u32 e = x + w;
    const BlockRegs kL = load_dna_block(ov.blocks, x >> 6);
    BlockRegs kR = kL;
    if ((e >> 6) != (x >> 6)) kR = load_dna_block(ov.blocks, e >> 6);
    BiChildren ch;
    u32 run = y + bidi_sentinel(ov, x, w);
#pragma unroll
    for (u32 a = 1; a <= 4; ++a) {
        const u32 lo = rank_in_block(kL, a, x, ov.primary), hi = rank_in_block(kR, a, e, ov.primary);
        ch.x[a - 1] = c5.c[a] + lo;
        ch.w[a - 1] = hi - lo;
        ch.y[a - 1] = run;
        run += hi - lo;
    }
    return ch;
}

// Byte layout: y_a, the start on the other index of the child of letter a (two O lookups per letter below a)
__device__ __forceinline__ u32 byte_bidi_run(const OccView &ov, u32 x, u32 w, u32 y, u32 a) {
    u32 run = y + bidi_sentinel(ov, x, w);
    for (u32 b = 1; b < a; ++b) run += occ_byte(ov, b, x + w) - occ_byte(ov, b, x);
    return run;
}

// Byte layout, one letter at a time in ascending order: the child of letter a.  `run` is y_a on entry (byte_bidi_run)
// and y_{a+1} on return, so a walk over the letters costs two O lookups per letter.
__device__ __forceinline__ void byte_bidi_child(const OccView &ov, const u32 *c, u32 a, u32 x, u32 w, u32 &run,
                                                u32 &cx, u32 &cw, u32 &cy) {
    const u32 lo = occ_byte(ov, a, x), hi = occ_byte(ov, a, x + w);
    cx = c[a] + lo;
    cw = hi - lo;
    cy = run;
    run += cw;
}

// The child of letter a alone (an exact step) on either layout; `c` is the C table (byte layout).  Without `need_y`
// the byte layout skips the letters below a, and cy is not the child's.
template <int LAYOUT>
__device__ __forceinline__ void bidi_child(const OccView &ov, const CTable5 &c5, const u32 *c, u32 a, u32 x, u32 w,
                                           u32 y, bool need_y, u32 &cx, u32 &cw, u32 &cy) {
    if (LAYOUT == 1) {
        const BiChildren ch = dna_bidi_children(ov, c5, x, w, y);
        cx = pick4(ch.x, a);
        cw = pick4(ch.w, a);
        cy = pick4(ch.y, a);
    } else {
        u32 run = byte_bidi_run(ov, x, w, y, need_y ? a : 1u);
        byte_bidi_child(ov, c, a, x, w, run, cx, cw, cy);
    }
}

// The index a step runs on: B (the reversed text) for a right extension, F (the text) for a left one.  The two
// indices share everything but their blocks and sentinel row.
__device__ __forceinline__ OccView step_index(const OccView &fv, const OccView &bv, bool right) {
    OccView ov = fv;
    if (right) {
        ov.blocks = bv.blocks;
        ov.primary = bv.primary;
    }
    return ov;
}

// The k + 1 parts of a search scheme: a pattern of m = (k + 1) qs + r symbols splits into parts of qs + 1 symbols
// (the r first) and of qs; part_start is the first position of part j, part_of the part of position pos.
__device__ __forceinline__ u32 part_start(u32 j, u32 qs, u32 r) { return j * qs + min(j, r); }
__device__ __forceinline__ u32 part_of(u32 pos, u32 qs, u32 r) {
    const u32 big = r * (qs + 1);
    return pos < big ? pos / (qs + 1) : r + (pos - big) / qs;
}

}  // namespace b200sa
