// bwt_occ.cu -- BWT rows, C table and the sampled occurrence table (sm_100a).
//
//   bwt[r] = sa[r] == 0 ? 0 : text[sa[r] - 1]                       stralg/bwt.c:13-20
//   C[a]   = #{symbols of text+sentinel smaller than a}             stralg/bwt.c:35-45 (pack_text)
//   O(a,i) = #{k < i : bwt[k] == a}                                 stralg/bwt.c:47-65
//
// The reference materialises O as a dense (len+1) x sigma u32 matrix (it cannot be allocated
// above ~214 M rows, bwt.c:50); here O is stored as 64-row blocks (occ.cuh) and queried with
// popcounts.  occ_dense() re-creates the reference layout for small inputs (compat shims, tests).
#include "engine.h"
#include "occ.cuh"
#include "scan.cuh"

namespace b200sa {

// ---- BWT rows by gather (only for tables added to an existing SA; builds carry them in the keys) ----
__global__ void __launch_bounds__(256) bwt_gather_kernel(const u32 *__restrict__ sa, const u64 *__restrict__ packed,
                                                         u32 len, int bits, u8 *__restrict__ bwt,
                                                         u32 *__restrict__ primary) {
    u64 r0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (r0 >= len) return;
    u32 out = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        u32 code = 0;
        if (r0 + q < len) {
            u32 s = sa[r0 + q];
            if (s == 0) {
                *primary = (u32)(r0 + q);
            } else {
                code = sym_at(packed, s - 1, bits) + 1u;
            }
        }
        out |= code << (8 * q);
    }
    *(u32 *)(bwt + r0) = out;  // the buffer is padded to a multiple of 64 rows
}

void gather_bwt(DeviceIndex &ix) {
    cudaStream_t st = ix.stream;
    size_t bwt_bytes = (((size_t)ix.len + 63) / 64 + 1) * 64;
    if (!ix.bwt.ptr) {
        ix.bwt.alloc_output(bwt_bytes, st);
        CUDA_CHECK(cudaMemsetAsync(ix.bwt.ptr + (bwt_bytes - 128), 0, 128, st));
    }
    DevBuf<u32> d_primary(1, st);
    int t = ix.timer.begin("bwt_gather", (double)ix.len * 6.0);
    bwt_gather_kernel<<<div_up_u(((u64)ix.len + 3) / 4, 256), 256, 0, st>>>(ix.sa.ptr, ix.packed, ix.len, ix.pk.bits,
                                                                             ix.bwt.ptr, d_primary.ptr);
    KERNEL_CHECK();
    ix.timer.end(t);
    CUDA_CHECK(cudaMemcpyAsync(&ix.primary, d_primary.ptr, 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
}

// ---- OCC_DNA32 --------------------------------------------------------------------------------
static constexpr int OD_NT = 256;  // blocks per tile

__global__ void __launch_bounds__(OD_NT) occ_dna_count_kernel(const u8 *__restrict__ bwt, u64 nblocks,
                                                              DnaBlock *__restrict__ blocks,
                                                              u32 *__restrict__ tile_counts) {
    __shared__ u32 wsum[OD_NT / 32][4];
    u64 b = (u64)blockIdx.x * OD_NT + threadIdx.x;
    u32 cnt[4] = {0, 0, 0, 0};
    if (b < nblocks) {
        const uint4 *src = (const uint4 *)(bwt + b * 64);
        u64 w[2] = {0, 0};
        u32 zero_rows = 0;  // rows holding code 0 (the sentinel row, padding after the last row): packed as 0
        const u64 ones = 0x0101010101010101ull, high = 0x8080808080808080ull;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const uint4 x = ld_stream_u128(src + v);
            const u64 half[2] = {((u64)x.y << 32) | x.x, ((u64)x.w << 32) | x.z};
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                // eight rows at a time: symbol = code - 1 (rows with code 0 are patched to code 1 first),
                // row k of the block at bits [2k, 2k+1] of word k / 32
                u64 c8 = half[hh];
                const u64 low7 = 0x7f7f7f7f7f7f7f7full;
                const u64 z = ~(((c8 & low7) + low7) | c8) & high;  // 0x80 exactly in the bytes that are zero
                if (z) {
                    c8 |= z >> 7;  // 0 -> 1
                    zero_rows += (u32)__popcll(z);
                }
                u64 y = (c8 - ones) & 0x0303030303030303ull;
                y = (y | (y >> 6)) & 0x000F000F000F000Full;
                y = (y | (y >> 12)) & 0x000000FF000000FFull;
                y = (y | (y >> 24)) & 0xFFFFull;
                const int k0 = v * 16 + hh * 8;
                w[k0 >> 5] |= y << (2 * (k0 & 31));
            }
        }
#pragma unroll
        for (u32 c = 0; c < 4; ++c) {
            const u64 p = c * 0x5555555555555555ull;
            const u64 y0 = w[0] ^ p, y1 = w[1] ^ p;
            cnt[c] = (u32)__popcll(~(y0 | (y0 >> 1)) & 0x5555555555555555ull) +
                     (u32)__popcll(~(y1 | (y1 >> 1)) & 0x5555555555555555ull);
        }
        cnt[0] -= zero_rows;  // they are not occurrences of code 1
        DnaBlock blk;
        blk.cnt[0] = cnt[0]; blk.cnt[1] = cnt[1]; blk.cnt[2] = cnt[2]; blk.cnt[3] = cnt[3];
        blk.bits[0] = w[0];
        blk.bits[1] = w[1];
        blocks[b] = blk;
    }
    u32 r[4] = {cnt[0], cnt[1], cnt[2], cnt[3]};
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r[x] += __shfl_xor_sync(0xffffffffu, r[x], o);
    if (lane_id() == 0)
        for (int x = 0; x < 4; ++x) wsum[threadIdx.x >> 5][x] = r[x];
    __syncthreads();
    if (threadIdx.x < 4) {
        u32 t = 0;
        for (int w = 0; w < OD_NT / 32; ++w) t += wsum[w][threadIdx.x];
        tile_counts[(size_t)blockIdx.x * 4 + threadIdx.x] = t;
    }
}

// grid = nsym blocks; block x scans tile_counts[tile * nsym + x] over tiles (exclusive, in place)
__global__ void __launch_bounds__(1024) occ_scan_tiles_kernel(u32 *__restrict__ tile_counts, u32 ntiles, u32 nsym) {
    u32 *col = tile_counts + blockIdx.x;
    cta_exclusive_scan(
        ntiles, [=](u32 i) { return col[(size_t)i * nsym]; }, [=](u32 i, u32 e) { col[(size_t)i * nsym] = e; }, SumOp(),
        0u);
}

__global__ void __launch_bounds__(OD_NT) occ_dna_finalize_kernel(DnaBlock *__restrict__ blocks, u64 nblocks,
                                                                 const u32 *__restrict__ tile_prefix) {
    __shared__ u32 wsum[OD_NT / 32][4];
    u64 b = (u64)blockIdx.x * OD_NT + threadIdx.x;
    u32 v[4] = {0, 0, 0, 0};
    if (b < nblocks) {
        uint4 h = *(const uint4 *)&blocks[b];
        v[0] = h.x; v[1] = h.y; v[2] = h.z; v[3] = h.w;
    }
    u32 incl[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) incl[x] = warp_inclusive(v[x], SumOp());
    if (lane_id() == 31)
        for (int x = 0; x < 4; ++x) wsum[threadIdx.x >> 5][x] = incl[x];
    __syncthreads();
    if (b < nblocks) {
        u32 out[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            u32 wb = 0;
            for (unsigned w = 0; w < (threadIdx.x >> 5); ++w) wb += wsum[w][x];
            out[x] = tile_prefix[(size_t)blockIdx.x * 4 + x] + wb + incl[x] - v[x];
        }
        *(uint4 *)&blocks[b] = make_uint4(out[0], out[1], out[2], out[3]);
    }
}

// ---- OCC_BYTE ---------------------------------------------------------------------------------
static constexpr int OB_BLOCKS = 16;  // 64-row blocks per tile (1024 rows, 256 threads x 4 rows)

__global__ void __launch_bounds__(256) occ_byte_count_kernel(const u8 *__restrict__ bwt, u32 len, u64 nblocks,
                                                             u32 sigma, u32 hdr_words, u32 block_bytes,
                                                             u8 *__restrict__ blocks, u32 *__restrict__ tile_counts) {
    __shared__ u32 cnt[OB_BLOCKS][256];
    for (int i = threadIdx.x; i < OB_BLOCKS * 256; i += 256) (&cnt[0][0])[i] = 0;
    __syncthreads();
    u64 row0 = (u64)blockIdx.x * (OB_BLOCKS * 64) + (u64)threadIdx.x * 4;
    u32 four = row0 < (((u64)len + 63) & ~63ull) ? *(const u32 *)(bwt + row0) : 0;
    u32 bt = threadIdx.x >> 4;  // block inside the tile
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        u32 code = (four >> (8 * q)) & 0xffu;
        if (row0 + q < len && code) atomicAdd(&cnt[bt][code], 1u);
    }
    u64 gb = (u64)blockIdx.x * OB_BLOCKS + bt;
    if (gb < nblocks) *(u32 *)(blocks + gb * block_bytes + (size_t)hdr_words * 4 + (threadIdx.x & 15) * 4) = four;
    __syncthreads();
    // per symbol: exclusive running count over the tile's blocks
    for (u32 a = 1 + threadIdx.x; a < sigma; a += 256) {
        u32 run = 0;
        for (int k = 0; k < OB_BLOCKS; ++k) {
            u64 g = (u64)blockIdx.x * OB_BLOCKS + k;
            if (g < nblocks) ((u32 *)(blocks + g * block_bytes))[a - 1] = run;
            run += cnt[k][a];
        }
        tile_counts[(size_t)blockIdx.x * (sigma - 1) + (a - 1)] = run;
    }
}

__global__ void __launch_bounds__(256) occ_byte_finalize_kernel(u8 *__restrict__ blocks, u64 nblocks, u32 sigma,
                                                                u32 block_bytes,
                                                                const u32 *__restrict__ tile_prefix) {
    for (u32 a = 1 + threadIdx.x; a < sigma; a += 256) {
        u32 add = tile_prefix[(size_t)blockIdx.x * (sigma - 1) + (a - 1)];
        for (int k = 0; k < OB_BLOCKS; ++k) {
            u64 g = (u64)blockIdx.x * OB_BLOCKS + k;
            if (g < nblocks) ((u32 *)(blocks + g * block_bytes))[a - 1] += add;
        }
    }
}

// ---- queries ----------------------------------------------------------------------------------
static OccView make_view(const DeviceIndex &ix) {
    OccView ov;
    ov.blocks = ix.occ.ptr;
    ov.block_bytes = ix.occ_block_bytes;
    ov.hdr_words = ix.occ_layout == OCC_BYTE ? (ix.occ_block_bytes - 64) / 4 : 4;
    ov.primary = ix.primary;
    ov.sigma = ix.sigma;
    ov.layout = (int)ix.occ_layout;
    return ov;
}
OccView occ_view(const DeviceIndex &ix) { return make_view(ix); }

__global__ void occ_probe_kernel(OccView ov, const u8 *__restrict__ a, const u32 *__restrict__ i, u64 count,
                                 u32 *__restrict__ out) {
    u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < count) out[q] = occ_any(ov, a[q], i[q]);
}

__global__ void occ_dense_kernel(OccView ov, u32 len, u32 *__restrict__ out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > len) return;
    for (u32 a = 0; a < ov.sigma; ++a) out[i * ov.sigma + a] = occ_any(ov, a, (u32)i);
}

void occ_probe(const DeviceIndex &ix, const u8 *d_a, const u32 *d_i, u64 count, u32 *d_out) {
    if (!count) return;
    occ_probe_kernel<<<div_up_u(count, 256), 256, 0, ix.stream>>>(make_view(ix), d_a, d_i, count, d_out);
    KERNEL_CHECK();
}

void occ_dense(const DeviceIndex &ix, u32 *d_out) {
    occ_dense_kernel<<<div_up_u((u64)ix.len + 1, 256), 256, 0, ix.stream>>>(make_view(ix), ix.len, d_out);
    KERNEL_CHECK();
}

// ---- host orchestration -----------------------------------------------------------------------
void build_bwt_tables(DeviceIndex &ix, bool keep_bwt) {
    // ix.bwt (rows padded to a multiple of 64 with zeros) and ix.primary come from the SA build
    cudaStream_t st = ix.stream;
    const u32 len = ix.len;
    DevBuf<u8> &bwt = ix.bwt;
    int t;

    const u64 nblocks = (u64)len / 64 + 1;  // O(a, len) may address one block past the last row
    ix.occ_blocks = nblocks;
    t = ix.timer.begin("occ_build", (double)len * 1.5);
    if (ix.sigma <= 5) {
        ix.occ_layout = OCC_DNA32;
        ix.occ_block_bytes = 32;
        ix.occ.alloc_output(nblocks * 32, st);
        u32 ntiles = div_up_u(nblocks, OD_NT);
        DevBuf<u32> tile_counts((size_t)ntiles * 4, st);
        occ_dna_count_kernel<<<ntiles, OD_NT, 0, st>>>(bwt.ptr, nblocks, (DnaBlock *)ix.occ.ptr, tile_counts.ptr);
        KERNEL_CHECK();
        occ_scan_tiles_kernel<<<4, 1024, 0, st>>>(tile_counts.ptr, ntiles, 4);
        KERNEL_CHECK();
        occ_dna_finalize_kernel<<<ntiles, OD_NT, 0, st>>>((DnaBlock *)ix.occ.ptr, nblocks, tile_counts.ptr);
        KERNEL_CHECK();
    } else {
        ix.occ_layout = OCC_BYTE;
        u32 hdr_words = ((ix.sigma - 1) + 3) & ~3u;
        ix.occ_block_bytes = hdr_words * 4 + 64;
        ix.occ.alloc_output(nblocks * ix.occ_block_bytes, st);
        u32 ntiles = div_up_u(nblocks, OB_BLOCKS);
        DevBuf<u32> tile_counts((size_t)ntiles * (ix.sigma - 1), st);
        occ_byte_count_kernel<<<ntiles, 256, 0, st>>>(bwt.ptr, len, nblocks, ix.sigma, hdr_words, ix.occ_block_bytes,
                                                      ix.occ.ptr, tile_counts.ptr);
        KERNEL_CHECK();
        occ_scan_tiles_kernel<<<ix.sigma - 1, 1024, 0, st>>>(tile_counts.ptr, ntiles, ix.sigma - 1);
        KERNEL_CHECK();
        occ_byte_finalize_kernel<<<ntiles, 256, 0, st>>>(ix.occ.ptr, nblocks, ix.sigma, ix.occ_block_bytes,
                                                         tile_counts.ptr);
        KERNEL_CHECK();
    }
    ix.timer.end(t);
    if (!keep_bwt) ix.bwt.release();
}

}  // namespace b200sa
