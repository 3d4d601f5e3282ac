// records.cu -- one index over many records (sm_100a).
//
// A records index holds the records r0, r1, ..., r(k-1) of a multi-record reference in one text,
// each followed by the separator code 1:  r0 # r1 # ... r(k-1) # $.  The separator sorts below
// every letter (codes 2..sigma-1), just like a record's own sentinel, so two suffixes of the same
// record compare in the concatenation exactly as they do in the record alone: they differ at a
// letter, or the shorter one reaches its record's separator first.  The global suffix array
// restricted to the positions of one record is therefore that record's own suffix array, in
// order.  Record r starts at start[r] = rec_off[r] + r; start[k] = n is the global sentinel.
//
//   records_assemble   codes back to back -> the text with separators (code i lands at i + record(i))
//   record_sas         every record's own suffix array: record id per row, stable partition by it
//   locate_records     (pattern, global position) -> (record, local position), grouped by record
//                      inside every pattern by one stable sort keyed [pattern | record]
#include "engine.h"
#include "radix_sort.cuh"

namespace b200sa {

// the largest r < nrec with bound[r] <= p, for bound[0] <= p < bound[nrec] (bound: rec_off or start)
__device__ __forceinline__ u32 record_of(const u64 *__restrict__ bound, u32 nrec, u64 p) {
    u32 lo = 0, hi = nrec;
    while (hi - lo > 1) {
        const u32 mid = lo + (hi - lo) / 2;
        if (__ldg(bound + mid) <= p) lo = mid;
        else hi = mid;
    }
    return lo;
}

// thread t < ncodes: code t goes to t + record(t); thread ncodes + r: the separator after record r
__global__ void __launch_bounds__(256) records_assemble_kernel(const u8 *__restrict__ codes, u64 ncodes,
                                                               const u64 *__restrict__ rec_off, u32 nrec, u32 sigma,
                                                               u8 *__restrict__ text, int *__restrict__ err) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ncodes) {
        const u32 c = codes[t];
        if (c < 2u || c >= sigma) atomicOr(err, 1);
        text[t + record_of(rec_off, nrec, t)] = (u8)c;
    } else if (t < ncodes + nrec) {
        const u32 r = (u32)(t - ncodes);
        text[rec_off[r + 1] + r] = 1;
    } else if (t == ncodes + nrec) {
        text[t] = 0;
    }
}

void records_assemble(const u8 *d_codes, u64 ncodes, const u64 *d_rec_off, u32 nrec, u32 sigma, u8 *d_text,
                      int *d_err, cudaStream_t st) {
    const u64 threads = ncodes + nrec + 1;
    records_assemble_kernel<<<div_up_u(threads, 256), 256, 0, st>>>(d_codes, ncodes, d_rec_off, nrec, sigma, d_text,
                                                                    d_err);
    KERNEL_CHECK();
}

// key = record of the suffix of row 1 + t (row 0, the global sentinel, belongs to no record), value = its local start
__global__ void __launch_bounds__(256) record_rows_kernel(const u32 *__restrict__ sa, u64 rows,
                                                          const u64 *__restrict__ start, u32 nrec,
                                                          u64 *__restrict__ keys, u32 *__restrict__ vals) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows) return;
    const u32 p = ld_stream_u32(sa + 1 + t);
    const u32 r = record_of(start, nrec, p);
    keys[t] = r;
    vals[t] = (u32)(p - __ldg(start + r));
}

// (pattern, global position) -> key [pattern | record], value = local position
__global__ void __launch_bounds__(256) record_keys_kernel(const u32 *__restrict__ pos, const u64 *__restrict__ pos_off,
                                                          u64 npat, u64 total, const u64 *__restrict__ start, u32 nrec,
                                                          int rbits, u64 *__restrict__ keys, u32 *__restrict__ vals) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    u64 lo = 0, hi = npat;  // largest q with pos_off[q] <= t
    while (hi - lo > 1) {
        const u64 mid = lo + (hi - lo) / 2;
        if (pos_off[mid] <= t) lo = mid;
        else hi = mid;
    }
    const u32 p = pos[t];
    const u32 r = record_of(start, nrec, p);
    keys[t] = (lo << rbits) | r;
    vals[t] = (u32)(p - __ldg(start + r));
}

__global__ void __launch_bounds__(256) record_take_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ vals,
                                                          u64 total, u64 rmask, u32 *__restrict__ rec,
                                                          u32 *__restrict__ local) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    rec[t] = (u32)(keys[t] & rmask);
    local[t] = vals[t];
}

// L'[q] = max(L[q], 1): row 0 (the global sentinel) is no record's row
__global__ void __launch_bounds__(256) record_clamp_kernel(const u32 *__restrict__ L, u64 npat, u32 *__restrict__ out) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < npat) out[t] = max(L[t], 1u);
}

static int bits_for(u64 count) {  // bits of the largest value below `count`
    int b = 0;
    while (count > 1 && (1ull << b) < count) ++b;
    return b;
}

void record_sas(const DeviceIndex &ix, u32 *d_out, cudaStream_t st) {
    const u64 rows = (u64)ix.len - 1;  // = n, the entries of all records' arrays together
    if (!rows) return;
    DevBuf<u64> kA(rows, st), kB(rows, st);
    DevBuf<u32> vA(rows, st), vB(rows, st);
    record_rows_kernel<<<div_up_u(rows, 256), 256, 0, st>>>(ix.sa.ptr, rows, ix.rec_start.ptr, ix.nrec, kA.ptr, vA.ptr);
    KERNEL_CHECK();
    u64 *kb[2] = {kA.ptr, kB.ptr};
    u32 *vb[2] = {vA.ptr, vB.ptr};
    const auto sorted = rs::Sorter<8>::sort(kb, vb, (u32)rows, bits_for(ix.nrec), st);
    // record r's rows, in the global order, are entries start[r] .. start[r + 1] - 1 of the partition
    CUDA_CHECK(cudaMemcpyAsync(d_out, sorted.vals, rows * 4, cudaMemcpyDeviceToDevice, st));
}

void records_clamp_rows(const u32 *d_L, u64 npat, u32 *d_out, cudaStream_t st) {
    if (!npat) return;
    record_clamp_kernel<<<div_up_u(npat, 256), 256, 0, st>>>(d_L, npat, d_out);
    KERNEL_CHECK();
}

void locate_records_group(const DeviceIndex &ix, u64 npat, const u64 *d_pos_off, u64 total, const u32 *d_pos,
                          u32 *d_rec, u32 *d_local, cudaStream_t st) {
    if (!total) return;
    if (total > 0xFFFFFFFFull || npat > 0xFFFFFFFFull)
        throw std::runtime_error("locate_records: more than 2^32 - 1 positions or patterns in one batch");
    const int rbits = bits_for(ix.nrec), qbits = bits_for(npat);
    DevBuf<u64> kA(total, st), kB(total, st);
    DevBuf<u32> vA(total, st), vB(total, st);
    record_keys_kernel<<<div_up_u(total, 256), 256, 0, st>>>(d_pos, d_pos_off, npat, total, ix.rec_start.ptr, ix.nrec,
                                                             rbits, kA.ptr, vA.ptr);
    KERNEL_CHECK();
    u64 *kb[2] = {kA.ptr, kB.ptr};
    u32 *vb[2] = {vA.ptr, vB.ptr};
    const auto sorted = rs::Sorter<8>::sort(kb, vb, (u32)total, qbits + rbits, st);
    record_take_kernel<<<div_up_u(total, 256), 256, 0, st>>>(sorted.keys, sorted.vals, total, (1ull << rbits) - 1ull,
                                                             d_rec, d_local);
    KERNEL_CHECK();
}

}  // namespace b200sa
