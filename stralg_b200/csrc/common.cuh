// common.cuh -- shared helpers for the b200sa kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <cstdlib>
#include <mutex>
#include <stdexcept>
#include <string>

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

namespace b200sa {

struct CudaFailure : public std::runtime_error {
    cudaError_t code;
    CudaFailure(cudaError_t c, const char *what, const char *file, int line)
        : std::runtime_error(std::string(what) + ": " + cudaGetErrorString(c) + " at " + file + ":" +
                             std::to_string(line)),
          code(c) {}
};

#define CUDA_CHECK(expr)                                                          \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) throw ::b200sa::CudaFailure(_e, #expr, __FILE__, __LINE__); \
    } while (0)

// every kernel launch of the library is counted (b200sa_launch_count, bench.py "gpu_launches")
extern unsigned long long g_kernel_launches;
#define KERNEL_CHECK()                      \
    do {                                    \
        ++::b200sa::g_kernel_launches;      \
        CUDA_CHECK(cudaGetLastError());     \
    } while (0)

// exact-size cache of large device blocks (api.cu); get throws CudaFailure when the device is out of memory
// the library's own stream-ordered memory pool of the current device (api.cu): freed blocks are kept
// (release threshold "never"), and the process's default pool -- shared with every other
// cudaMallocAsync user, e.g. torch's async allocator -- is left alone
cudaMemPool_t library_pool();
void *output_cache_get(size_t bytes);
void output_cache_put(void *ptr, size_t bytes);
void output_cache_purge(int device);

// Stream-ordered device buffer from the library's own pool, which keeps freed blocks (release
// threshold "never", api.cu), so steady-state builds do not pay cudaMalloc.
template <typename T>
struct DevBuf {
    T *ptr = nullptr;
    size_t count = 0;
    cudaStream_t stream = 0;
    bool cached = false;
    DevBuf() {}
    DevBuf(size_t n, cudaStream_t s) { alloc(n, s); }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : ptr(o.ptr), count(o.count), stream(o.stream), cached(o.cached) {
        o.ptr = nullptr;
        o.count = 0;
        o.cached = false;
    }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) {
            release();
            ptr = o.ptr; count = o.count; stream = o.stream; cached = o.cached;
            o.ptr = nullptr; o.count = 0; o.cached = false;
        }
        return *this;
    }
    void alloc(size_t n, cudaStream_t s) {
        release();
        stream = s;
        count = n;
        if (n) CUDA_CHECK(cudaMallocFromPoolAsync((void **)&ptr, n * sizeof(T), library_pool(), s));
    }
    // For the large tables an index OWNS (SA, BWT, O, ISA, LCP ...): blocks come from an exact-size
    // cache of plain device allocations (output_cache_get / _put, api.cu) instead of the
    // stream-ordered pool.  The pool reuses freed memory well only while the same sequence of
    // requests repeats; a caller that keeps one index alive while the next is built (transfer of
    // one result next to the construction of the next) breaks that sequence, and the pool then maps
    // gigabytes of fresh memory in the middle of a build.  Exact sizes repeat from build to build.
    void alloc_output(size_t n, cudaStream_t s) {
        release();
        stream = s;
        count = n;
        if (n * sizeof(T) < ((size_t)1 << 20)) {  // small tables: the pool is fine
            if (n) CUDA_CHECK(cudaMallocFromPoolAsync((void **)&ptr, n * sizeof(T), library_pool(), s));
        } else {
            ptr = (T *)output_cache_get(n * sizeof(T));
            cached = true;
        }
    }
    void release() {
        if (ptr) {
            if (cached) {
                cudaStreamSynchronize(stream);  // an index is released by its owner: its work is done
                output_cache_put(ptr, count * sizeof(T));
            } else {
                cudaFreeAsync(ptr, stream);
            }
        }
        ptr = nullptr;
        count = 0;
        cached = false;
    }
    T *detach() {
        T *p = ptr;
        ptr = nullptr;
        count = 0;
        cached = false;
        return p;
    }
    ~DevBuf() { release(); }
    size_t bytes() const { return count * sizeof(T); }
};

// Build workspace: a few large device allocations that persist across builds (per device) and
// are carved with a bump pointer, so a steady-state build issues no cudaMalloc at all and the
// driver never has to re-map physical pages between differently sized requests.
// cudaMalloc that gives the cached output blocks back before it reports out-of-memory
static inline void *malloc_or_purge(size_t bytes) {
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        int device = 0;
        cudaGetDevice(&device);
        output_cache_purge(device);
        e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) throw CudaFailure(e, "cudaMalloc", __FILE__, __LINE__);
    return p;
}

struct Arena {
    struct Chunk {
        u8 *base;
        size_t cap, top;
    };
    static const int MAX_CHUNKS = 16;
    Chunk chunks[MAX_CHUNKS];
    int nchunks = 0;
    void reset() {
        for (int i = 0; i < nchunks; ++i) chunks[i].top = 0;
    }
    // make sure the FIRST chunk can hold `bytes` (called before anything is carved)
    void reserve_first(size_t bytes) {
        bytes = (bytes + ((size_t)64 << 20)) & ~(((size_t)1 << 20) - 1);
        if (nchunks > 0 && chunks[0].cap >= bytes) return;
        release_chunks();  // (the side buffer may already hold the staged text of this build)
        u8 *p = (u8 *)malloc_or_purge(bytes);
        chunks[0] = Chunk{p, bytes, 0};
        nchunks = 1;
    }
    void *alloc(size_t bytes) {
        bytes = (bytes + 511) & ~(size_t)511;
        for (int i = 0; i < nchunks; ++i)
            if (chunks[i].top + bytes <= chunks[i].cap) {
                void *p = chunks[i].base + chunks[i].top;
                chunks[i].top += bytes;
                return p;
            }
        if (nchunks == MAX_CHUNKS) throw std::runtime_error("workspace arena exhausted");
        size_t cap = (bytes + ((size_t)256 << 20)) & ~(((size_t)1 << 20) - 1);
        u8 *p = (u8 *)malloc_or_purge(cap);
        chunks[nchunks] = Chunk{p, cap, bytes};
        return chunks[nchunks++].base;
    }
    template <typename T>
    T *get(size_t count) { return (T *)alloc(count * sizeof(T)); }
    // would alloc(bytes) succeed -- in a chunk that exists, or in a new one with `margin` bytes of device memory
    // to spare?  (optional buffers of a build are dropped instead of running the device out of memory)
    bool can_fit(size_t bytes, size_t margin) const {
        bytes = (bytes + 511) & ~(size_t)511;
        for (int i = 0; i < nchunks; ++i)
            if (chunks[i].top + bytes <= chunks[i].cap) return true;
        if (nchunks == MAX_CHUNKS) return false;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return false;
        return free_b >= bytes + ((size_t)256 << 20) + margin;
    }
    struct Mark {
        size_t tops[MAX_CHUNKS];
        int n;
    };
    Mark mark() const {
        Mark m;
        m.n = nchunks;
        for (int i = 0; i < nchunks; ++i) m.tops[i] = chunks[i].top;
        return m;
    }
    void release_to(const Mark &m) {
        for (int i = 0; i < nchunks; ++i) chunks[i].top = i < m.n ? m.tops[i] : 0;
    }
    // grow-only side buffer (staging of a host text): kept out of the stream-ordered pool so that
    // the pool only ever sees the same sequence of output allocations, build after build
    u8 *side = nullptr;
    size_t side_cap = 0;
    void *side_alloc(size_t bytes) {
        if (bytes > side_cap) {
            if (side) {
                cudaDeviceSynchronize();
                cudaFree(side);
                side = nullptr;
                side_cap = 0;
            }
            size_t cap = (bytes + ((size_t)1 << 20)) & ~(((size_t)1 << 20) - 1);
            side = (u8 *)malloc_or_purge(cap);
            side_cap = cap;
        }
        return side;
    }
    void release_chunks() {
        if (nchunks) cudaDeviceSynchronize();
        for (int i = 0; i < nchunks; ++i) cudaFree(chunks[i].base);
        nchunks = 0;
    }
    void release_all() {
        release_chunks();
        if (side) cudaDeviceSynchronize();
        if (side) cudaFree(side);
        side = nullptr;
        side_cap = 0;
    }
    size_t reserved() const {
        size_t t = 0;
        for (int i = 0; i < nchunks; ++i) t += chunks[i].cap;
        return t + side_cap;
    }
};

static inline unsigned div_up_u(u64 a, u64 b) { return (unsigned)((a + b - 1) / b); }

// integer value of environment variable `name`; `dflt` when it is unset or empty
static inline int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// cudaFuncSetAttribute (the opt-in for more than 48 KB of dynamic shared memory) is per device, i.e.
// per context: a process that builds on several devices has to repeat it on each one.  first()
// is true exactly once per CUDA device (the current one when `device` < 0).
struct PerDeviceOnce {
    bool done[64] = {};
    std::mutex mu;
    bool first(int device = -1) {
        if (device < 0) CUDA_CHECK(cudaGetDevice(&device));
        std::lock_guard<std::mutex> lock(mu);
        bool &d = done[device & 63];
        if (d) return false;
        d = true;
        return true;
    }
};

// Small device-to-host read-back (<= 4 KB, a multiple of 4 bytes) that stays off the copy engines: a
// one-warp kernel stores the words into mapped pinned host memory, the stream is synchronised, the
// words are handed to `dst`.  The copy engines serve transfers in submission order, so a build that
// runs next to a multi-gigabyte device-to-host transfer (b200sa_copy_async) would otherwise wait
// for it every time it looks at a counter.  Defined in api.cu.
void read_back(void *dst, const void *dev_src, size_t bytes, cudaStream_t st);

// packed symbol t (its code - 1) of the big-endian packed text
__device__ __forceinline__ u32 sym_at(const u64 *__restrict__ packed, u32 t, int bits) {
    u64 bitpos = (u64)t * bits;
    return (u32)((packed[bitpos >> 6] >> (64 - bits - (unsigned)(bitpos & 63))) & ((1u << bits) - 1u));
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// streaming (read-once) loads/stores: keep them out of L1
__device__ __forceinline__ u64 ld_stream_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ u32 ld_stream_u32(const u32 *p) {
    u32 v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream_u128(const void *p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p));
    return v;
}

__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(u64 *p, u64 v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// bulk prefetch of [src, src + bytes) into L2 (bytes: multiple of 16, src 16-byte aligned)
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, u32 bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// ---- mbarrier + bulk asynchronous copy (TMA engine, 1-D) : global -> shared ----------------
__device__ __forceinline__ u32 smem_addr_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 arrivals) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(u64 *bar, u32 parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra MBAR_DONE;\n"
        "bra MBAR_WAIT;\n"
        "MBAR_DONE:\n"
        "}" ::"r"(smem_addr_u32(bar)), "r"(parity) : "memory");
}
// bytes: multiple of 16; dst and src 16-byte aligned; completion is signalled on `bar`
__device__ __forceinline__ void bulk_copy_g2s(void *dst, const void *src, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr_u32(bar))
                 : "memory");
}

// Per-stage device timing (optional; enabled with B200SA_PROFILE).
struct StageTimer {
    static const int MAX = 1024;
    cudaEvent_t ev[MAX][2];
    const char *name[MAX];
    double bytes[MAX];
    int n = 0;
    bool on = false;
    cudaStream_t stream = 0;
    void enable(cudaStream_t s) { on = true; stream = s; }
    int begin(const char *nm, double algorithmic_bytes) {
        if (!on || n >= MAX) return -1;
        cudaEventCreate(&ev[n][0]);
        cudaEventCreate(&ev[n][1]);
        name[n] = nm;
        bytes[n] = algorithmic_bytes;
        cudaEventRecord(ev[n][0], stream);
        return n++;
    }
    void end(int id) {
        if (id >= 0) cudaEventRecord(ev[id][1], stream);
    }
    void clear() {
        for (int i = 0; i < n; ++i) {
            cudaEventDestroy(ev[i][0]);
            cudaEventDestroy(ev[i][1]);
        }
        n = 0;
    }
};

}  // namespace b200sa
