// api.cu -- the C ABI declared in include/b200sa.h.
#include "../../include/b200sa.h"
#include "engine.h"
#include "round0_msd.cuh"

#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string.h>
#include <algorithm>
#include <type_traits>
#include <atomic>
#include <chrono>
#include <vector>

using namespace b200sa;

struct b200sa_index {
    DeviceIndex ix;
    uint32_t flags = 0;
    float prof_ms[StageTimer::MAX];
    const char *prof_name[StageTimer::MAX];
    double prof_bytes[StageTimer::MAX];
    int prof_n = 0;
};

namespace b200sa { unsigned long long g_kernel_launches = 0; }

static thread_local std::string g_last_error;

static int fail(enum b200sa_error code, const std::string &msg, enum b200sa_error *err) {
    g_last_error = msg;
    if (err) *err = code;
    return (int)code;
}
static int ok(enum b200sa_error *err) {
    if (err) *err = B200SA_OK;
    return 0;
}

static enum b200sa_error code_of(cudaError_t e) {
    return e == cudaErrorMemoryAllocation ? B200SA_ERR_OUT_OF_MEMORY : B200SA_ERR_CUDA;
}

// Runs `body`, which returns 0 or a code it has reported through fail(), and turns what it throws into the
// entry point's error code.  (A template, not std::function: the one-pattern search is a microsecond path.)
template <class F>
static int guarded(enum b200sa_error *err, F &&body) {
    try {
        return body();
    } catch (const CudaFailure &e) {
        cudaGetLastError();
        return fail(code_of(e.code), e.what(), err);
    } catch (const std::bad_alloc &) {
        return fail(B200SA_ERR_OUT_OF_MEMORY, "host allocation failed", err);
    } catch (const std::invalid_argument &e) {  // (a malformed index file)
        return fail(B200SA_ERR_BAD_ARGUMENT, e.what(), err);
    } catch (const std::exception &e) {
        return fail(B200SA_ERR_INTERNAL, e.what(), err);
    }
}

// The pointer-returning entry points: a new T filled by `fill(T *)` under guarded().  On any error the object
// is freed and the result is nullptr; on success `err` is written with B200SA_OK.
template <class T, class F>
static T *new_handle(enum b200sa_error *err, F &&fill) {
    T *h = new (std::nothrow) T();
    if (!h) {
        fail(B200SA_ERR_OUT_OF_MEMORY, "host allocation failed", err);
        return nullptr;
    }
    if (guarded(err, [&] { return fill(h); }) != 0) {
        if constexpr (std::is_same<T, b200sa_index>::value) b200sa_free(h);  // (frees its tables on its device)
        else delete h;
        return nullptr;
    }
    ok(err);
    return h;
}

namespace b200sa {
__global__ void read_back_kernel(const u32 *__restrict__ src, u32 *__restrict__ dst, u32 words) {
    for (u32 i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
}
namespace {
// One buffer of mapped pinned memory per host thread and device (0 <= device < 64), allocated on first use:
// read_back uses its first 4 KB, the small-batch search (b200sa_search_batch) all 8 KB.
const size_t kStagingBytes = 8192;
struct MappedStaging {
    u8 *host[64] = {};
    u8 *dev[64] = {};
    ~MappedStaging() {
        for (auto p : host)
            if (p) cudaFreeHost(p);
    }
};
thread_local MappedStaging t_staging;
}  // namespace
static void mapped_staging(int device, u8 *&host, u8 *&dev) {
    MappedStaging &ms = t_staging;
    if (!ms.host[device]) {
        CUDA_CHECK(cudaHostAlloc((void **)&ms.host[device], kStagingBytes, cudaHostAllocMapped));
        CUDA_CHECK(cudaHostGetDevicePointer((void **)&ms.dev[device], ms.host[device], 0));
    }
    host = ms.host[device];
    dev = ms.dev[device];
}
void read_back(void *dst, const void *dev_src, size_t bytes, cudaStream_t st) {
    int device = 0;
    CUDA_CHECK(cudaGetDevice(&device));
    if (bytes > 4096 || (bytes & 3) || device < 0 || device >= 64) {  // not a mailbox case: plain copy
        CUDA_CHECK(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        return;
    }
    u8 *host, *dev;
    mapped_staging(device, host, dev);
    read_back_kernel<<<1, 64, 0, st>>>((const u32 *)dev_src, (u32 *)dev, (u32)(bytes / 4));
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(st));
    memcpy(dst, host, bytes);
}
}  // namespace b200sa

namespace b200sa {
namespace {
std::mutex g_cache_mu;
std::multimap<std::pair<int, size_t>, void *> g_cache;  // (device, bytes) -> free block
}  // namespace
void *output_cache_get(size_t bytes) {
    int device = 0;
    CUDA_CHECK(cudaGetDevice(&device));
    {
        std::lock_guard<std::mutex> lock(g_cache_mu);
        auto it = g_cache.find({device, bytes});
        if (it != g_cache.end()) {
            void *p = it->second;
            g_cache.erase(it);
            return p;
        }
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaErrorMemoryAllocation) {  // give the cached blocks back and try once more
        cudaGetLastError();
        output_cache_purge(device);
        e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) throw CudaFailure(e, "cudaMalloc (output table)", __FILE__, __LINE__);
    return p;
}
void output_cache_put(void *ptr, size_t bytes) {
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) == cudaSuccess) device = at.device;
    std::lock_guard<std::mutex> lock(g_cache_mu);
    // keep at most two blocks of a size (one index alive + one being built) and 40 GB per device; the
    // rest goes back to the driver
    size_t held = 0;
    for (auto &kv : g_cache)
        if (kv.first.first == device) held += kv.first.second;
    if (g_cache.count({device, bytes}) >= 2 || held + bytes > ((size_t)40 << 30)) {
        cudaFree(ptr);
        return;
    }
    g_cache.insert({{device, bytes}, ptr});
}
void output_cache_purge(int device) {
    std::lock_guard<std::mutex> lock(g_cache_mu);
    for (auto it = g_cache.begin(); it != g_cache.end();) {
        if (it->first.first == device) {
            cudaFree(it->second);
            it = g_cache.erase(it);
        } else {
            ++it;
        }
    }
}
}  // namespace b200sa

static Arena g_arena[64];
static std::mutex g_arena_mu[64];

namespace b200sa {
namespace {
std::mutex g_pool_mu;
cudaMemPool_t g_pool[64] = {};
}  // namespace
cudaMemPool_t library_pool() {
    int device = 0;
    CUDA_CHECK(cudaGetDevice(&device));
    std::lock_guard<std::mutex> lock(g_pool_mu);
    cudaMemPool_t &p = g_pool[device & 63];
    if (!p) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        CUDA_CHECK(cudaMemPoolCreate(&p, &props));
        uint64_t never = UINT64_MAX;
        CUDA_CHECK(cudaMemPoolSetAttribute(p, cudaMemPoolAttrReleaseThreshold, &never));
    }
    return p;
}
}  // namespace b200sa

// Restores the caller's current device when an entry point returns (ADVICE r1: the library must not
// silently switch the device of the process that hosts it).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            cudaGetLastError();
            prev = -1;
        }
        CUDA_CHECK(cudaSetDevice(device));
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Per-device staging for the host-buffer search entry points: two non-blocking streams and grow-only
// device buffers, created once -- a call costs no cudaMalloc / stream creation in the steady state.
struct SearchLanes {
    std::mutex mu;
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t ready = nullptr;
    u8 *patterns = nullptr;
    size_t pat_cap = 0;
    u32 *L = nullptr, *R = nullptr;
    size_t lr_cap = 0;
    void reserve(size_t pat_bytes, size_t npat) {
        if (!s[0]) {
            CUDA_CHECK(cudaStreamCreateWithFlags(&s[0], cudaStreamNonBlocking));
            CUDA_CHECK(cudaStreamCreateWithFlags(&s[1], cudaStreamNonBlocking));
            CUDA_CHECK(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
        }
        if (pat_bytes > pat_cap) {
            if (patterns) CUDA_CHECK(cudaFree(patterns));
            patterns = nullptr;
            pat_cap = (pat_bytes + ((size_t)1 << 20)) & ~(((size_t)1 << 20) - 1);
            patterns = (u8 *)malloc_or_purge(pat_cap);
        }
        if (npat > lr_cap) {
            if (L) CUDA_CHECK(cudaFree(L));
            if (R) CUDA_CHECK(cudaFree(R));
            L = R = nullptr;
            lr_cap = (npat + 4095) & ~(size_t)4095;
            L = (u32 *)malloc_or_purge(lr_cap * 4);
            R = (u32 *)malloc_or_purge(lr_cap * 4);
        }
    }
    void release() {
        if (patterns) cudaFree(patterns);
        if (L) cudaFree(L);
        if (R) cudaFree(R);
        patterns = nullptr;
        L = R = nullptr;
        pat_cap = lr_cap = 0;
    }
};
static SearchLanes g_lanes[64];
static SearchLanes &search_lanes(int device) { return g_lanes[device & 63]; }

// Runs `search(d_counters)`.  With `counts`, the kernel counts its traffic into four zeroed device counters,
// which are read back into `counts`; without, d_counters is null.
template <class Search>
static void count_traffic(uint64_t *counts, cudaStream_t st, Search &&search) {
    if (!counts) return search(nullptr);
    DevBuf<unsigned long long> d(4, st);
    CUDA_CHECK(cudaMemsetAsync(d.ptr, 0, 4 * sizeof(unsigned long long), st));
    search(d.ptr);
    unsigned long long h[4];
    CUDA_CHECK(cudaMemcpyAsync(h, d.ptr, sizeof h, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    for (int i = 0; i < 4; ++i) counts[i] = h[i];
}

// The pipeline of the host-buffer searches: the batch is cut into pieces that alternate between the device's
// two lanes, so that while the kernel of one piece runs the next piece's patterns cross PCIe and the previous
// piece's (L, R) return (pinned host memory makes the copies truly asynchronous; pageable memory still works,
// staged by the driver).  Pieces hold about `piece_bytes` of patterns and start at multiples of 8 patterns.
// `piece(q0, q1, lane, d_patterns, d_L, d_R)` copies the patterns of [q0, q1) in on `lane` and searches them
// into d_L / d_R (the piece's slices); the lanes first wait for the work `st` holds.
template <class Piece>
static void search_pieces(int device, cudaStream_t st, uint64_t npat, uint64_t total, uint64_t piece_bytes, uint32_t *L,
                          uint32_t *R, Piece &&piece) {
    SearchLanes &ln = search_lanes(device);
    std::lock_guard<std::mutex> lock(ln.mu);
    ln.reserve(total + 16, npat);
    uint64_t per = npat;
    if (total > 2 * piece_bytes) {
        const uint64_t avg = std::max<uint64_t>(1, total / npat);
        per = std::max<uint64_t>(1024, (piece_bytes / avg) & ~(uint64_t)7);
    }
    CUDA_CHECK(cudaEventRecord(ln.ready, st));
    CUDA_CHECK(cudaStreamWaitEvent(ln.s[0], ln.ready, 0));
    CUDA_CHECK(cudaStreamWaitEvent(ln.s[1], ln.ready, 0));
    uint64_t k = 0;
    for (uint64_t q0 = 0; q0 < npat; q0 += per, ++k) {
        const uint64_t q1 = std::min(npat, q0 + per);
        cudaStream_t ls = ln.s[k & 1];
        piece(q0, q1, ls, ln.patterns, ln.L + q0, ln.R + q0);
        CUDA_CHECK(cudaMemcpyAsync(L + q0, ln.L + q0, (q1 - q0) * 4, cudaMemcpyDeviceToHost, ls));
        CUDA_CHECK(cudaMemcpyAsync(R + q0, ln.R + q0, (q1 - q0) * 4, cudaMemcpyDeviceToHost, ls));
    }
    CUDA_CHECK(cudaStreamSynchronize(ln.s[0]));
    CUDA_CHECK(cudaStreamSynchronize(ln.s[1]));
}

// ---- native index file ---------------------------------------------------------------------------
// [header][section]*: the header carries the scalars, every section is {tag, element size, count}
// + the raw device array, padded to 8 bytes.  Host-endian like the reference's own dumps
// (suffix_array.c:238-241); `endian` lets a reader on the other byte order refuse the file.
namespace {
struct IndexFileHeader {
    char magic[8];          // "B200SAIX"
    uint32_t version;       // 1
    uint32_t endian;        // 0x01020304 as written by the producer
    uint64_t n;
    uint32_t sigma, primary;
    uint32_t occ_layout, occ_block_bytes;
    uint64_t occ_blocks;
    uint32_t ktable_k, ssa_rate;
    uint32_t flags, nsections;
    uint32_t pack_bits, reserved;
    uint32_t c_table[256];
    uint64_t sym_counts[256];
    BuildStats stats;
};
struct SectionHeader {
    char tag[8];
    uint64_t elem_bytes, count;
};
const size_t kIoChunk = (size_t)64 << 20;

struct CloseFile {
    void operator()(FILE *f) const { fclose(f); }
};
using File = std::unique_ptr<FILE, CloseFile>;

struct Section {
    const char *tag;
    const void *dptr;
    size_t elem, count;
};

void write_section(FILE *f, const Section &sc, std::vector<char> &buf, cudaStream_t st) {
    SectionHeader sh{};
    strncpy(sh.tag, sc.tag, 8);
    sh.elem_bytes = sc.elem;
    sh.count = sc.count;
    if (fwrite(&sh, sizeof sh, 1, f) != 1) throw std::runtime_error("index file: short write");
    const size_t bytes = sc.elem * sc.count;
    for (size_t at = 0; at < bytes; at += kIoChunk) {
        const size_t k = std::min(kIoChunk, bytes - at);
        CUDA_CHECK(cudaMemcpyAsync(buf.data(), (const char *)sc.dptr + at, k, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        if (fwrite(buf.data(), 1, k, f) != k) throw std::runtime_error("index file: short write");
    }
    const char zeros[8] = {0};
    if (bytes % 8 && fwrite(zeros, 1, 8 - bytes % 8, f) != 8 - bytes % 8) throw std::runtime_error("index file: short write");
}

template <typename T>
void read_section(FILE *f, const SectionHeader &sh, DevBuf<T> &dst, size_t expect_count, std::vector<char> &buf,
                  cudaStream_t st) {
    if (sh.elem_bytes != sizeof(T) || sh.count != expect_count)
        throw std::runtime_error(std::string("index file: section ") + std::string(sh.tag, strnlen(sh.tag, 8)) +
                                 " has an unexpected shape");
    dst.alloc(sh.count, st);
    const size_t bytes = sh.elem_bytes * sh.count;
    for (size_t at = 0; at < bytes; at += kIoChunk) {
        const size_t k = std::min(kIoChunk, bytes - at);
        if (fread(buf.data(), 1, k, f) != k) throw std::runtime_error("index file: truncated section");
        CUDA_CHECK(cudaMemcpyAsync((char *)dst.ptr + at, buf.data(), k, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
    if (bytes % 8 && fseek(f, (long)(8 - bytes % 8), SEEK_CUR) != 0) throw std::runtime_error("index file: truncated section");
}
}  // namespace

static int needs_o_table(const DeviceIndex &ix, enum b200sa_error *err = nullptr) {
    if (ix.occ_layout != OCC_NONE) return 0;
    return fail(B200SA_ERR_NOT_BUILT, "O table was not requested at build time", err);
}

static bool can_locate(const b200sa_index *idx) {
    return idx->ix.sa.ptr || (idx->ix.ssa_rate && idx->ix.occ_layout != OCC_NONE);
}
// positions through the full suffix array when it is resident, else through the sampled one
static void locate_fill_any(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, const u64 *d_pos_off,
                            u64 total, u32 *d_pos, cudaStream_t st) {
    const bool force_ssa = getenv("B200SA_LOCATE_SAMPLED") != nullptr;  // measurement aid (bench.py)
    if (ix.sa.ptr && !(force_ssa && ix.ssa_rate)) fm_locate_fill(ix, d_L, d_R, npat, d_pos_off, total, d_pos, st);
    else fm_locate_fill_ssa(ix, d_L, npat, d_pos_off, total, d_pos, st);
}

template <typename T>
static void replicate_buf(const DevBuf<T> &src, int src_dev, DevBuf<T> &dst, int dst_dev, cudaStream_t st, bool output) {
    if (!src.ptr) return;
    if (output) dst.alloc_output(src.count, st);
    else dst.alloc(src.count, st);
    CUDA_CHECK(cudaMemcpyPeerAsync(dst.ptr, dst_dev, src.ptr, src_dev, src.count * sizeof(T), st));
}

// device bytes from cudaMalloc, freed with cudaFree (which waits for the device) when released or destroyed
struct DeviceBytes {
    u8 *ptr = nullptr;
    void alloc(size_t bytes) { ptr = (u8 *)malloc_or_purge(bytes); }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
    }
    ~DeviceBytes() { release(); }
};

// records index (records.cu): the host offsets and the device record starts start[r] = rec_off[r] + r
static void set_records(DeviceIndex &ix, const std::vector<u64> &rec_off, cudaStream_t st) {
    ix.nrec = (u32)(rec_off.size() - 1);
    ix.rec_off = rec_off;
    std::vector<u64> start(rec_off.size());
    for (size_t r = 0; r < rec_off.size(); ++r) start[r] = rec_off[r] + r;
    ix.rec_start.alloc(start.size(), st);
    CUDA_CHECK(cudaMemcpyAsync(ix.rec_start.ptr, start.data(), start.size() * 8, cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaStreamSynchronize(st));  // (`start` is pageable host memory)
}

// a pattern of a host batch that holds the separator (code 1) of a records index
static bool holds_separator(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                            uint64_t npat) {
    if (!idx->ix.nrec || !npat) return false;
    const uint64_t b0 = offsets ? offsets[0] : 0, b1 = offsets ? offsets[npat] : (uint64_t)fixed_len * npat;
    return b1 > b0 && memchr(patterns + b0, 1, (size_t)(b1 - b0)) != nullptr;
}

// The refusals of a host batch's pattern lengths: offsets that decrease, then a pattern longer than `limit` symbols
// (B200SA_ERR_TOO_LARGE with `msg`); max_m gets the longest pattern.
static int pattern_lengths_ok(const uint64_t *offsets, uint32_t fixed_len, uint64_t npat, uint64_t limit,
                              const std::string &msg, uint32_t &max_m, enum b200sa_error *err) {
    uint64_t longest = offsets ? 0 : fixed_len;
    if (offsets)
        for (uint64_t q = 0; q < npat; ++q) {
            if (offsets[q + 1] < offsets[q]) return fail(B200SA_ERR_BAD_ARGUMENT, "pattern offsets must not decrease", err);
            longest = std::max(longest, offsets[q + 1] - offsets[q]);
        }
    if (longest > limit) return fail(B200SA_ERR_TOO_LARGE, msg, err);
    max_m = (uint32_t)longest;
    return 0;
}

// A piece's n results, one device column per host vector, appended after the `base` results of the earlier pieces
// (asynchronous on st)
struct Column {
    std::vector<uint32_t> &host;
    const u32 *dev;
};
static void append_columns(uint64_t base, uint64_t n, std::initializer_list<Column> cols, cudaStream_t st) {
    for (const Column &c : cols) {
        c.host.resize(base + n);
        if (n) CUDA_CHECK(cudaMemcpyAsync(c.host.data() + base, c.dev, n * 4, cudaMemcpyDeviceToHost, st));
    }
}

// ---- the text of a build or an extension: staged, packed with its bad-symbol check, kept for TEXTCMP ----
static size_t packed_words(const DeviceIndex &ix) { return ((size_t)ix.len + ix.pk.cpw - 1) / ix.pk.cpw + 4; }

// the caller's device text as given, or the host text copied into the arena's side buffer (text[n] = 0)
static void stage_text(DeviceIndex &ix, Arena &arena, const uint8_t *codes, uint32_t flags) {
    if (flags & B200SA_TEXT_ON_DEVICE) {
        ix.text_ptr = codes;
        return;
    }
    u8 *stage = (u8 *)arena.side_alloc((size_t)ix.n + 1);
    if (ix.n) CUDA_CHECK(cudaMemcpyAsync(stage, codes, ix.n, cudaMemcpyHostToDevice, ix.stream));
    CUDA_CHECK(cudaMemsetAsync(stage + ix.n, 0, 1, ix.stream));
    ix.text_ptr = stage;
}

// pack_text; false when the text holds a code outside 1..sigma-1
static bool pack_text_checked(DeviceIndex &ix) {
    DevBuf<int> d_err(1, ix.stream);
    CUDA_CHECK(cudaMemsetAsync(d_err.ptr, 0, 4, ix.stream));
    pack_text(ix, d_err.ptr);
    int herr = 0;
    read_back(&herr, d_err.ptr, 4, ix.stream);
    return herr == 0;
}

static void keep_packed_text(DeviceIndex &ix) {
    const size_t words = packed_words(ix);
    ix.text_packed.alloc_output(words, ix.stream);
    CUDA_CHECK(cudaMemcpyAsync(ix.text_packed.ptr, ix.packed, words * 8, cudaMemcpyDeviceToDevice, ix.stream));
}

#pragma GCC visibility push(default)
extern "C" {

const char *b200sa_last_error(void) { return g_last_error.c_str(); }

int b200sa_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// (called under guarded(): throws on a CUDA failure)
static int build_into(b200sa_index *h, const uint8_t *codes, uint64_t n, uint32_t sigma, uint32_t flags, int device,
                      void *stream, enum b200sa_error *err) {
    DeviceGuard guard(device);
    DeviceIndex &ix = h->ix;
    ix.stream = (cudaStream_t)stream;
    ix.device = device;
    ix.n = (u32)n;
    ix.len = (u32)n + 1;
    ix.sigma = sigma;
    ix.pk = packing_for_sigma(sigma);
    h->flags = flags;
    cudaStream_t st = ix.stream;
    if (flags & B200SA_PROFILE) ix.timer.enable(st);

    // one build at a time per device: the workspace arena is shared and persistent
    std::lock_guard<std::mutex> arena_lock(g_arena_mu[device & 63]);
    Arena &arena = g_arena[device & 63];
    stage_text(ix, arena, codes, flags);
    arena.reset();
    arena.reserve_first(build_workspace_estimate(ix.len, ix.pk.bits));
    ix.arena = &arena;

    if (!pack_text_checked(ix)) {
        ix.arena = nullptr;
        return fail(B200SA_ERR_BAD_SYMBOL, "text holds a code outside 1..sigma-1", err);
    }
    ix.text.release();  // everything downstream reads the packed text
    ix.text_ptr = nullptr;

    const bool want_tables = flags & (B200SA_BUILD_OCC | B200SA_BUILD_BWT);
    Arena::Mark after_pack = arena.mark();
    build_suffix_array(ix, want_tables);
    arena.release_to(after_pack);  // the sort workspace is dead; LCP reuses it (same stream)
    if (flags & (B200SA_BUILD_ISA | B200SA_BUILD_TEXTCMP)) build_inverse(ix);
    if (flags & B200SA_BUILD_LCP) build_lcp(ix);
    if (flags & B200SA_BUILD_OCC) build_bwt_tables(ix, flags & B200SA_BUILD_BWT);
    if (flags & B200SA_BUILD_TEXTCMP) keep_packed_text(ix);
    ix.packed = nullptr;
    ix.arena = nullptr;
    if ((flags & B200SA_BUILD_KTABLE) && (flags & B200SA_BUILD_OCC)) build_ktable(ix);
    if ((flags & B200SA_DROP_SA) && !(flags & B200SA_BUILD_TEXTCMP)) ix.sa.release();
    CUDA_CHECK(cudaStreamSynchronize(st));
    if (flags & B200SA_PROFILE) {
        h->prof_n = ix.timer.n;
        for (int i = 0; i < ix.timer.n; ++i) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ix.timer.ev[i][0], ix.timer.ev[i][1]);
            h->prof_ms[i] = ms;
            h->prof_name[i] = ix.timer.name[i];
            h->prof_bytes[i] = ix.timer.bytes[i];
        }
        ix.timer.clear();
    }
    return 0;
}

b200sa_index *b200sa_build(const uint8_t *codes, uint64_t n, uint32_t sigma, uint32_t flags, int device,
                           void *stream, enum b200sa_error *err) {
    if ((!codes && n) || sigma < 1 || sigma > 256) {
        fail(B200SA_ERR_BAD_ARGUMENT, "bad text pointer or sigma outside 1..256", err);
        return nullptr;
    }
    if (n > 0xFFFFFFFEull) {
        fail(B200SA_ERR_TOO_LARGE, "n exceeds 2^32 - 2 (uint32 suffix arrays, suffix_array.h:10-20)", err);
        return nullptr;
    }
    return new_handle<b200sa_index>(
        err, [&](b200sa_index *h) { return build_into(h, codes, n, sigma, flags, device, stream, err); });
}

b200sa_index *b200sa_build_records(const uint8_t *codes, const uint64_t *rec_off, uint32_t nrec, uint32_t sigma,
                                   uint32_t flags, int device, void *stream, enum b200sa_error *err) {
    const uint32_t accepted = B200SA_BUILD_OCC | B200SA_BUILD_TEXTCMP | B200SA_BUILD_KTABLE | B200SA_DROP_SA |
                              B200SA_PROFILE | B200SA_TEXT_ON_DEVICE;
    if (!rec_off || nrec == 0 || sigma < 3 || sigma > 256 || (flags & ~accepted)) {
        fail(B200SA_ERR_BAD_ARGUMENT,
             "b200sa_build_records: null offsets, no record, sigma outside 3..256, or a flag other than OCC, TEXTCMP, "
             "KTABLE, DROP_SA, PROFILE, TEXT_ON_DEVICE (per-record ISA, LCP and BWT do not exist)", err);
        return nullptr;
    }
    if (rec_off[0] != 0) {
        fail(B200SA_ERR_BAD_ARGUMENT, "b200sa_build_records: rec_off[0] must be 0", err);
        return nullptr;
    }
    for (uint32_t r = 0; r < nrec; ++r)
        if (rec_off[r + 1] < rec_off[r]) {
            fail(B200SA_ERR_BAD_ARGUMENT, "b200sa_build_records: record offsets decrease", err);
            return nullptr;
        }
    const uint64_t ncodes = rec_off[nrec];
    if (!codes && ncodes) {
        fail(B200SA_ERR_BAD_ARGUMENT, "b200sa_build_records: null codes", err);
        return nullptr;
    }
    if (ncodes > 0xFFFFFFFEull || ncodes + nrec > 0xFFFFFFFEull) {
        fail(B200SA_ERR_TOO_LARGE, "records and separators exceed 2^32 - 2 symbols (uint32 suffix arrays)", err);
        return nullptr;
    }
    const uint64_t n = ncodes + nrec;
    return new_handle<b200sa_index>(err, [&](b200sa_index *h) {
        DeviceGuard guard(device);
        cudaStream_t st = (cudaStream_t)stream;
        const std::vector<u64> off(rec_off, rec_off + nrec + 1);
        // The text with separators, assembled on the device; it then takes the path of any other text.  The two
        // byte buffers are plain allocations given back to the driver as soon as they are dead (the staged records
        // right after the assembly), not blocks of the library's pool, which keeps what it is given.
        DeviceBytes text, staged;
        text.alloc(n + 1);
        DevBuf<u64> d_off(nrec + 1, st);
        DevBuf<int> d_err(1, st);
        const u8 *d_codes = codes;
        if (!(flags & B200SA_TEXT_ON_DEVICE)) {
            staged.alloc(ncodes ? ncodes : 1);
            if (ncodes) CUDA_CHECK(cudaMemcpyAsync(staged.ptr, codes, ncodes, cudaMemcpyHostToDevice, st));
            d_codes = staged.ptr;
        }
        CUDA_CHECK(cudaMemcpyAsync(d_off.ptr, off.data(), (nrec + 1) * 8, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(d_err.ptr, 0, 4, st));
        records_assemble(d_codes, ncodes, d_off.ptr, nrec, sigma, text.ptr, d_err.ptr, st);
        int herr = 0;
        read_back(&herr, d_err.ptr, 4, st);  // (synchronises the stream: the assembly is done)
        staged.release();
        d_off.release();
        if (herr) return fail(B200SA_ERR_BAD_SYMBOL, "a record holds a code outside 2..sigma-1 (1 is the separator)", err);
        if (int rc = build_into(h, text.ptr, n, sigma, flags | B200SA_TEXT_ON_DEVICE, device, stream, err)) return rc;
        h->flags = flags & ~B200SA_TEXT_ON_DEVICE;
        set_records(h->ix, off, st);
        return 0;
    });
}

int b200sa_records(const b200sa_index *idx, uint32_t *nrec, uint64_t *rec_off) {
    if (!idx || !nrec) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    *nrec = idx->ix.nrec;
    if (rec_off && idx->ix.nrec) memcpy(rec_off, idx->ix.rec_off.data(), idx->ix.rec_off.size() * 8);
    return 0;
}

namespace {
void mail_server_release(const b200sa_index *idx);  // (the resident one-pattern search holds pointers into the index)
}
int b200sa_extend(b200sa_index *idx, const uint8_t *codes, uint32_t flags) {
    if (!idx || (!codes && idx->ix.n)) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    DeviceIndex &ix = idx->ix;
    if (ix.nrec) return fail(B200SA_ERR_BAD_ARGUMENT, "b200sa_extend does not apply to a records index", nullptr);
    if (!ix.sa.ptr) return fail(B200SA_ERR_NOT_BUILT, "suffix array was dropped (B200SA_DROP_SA)", nullptr);
    const bool need_textcmp = (flags & B200SA_BUILD_TEXTCMP) && !ix.text_packed.ptr;
    const bool need_isa = ((flags & B200SA_BUILD_ISA) || need_textcmp) && !ix.isa.ptr;
    const bool need_lcp = (flags & B200SA_BUILD_LCP) && !ix.lcp.ptr;
    const bool need_occ = (flags & B200SA_BUILD_OCC) && ix.occ_layout == OCC_NONE;
    const bool need_bwt = ((flags & B200SA_BUILD_BWT) && !ix.bwt.ptr) || need_occ;
    const bool need_ktable = (flags & B200SA_BUILD_KTABLE) && !ix.ktable.ptr && (need_occ || ix.occ_layout != OCC_NONE);
    if (!need_isa && !need_lcp && !need_bwt && !need_textcmp && !need_ktable) return 0;
    mail_server_release(idx);  // (the resident one-pattern search was launched with the tables as they were)
    return guarded(nullptr, [&] {
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        std::lock_guard<std::mutex> arena_lock(g_arena_mu[ix.device & 63]);
        Arena &arena = g_arena[ix.device & 63];
        arena.reset();
        arena.reserve_first((size_t)ix.len * ix.pk.bits / 8 + (need_lcp ? (size_t)ix.len * 13 : 0) + ((size_t)64 << 20));
        ix.arena = &arena;
        stage_text(ix, arena, codes, flags);
        // the text must be the one the suffix array was built from: same symbol counts, no bad code
        // (pack_text recomputes the C table; the index keeps its own until the text has been accepted)
        u32 c_saved[256];
        u64 counts_saved[256];
        memcpy(c_saved, ix.c_host, sizeof c_saved);
        memcpy(counts_saved, ix.sym_counts_host, sizeof counts_saved);
        DevBuf<u32> c_table_saved = std::move(ix.c_table);
        const bool good_symbols = pack_text_checked(ix);
        const bool same_text = memcmp(counts_saved, ix.sym_counts_host, sizeof counts_saved) == 0;
        if (!good_symbols || !same_text) {
            memcpy(ix.c_host, c_saved, sizeof c_saved);
            memcpy(ix.sym_counts_host, counts_saved, sizeof counts_saved);
            ix.c_table = std::move(c_table_saved);
            ix.text_ptr = nullptr;
            ix.packed = nullptr;
            ix.arena = nullptr;
            if (!good_symbols) return fail(B200SA_ERR_BAD_SYMBOL, "text holds a code outside 1..sigma-1", nullptr);
            return fail(B200SA_ERR_BAD_ARGUMENT, "b200sa_extend: not the text this index was built from (symbol counts differ)", nullptr);
        }
        ix.text.release();
        ix.text_ptr = nullptr;
        if (need_isa) build_inverse(ix);
        if (need_lcp) build_lcp(ix);
        if (need_bwt) {
            const bool had_bwt = ix.bwt.ptr != nullptr;
            if (!had_bwt) gather_bwt(ix);
            if (need_occ) build_bwt_tables(ix, had_bwt || (flags & B200SA_BUILD_BWT));
        }
        if (need_textcmp) keep_packed_text(ix);
        ix.packed = nullptr;
        ix.arena = nullptr;
        if (need_ktable) build_ktable(ix);
        CUDA_CHECK(cudaStreamSynchronize(st));
        idx->flags |= flags & (B200SA_BUILD_ISA | B200SA_BUILD_LCP | B200SA_BUILD_BWT | B200SA_BUILD_OCC);
        if (ix.text_packed.ptr) idx->flags |= B200SA_BUILD_TEXTCMP;
        if (ix.ktable.ptr) idx->flags |= B200SA_BUILD_KTABLE;
        return 0;
    });
}

// ---- resident one-pattern search (fm_search.cu: fm_mailbox_server_kernel) --------------------------------
namespace {
struct MailServer {  // one per device: a slot of mapped pinned memory, a stream of its own, the index it serves
    std::mutex mu;
    u8 *host = nullptr, *dev = nullptr;
    cudaStream_t st = nullptr;
    const b200sa_index *bound = nullptr;
    u32 tag = 0;
    bool broken = false;  // a request timed out once: the launch path is used from then on
};
MailServer g_mail[64];
const size_t kSlotBytes = 512;
const u32 kMailMaxPat = 31 * 6;
inline volatile unsigned long long *slot_words(MailServer &ms) { return (volatile unsigned long long *)ms.host; }

// asks the resident kernel to leave and waits for it (the caller holds ms.mu)
void mail_server_stop(MailServer &ms) {
    if (!ms.host) return;
    volatile unsigned long long *w = slot_words(ms);
    if (w[40]) {
        w[41] = 1;
        const auto t0 = std::chrono::steady_clock::now();
        while (w[40] && std::chrono::steady_clock::now() - t0 < std::chrono::seconds(2)) {
        }
        if (w[40]) cudaStreamSynchronize(ms.st);  // (never seen: the kernel polls the flag every 16 reads of the slot)
        w[41] = 0;
    }
    ms.bound = nullptr;
}

void mail_server_release(const b200sa_index *idx) {
    const int d = idx->ix.device;
    if (d < 0 || d >= 64) return;
    MailServer &ms = g_mail[d];
    std::lock_guard<std::mutex> lock(ms.mu);
    if (ms.bound == idx) mail_server_stop(ms);
}

// one pattern through the resident kernel; false: not served (the caller takes the launch path)
bool mail_server_search(const b200sa_index *idx, const uint8_t *pat, uint32_t m, uint32_t *L, uint32_t *R) {
    static const int enabled = getenv("B200SA_MAIL_SERVER") ? atoi(getenv("B200SA_MAIL_SERVER")) : 1;
    const DeviceIndex &ix = idx->ix;
    if (!enabled || m > kMailMaxPat || ix.occ_layout != OCC_DNA32 || ix.device < 0 || ix.device >= 64) return false;
    MailServer &ms = g_mail[ix.device];
    std::lock_guard<std::mutex> lock(ms.mu);
    if (ms.broken) return false;
    if (!ms.host) {
        if (cudaHostAlloc((void **)&ms.host, kSlotBytes, cudaHostAllocMapped) != cudaSuccess) {
            cudaGetLastError();
            ms.host = nullptr;
            ms.broken = true;
            return false;
        }
        memset(ms.host, 0, kSlotBytes);
        CUDA_CHECK(cudaHostGetDevicePointer((void **)&ms.dev, ms.host, 0));
        CUDA_CHECK(cudaStreamCreateWithFlags(&ms.st, cudaStreamNonBlocking));
    }
    volatile unsigned long long *w = slot_words(ms);
    static const u32 idle_limit = (u32)std::max(16, getenv("B200SA_MAIL_IDLE") ? atoi(getenv("B200SA_MAIL_IDLE")) : 2000);
    auto launch = [&]() {
        // (what the index holds must have been written before the kernel reads it: builds run in the index's stream)
        CUDA_CHECK(cudaStreamSynchronize(ix.stream));
        w[40] = 1;
        w[41] = 0;
        fm_mailbox_server_launch(ix, ms.dev, ms.tag, idle_limit, ms.st);
        ms.bound = idx;
    };
    if (ms.bound != idx || !w[40]) {
        if (w[40]) mail_server_stop(ms);
        launch();
    }
    const u32 tag = (ms.tag + 1u) & 0xffffu;
    const unsigned long long t48 = (unsigned long long)tag << 48;
    const u32 nw = 1u + (m + 5u) / 6u;
    for (u32 k = 1; k < nw; ++k) {
        unsigned long long v = 0;
        for (u32 b = 0; b < 6 && (k - 1) * 6 + b < m; ++b) v |= (unsigned long long)pat[(k - 1) * 6 + b] << (8 * b);
        w[k] = v | t48;
    }
    std::atomic_thread_fence(std::memory_order_release);
    w[0] = t48 | ((unsigned long long)m << 32);
    const auto t0 = std::chrono::steady_clock::now();
    u32 spins = 0;
    for (;;) {
        const unsigned long long r0 = w[32], r1 = w[33];
        if ((r0 >> 48) == tag && (r1 >> 48) == tag) {
            *L = (uint32_t)r0;
            *R = (uint32_t)r1;
            ms.tag = tag;
            static const bool dbg = getenv("B200SA_MAIL_DEBUG") != nullptr;
            if (dbg) {
                static double sum_search = 0, sum_total = 0;
                static unsigned cnt = 0;
                sum_search += (double)w[34];
                sum_total += std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - t0).count();
                if (++cnt % 4096 == 0) {
                    fprintf(stderr, "[b200sa mail] %u requests: %.1f us round trip, %.1f us inside the search\n", cnt,
                            sum_total / cnt / 1e3, sum_search / cnt / 1e3);
                }
            }
            return true;
        }
        if ((++spins & 1023u) == 0) {
            if (!w[40]) {  // the kernel left (idle) before it saw the request: the request is still in the slot
                const unsigned long long q0 = w[32], q1 = w[33];
                if ((q0 >> 48) == tag && (q1 >> 48) == tag) continue;
                launch();
            }
            if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(5)) {
                ms.broken = true;
                w[41] = 1;
                return false;
            }
        }
    }
}
}  // namespace

void b200sa_free(b200sa_index *idx) {
    if (!idx) return;
    mail_server_release(idx);
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    cudaSetDevice(idx->ix.device);
    delete idx;
    if (prev >= 0) cudaSetDevice(prev);
}

int b200sa_stats(const b200sa_index *idx, struct b200sa_stats *out) {
    if (!idx || !out) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const DeviceIndex &ix = idx->ix;
    out->length = ix.len;
    out->sigma = ix.sigma;
    out->primary = ix.primary;
    out->rounds = ix.stats.rounds;
    out->k0 = ix.stats.k0;
    out->radix_bits = ix.stats.radix_bits;
    out->passes0 = ix.stats.passes0;
    out->occ_layout = (uint32_t)ix.occ_layout;
    out->sorted_total = ix.stats.sorted_total;
    out->passes_elems = ix.stats.passes_elems;
    out->occ_bytes = ix.occ.bytes();
    out->round0_mode = ix.stats.round0_mode;
    out->bucket_bits = ix.stats.bucket_bits;
    out->sa_sample_rate = ix.ssa_rate;
    out->sa_resident = ix.sa.ptr ? 1u : 0u;
    out->shallow_buckets = ix.stats.shallow_buckets;
    out->chain_rounds = ix.stats.chain_rounds;
    out->shallow_elems = ix.stats.shallow_elems;
    out->chain_elems = ix.stats.chain_elems;
    out->lazy_lookups = ix.stats.lazy_lookups;
    out->resolved_small = ix.stats.resolved_small;
    out->small_path_elems = ix.stats.small_path_elems;
    out->pivot_elems = ix.stats.pivot_elems;
    out->pivot_rounds = ix.stats.pivot_rounds;
    out->pair_placed = ix.stats.pair_placed;
    out->ktable_k = ix.ktable.ptr ? (uint32_t)ix.ktable_k : 0u;
    out->dense_keys = ix.stats.dense_keys;
    return 0;
}

int b200sa_profile(const b200sa_index *idx, const char **names, float *ms, double *bytes, int cap) {
    if (!idx) return 0;
    int n = idx->prof_n < cap ? idx->prof_n : cap;
    for (int i = 0; i < n; ++i) {
        if (names) names[i] = idx->prof_name[i];
        if (ms) ms[i] = idx->prof_ms[i];
        if (bytes) bytes[i] = idx->prof_bytes[i];
    }
    return idx->prof_n;
}

const uint32_t *b200sa_device_sa(const b200sa_index *idx) { return idx ? idx->ix.sa.ptr : nullptr; }
const uint32_t *b200sa_device_isa(const b200sa_index *idx) { return idx ? idx->ix.isa.ptr : nullptr; }
const uint32_t *b200sa_device_lcp(const b200sa_index *idx) { return idx ? idx->ix.lcp.ptr : nullptr; }
const uint8_t *b200sa_device_bwt(const b200sa_index *idx) { return idx ? idx->ix.bwt.ptr : nullptr; }
const uint8_t *b200sa_device_occ(const b200sa_index *idx) { return idx ? idx->ix.occ.ptr : nullptr; }

// (device pointer, bytes, name) of a table; false for an unknown table id
static bool table_of(const DeviceIndex &ix, int what, const void *&dptr, size_t &bytes, const char *&name) {
    switch (what) {
        case B200SA_TABLE_SA: dptr = ix.sa.ptr; bytes = (size_t)ix.len * 4; name = "SA"; return true;
        case B200SA_TABLE_ISA: dptr = ix.isa.ptr; bytes = (size_t)ix.len * 4; name = "ISA"; return true;
        case B200SA_TABLE_LCP: dptr = ix.lcp.ptr; bytes = (size_t)ix.len * 4; name = "LCP"; return true;
        case B200SA_TABLE_BWT: dptr = ix.bwt.ptr; bytes = (size_t)ix.len; name = "BWT"; return true;
        case B200SA_TABLE_OCC: dptr = ix.occ.ptr; bytes = ix.occ.bytes(); name = "O table"; return true;
        default: return false;
    }
}

// One table into host memory: ordered on `stream`, or on the index's stream and waited for (`wait`).
static int copy_table(const b200sa_index *idx, int what, void *host, void *stream, bool wait) {
    if (!idx || !host) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const void *src = nullptr;
    size_t bytes = 0;
    const char *name = nullptr;
    if (!table_of(idx->ix, what, src, bytes, name)) return fail(B200SA_ERR_BAD_ARGUMENT, "unknown table", nullptr);
    if (!src) return fail(B200SA_ERR_NOT_BUILT, std::string(name) + " was not requested at build time (or was dropped)", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        const cudaStream_t st = wait ? idx->ix.stream : (cudaStream_t)stream;
        // in pieces: they measured faster than one multi-gigabyte copy (57 vs 52 GB/s), and the device-to-host
        // copy engine serves one copy at a time -- a build running next to this transfer reads a few words back
        // per stage, and those must not queue behind gigabytes
        const size_t piece = (size_t)32 << 20;
        for (size_t at = 0; at < bytes; at += piece)
            CUDA_CHECK(cudaMemcpyAsync((char *)host + at, (const char *)src + at, std::min(piece, bytes - at),
                                       cudaMemcpyDeviceToHost, st));
        if (wait) CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

int b200sa_copy_sa(const b200sa_index *idx, uint32_t *host) { return copy_table(idx, B200SA_TABLE_SA, host, nullptr, true); }
int b200sa_copy_isa(const b200sa_index *idx, uint32_t *host) { return copy_table(idx, B200SA_TABLE_ISA, host, nullptr, true); }
int b200sa_copy_lcp(const b200sa_index *idx, uint32_t *host) { return copy_table(idx, B200SA_TABLE_LCP, host, nullptr, true); }
int b200sa_copy_bwt(const b200sa_index *idx, uint8_t *host) { return copy_table(idx, B200SA_TABLE_BWT, host, nullptr, true); }
int b200sa_copy_occ(const b200sa_index *idx, uint8_t *host) { return copy_table(idx, B200SA_TABLE_OCC, host, nullptr, true); }
// Asynchronous copy of one table into caller-owned (pinned) host memory, ordered on `stream`.
int b200sa_copy_async(const b200sa_index *idx, int what, void *host, void *stream) {
    return copy_table(idx, what, host, stream, false);
}
uint64_t b200sa_launch_count(void) { return b200sa::g_kernel_launches; }
int b200sa_plan_round0(uint32_t len, uint32_t sigma, const uint64_t *sym_counts, uint64_t out[16]) {
    b200sa::MsdPlan pl{};
    const b200sa::Packing pk = b200sa::packing_for_sigma(sigma);
    const bool ok = b200sa::msd_make_plan(len, sigma, pk.bits, pl, sym_counts);
    const uint64_t v[16] = {ok ? 1ull : 0ull, (uint64_t)pl.nlevels, (uint64_t)pl.D[0], (uint64_t)pl.D[1], (uint64_t)pl.D[2],
                            (uint64_t)pl.BB, (uint64_t)pl.K, (uint64_t)pl.KB, (uint64_t)pl.pb, (uint64_t)pl.R,
                            pl.dense.nsym, pl.dense.Khi, pl.dense.Klo, pl.dense.powlo, (uint64_t)pk.bits, 0ull};
    for (int i = 0; i < 16; ++i) out[i] = ok || i == 14 ? v[i] : 0ull;
    return 0;
}
uint64_t b200sa_workspace_bytes(int device) { return g_arena[device & 63].reserved(); }
int b200sa_release_workspace(int device) {
    return guarded(nullptr, [&] {
        DeviceGuard guard(device);
        std::lock_guard<std::mutex> lock(g_arena_mu[device & 63]);
        g_arena[device & 63].release_all();
        output_cache_purge(device);
        cudaDeviceSynchronize();
        cudaMemPoolTrimTo(library_pool(), 0);
        {
            SearchLanes &ln = search_lanes(device);
            std::lock_guard<std::mutex> l2(ln.mu);
            ln.release();
        }
        return 0;
    });
}
int b200sa_copy_c_table(const b200sa_index *idx, uint32_t *host) {
    if (!idx || !host) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    memcpy(host, idx->ix.c_host, (size_t)idx->ix.sigma * 4);
    return 0;
}

int b200sa_copy_o_dense(const b200sa_index *idx, uint32_t *host) {
    if (!idx || !host) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const DeviceIndex &ix = idx->ix;
    if (int rc = needs_o_table(ix)) return rc;
    uint64_t entries = ((uint64_t)ix.len + 1) * ix.sigma;
    if (entries * 4 > 0xFFFFFFFFull)
        return fail(B200SA_ERR_TOO_LARGE, "dense O table exceeds the reference's u32 byte size (bwt.c:50)", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(ix.device);
        DevBuf<u32> d(entries, ix.stream);
        occ_dense(ix, d.ptr);
        CUDA_CHECK(cudaMemcpyAsync(host, d.ptr, entries * 4, cudaMemcpyDeviceToHost, ix.stream));
        CUDA_CHECK(cudaStreamSynchronize(ix.stream));
        return 0;
    });
}

int b200sa_occ(const b200sa_index *idx, const uint8_t *a, const uint32_t *i, uint64_t count, uint32_t *out) {
    if (!idx || (count && (!a || !i || !out))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const DeviceIndex &ix = idx->ix;
    if (int rc = needs_o_table(ix)) return rc;
    for (uint64_t q = 0; q < count; ++q)
        if (a[q] >= ix.sigma || i[q] > ix.len) return fail(B200SA_ERR_BAD_ARGUMENT, "O(a,i) query out of range", nullptr);
    if (!count) return 0;
    return guarded(nullptr, [&] {
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        DevBuf<u8> da(count, st);
        DevBuf<u32> di(count, st), dout(count, st);
        CUDA_CHECK(cudaMemcpyAsync(da.ptr, a, count, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(di.ptr, i, count * 4, cudaMemcpyHostToDevice, st));
        occ_probe(ix, da.ptr, di.ptr, count, dout.ptr);
        CUDA_CHECK(cudaMemcpyAsync(out, dout.ptr, count * 4, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

// b200sa_search_device and, with `traffic`, b200sa_search_traffic
static int search_device(const b200sa_index *idx, const uint8_t *d_patterns, const uint64_t *d_offsets, uint32_t fixed_len,
                         uint64_t npat, uint32_t *d_L, uint32_t *d_R, bool traffic, uint64_t *counts, void *stream) {
    if (!idx || (traffic && !counts) || (npat && (!d_patterns || !d_L || !d_R)))
        return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (int rc = needs_o_table(idx->ix)) return rc;
    if (traffic && (idx->ix.occ_layout != OCC_DNA32 || (((uintptr_t)d_patterns) & 7)))
        return fail(B200SA_ERR_NOT_BUILT, "traffic counters exist for the DNA search kernel (8-byte aligned patterns) only", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        const cudaStream_t st = (cudaStream_t)stream;
        count_traffic(counts, st, [&](unsigned long long *d_counts) {
            fm_search(idx->ix, d_patterns, d_offsets, fixed_len, npat, d_L, d_R, st, d_counts);
        });
        return 0;
    });
}

int b200sa_search_device(const b200sa_index *idx, const uint8_t *d_patterns, const uint64_t *d_offsets,
                         uint32_t fixed_len, uint64_t npat, uint32_t *d_L, uint32_t *d_R, void *stream) {
    return search_device(idx, d_patterns, d_offsets, fixed_len, npat, d_L, d_R, false, nullptr, stream);
}

int b200sa_search_traffic(const b200sa_index *idx, const uint8_t *d_patterns, const uint64_t *d_offsets,
                          uint32_t fixed_len, uint64_t npat, uint32_t *d_L, uint32_t *d_R, uint64_t counts[4],
                          void *stream) {
    return search_device(idx, d_patterns, d_offsets, fixed_len, npat, d_L, d_R, true, counts, stream);
}

// Host buffers in, host (L, R) out.
//  * A handful of short patterns (the reference's one-pattern iterator, bwt.c:164-199, through the
//    drop-in): the patterns are written into mapped pinned memory, one kernel reads them there and
//    stores (L, R) next to them -- one launch and one stream synchronisation, no cudaMemcpy.
//  * Otherwise the batch goes through search_pieces (two internal streams per device, SearchLanes).
namespace {
const size_t kMailPat = 4096, kMailOff = 4096, kMailL = 4096 + 65 * 8, kMailR = kMailL + 64 * 4;
static_assert(kMailR + 64 * 4 <= kStagingBytes, "the small-batch layout fits the mapped staging buffer");
}  // namespace

int b200sa_search_batch(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets,
                        uint32_t fixed_len, uint64_t npat, uint32_t *L, uint32_t *R) {
    if (!idx || (npat && (!patterns || !L || !R))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (int rc = needs_o_table(idx->ix)) return rc;
    if (!npat) return 0;
    if (holds_separator(idx, patterns, offsets, fixed_len, npat))
        return fail(B200SA_ERR_BAD_SYMBOL, "a pattern holds code 1, the record separator of this records index", nullptr);
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        const uint64_t total = offsets ? offsets[npat] : (uint64_t)fixed_len * npat;
        if (npat == 1) {  // one pattern: the resident kernel, when there is one to be had
            const uint64_t b0 = offsets ? offsets[0] : 0;
            if (total - b0 <= kMailMaxPat && mail_server_search(idx, patterns + b0, (uint32_t)(total - b0), L, R)) return 0;
        }
        if (npat <= 64 && total + 16 <= kMailPat && ix.device >= 0 && ix.device < 64) {
            u8 *h, *d;
            mapped_staging(ix.device, h, d);
            const uint64_t base = offsets ? offsets[0] : 0;
            memcpy(h, patterns + base, (size_t)(total - base));
            memset(h + (total - base), 0, 16);
            uint64_t *ho = (uint64_t *)(h + kMailOff);
            if (offsets)
                for (uint64_t q = 0; q <= npat; ++q) ho[q] = offsets[q] - base;
            fm_search(ix, d, offsets ? (const u64 *)(d + kMailOff) : nullptr, fixed_len, npat, (u32 *)(d + kMailL),
                      (u32 *)(d + kMailR), st);
            CUDA_CHECK(cudaStreamSynchronize(st));
            memcpy(L, h + kMailL, npat * 4);
            memcpy(R, h + kMailR, npat * 4);
            return 0;
        }
        DevBuf<u64> doff;
        if (offsets) {  // (copied in `st`, which the lanes wait for)
            doff.alloc(npat + 1, st);
            CUDA_CHECK(cudaMemcpyAsync(doff.ptr, offsets, (npat + 1) * 8, cudaMemcpyHostToDevice, st));
        }
        // pieces of ~64 MB of pattern bytes; with a fixed length, multiples of 8 patterns keep every piece's first
        // byte 8-byte aligned (variable-length patterns share one base pointer)
        search_pieces(ix.device, st, npat, total, (uint64_t)64 << 20, L, R,
                      [&](uint64_t q0, uint64_t q1, cudaStream_t ls, u8 *dp, u32 *dL, u32 *dR) {
                          const uint64_t b0 = offsets ? offsets[q0] : q0 * fixed_len;
                          const uint64_t b1 = offsets ? offsets[q1] : q1 * fixed_len;
                          if (b1 > b0) CUDA_CHECK(cudaMemcpyAsync(dp + b0, patterns + b0, b1 - b0, cudaMemcpyHostToDevice, ls));
                          if (offsets)  // absolute offsets: same pattern base, the piece's slice of the offset array
                              fm_search(ix, dp, doff.ptr + q0, 0, q1 - q0, dL, dR, ls);
                          else
                              fm_search(ix, dp + b0, nullptr, fixed_len, q1 - q0, dL, dR, ls);
                      });
        CUDA_CHECK(cudaStreamSynchronize(st));  // (the offsets' buffer is freed on return)
        return 0;
    });
}

// ---- packed reads ---------------------------------------------------------------------------------
// stride 0 stands for ceil(read_len / 4), the least a read of read_len bases takes
static int packed_stride_ok(uint32_t read_len, uint32_t &stride) {
    const uint32_t need = (read_len + 3u) / 4u;
    if (stride == 0) stride = need;
    if (stride < need) return fail(B200SA_ERR_BAD_ARGUMENT, "stride_bytes smaller than ceil(read_len / 4)", nullptr);
    return 0;
}

static int packed_args_ok(const b200sa_index *idx, uint32_t read_len, uint32_t &stride) {
    if (!idx) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (idx->ix.occ_layout != OCC_DNA32)
        return fail(B200SA_ERR_NOT_BUILT, "packed reads need a DNA index (sigma <= 5) with the O table", nullptr);
    // (packed base 0 is code 1, the separator of a records index: a packed read could match across records)
    if (idx->ix.nrec)
        return fail(B200SA_ERR_NOT_BUILT, "packed reads do not apply to a records index (code 1 is its separator)", nullptr);
    if (read_len == 0) return fail(B200SA_ERR_BAD_ARGUMENT, "empty reads", nullptr);
    return packed_stride_ok(read_len, stride);
}

// b200sa_search_device_packed and, with `traffic`, b200sa_search_traffic_packed
static int search_device_packed(const b200sa_index *idx, const uint8_t *d_packed, uint32_t read_len, uint32_t stride,
                                uint64_t npat, uint32_t *d_L, uint32_t *d_R, bool traffic, uint64_t *counts, void *stream) {
    if (int rc = packed_args_ok(idx, read_len, stride)) return rc;
    if ((traffic && !counts) || (npat && (!d_packed || !d_L || !d_R)))
        return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (((uintptr_t)d_packed) & 7) return fail(B200SA_ERR_BAD_ARGUMENT, "packed reads must be 8-byte aligned", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        const cudaStream_t st = (cudaStream_t)stream;
        count_traffic(counts, st, [&](unsigned long long *d_counts) {
            fm_search_packed(idx->ix, d_packed, read_len, stride, npat, d_L, d_R, st, d_counts);
        });
        return 0;
    });
}

int b200sa_search_device_packed(const b200sa_index *idx, const uint8_t *d_packed, uint32_t read_len, uint32_t stride,
                                uint64_t npat, uint32_t *d_L, uint32_t *d_R, void *stream) {
    return search_device_packed(idx, d_packed, read_len, stride, npat, d_L, d_R, false, nullptr, stream);
}

int b200sa_search_traffic_packed(const b200sa_index *idx, const uint8_t *d_packed, uint32_t read_len, uint32_t stride,
                                 uint64_t npat, uint32_t *d_L, uint32_t *d_R, uint64_t counts[4], void *stream) {
    return search_device_packed(idx, d_packed, read_len, stride, npat, d_L, d_R, true, counts, stream);
}

int b200sa_pack_reads(const uint8_t *codes, uint32_t read_len, uint32_t stride, uint64_t npat, uint8_t *packed) {
    if ((npat && (!codes || !packed)) || read_len == 0) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (int rc = packed_stride_ok(read_len, stride)) return rc;
    bool bad = false;
    for (uint64_t q = 0; q < npat; ++q) {
        const uint8_t *r = codes + q * (uint64_t)read_len;
        uint8_t *o = packed + q * (uint64_t)stride;
        for (uint32_t b = 0; b < stride; ++b) {
            uint32_t v = 0;
            for (uint32_t x = 0; x < 4; ++x) {
                const uint32_t j = 4 * b + x;
                uint32_t sym = 0;
                if (j < read_len) {
                    const uint32_t c = r[j];
                    bad |= (c - 1u) > 3u;
                    sym = (c - 1u) & 3u;
                }
                v |= sym << (6u - 2u * x);
            }
            o[b] = (uint8_t)v;
        }
    }
    if (bad) return fail(B200SA_ERR_BAD_SYMBOL, "a read holds a code outside 1..4", nullptr);
    return 0;
}

int b200sa_pack_reads_device(const uint8_t *d_codes, uint32_t read_len, uint32_t stride, uint64_t npat,
                             uint8_t *d_packed, int device, void *stream) {
    if ((npat && (!d_codes || !d_packed)) || read_len == 0) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (int rc = packed_stride_ok(read_len, stride)) return rc;
    return guarded(nullptr, [&] {
        DeviceGuard guard(device);
        cudaStream_t st = (cudaStream_t)stream;
        DevBuf<int> d_err(1, st);
        CUDA_CHECK(cudaMemsetAsync(d_err.ptr, 0, 4, st));
        pack_reads(d_codes, read_len, stride, npat, d_packed, d_err.ptr, st);
        int herr = 0;
        read_back(&herr, d_err.ptr, 4, st);
        if (herr) return fail(B200SA_ERR_BAD_SYMBOL, "a read holds a code outside 1..4", nullptr);
        return 0;
    });
}

// Host packed reads in, host (L, R) out, through search_pieces in pieces of ~16 MB of packed reads.
int b200sa_search_batch_packed(const b200sa_index *idx, const uint8_t *packed, uint32_t read_len, uint32_t stride,
                               uint64_t npat, uint32_t *L, uint32_t *R) {
    if (int rc = packed_args_ok(idx, read_len, stride)) return rc;
    if (npat && (!packed || !L || !R)) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!npat) return 0;
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        // a piece starts at a multiple of 8 reads, hence (any stride) at a multiple of 8 bytes
        search_pieces(ix.device, ix.stream, npat, (uint64_t)stride * npat, (uint64_t)16 << 20, L, R,
                      [&](uint64_t q0, uint64_t q1, cudaStream_t ls, u8 *dp, u32 *dL, u32 *dR) {
                          const uint64_t b0 = q0 * stride, b1 = q1 * stride;
                          CUDA_CHECK(cudaMemcpyAsync(dp + b0, packed + b0, b1 - b0, cudaMemcpyHostToDevice, ls));
                          fm_search_packed(ix, dp + b0, read_len, stride, q1 - q0, dL, dR, ls);
                      });
        return 0;
    });
}

// ---- several devices in one process ------------------------------------------------------------------
b200sa_index *b200sa_replicate(const b200sa_index *src, int device, void *stream, enum b200sa_error *err) {
    if (!src) {
        fail(B200SA_ERR_BAD_ARGUMENT, "null argument", err);
        return nullptr;
    }
    return new_handle<b200sa_index>(err, [&](b200sa_index *h) {
        {
            DeviceGuard gs(src->ix.device);
            CUDA_CHECK(cudaStreamSynchronize(src->ix.stream));  // the source tables are complete
        }
        DeviceGuard guard(device);
        const DeviceIndex &a = src->ix;
        DeviceIndex &ix = h->ix;
        cudaStream_t st = (cudaStream_t)stream;
        ix.stream = st;
        ix.device = device;
        ix.n = a.n; ix.len = a.len; ix.sigma = a.sigma; ix.pk = a.pk;
        ix.primary = a.primary;
        ix.occ_layout = a.occ_layout; ix.occ_blocks = a.occ_blocks; ix.occ_block_bytes = a.occ_block_bytes;
        ix.ktable_k = a.ktable_k; ix.ssa_rate = a.ssa_rate;
        ix.stats = a.stats;
        h->flags = src->flags;
        memcpy(ix.c_host, a.c_host, sizeof ix.c_host);
        memcpy(ix.sym_counts_host, a.sym_counts_host, sizeof ix.sym_counts_host);
        const int sd = a.device;
        replicate_buf(a.sa, sd, ix.sa, device, st, true);
        replicate_buf(a.isa, sd, ix.isa, device, st, true);
        replicate_buf(a.lcp, sd, ix.lcp, device, st, true);
        replicate_buf(a.bwt, sd, ix.bwt, device, st, true);
        replicate_buf(a.occ, sd, ix.occ, device, st, true);
        replicate_buf(a.text_packed, sd, ix.text_packed, device, st, true);
        replicate_buf(a.ktable, sd, ix.ktable, device, st, false);
        replicate_buf(a.ssa_marks, sd, ix.ssa_marks, device, st, false);
        replicate_buf(a.ssa_vals, sd, ix.ssa_vals, device, st, false);
        replicate_buf(a.c_table, sd, ix.c_table, device, st, false);
        if (a.nrec) set_records(ix, a.rec_off, st);
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

int b200sa_search_sharded_packed(const b200sa_index *const *replicas, int nrep, const uint8_t *packed,
                                 uint32_t read_len, uint32_t stride, uint64_t npat, uint32_t *L, uint32_t *R) {
    if (!replicas || nrep < 1 || nrep > 64) return fail(B200SA_ERR_BAD_ARGUMENT, "bad replica list", nullptr);
    for (int g = 0; g < nrep; ++g) {
        if (!replicas[g]) return fail(B200SA_ERR_BAD_ARGUMENT, "null replica", nullptr);
        if (replicas[g]->ix.nrec)
            return fail(B200SA_ERR_NOT_BUILT, "packed reads do not apply to a records index (code 1 is its separator)", nullptr);
        if (replicas[g]->ix.len != replicas[0]->ix.len || replicas[g]->ix.primary != replicas[0]->ix.primary)
            return fail(B200SA_ERR_BAD_ARGUMENT, "replicas are not copies of one index", nullptr);
        for (int k = 0; k < g; ++k)
            if (replicas[k]->ix.device == replicas[g]->ix.device)
                return fail(B200SA_ERR_BAD_ARGUMENT, "two replicas on one device", nullptr);
    }
    if (int rc = packed_args_ok(replicas[0], read_len, stride)) return rc;
    if (npat && (!packed || !L || !R)) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!npat) return 0;
    if (nrep == 1) return b200sa_search_batch_packed(replicas[0], packed, read_len, stride, npat, L, R);
    return guarded(nullptr, [&] {
        int prev = -1;
        cudaGetDevice(&prev);
        struct Restore {
            int d;
            ~Restore() { if (d >= 0) cudaSetDevice(d); }
        } restore{prev};
        const int dev0 = replicas[0]->ix.device;
        // shards: contiguous, boundaries at multiples of 8 reads (every shard's first byte 8-byte aligned)
        std::vector<uint64_t> lo(nrep + 1);
        const uint64_t per = ((npat + nrep - 1) / nrep + 7) & ~(uint64_t)7;
        for (int g = 0; g <= nrep; ++g) lo[g] = std::min(npat, per * (uint64_t)g);
        // result array in the first replica's HBM
        std::vector<std::unique_lock<std::mutex>> locks;
        for (int g = 0; g < nrep; ++g) locks.emplace_back(search_lanes(replicas[g]->ix.device).mu);
        CUDA_CHECK(cudaSetDevice(dev0));
        SearchLanes &l0 = search_lanes(dev0);
        l0.reserve((lo[1] - lo[0]) * stride + 16, npat);
        std::vector<cudaEvent_t> done(nrep, nullptr);
        std::vector<char> direct(nrep, 0);
        for (int g = 0; g < nrep; ++g) {
            const int dev = replicas[g]->ix.device;
            CUDA_CHECK(cudaSetDevice(dev));
            SearchLanes &ln = search_lanes(dev);
            const uint64_t cnt = lo[g + 1] - lo[g];
            if (g) ln.reserve(cnt * stride + 16, cnt);
            else ln.reserve(cnt * stride + 16, npat);
            u32 *outL = ln.L, *outR = ln.R;
            if (g) {
                int can = 0;
                CUDA_CHECK(cudaDeviceCanAccessPeer(&can, dev, dev0));
                if (can) {
                    cudaError_t e = cudaDeviceEnablePeerAccess(dev0, 0);
                    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                    else if (e != cudaSuccess) can = 0, cudaGetLastError();
                }
                if (can) {  // the kernel stores this shard's (L, R) straight into the first replica's HBM
                    outL = l0.L + lo[g];
                    outR = l0.R + lo[g];
                    direct[g] = 1;
                }
            }
            cudaStream_t ls = ln.s[0];
            if (cnt) {
                CUDA_CHECK(cudaMemcpyAsync(ln.patterns, packed + lo[g] * stride, cnt * stride, cudaMemcpyHostToDevice, ls));
                fm_search_packed(replicas[g]->ix, ln.patterns, read_len, stride, cnt, outL, outR, ls);
                if (g && !direct[g]) {
                    CUDA_CHECK(cudaMemcpyAsync(L + lo[g], outL, cnt * 4, cudaMemcpyDeviceToHost, ls));
                    CUDA_CHECK(cudaMemcpyAsync(R + lo[g], outR, cnt * 4, cudaMemcpyDeviceToHost, ls));
                }
            }
            CUDA_CHECK(cudaEventCreateWithFlags(&done[g], cudaEventDisableTiming));
            CUDA_CHECK(cudaEventRecord(done[g], ls));
        }
        // the first replica's stream waits for every peer's kernel, then the result goes home in one piece per range
        CUDA_CHECK(cudaSetDevice(dev0));
        for (int g = 1; g < nrep; ++g) CUDA_CHECK(cudaStreamWaitEvent(l0.s[0], done[g], 0));
        for (int g = 0; g < nrep; ++g) {
            const uint64_t cnt = lo[g + 1] - lo[g];
            if (!cnt || (g && !direct[g])) continue;
            CUDA_CHECK(cudaMemcpyAsync(L + lo[g], l0.L + lo[g], cnt * 4, cudaMemcpyDeviceToHost, l0.s[0]));
            CUDA_CHECK(cudaMemcpyAsync(R + lo[g], l0.R + lo[g], cnt * 4, cudaMemcpyDeviceToHost, l0.s[0]));
        }
        for (int g = 0; g < nrep; ++g) {
            CUDA_CHECK(cudaSetDevice(replicas[g]->ix.device));
            CUDA_CHECK(cudaStreamSynchronize(search_lanes(replicas[g]->ix.device).s[0]));
            cudaEventDestroy(done[g]);
        }
        return 0;
    });
}

int b200sa_locate_device(const b200sa_index *idx, const uint32_t *d_L, const uint32_t *d_R, uint64_t npat,
                         uint64_t *d_pos_off, uint32_t *d_pos, uint64_t pos_capacity, uint64_t *total, void *stream) {
    if (!idx || !d_pos_off || (npat && (!d_L || !d_R))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!can_locate(idx)) return fail(B200SA_ERR_NOT_BUILT, "no suffix array to locate with (dropped and not sampled)", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        cudaStream_t st = (cudaStream_t)stream;
        u64 t = fm_locate_count(idx->ix, d_L, d_R, npat, d_pos_off, st);
        if (total) *total = t;
        if (d_pos) {
            if (t > pos_capacity) return fail(B200SA_ERR_BAD_ARGUMENT, "position buffer too small", nullptr);
            locate_fill_any(idx->ix, d_L, d_R, npat, d_pos_off, t, d_pos, st);
        }
        return 0;
    });
}

int b200sa_sort_positions_device(const b200sa_index *idx, uint64_t npat, const uint64_t *d_pos_off, uint64_t total,
                                 uint32_t *d_pos, void *stream) {
    if (!idx || !d_pos_off || (total && !d_pos)) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (total > 0xFFFFFFFFull || npat > 0xFFFFFFFFull)
        return fail(B200SA_ERR_TOO_LARGE, "more than 2^32 - 1 positions or patterns in one batch", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        sort_positions(idx->ix, npat, d_pos_off, total, d_pos, (cudaStream_t)stream);
        return 0;
    });
}

static int locate_batch_impl(const b200sa_index *idx, const uint32_t *L, const uint32_t *R, uint64_t npat,
                        uint64_t *pos_off, uint32_t *pos, uint64_t pos_capacity, uint64_t *total, bool sorted) {
    if (!idx || !pos_off || (npat && (!L || !R))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!can_locate(idx)) return fail(B200SA_ERR_NOT_BUILT, "no suffix array to locate with (dropped and not sampled)", nullptr);
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        DevBuf<u32> dL(npat ? npat : 1, st), dR(npat ? npat : 1, st);
        DevBuf<u64> doff(npat + 1, st);
        if (npat) {
            CUDA_CHECK(cudaMemcpyAsync(dL.ptr, L, npat * 4, cudaMemcpyHostToDevice, st));
            CUDA_CHECK(cudaMemcpyAsync(dR.ptr, R, npat * 4, cudaMemcpyHostToDevice, st));
        }
        u64 t = fm_locate_count(ix, dL.ptr, dR.ptr, npat, doff.ptr, st);
        if (total) *total = t;
        CUDA_CHECK(cudaMemcpyAsync(pos_off, doff.ptr, (npat + 1) * 8, cudaMemcpyDeviceToHost, st));
        if (pos && t) {
            if (t > pos_capacity) return fail(B200SA_ERR_BAD_ARGUMENT, "position buffer too small", nullptr);
            DevBuf<u32> dpos(t, st);
            locate_fill_any(ix, dL.ptr, dR.ptr, npat, doff.ptr, t, dpos.ptr, st);
            if (sorted) {
                if (t > 0xFFFFFFFFull) return fail(B200SA_ERR_TOO_LARGE, "more than 2^32 - 1 positions in one batch", nullptr);
                sort_positions(ix, npat, doff.ptr, t, dpos.ptr, st);
            }
            CUDA_CHECK(cudaMemcpyAsync(pos, dpos.ptr, t * 4, cudaMemcpyDeviceToHost, st));
        }
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

int b200sa_locate_batch(const b200sa_index *idx, const uint32_t *L, const uint32_t *R, uint64_t npat,
                        uint64_t *pos_off, uint32_t *pos, uint64_t pos_capacity, uint64_t *total) {
    return locate_batch_impl(idx, L, R, npat, pos_off, pos, pos_capacity, total, false);
}
int b200sa_locate_batch_sorted(const b200sa_index *idx, const uint32_t *L, const uint32_t *R, uint64_t npat,
                               uint64_t *pos_off, uint32_t *pos, uint64_t pos_capacity, uint64_t *total) {
    return locate_batch_impl(idx, L, R, npat, pos_off, pos, pos_capacity, total, true);
}

// ---- records index (records.cu) ----
int b200sa_record_sas_device(const b200sa_index *idx, uint32_t *d_out, void *stream) {
    if (!idx || !d_out) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!idx->ix.nrec) return fail(B200SA_ERR_BAD_ARGUMENT, "not a records index (b200sa_build_records)", nullptr);
    if (!idx->ix.sa.ptr) return fail(B200SA_ERR_NOT_BUILT, "the record suffix arrays need the full suffix array (dropped)", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(idx->ix.device);
        record_sas(idx->ix, d_out, (cudaStream_t)stream);
        return 0;
    });
}

int b200sa_copy_record_sas(const b200sa_index *idx, uint32_t *host) {
    if (!idx || !host) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (!idx->ix.nrec) return fail(B200SA_ERR_BAD_ARGUMENT, "not a records index (b200sa_build_records)", nullptr);
    if (!idx->ix.sa.ptr) return fail(B200SA_ERR_NOT_BUILT, "the record suffix arrays need the full suffix array (dropped)", nullptr);
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        DevBuf<u32> d(ix.n, st);
        record_sas(ix, d.ptr, st);
        if (ix.n) CUDA_CHECK(cudaMemcpyAsync(host, d.ptr, (size_t)ix.n * 4, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

// The rows [max(L, 1), R): row 0 is the global sentinel, which belongs to no record.  The count clamps L into d_L1
// and fills d_pos_off; the fill locates the global positions and turns them into (record, local position) pairs.
static u64 locate_records_count(const DeviceIndex &ix, const u32 *d_L, const u32 *d_R, u64 npat, u64 *d_pos_off,
                                u32 *d_L1, cudaStream_t st) {
    records_clamp_rows(d_L, npat, d_L1, st);
    return fm_locate_count(ix, d_L1, d_R, npat, d_pos_off, st);
}
static void locate_records_fill(const DeviceIndex &ix, const u32 *d_L1, const u32 *d_R, u64 npat, const u64 *d_pos_off,
                                u64 total, u32 *d_rec, u32 *d_pos, cudaStream_t st) {
    if (!total) return;
    DevBuf<u32> global(total, st);
    locate_fill_any(ix, d_L1, d_R, npat, d_pos_off, total, global.ptr, st);
    locate_records_group(ix, npat, d_pos_off, total, global.ptr, d_rec, d_pos, st);
}

static int locate_records_args_ok(const b200sa_index *idx, const void *L, const void *R, uint64_t npat, const void *pos_off,
                                  const void *rec, const void *pos) {
    if (!idx || !pos_off || (npat && (!L || !R)) || (!rec != !pos))
        return fail(B200SA_ERR_BAD_ARGUMENT, "null argument (rec and pos are given together)", nullptr);
    if (!idx->ix.nrec) return fail(B200SA_ERR_BAD_ARGUMENT, "not a records index (b200sa_build_records)", nullptr);
    if (!can_locate(idx)) return fail(B200SA_ERR_NOT_BUILT, "no suffix array to locate with (dropped and not sampled)", nullptr);
    return 0;
}

static int locate_records_fits(u64 t, u64 npat, u64 capacity) {
    if (t > capacity) return fail(B200SA_ERR_BAD_ARGUMENT, "position buffer too small", nullptr);
    if (t > 0xFFFFFFFFull || npat > 0xFFFFFFFFull)
        return fail(B200SA_ERR_TOO_LARGE, "more than 2^32 - 1 positions or patterns in one batch", nullptr);
    return 0;
}

int b200sa_locate_records_device(const b200sa_index *idx, const uint32_t *d_L, const uint32_t *d_R, uint64_t npat,
                                 uint64_t *d_pos_off, uint32_t *d_rec, uint32_t *d_pos, uint64_t capacity,
                                 uint64_t *total, void *stream) {
    if (int rc = locate_records_args_ok(idx, d_L, d_R, npat, d_pos_off, d_rec, d_pos)) return rc;
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        cudaStream_t st = (cudaStream_t)stream;
        DevBuf<u32> dL1(npat ? npat : 1, st);
        const u64 t = locate_records_count(ix, d_L, d_R, npat, d_pos_off, dL1.ptr, st);
        if (total) *total = t;
        if (d_pos && t) {
            if (int rc = locate_records_fits(t, npat, capacity)) return rc;
            locate_records_fill(ix, dL1.ptr, d_R, npat, d_pos_off, t, d_rec, d_pos, st);
        }
        return 0;
    });
}

int b200sa_locate_records(const b200sa_index *idx, const uint32_t *L, const uint32_t *R, uint64_t npat,
                          uint64_t *pos_off, uint32_t *rec, uint32_t *pos, uint64_t capacity, uint64_t *total) {
    if (int rc = locate_records_args_ok(idx, L, R, npat, pos_off, rec, pos)) return rc;
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        DevBuf<u32> dL(npat ? npat : 1, st), dR(npat ? npat : 1, st), dL1(npat ? npat : 1, st);
        DevBuf<u64> doff(npat + 1, st);
        if (npat) {
            CUDA_CHECK(cudaMemcpyAsync(dL.ptr, L, npat * 4, cudaMemcpyHostToDevice, st));
            CUDA_CHECK(cudaMemcpyAsync(dR.ptr, R, npat * 4, cudaMemcpyHostToDevice, st));
        }
        const u64 t = locate_records_count(ix, dL.ptr, dR.ptr, npat, doff.ptr, dL1.ptr, st);
        if (total) *total = t;
        CUDA_CHECK(cudaMemcpyAsync(pos_off, doff.ptr, (npat + 1) * 8, cudaMemcpyDeviceToHost, st));
        if (pos && t) {
            if (int rc = locate_records_fits(t, npat, capacity)) return rc;
            DevBuf<u32> drec(t, st), dpos(t, st);
            locate_records_fill(ix, dL1.ptr, dR.ptr, npat, doff.ptr, t, drec.ptr, dpos.ptr, st);
            CUDA_CHECK(cudaMemcpyAsync(rec, drec.ptr, t * 4, cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaMemcpyAsync(pos, dpos.ptr, t * 4, cudaMemcpyDeviceToHost, st));
        }
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

int b200sa_sample_sa(b200sa_index *idx, uint32_t rate, int drop_sa) {
    if (!idx || rate < 1) return fail(B200SA_ERR_BAD_ARGUMENT, "null index or sampling rate 0", nullptr);
    mail_server_release(idx);
    DeviceIndex &ix = idx->ix;
    if (!ix.sa.ptr) return fail(B200SA_ERR_NOT_BUILT, "suffix array was dropped (B200SA_DROP_SA)", nullptr);
    if (ix.occ_layout == OCC_NONE) return fail(B200SA_ERR_NOT_BUILT, "the sampled suffix array needs the O table (B200SA_BUILD_OCC)", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(ix.device);
        build_sampled_sa(ix, rate);
        if (drop_sa && !(idx->flags & B200SA_BUILD_TEXTCMP)) ix.sa.release();
        CUDA_CHECK(cudaStreamSynchronize(ix.stream));
        return 0;
    });
}

int b200sa_sa_lookup(const b200sa_index *idx, const uint32_t *rows, uint64_t count, uint32_t *out, int force_sampled) {
    if (!idx || (count && (!rows || !out))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const DeviceIndex &ix = idx->ix;
    if (force_sampled ? !ix.ssa_rate : !can_locate(idx))
        return fail(B200SA_ERR_NOT_BUILT, "no (sampled) suffix array", nullptr);
    for (uint64_t q = 0; q < count; ++q)
        if (rows[q] >= ix.len) return fail(B200SA_ERR_BAD_ARGUMENT, "row out of range", nullptr);
    if (!count) return 0;
    return guarded(nullptr, [&] {
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        DevBuf<u32> dr(count, st), dout(count, st);
        CUDA_CHECK(cudaMemcpyAsync(dr.ptr, rows, count * 4, cudaMemcpyHostToDevice, st));
        sa_lookup_rows(ix, dr.ptr, count, dout.ptr, force_sampled != 0, st);
        CUDA_CHECK(cudaMemcpyAsync(out, dout.ptr, count * 4, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

// ---- native index file: b200sa_save / b200sa_load (layout above, next to the helpers) ----

int b200sa_save(const b200sa_index *idx, const char *path) {
    if (!idx || !path) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    const DeviceIndex &ix = idx->ix;
    File file(fopen(path, "wb"));
    if (!file) return fail(B200SA_ERR_BAD_ARGUMENT, std::string("cannot open ") + path + " for writing", nullptr);
    return guarded(nullptr, [&] {
        FILE *f = file.get();
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        const size_t words = packed_words(ix);
        std::vector<Section> secs;
        if (ix.sa.ptr) secs.push_back({"SA", ix.sa.ptr, 4, ix.len});
        if (ix.isa.ptr) secs.push_back({"ISA", ix.isa.ptr, 4, ix.len});
        if (ix.lcp.ptr) secs.push_back({"LCP", ix.lcp.ptr, 4, ix.len});
        if (ix.bwt.ptr) secs.push_back({"BWT", ix.bwt.ptr, 1, ix.bwt.count});
        if (ix.occ.ptr) secs.push_back({"OCC", ix.occ.ptr, 1, ix.occ.count});
        if (ix.text_packed.ptr) secs.push_back({"TEXT", ix.text_packed.ptr, 8, words});
        if (ix.ktable.ptr) secs.push_back({"KTABLE", ix.ktable.ptr, 8, ix.ktable.count});
        if (ix.ssa_rate) {
            secs.push_back({"SSAMARK", ix.ssa_marks.ptr, 16, ix.ssa_marks.count});
            secs.push_back({"SSAVAL", ix.ssa_vals.ptr, 4, ix.ssa_vals.count});
        }
        DevBuf<u64> d_recoff;  // (sections are written from device memory)
        if (ix.nrec) {
            d_recoff.alloc(ix.rec_off.size(), st);
            CUDA_CHECK(cudaMemcpyAsync(d_recoff.ptr, ix.rec_off.data(), ix.rec_off.size() * 8, cudaMemcpyHostToDevice, st));
            secs.push_back({"RECOFF", d_recoff.ptr, 8, ix.rec_off.size()});
        }
        IndexFileHeader h{};
        memcpy(h.magic, "B200SAIX", 8);
        h.version = 2;
        h.endian = 0x01020304u;
        h.n = ix.n;
        h.sigma = ix.sigma;
        h.primary = ix.primary;
        h.occ_layout = (uint32_t)ix.occ_layout;
        h.occ_block_bytes = ix.occ_block_bytes;
        h.occ_blocks = ix.occ_blocks;
        h.ktable_k = (uint32_t)ix.ktable_k;
        h.ssa_rate = ix.ssa_rate;
        h.flags = idx->flags & (B200SA_BUILD_ISA | B200SA_BUILD_LCP | B200SA_BUILD_BWT | B200SA_BUILD_OCC |
                                B200SA_BUILD_TEXTCMP | B200SA_BUILD_KTABLE | B200SA_DROP_SA);
        h.nsections = (uint32_t)secs.size();
        h.pack_bits = (uint32_t)ix.pk.bits;
        memcpy(h.c_table, ix.c_host, sizeof h.c_table);
        memcpy(h.sym_counts, ix.sym_counts_host, sizeof h.sym_counts);
        h.stats = ix.stats;
        if (fwrite(&h, sizeof h, 1, f) != 1) throw std::runtime_error("index file: short write");
        std::vector<char> buf(kIoChunk);
        for (const Section &sc : secs) write_section(f, sc, buf, st);
        if (fclose(file.release()) != 0) throw std::runtime_error("index file: close failed");  // (buffered data not written)
        return 0;
    });
}

b200sa_index *b200sa_load(const char *path, int device, void *stream, enum b200sa_error *err) {
    if (!path) {
        fail(B200SA_ERR_BAD_ARGUMENT, "null path", err);
        return nullptr;
    }
    File file(fopen(path, "rb"));
    if (!file) {
        fail(B200SA_ERR_BAD_ARGUMENT, std::string("cannot open ") + path, err);
        return nullptr;
    }
    return new_handle<b200sa_index>(err, [&](b200sa_index *h) {
        FILE *f = file.get();
        DeviceGuard guard(device);
        IndexFileHeader fh;
        if (fread(&fh, sizeof fh, 1, f) != 1 || memcmp(fh.magic, "B200SAIX", 8) != 0)
            throw std::invalid_argument("not a b200sa index file");
        if (fh.endian != 0x01020304u) throw std::invalid_argument("index file was written on the other byte order");
        if (fh.version != 2) throw std::invalid_argument("unsupported index file version");
        if (fh.n > 0xFFFFFFFEull || fh.sigma < 1 || fh.sigma > 256 || fh.primary > fh.n)
            throw std::invalid_argument("index file header is inconsistent");
        // every layout field is checked before a kernel may index with it
        {
            const uint64_t blocks = (fh.n + 1) / 64 + 1;  // build_bwt_tables: len / 64 + 1
            const uint32_t hdr_words = ((fh.sigma - 1) + 3u) & ~3u;
            bool good = fh.occ_layout <= 2;
            if (fh.occ_layout == 1) good = good && fh.sigma <= 5 && fh.occ_block_bytes == 32;
            if (fh.occ_layout == 2) good = good && fh.sigma > 5 && fh.occ_block_bytes == hdr_words * 4 + 64;
            if (fh.occ_layout != 0) good = good && fh.occ_blocks == blocks;
            if (fh.occ_layout == 0) good = good && fh.occ_blocks == 0;
            good = good && fh.ktable_k <= 16 && (fh.ktable_k == 0 || fh.occ_layout == 1 || fh.occ_layout == 2);
            if (!good) throw std::invalid_argument("index file header is inconsistent (O-table layout / k-mer table)");
        }
        DeviceIndex &ix = h->ix;
        cudaStream_t st = (cudaStream_t)stream;
        ix.stream = st;
        ix.device = device;
        ix.n = (u32)fh.n;
        ix.len = ix.n + 1;
        ix.sigma = fh.sigma;
        ix.pk = packing_for_sigma(fh.sigma);
        if ((uint32_t)ix.pk.bits != fh.pack_bits) throw std::invalid_argument("index file header is inconsistent");
        ix.primary = fh.primary;
        ix.occ_layout = (OccLayout)fh.occ_layout;
        ix.occ_block_bytes = fh.occ_block_bytes;
        ix.occ_blocks = fh.occ_blocks;
        ix.ktable_k = (int)fh.ktable_k;
        ix.stats = fh.stats;
        h->flags = fh.flags;
        memcpy(ix.c_host, fh.c_table, sizeof fh.c_table);
        memcpy(ix.sym_counts_host, fh.sym_counts, sizeof fh.sym_counts);
        ix.c_table.alloc(ix.sigma, st);
        CUDA_CHECK(cudaMemcpyAsync(ix.c_table.ptr, ix.c_host, (size_t)ix.sigma * 4, cudaMemcpyHostToDevice, st));
        const size_t words = packed_words(ix);
        const size_t bwt_bytes = (((size_t)ix.len + 63) / 64 + 1) * 64;
        std::vector<char> buf(kIoChunk);
        bool have_occ = false, have_marks = false, have_vals = false;
        for (uint32_t k = 0; k < fh.nsections; ++k) {
            SectionHeader sh;
            if (fread(&sh, sizeof sh, 1, f) != 1) throw std::invalid_argument("index file: truncated");
            const std::string tag(sh.tag, strnlen(sh.tag, 8));
            if (tag == "SA") read_section(f, sh, ix.sa, ix.len, buf, st);
            else if (tag == "ISA") read_section(f, sh, ix.isa, ix.len, buf, st);
            else if (tag == "LCP") read_section(f, sh, ix.lcp, ix.len, buf, st);
            else if (tag == "BWT") read_section(f, sh, ix.bwt, bwt_bytes, buf, st);
            else if (tag == "OCC") {
                read_section(f, sh, ix.occ, (size_t)fh.occ_blocks * fh.occ_block_bytes, buf, st);
                have_occ = true;
            } else if (tag == "TEXT") read_section(f, sh, ix.text_packed, words, buf, st);
            else if (tag == "KTABLE") {
                // 4^k entries over 2-bit symbols, (sigma - 1)^k over any other alphabet
                size_t entries = (size_t)1 << (2 * fh.ktable_k);
                if (fh.occ_layout == 2) {
                    entries = 1;
                    for (uint32_t j = 0; j < fh.ktable_k; ++j) entries *= (size_t)(fh.sigma - 1);
                }
                read_section(f, sh, ix.ktable, entries, buf, st);
            }
            else if (tag == "SSAMARK") {
                read_section(f, sh, ix.ssa_marks, ((size_t)ix.len + 63) / 64, buf, st);
                have_marks = true;
            } else if (tag == "SSAVAL") {
                if (!fh.ssa_rate) throw std::invalid_argument("index file header is inconsistent");
                read_section(f, sh, ix.ssa_vals, (size_t)ix.n / fh.ssa_rate + 1, buf, st);
                have_vals = true;
            } else if (tag == "RECOFF") {
                if (sh.elem_bytes != 8 || sh.count < 2 || sh.count - 1 > fh.n)
                    throw std::invalid_argument("index file: section RECOFF has an unexpected shape");
                std::vector<u64> off(sh.count);
                if (fread(off.data(), 8, sh.count, f) != sh.count) throw std::invalid_argument("index file: truncated section");
                bool good = off[0] == 0 && off.back() + (sh.count - 1) == fh.n;
                for (size_t r = 1; r < off.size() && good; ++r) good = off[r] >= off[r - 1];
                if (!good) throw std::invalid_argument("index file: record offsets are inconsistent");
                set_records(ix, off, st);
            } else
                throw std::invalid_argument("index file: unknown section " + tag);
        }
        if ((ix.occ_layout != OCC_NONE) != have_occ || (fh.ssa_rate != 0) != (have_marks && have_vals) ||
            (fh.ktable_k != 0) != (ix.ktable.ptr != nullptr))
            throw std::invalid_argument("index file: sections do not match the header");
        ix.ssa_rate = fh.ssa_rate;
        CUDA_CHECK(cudaStreamSynchronize(st));
        return 0;
    });
}

// ---- approximate search ------------------------------------------------------------------------
struct b200sa_approx_result {
    std::vector<uint64_t> hit_off;   // npat + 1
    std::vector<uint32_t> L, R, mlen;
    std::vector<uint64_t> cig_off;   // nhits + 1
    std::vector<char> cigars;        // NUL-terminated, back to back
};

b200sa_approx_result *b200sa_approx_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                          const uint8_t *d_table, const uint8_t *patterns, const uint64_t *offsets,
                                          uint32_t fixed_len, uint64_t npat, int max_edits, enum b200sa_error *err) {
    if (!idx || (npat && !patterns) || max_edits < 0 || max_edits > 255) {
        fail(B200SA_ERR_BAD_ARGUMENT, "null argument or max_edits outside 0..255", err);
        return nullptr;
    }
    const DeviceIndex &ix = idx->ix;
    if (needs_o_table(ix, err)) return nullptr;
    if (rev_idx && (rev_idx->ix.occ_layout == OCC_NONE || rev_idx->ix.len != ix.len || rev_idx->ix.sigma != ix.sigma ||
                    rev_idx->ix.device != ix.device)) {
        fail(B200SA_ERR_BAD_ARGUMENT, "the reverse index must be an O-table index of the reversed text on the same device", err);
        return nullptr;
    }
    uint64_t total = offsets ? offsets[npat] : (uint64_t)fixed_len * npat;
    uint32_t max_m = 0;
    if (pattern_lengths_ok(offsets, fixed_len, npat, 65000, "approximate search takes patterns of up to 65000 symbols",
                           max_m, err))
        return nullptr;
    if (holds_separator(idx, patterns, offsets, fixed_len, npat)) {
        fail(B200SA_ERR_BAD_SYMBOL, "a pattern holds code 1, the record separator of this records index", err);
        return nullptr;
    }
    return new_handle<b200sa_approx_result>(err, [&](b200sa_approx_result *res) {
        DeviceGuard guard(ix.device);
        cudaStream_t st = ix.stream;
        res->hit_off.assign(npat + 1, 0);
        res->cig_off.assign(1, 0);
        if (npat) {
            DevBuf<u8> dp(total + 16, st), ddt;
            DevBuf<u64> doff, d_hit_off(npat + 1, st), d_ops_off(npat + 1, st);
            if (total) CUDA_CHECK(cudaMemcpyAsync(dp.ptr, patterns, total, cudaMemcpyHostToDevice, st));
            if (offsets) {
                doff.alloc(npat + 1, st);
                CUDA_CHECK(cudaMemcpyAsync(doff.ptr, offsets, (npat + 1) * 8, cudaMemcpyHostToDevice, st));
            }
            if (d_table) {
                ddt.alloc(total + 16, st);
                if (total) CUDA_CHECK(cudaMemcpyAsync(ddt.ptr, d_table, total, cudaMemcpyHostToDevice, st));
            } else if (rev_idx) {
                ddt.alloc(total + 16, st);
                approx_dtable(rev_idx->ix, dp.ptr, doff.ptr, fixed_len, npat, ddt.ptr, st);
            }
            u64 hits = 0, ops = 0;
            approx_count(ix, dp.ptr, doff.ptr, fixed_len, npat, max_m, ddt.ptr, max_edits, d_hit_off.ptr, d_ops_off.ptr,
                         &hits, &ops, st);
            CUDA_CHECK(cudaMemcpyAsync(res->hit_off.data(), d_hit_off.ptr, (npat + 1) * 8, cudaMemcpyDeviceToHost, st));
            res->L.resize(hits);
            res->R.resize(hits);
            res->mlen.resize(hits);
            // the emitting pass writes the run-length CIGAR strings (stralg/cigar.c:8-31) themselves
            res->cig_off.assign(hits + 1, 0);
            res->cigars.assign(ops + 1, 0);
            if (hits) {
                DevBuf<u32> dL(hits, st), dR(hits, st), dM(hits, st);
                DevBuf<u64> dho(hits, st);
                DevBuf<char> dops(ops + 1, st);
                approx_emit(ix, dp.ptr, doff.ptr, fixed_len, npat, max_m, ddt.ptr, max_edits, d_hit_off.ptr, d_ops_off.ptr,
                            dL.ptr, dR.ptr, dM.ptr, dho.ptr, dops.ptr, st);
                CUDA_CHECK(cudaMemcpyAsync(res->L.data(), dL.ptr, hits * 4, cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaMemcpyAsync(res->R.data(), dR.ptr, hits * 4, cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaMemcpyAsync(res->mlen.data(), dM.ptr, hits * 4, cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaMemcpyAsync(res->cig_off.data(), dho.ptr, hits * 8, cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaMemcpyAsync(res->cigars.data(), dops.ptr, ops, cudaMemcpyDeviceToHost, st));
            }
            CUDA_CHECK(cudaStreamSynchronize(st));
            res->cig_off[hits] = ops;
        }
        return 0;
    });
}

uint64_t b200sa_approx_hits(const b200sa_approx_result *r) { return r ? r->L.size() : 0; }
const uint64_t *b200sa_approx_hit_offsets(const b200sa_approx_result *r) { return r ? r->hit_off.data() : nullptr; }
const uint32_t *b200sa_approx_L(const b200sa_approx_result *r) { return r ? r->L.data() : nullptr; }
const uint32_t *b200sa_approx_R(const b200sa_approx_result *r) { return r ? r->R.data() : nullptr; }
const uint32_t *b200sa_approx_match_length(const b200sa_approx_result *r) { return r ? r->mlen.data() : nullptr; }
const uint64_t *b200sa_approx_cigar_offsets(const b200sa_approx_result *r) { return r ? r->cig_off.data() : nullptr; }
const char *b200sa_approx_cigars(const b200sa_approx_result *r) { return r ? r->cigars.data() : nullptr; }
void b200sa_approx_free(b200sa_approx_result *r) { delete r; }

}  // extern "C"
#pragma GCC visibility pop

// ---- matching statistics and SMEMs ---------------------------------------------------------------
// the refusals of b200sa_matching_stats and b200sa_smem_batch that come before any CUDA call
static int mems_args_ok(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                        uint64_t npat, enum b200sa_error *err) {
    if (int rc = needs_o_table(idx->ix, err)) return rc;
    uint32_t max_m = 0;
    if (int rc = pattern_lengths_ok(offsets, fixed_len, npat, 0xFFFFFFFFull, "a pattern longer than 2^32 - 1 symbols",
                                    max_m, err))
        return rc;
    if (holds_separator(idx, patterns, offsets, fixed_len, npat))
        return fail(B200SA_ERR_BAD_SYMBOL, "a pattern holds code 1, the record separator of this records index", err);
    return 0;
}

// The end of the piece of a host batch that starts at pattern q0: whole patterns of about 64 MB of symbols in all (a
// longer pattern is a piece of its own), so that device memory stays bounded whatever the batch.
static uint64_t piece_end(const uint64_t *offsets, uint32_t fixed_len, uint64_t npat, uint64_t q0) {
    const uint64_t kPieceBytes = (uint64_t)64 << 20;
    uint64_t q1 = q0 + 1;
    if (offsets)
        while (q1 < npat && offsets[q1 + 1] - offsets[q0] <= kPieceBytes) ++q1;
    else
        q1 = std::min(npat, q0 + std::max<uint64_t>(1, kPieceBytes / std::max<uint32_t>(1, fixed_len)));
    return q1;
}

// The first pass over a host batch, in pieces (piece_end): a piece's patterns are copied in (8-byte aligned and
// padded, as the kernels read whole words), its offsets rebased to the piece, and mems_stats stores ms / L / R per
// symbol and, with `count`, the SMEMs of each pattern.  Then `piece(q0, q1, b0, d_off, d_ms, d_L, d_R, d_count)`
// takes over the results of patterns [q0, q1), whose symbols start at b0 in the batch, on the index's stream; it
// returns when it no longer needs them.
template <class Piece>
static void mems_pieces(const DeviceIndex &ix, const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                        uint64_t npat, uint32_t min_len, bool count, Piece &&piece) {
    const cudaStream_t st = ix.stream;
    auto at = [&](uint64_t q) { return offsets ? offsets[q] : q * (uint64_t)fixed_len; };
    std::vector<uint64_t> hoff;
    for (uint64_t q0 = 0, q1; q0 < npat; q0 = q1) {
        q1 = piece_end(offsets, fixed_len, npat, q0);
        const uint64_t b0 = at(q0), bytes = at(q1) - b0;
        DevBuf<u8> dp(bytes + 16, st);
        DevBuf<u32> dms(bytes, st), dL(bytes, st), dR(bytes, st);
        DevBuf<u64> doff, dcnt;
        if (bytes) CUDA_CHECK(cudaMemcpyAsync(dp.ptr, patterns + b0, bytes, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(dp.ptr + bytes, 0, 16, st));
        if (offsets) {
            hoff.resize(q1 - q0 + 1);
            for (uint64_t q = q0; q <= q1; ++q) hoff[q - q0] = offsets[q] - b0;
            doff.alloc(hoff.size(), st);
            CUDA_CHECK(cudaMemcpyAsync(doff.ptr, hoff.data(), hoff.size() * 8, cudaMemcpyHostToDevice, st));
        }
        if (count) dcnt.alloc(q1 - q0 + 1, st);  // (+1: the scan's total)
        mems_stats(ix, dp.ptr, doff.ptr, fixed_len, q1 - q0, min_len, dms.ptr, dL.ptr, dR.ptr, dcnt.ptr, st);
        piece(q0, q1, b0, doff.ptr, dms.ptr, dL.ptr, dR.ptr, dcnt.ptr);
        CUDA_CHECK(cudaStreamSynchronize(st));  // (`hoff` and the piece's buffers are reused or freed next)
    }
}

struct b200sa_smem_result {
    std::vector<uint64_t> off;  // npat + 1
    std::vector<uint32_t> start, length, L, R;
};

#pragma GCC visibility push(default)
extern "C" {

int b200sa_matching_stats(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                          uint64_t npat, uint32_t *ms, uint32_t *L, uint32_t *R) {
    if (!idx || (npat && (!patterns || !ms))) return fail(B200SA_ERR_BAD_ARGUMENT, "null argument", nullptr);
    if (int rc = mems_args_ok(idx, patterns, offsets, fixed_len, npat, nullptr)) return rc;
    if (!npat) return 0;
    return guarded(nullptr, [&] {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        const cudaStream_t st = ix.stream;
        mems_pieces(ix, patterns, offsets, fixed_len, npat, 1, false,
                    [&](uint64_t q0, uint64_t q1, uint64_t b0, const u64 *, const u32 *dms, const u32 *dL, const u32 *dR,
                        u64 *) {
                        const size_t bytes = (size_t)((offsets ? offsets[q1] : q1 * (uint64_t)fixed_len) - b0) * 4;
                        if (!bytes) return;
                        CUDA_CHECK(cudaMemcpyAsync(ms + b0, dms, bytes, cudaMemcpyDeviceToHost, st));
                        if (L) CUDA_CHECK(cudaMemcpyAsync(L + b0, dL, bytes, cudaMemcpyDeviceToHost, st));
                        if (R) CUDA_CHECK(cudaMemcpyAsync(R + b0, dR, bytes, cudaMemcpyDeviceToHost, st));
                    });
        return 0;
    });
}

b200sa_smem_result *b200sa_smem_batch(const b200sa_index *idx, const uint8_t *patterns, const uint64_t *offsets,
                                      uint32_t fixed_len, uint64_t npat, uint32_t min_len, enum b200sa_error *err) {
    if (!idx || (npat && !patterns) || min_len == 0) {
        fail(B200SA_ERR_BAD_ARGUMENT, "null argument or min_len 0", err);
        return nullptr;
    }
    if (mems_args_ok(idx, patterns, offsets, fixed_len, npat, err)) return nullptr;
    return new_handle<b200sa_smem_result>(err, [&](b200sa_smem_result *res) {
        const DeviceIndex &ix = idx->ix;
        DeviceGuard guard(ix.device);
        const cudaStream_t st = ix.stream;
        res->off.assign(npat + 1, 0);
        mems_pieces(ix, patterns, offsets, fixed_len, npat, min_len, true,
                    [&](uint64_t q0, uint64_t q1, uint64_t, const u64 *doff, const u32 *dms, const u32 *dL, const u32 *dR,
                        u64 *dcnt) {
                        const uint64_t np = q1 - q0, base = res->start.size();
                        scan_u64(dcnt, np, st);
                        CUDA_CHECK(cudaMemcpyAsync(res->off.data() + q0, dcnt, (np + 1) * 8, cudaMemcpyDeviceToHost, st));
                        CUDA_CHECK(cudaStreamSynchronize(st));
                        for (uint64_t q = q0; q <= q1; ++q) res->off[q] += base;
                        const uint64_t total = res->off[q1] - base;
                        if (!total) return;
                        DevBuf<u32> ds(total, st), dn(total, st), dsL(total, st), dsR(total, st);
                        mems_emit(ix, doff, fixed_len, np, min_len, dms, dL, dR, dcnt, ds.ptr, dn.ptr, dsL.ptr, dsR.ptr, st);
                        append_columns(base, total, {{res->start, ds.ptr}, {res->length, dn.ptr}, {res->L, dsL.ptr},
                                                     {res->R, dsR.ptr}}, st);
                        CUDA_CHECK(cudaStreamSynchronize(st));  // (the output buffers are freed on return)
                    });
        return 0;
    });
}

uint64_t b200sa_smem_count(const b200sa_smem_result *r) { return r ? r->start.size() : 0; }
const uint64_t *b200sa_smem_offsets(const b200sa_smem_result *r) { return r ? r->off.data() : nullptr; }
const uint32_t *b200sa_smem_start(const b200sa_smem_result *r) { return r ? r->start.data() : nullptr; }
const uint32_t *b200sa_smem_length(const b200sa_smem_result *r) { return r ? r->length.data() : nullptr; }
const uint32_t *b200sa_smem_L(const b200sa_smem_result *r) { return r ? r->L.data() : nullptr; }
const uint32_t *b200sa_smem_R(const b200sa_smem_result *r) { return r ? r->R.data() : nullptr; }
void b200sa_smem_free(b200sa_smem_result *r) { delete r; }

}  // extern "C"
#pragma GCC visibility pop

// ---- k-mismatch and edit-distance search on an index pair --------------------------------------------
// the refusals of b200sa_hamming_batch and b200sa_levenshtein_batch that come before any CUDA call; max_m gets the
// longest pattern
static int pair_args_ok(const b200sa_index *idx, const b200sa_index *rev_idx, const uint8_t *patterns,
                        const uint64_t *offsets, uint32_t fixed_len, uint64_t npat, uint32_t k, uint32_t max_k,
                        const char *what, const char *k_name, uint32_t &max_m, enum b200sa_error *err) {
    if (!idx || !rev_idx || (npat && !patterns) || k > max_k)
        return fail(B200SA_ERR_BAD_ARGUMENT,
                    std::string("null argument or ") + k_name + " above " + std::to_string(max_k), err);
    if (int rc = pattern_lengths_ok(offsets, fixed_len, npat, 65000,
                                    std::string(what) + " search takes patterns of up to 65000 symbols", max_m, err))
        return rc;
    const DeviceIndex &ix = idx->ix, &rv = rev_idx->ix;
    if (int rc = needs_o_table(ix, err)) return rc;
    if (int rc = needs_o_table(rv, err)) return rc;
    if (rv.len != ix.len || rv.sigma != ix.sigma || rv.device != ix.device ||
        memcmp(rv.c_host, ix.c_host, (size_t)ix.sigma * 4) != 0)
        return fail(B200SA_ERR_BAD_ARGUMENT,
                    "the reverse index must be an O-table index of the reversed text on the same device", err);
    if (ix.nrec || rv.nrec)
        return fail(B200SA_ERR_BAD_ARGUMENT, std::string(what) + " search does not take a records index", err);
    return 0;
}

// A host batch searched on an index pair, in pieces (piece_end, and at most max_np patterns each): a piece's
// patterns are copied in and its offsets rebased to the piece; `piece(np, d_pat, d_off, d_pat_off, base)` runs the
// search of its np patterns, copies its hits back after the `base` hits of the earlier pieces and leaves the CSR of
// its hits in d_pat_off (np + 1 entries), or returns an error code; res_off (npat + 1) gets the CSR of the batch.
template <class Piece>
static int pair_pieces(const DeviceIndex &ix, const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                       uint64_t npat, uint64_t max_np, std::vector<uint64_t> &res_off, Piece &&piece) {
    const cudaStream_t st = ix.stream;
    res_off.assign(npat + 1, 0);
    auto at = [&](uint64_t q) { return offsets ? offsets[q] : q * (uint64_t)fixed_len; };
    std::vector<uint64_t> hoff;
    for (uint64_t q0 = 0, q1; q0 < npat; q0 = q1) {
        q1 = std::min(piece_end(offsets, fixed_len, npat, q0), q0 + max_np);
        const uint64_t np = q1 - q0, b0 = at(q0), bytes = at(q1) - b0;
        DevBuf<u8> dp(bytes + 16, st);
        DevBuf<u64> doff, dpo(np + 1, st);
        if (bytes) CUDA_CHECK(cudaMemcpyAsync(dp.ptr, patterns + b0, bytes, cudaMemcpyHostToDevice, st));
        if (offsets) {
            hoff.resize(np + 1);
            for (uint64_t q = q0; q <= q1; ++q) hoff[q - q0] = offsets[q] - b0;
            doff.alloc(np + 1, st);
            CUDA_CHECK(cudaMemcpyAsync(doff.ptr, hoff.data(), (np + 1) * 8, cudaMemcpyHostToDevice, st));
        }
        uint64_t base = 0;
        if (int rc = piece(np, dp.ptr, doff.ptr, dpo.ptr, base)) return rc;
        CUDA_CHECK(cudaMemcpyAsync(res_off.data() + q0, dpo.ptr, (np + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));  // (`hoff` and the piece's buffers are reused or freed next)
        for (uint64_t q = q0; q <= q1; ++q) res_off[q] += base;
    }
    return 0;
}

struct b200sa_hamming_result {
    std::vector<uint64_t> off;  // npat + 1
    std::vector<uint32_t> L, R, d;
};

struct b200sa_levenshtein_result {
    std::vector<uint64_t> off;  // npat + 1
    std::vector<uint32_t> L, R, length, d;
};

#pragma GCC visibility push(default)
extern "C" {

b200sa_hamming_result *b200sa_hamming_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                            const uint8_t *patterns, const uint64_t *offsets, uint32_t fixed_len,
                                            uint64_t npat, uint32_t max_mismatches, enum b200sa_error *err) {
    uint32_t max_m = 0;
    if (pair_args_ok(idx, rev_idx, patterns, offsets, fixed_len, npat, max_mismatches, 8, "k-mismatch", "max_mismatches",
                     max_m, err))
        return nullptr;
    const DeviceIndex &ix = idx->ix, &rv = rev_idx->ix;
    const uint32_t k = max_mismatches;
    return new_handle<b200sa_hamming_result>(err, [&](b200sa_hamming_result *res) {
        DeviceGuard guard(ix.device);
        const cudaStream_t st = ix.stream;
        return pair_pieces(ix, patterns, offsets, fixed_len, npat, npat, res->off,
                           [&](uint64_t np, const u8 *dp, const u64 *doff, u64 *dpo, uint64_t &base) {
            base = res->L.size();
            DevBuf<u64> duo(np * (k + 1) + 1, st);
            const u64 hits = pair_count(PairSearch::HAMMING, ix, rv, dp, doff, fixed_len, np, max_m, k, duo.ptr, st);
            if (hits > 0xFFFFFFFFull || np > 0xFFFFFFFFull)
                return fail(B200SA_ERR_TOO_LARGE, "more than 2^32 - 1 hits or patterns in one piece of the batch", err);
            DevBuf<u32> dL(hits ? hits : 1, st), dR(hits ? hits : 1, st), dd(hits ? hits : 1, st);
            hamming_emit(ix, rv, dp, doff, fixed_len, np, max_m, k, duo.ptr, hits, dpo, dL.ptr, dR.ptr, dd.ptr, st);
            append_columns(base, hits, {{res->L, dL.ptr}, {res->R, dR.ptr}, {res->d, dd.ptr}}, st);
            return 0;
        });
    });
}

uint64_t b200sa_hamming_hits(const b200sa_hamming_result *r) { return r ? r->L.size() : 0; }
const uint64_t *b200sa_hamming_offsets(const b200sa_hamming_result *r) { return r ? r->off.data() : nullptr; }
const uint32_t *b200sa_hamming_L(const b200sa_hamming_result *r) { return r ? r->L.data() : nullptr; }
const uint32_t *b200sa_hamming_R(const b200sa_hamming_result *r) { return r ? r->R.data() : nullptr; }
const uint32_t *b200sa_hamming_mismatches(const b200sa_hamming_result *r) { return r ? r->d.data() : nullptr; }
void b200sa_hamming_free(b200sa_hamming_result *r) { delete r; }

b200sa_levenshtein_result *b200sa_levenshtein_batch(const b200sa_index *idx, const b200sa_index *rev_idx,
                                                    const uint8_t *patterns, const uint64_t *offsets,
                                                    uint32_t fixed_len, uint64_t npat, uint32_t max_edits,
                                                    enum b200sa_error *err) {
    uint32_t max_m = 0;
    if (pair_args_ok(idx, rev_idx, patterns, offsets, fixed_len, npat, max_edits, 4, "edit-distance", "max_edits", max_m,
                     err))
        return nullptr;
    const DeviceIndex &ix = idx->ix, &rv = rev_idx->ix;
    const uint32_t k = max_edits;
    return new_handle<b200sa_levenshtein_result>(err, [&](b200sa_levenshtein_result *res) {
        DeviceGuard guard(ix.device);
        const cudaStream_t st = ix.stream;
        // a raw hit's sort key is [pattern | L | length - (m - k)]: 64 - 32 - 4 bits for the pattern
        return pair_pieces(ix, patterns, offsets, fixed_len, npat, (uint64_t)1 << 28, res->off,
                           [&](uint64_t np, const u8 *dp, const u64 *doff, u64 *dpo, uint64_t &base) {
            base = res->L.size();
            DevBuf<u64> duo(np * (k + 1) + 1, st);
            const u64 raw = pair_count(PairSearch::LEVENSHTEIN, ix, rv, dp, doff, fixed_len, np, max_m, k, duo.ptr, st);
            if (raw > 0xFFFFFFFFull)
                return fail(B200SA_ERR_TOO_LARGE, "more than 2^32 - 1 raw hits in one piece of the batch", err);
            DevBuf<u32> dL(raw ? raw : 1, st), dR(raw ? raw : 1, st), dn(raw ? raw : 1, st), dd(raw ? raw : 1, st);
            const u64 hits =
                levenshtein_emit(ix, rv, dp, doff, fixed_len, np, max_m, k, duo.ptr, raw, dpo, dL.ptr, dR.ptr, dn.ptr,
                                 dd.ptr, st);
            append_columns(base, hits, {{res->L, dL.ptr}, {res->R, dR.ptr}, {res->length, dn.ptr}, {res->d, dd.ptr}}, st);
            return 0;
        });
    });
}

uint64_t b200sa_levenshtein_hits(const b200sa_levenshtein_result *r) { return r ? r->L.size() : 0; }
const uint64_t *b200sa_levenshtein_offsets(const b200sa_levenshtein_result *r) { return r ? r->off.data() : nullptr; }
const uint32_t *b200sa_levenshtein_L(const b200sa_levenshtein_result *r) { return r ? r->L.data() : nullptr; }
const uint32_t *b200sa_levenshtein_R(const b200sa_levenshtein_result *r) { return r ? r->R.data() : nullptr; }
const uint32_t *b200sa_levenshtein_length(const b200sa_levenshtein_result *r) { return r ? r->length.data() : nullptr; }
const uint32_t *b200sa_levenshtein_distance(const b200sa_levenshtein_result *r) { return r ? r->d.data() : nullptr; }
void b200sa_levenshtein_free(b200sa_levenshtein_result *r) { delete r; }

int b200sa_synth_codes(uint8_t *d_text, uint64_t n, uint32_t nsym, uint64_t seed, int device, void *stream) {
    if (!d_text || nsym < 1 || nsym > 255) return fail(B200SA_ERR_BAD_ARGUMENT, "bad argument", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(device);
        synth_codes(d_text, n, nsym, seed, (cudaStream_t)stream);
        return 0;
    });
}

int b200sa_synth_reads(const uint8_t *d_text, uint64_t n, uint32_t nsym, uint8_t *d_reads, uint64_t nreads,
                       uint32_t m, uint32_t miss_per_1024, uint64_t seed, int device, void *stream) {
    if (!d_text || !d_reads || nsym < 1 || nsym > 255) return fail(B200SA_ERR_BAD_ARGUMENT, "bad argument", nullptr);
    return guarded(nullptr, [&] {
        DeviceGuard guard(device);
        synth_reads(d_text, n, nsym, d_reads, nreads, m, miss_per_1024, seed, (cudaStream_t)stream);
        return 0;
    });
}

}  // extern "C"
#pragma GCC visibility pop
