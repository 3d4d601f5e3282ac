// scan.cuh -- the prefix scans of the kernels (sm_100a): warp, block and single-CTA forms.
#pragma once
#include "common.cuh"

namespace b200sa {

struct SumOp {
    template <typename T>
    __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};
struct MaxOp {
    template <typename T>
    __device__ __forceinline__ T operator()(T a, T b) const { return max(a, b); }
};

// Inclusive scan over lanes 0 .. W - 1 of a warp (every lane of the warp takes part).  The value t of the
// lower lane combines as op(t, v), so an operator that does not commute keeps its order.
template <int W = 32, typename T, typename Op>
__device__ __forceinline__ T warp_inclusive(T v, Op op) {
    const unsigned lane = lane_id();
#pragma unroll
    for (int o = 1; o < W; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= (unsigned)o) v = op(t, v);
    }
    return v;
}

// A lane's exclusive value from its inclusive one `incl` and its own value `v`: the lower lane's inclusive
// value, `identity` in lane 0.  A sum subtracts `v` instead.
template <typename T, typename Op>
__device__ __forceinline__ T warp_exclusive(T incl, T v, Op, T identity) {
    const T t = __shfl_up_sync(0xffffffffu, incl, 1);
    (void)v;
    return lane_id() == 0 ? identity : t;
}
template <typename T>
__device__ __forceinline__ T warp_exclusive(T incl, T v, SumOp, T) { return incl - v; }

// Exclusive prefix sum of `v` over an NT-thread block.  wsum: NT / 32 words of shared memory, which hold the
// warp totals afterwards; one barrier inside.  *total (optional): the sum over the block.
template <int NT, typename T>
__device__ __forceinline__ T block_exclusive(T v, T *wsum, T *total = nullptr) {
    constexpr int NW = NT / 32;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const T incl = warp_inclusive(v, SumOp());
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    const T ws = lane < (unsigned)NW ? wsum[lane] : T(0);
    const T wi = warp_inclusive<NW>(ws, SumOp());
    if (total) *total = __shfl_sync(0xffffffffu, wi, NW - 1);
    return __shfl_sync(0xffffffffu, wi - ws, warp) + incl - v;
}

// Exclusive scan of `count` values by one CTA of 1024 threads, 1024 values per step with a carry between
// steps: load(i) gives value i < count, store(i, e) takes its exclusive prefix.  Returns the total to every
// thread.  The index type I is the caller's: a 32-bit count keeps 32-bit index arithmetic.
template <typename T, typename I, typename Load, typename Store, typename Op>
__device__ __forceinline__ T cta_exclusive_scan(I count, Load load, Store store, Op op, T identity) {
    __shared__ T wsum[32];
    __shared__ T carry;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = identity;
    __syncthreads();
    for (I base = 0; base < count; base += 1024) {
        const I i = base + threadIdx.x;
        const T v = i < count ? load(i) : identity;
        const T incl = warp_inclusive(v, op);
        if (lane == 31) wsum[warp] = incl;
        const T ex = warp_exclusive(incl, v, op, identity);
        __syncthreads();
        T pre = carry;
        for (unsigned w = 0; w < warp; ++w) pre = op(pre, wsum[w]);
        const T excl = op(pre, ex);
        if (i < count) store(i, excl);
        __syncthreads();
        if (threadIdx.x == 1023) carry = op(excl, v);
        __syncthreads();
    }
    return carry;
}

// exclusive sum of vals[0, count) in place by one CTA; *total (when not null) = the sum
template <typename T, typename I>
__global__ void __launch_bounds__(1024) scan_sum_kernel(T *__restrict__ vals, I count, T *__restrict__ total) {
    const T t = cta_exclusive_scan(count, [=](I i) { return vals[i]; }, [=](I i, T e) { vals[i] = e; }, SumOp(), T(0));
    if (total && threadIdx.x == 0) *total = t;
}

template <typename T, typename I>
static inline void scan_sum(T *vals, I count, cudaStream_t st, T *total = nullptr) {
    scan_sum_kernel<T, I><<<1, 1024, 0, st>>>(vals, count, total);
    KERNEL_CHECK();
}

}  // namespace b200sa
