// cta_scan.cuh -- the scan of the one-CTA kernels that walk a per-frame (or per-problem) array in blocks of
// CTA_SCAN_THREADS elements: a warp scan, a scan of the 32 warp totals by warp 0, then the carry of earlier blocks.
#ifndef PDA_CTA_SCAN_CUH
#define PDA_CTA_SCAN_CUH

namespace pda {
namespace {

constexpr int CTA_SCAN_THREADS = 1024;  // 32 warps, so one warp scans the warp totals

struct ScanSum {
    template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};
struct ScanMax {
    template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a < b ? b : a; }
};

// x: this thread's element of the current block (op's identity past the end of the array).  Returns op over every element
// up to and including it, earlier blocks included, and advances carry -- the same in every thread, op's identity before
// the first block -- to the total so far.  Every thread of the CTA must make every call; warpTot is 32 entries of shared
// memory.
template <class T, class Op>
__device__ __forceinline__ T cta_scan(T x, T& carry, T* warpTot, Op op) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = op(x, y);
    }
    if (lane == 31) warpTot[warp] = x;
    __syncthreads();
    if (warp == 0) {
        T w = warpTot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w = op(w, y);
        }
        warpTot[lane] = w;
    }
    __syncthreads();
    if (warp) x = op(warpTot[warp - 1], x);
    x = op(carry, x);
    carry = op(carry, warpTot[CTA_SCAN_THREADS / 32 - 1]);
    __syncthreads();  // every thread has read warpTot before the next call writes it
    return x;
}

}  // namespace
}  // namespace pda
#endif
