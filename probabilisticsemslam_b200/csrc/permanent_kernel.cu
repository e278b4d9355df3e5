// permanent_kernel.cu -- Nijenhuis-Wilf / Ryser matrix permanent for sm_100a.
//
// The reference (nwPerm.cpp:251-332) walks all 2^(n-1) Gray-code column subsets
// sequentially, updating x_j += +-a[j,k] and accumulating +-prod_j x_j.  Here the
// index range [0, 2^(n-1)) is cut into aligned power-of-two chunks, one per thread:
// a thread re-seeds x from the Gray code of its first index (base_j + sum of the set
// columns), then walks its chunk.  Because chunks are aligned, every thread of a CTA
// flips the SAME column at the same step, so the column is read from shared memory as
// a broadcast; x lives in registers (row count is a template parameter, rows padded
// with x == 1); the running sum is kept as an error-free double-double and reduced in
// a fixed order (lane, warp, CTA, then the CTAs of a matrix, added up by the last one
// to finish), so results are reproducible and slightly MORE accurate than the
// reference's single running double.
// Bound: FP64 pipe (n DFMA + n DMUL per subset per thread); the matrix is <= 8 KB.
//
// Rectangular input follows permanentExact (nwPerm.cpp:217-231): pad with ones to
// max(rows, cols), divide by (|rows - cols|)!.
#include "pda_internal.h"
#include "pda_host_stage.h"
#include "perm_device.cuh"
#include "perm_walk.cuh"

#include <algorithm>
#include <vector>

namespace pda {
namespace {

// dd, the walk variants, nw_unit, perm_ld, perm_min_blocks: perm_walk.cuh

struct PermArgs {
    const double* mats; const int64_t* matOff; const int32_t* rows; const int32_t* cols;
    int64_t nMats;
    // range mode (nMats == 1, square): Gray indices [begin, end)
    unsigned long long begin, end;
    int rangeMode;
    int chunk;          // alignment of the per-thread ranges (power of two): below it every thread of a CTA flips
                        // the same column at the same step, so the column read is a shared-memory broadcast
    int threadsPerMat;  // 32..256 (power of two): threads of one CTA that share a matrix
    int ctasPerMat;     // CTAs (blockIdx.x) that share a matrix
    int maxN;           // largest dimension in the batch (sizes the shared-memory slots)
    dd* partial;        // [nMats * ctasPerMat]
    int dpBits;         // matrices whose SMALLER side is <= dpBits go to perm_dp_kernel instead (-1: none)
    unsigned* done;     // [nMats] arrival counters (zero before the launch; the finishing CTA resets its counter)
    double* out; int32_t* status; double* rangePartial;
    int oneDim;         // > 0: a single oneDim x oneDim matrix at mats[0]; rows / cols / matOff are not read (range mode)
};

__device__ __forceinline__ bool perm_uses_dp(const int rows, const int cols, const int dpBits) {
    return (rows < cols ? rows : cols) <= dpBits;
}

// Lane 0 of the CTA that completes matrix m: the raw NW sum s in range mode, else the status and the permanent.
__device__ __forceinline__ void perm_finish(const PermArgs& a, const int64_t m, const dd s) {
    if (a.rangeMode) {
        a.rangePartial[0] = s.hi;
        a.rangePartial[1] = s.lo;
        return;
    }
    // read again rather than kept in registers over the walk
    const int rows = a.oneDim > 0 ? a.oneDim : a.rows[m], cols = a.oneDim > 0 ? a.oneDim : a.cols[m];
    const int n = rows > cols ? rows : cols;
    if (n > PDA_MAX_PERM_DIM) { a.out[m] = 0.0; if (a.status) a.status[m] = 1; return; }  // nwPerm.cpp:327-330 throws
    if (n > a.maxN) { a.out[m] = 0.0; if (a.status) a.status[m] = 2; return; }  // above the call's maxDim: not walked
    if (a.status) a.status[m] = 0;
    a.out[m] = n == 0 ? 1.0 : nw_value(s, rows, cols);  // nwPerm.cpp:261-264
}

// blockIdx.x is the CTA of a matrix, blockIdx.y the group of matrices.  The CTA that completes a matrix finishes it, so a
// large single matrix costs one launch.
template <int NP>
__global__ void __launch_bounds__(PERM_THREADS, perm_min_blocks(NP)) perm_kernel(const PermArgs a) {
    extern __shared__ __align__(16) double smemD[];
    const int tid = threadIdx.x, tpm = a.threadsPerMat, slot = tid / tpm, t = tid % tpm;
    const int64_t m = (int64_t)blockIdx.y * (PERM_THREADS / tpm) + slot;
    double* sA = smemD + (size_t)slot * (perm_ld(NP) * a.maxN + NP);
    const bool live = m < a.nMats;
    const int rows = live ? (a.oneDim > 0 ? a.oneDim : a.rows[m]) : 0, cols = live ? (a.oneDim > 0 ? a.oneDim : a.cols[m]) : 0;
    const int n = rows > cols ? rows : cols;
    const bool ok = live && n >= 1 && n <= NP && n <= PDA_MAX_PERM_DIM && n <= a.maxN && !perm_uses_dp(rows, cols, a.dpBits);
    const bool last = nw_unit<NP>(ok ? a.mats + (a.oneDim > 0 ? 0 : a.matOff[m]) : nullptr, rows, cols, live, ok, a.rangeMode,
                                  a.begin, a.end, a.chunk, tpm, a.ctasPerMat, blockIdx.x, sA, sA + perm_ld(NP) * a.maxN, m,
                                  a.partial, a.ctasPerMat, a.done);
    if (!last || (a.dpBits >= 0 && perm_uses_dp(rows, cols, a.dpBits))) return;
    const dd s = nw_partials_sum(a.partial + (size_t)m * a.ctasPerMat, a.ctasPerMat, t);
    if (t != 0) return;
    perm_finish(a, m, s);
    if (a.ctasPerMat > 1) a.done[m] = 0u;  // ready for the next launch on this stream
}

// ---- matrices with a small side: subset dynamic programme ---------------------------------------------------------
// permanentExact pads an m x n matrix (m < n) with ones to n x n and divides by (n-m)! (nwPerm.cpp:223-230); what that
// computes is the sum over all injective maps of the m short-side indices into the n long-side ones.  The NW walk
// over the padded matrix costs n * 2^(n-1) and -- alternating signs over products of row sums -- cancels: on the
// shapes permanentProb produces (3-8 detections against 10-30 landmark rows, entries spanning many decades) the
// reference's own result is good to 1e-8 at best.  The same sum by dynamic programming over subsets of the SHORT side,
// one long-side index at a time,
//     f_j[S] = f_{j-1}[S] + sum_{i in S} B[i, j] * f_{j-1}[S \ {i}],        perm = f_n[all],
// costs n * 2^m * m / 2 multiply-adds and, for the non-negative matrices of this path, adds only non-negative terms:
// no cancellation, relative error ~ (n + m) ulp.  One warp per matrix, f double-buffered in shared memory, states
// strided over the lanes (S ^ (1 << i) keeps the bank of S: conflict-free).  Used whenever the short side is at most
// PERM_DP_MAX (square matrices included); the reference's n > 32 limit is kept (status 1) so callers see the same
// "throws" behaviour.
__device__ __forceinline__ void perm_dp_warp(const PermArgs& a, const int64_t it, const int rows, const int cols,
                                             double* __restrict__ buf, const int lane) {
    const int n = rows < cols ? cols : rows;
    if (n > PDA_MAX_PERM_DIM) { if (lane == 0) { a.out[it] = 0.0; if (a.status) a.status[it] = 1; } return; }  // nwPerm.cpp:327-330
    const double r = perm_dp_subsets(a.mats + a.matOff[it], rows, cols, buf, 1 << a.dpBits, lane);
    if (lane == 0) { a.out[it] = r; if (a.status) a.status[it] = 0; }
}

// One warp per matrix: the short-sided matrices, which perm_kernel leaves alone.
__global__ void perm_dp_kernel(const PermArgs a) {
    extern __shared__ __align__(16) double smemD[];
    const int64_t m = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= a.nMats) return;
    const int rows = a.rows[m], cols = a.cols[m];
    if (!perm_uses_dp(rows, cols, a.dpBits)) return;
    perm_dp_warp(a, m, rows, cols, smemD + (size_t)(threadIdx.x >> 5) * (2 * ((size_t)1 << a.dpBits) + 16), threadIdx.x & 31);
}

template <int NP>
int launch_np(const PermArgs& a, cudaStream_t stream) {
    const int slots = PERM_THREADS / a.threadsPerMat;
    const size_t smem = (size_t)slots * (perm_ld(NP) * a.maxN + NP) * sizeof(double);
    PDA_CUDA_TRY(cudaFuncSetAttribute(perm_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)a.ctasPerMat, (unsigned)((a.nMats + slots - 1) / slots));
    perm_kernel<NP><<<grid, PERM_THREADS, smem, stream>>>(a);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int dispatch(const PermArgs& a, cudaStream_t stream) {
    return nw_dispatch<2>(a.maxN, [&](auto np) { return launch_np<decltype(np)::value>(a, stream); });
}

}  // namespace

// PermShape / perm_shape: perm_walk.cuh

int launch_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                           int64_t nMats, int32_t maxDim, double* out, int32_t* status, void* workspace,
                           int64_t workspaceBytes, cudaStream_t stream, int32_t maxSmall, int32_t minSmall) {
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    // 0 when maxDim is 0: every matrix with a side then ends as status 2 (perm_kernel)
    const int effDim = std::max(0, std::min<int>(maxDim, PDA_MAX_PERM_DIM));
    // maxSmall / minSmall: bounds on min(rows, cols) over the batch when the caller knows them (else maxDim / 0)
    const int dpBits = std::min(PERM_DP_MAX, std::max(0, std::min<int>(maxSmall < 0 ? maxDim : maxSmall, maxDim)));
    const bool noneDp = minSmall > dpBits;
    // nothing for the NW walk.  Never together with noneDp: the DP path then has no shared memory (dpSmem == 0)
    const bool allDp = !noneDp && (maxSmall >= 0 ? maxSmall : maxDim) <= dpBits;
    const size_t dpSmem = noneDp ? 0 : (size_t)4 * (2 * ((size_t)1 << dpBits) + 16) * sizeof(double);  // 4 warps per DP CTA
    if (dpSmem > 48 * 1024) PDA_CUDA_TRY(cudaFuncSetAttribute(perm_dp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dpSmem));
    if (allDp) {
        PermArgs d = {mats, matOff, rows, cols, nMats, 0, 0, 0, 1, 32, 0, effDim, nullptr, dpBits, nullptr, out, status, nullptr, 0};
        perm_dp_kernel<<<(unsigned)((nMats + 3) / 4), 128, dpSmem, stream>>>(d);
        PDA_CUDA_TRY(cudaGetLastError());
        return PDA_OK;
    }
    // workspace: arrival counters of the matrices, then the per-CTA partial sums
    const int64_t cntBytes = (nMats * 4 + 15) / 16 * 16;
    const int64_t partBytes = workspaceBytes - cntBytes;
    PermShape sh = perm_shape(nMats, effDim, dev.smCount, 0);
    while (sh.ctasPerMat > 1 && (int64_t)sh.ctasPerMat * nMats * (int64_t)sizeof(dd) > partBytes) sh.ctasPerMat >>= 1;
    if ((int64_t)sh.ctasPerMat * nMats * (int64_t)sizeof(dd) > partBytes)
        return fail(PDA_ERR_WORKSPACE, "permanent: workspace of %lld B too small (need %lld)", (long long)workspaceBytes,
                    (long long)(cntBytes + nMats * (int64_t)sizeof(dd)));
    unsigned* done = reinterpret_cast<unsigned*>(workspace);
    if (sh.ctasPerMat > 1) PDA_CUDA_TRY(cudaMemsetAsync(done, 0, (size_t)nMats * 4, stream));
    PermArgs a = {mats, matOff, rows, cols, nMats, 0, 0, 0, sh.chunk, sh.threadsPerMat, sh.ctasPerMat, effDim,
                  reinterpret_cast<dd*>(reinterpret_cast<unsigned char*>(workspace) + cntBytes), noneDp ? -1 : dpBits,
                  done, out, status, nullptr, 0};
    // blockIdx.y is limited to 65535: slice the batch
    const int64_t slots = PERM_THREADS / sh.threadsPerMat, perLaunch = 65535 * slots;
    for (int64_t m0 = 0; m0 < nMats; m0 += perLaunch) {
        PermArgs s = a;
        s.matOff = matOff + m0; s.rows = rows + m0; s.cols = cols + m0;
        s.nMats = std::min<int64_t>(perLaunch, nMats - m0);
        s.partial = a.partial + m0 * sh.ctasPerMat;
        s.done = done + m0;
        s.out = out + m0;
        s.status = status ? status + m0 : nullptr;
        PDA_TRY(dispatch(s, stream));
    }
    if (!noneDp) {  // the short-sided matrices
        perm_dp_kernel<<<(unsigned)((nMats + 3) / 4), 128, dpSmem, stream>>>(a);
        PDA_CUDA_TRY(cudaGetLastError());
    }
    return PDA_OK;
}

int launch_permanent_range(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial,
                           void* workspace, int64_t workspaceBytes, cudaStream_t stream) {
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    PermShape sh = perm_shape(1, n, dev.smCount, end - begin);
    // keep the ranges uniform inside a warp: the chunk must divide `begin`
    while (sh.chunk > 1 && (begin % (unsigned long long)sh.chunk) != 0) sh.chunk >>= 1;
    if ((int64_t)sh.ctasPerMat * (int64_t)sizeof(dd) + 64 > workspaceBytes) {
        sh.ctasPerMat = (int)std::max<int64_t>(1, (workspaceBytes - 64) / (int64_t)sizeof(dd));
        if (workspaceBytes < 64 + (int64_t)sizeof(dd)) return fail(PDA_ERR_WORKSPACE, "permanent_range: workspace too small");
    }
    // one launch: the matrix is described in the kernel arguments (oneDim), the CTA that arrives last adds the per-CTA
    // partials up; the arrival counter at the head of the workspace is zeroed by a memset node in front of the kernel
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    unsigned* done = reinterpret_cast<unsigned*>(ws);
    if (sh.ctasPerMat > 1) PDA_CUDA_TRY(cudaMemsetAsync(done, 0, 4, stream));
    PermArgs a = {A, nullptr, nullptr, nullptr, 1, begin, end, 1, sh.chunk, sh.threadsPerMat, sh.ctasPerMat, n,
                  reinterpret_cast<dd*>(ws + 64), -1, done, nullptr, nullptr, partial, n};
    return dispatch(a, stream);
}

}  // namespace pda

using namespace pda;

extern "C" {

int64_t pda_permanent_workspace_bytes(int64_t nMats) {
    const int64_t n = std::max<int64_t>(nMats, 1);
    return perm_partial_bytes(n) + (n * 4 + 15) / 16 * 16;  // per-CTA partials + arrival counters
}

int pda_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                        int64_t nMats, int32_t maxDim, double* out, int32_t* status,
                        void* workspace, int64_t workspaceBytes, void* stream) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "permanent: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out || !workspace) return fail(PDA_ERR_INVALID, "permanent: NULL argument");
    if (maxDim < 0) return fail(PDA_ERR_INVALID, "permanent: maxDim < 0");
    // the dimensions live on the device, so this entry cannot tell whether any matrix has a short side: it walks every
    // matrix the reference's way (NW on the ones-padded square), tiles 2..32 alike (minSmall above every dpBits keeps
    // perm_dp_warp out).  The *_host entries, which see the dimensions, send short-sided matrices to the
    // cancellation-free subset programme (perm_dp_warp).  A matrix above maxDim ends as status 2 (perm_kernel).
    return launch_permanent_batch(mats, matOff, rows, cols, nMats, maxDim, out, status, workspace, workspaceBytes,
                                  reinterpret_cast<cudaStream_t>(stream), -1, PDA_MAX_DIM + 1);
}

int pda_permanent_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                             int64_t nMats, double* out, int32_t* status, int32_t device) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "permanent: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out) return fail(PDA_ERR_INVALID, "permanent: NULL argument");
    size_t nEl = 0, loEl = ~(size_t)0;  // only [loEl, nEl) of `mats` is staged (a shard passes the whole array)
    int maxDim = 0;
    for (int64_t i = 0; i < nMats; ++i) {
        if (rows[i] < 0 || cols[i] < 0 || matOff[i] < 0) return fail(PDA_ERR_INVALID, "permanent: negative dimension or offset");
        nEl = std::max(nEl, (size_t)matOff[i] + (size_t)rows[i] * cols[i]);
        loEl = std::min(loEl, (size_t)matOff[i]);
        maxDim = std::max(maxDim, std::max(rows[i], cols[i]));
    }
    if (loEl > nEl) loEl = nEl;
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    const size_t n = (size_t)nMats;
    const size_t wsBytes = (size_t)pda_permanent_workspace_bytes(nMats);
    HostIO io(device);
    const size_t oM = io.in(mats + loEl, (nEl - loEl) * 8), oOff = io.in(matOff, n * 8), oR = io.in(rows, n * 4), oC = io.in(cols, n * 4);
    const size_t oOut = io.out(out, n * 8), oSt = io.out(status, n * 4), oWs = io.scratch(wsBytes);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    int maxSmall = 0, minSmall = PDA_MAX_DIM;
    for (int64_t i = 0; i < nMats; ++i) {
        const int sm = std::min(rows[i], cols[i]);
        maxSmall = std::max(maxSmall, sm); minSmall = std::min(minSmall, sm);
    }
    PDA_TRY(launch_permanent_batch(io.at<double>(oM) - loEl, io.at<int64_t>(oOff), io.at<int32_t>(oR), io.at<int32_t>(oC), nMats,
                                   maxDim, io.at<double>(oOut), io.at<int32_t>(oSt), io.at<unsigned char>(oWs),
                                   (int64_t)wsBytes, io.stream(), maxSmall, minSmall));
    return io.download();
}

int pda_permanent_range(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial,
                        void* workspace, int64_t workspaceBytes, void* stream) {
    if (!A || !partial || !workspace) return fail(PDA_ERR_INVALID, "permanent_range: NULL argument");
    if (n < 1 || n > PDA_MAX_PERM_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_range: n = %d outside 1..%d", n, PDA_MAX_PERM_DIM);
    if (begin > end || end > (1ULL << (n - 1))) return fail(PDA_ERR_INVALID, "permanent_range: bad Gray range");
    if (begin == end) {
        PDA_CUDA_TRY(cudaMemsetAsync(partial, 0, 16, reinterpret_cast<cudaStream_t>(stream)));
        return PDA_OK;
    }
    return launch_permanent_range(A, n, begin, end, partial, workspace, workspaceBytes, reinterpret_cast<cudaStream_t>(stream));
}

int pda_permanent_range_host(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial, int32_t device) {
    if (!A || !partial) return fail(PDA_ERR_INVALID, "permanent_range: NULL argument");
    if (n < 1 || n > PDA_MAX_PERM_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_range: n = %d outside 1..%d", n, PDA_MAX_PERM_DIM);
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    const size_t wsBytes = 64 + (size_t)16 * 8192;
    HostIO io(device);
    const size_t oA = io.in(A, (size_t)n * n * 8), oP = io.out(partial, 16), oWs = io.scratch(wsBytes);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    PDA_TRY(pda_permanent_range(io.at<double>(oA), n, begin, end, io.at<double>(oP), io.at<unsigned char>(oWs), (int64_t)wsBytes,
                                io.stream()));
    return io.download();
}

// ---- multi-device forms (SURVEY.md 8e): one host thread per device, no data-path collective except for the single
// large permanent, whose 16-byte partial sums are gathered by the host and added in device order ----------------------
int pda_permanent_batch_host_multi(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                   int64_t nMats, double* out, int32_t* status, const int32_t* devices, int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "permanent (multi): need at least one device");
    if (nMats < 0) return fail(PDA_ERR_INVALID, "permanent: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out || !status) return fail(PDA_ERR_INVALID, "permanent: NULL argument");
    return run_sharded(nMats, devices, nDevices, [&](int64_t m0, int64_t m1, int dev) {
        return pda_permanent_batch_host(mats, matOff + m0, rows + m0, cols + m0, m1 - m0, out + m0, status + m0, dev);
    });
}

int pda_permanent_sharded_host(const double* A, int32_t n, const int32_t* devices, int32_t nDevices, double* out) {
    if (!A || !out) return fail(PDA_ERR_INVALID, "permanent_sharded: NULL argument");
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "permanent_sharded: need at least one device");
    if (n < 1 || n > PDA_MAX_PERM_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_sharded: n = %d outside 1..%d", n, PDA_MAX_PERM_DIM);
    // Gray index range [0, 2^(n-1)) in a power-of-two number of equal pieces: every boundary is a multiple of a large
    // power of two, which keeps the kernel's column reads warp-uniform (launch_permanent_range)
    const uint64_t total = 1ULL << (n - 1);
    int parts = 1;
    while (parts * 2 <= nDevices && (uint64_t)parts * 2 <= total) parts *= 2;
    std::vector<double> partial((size_t)parts * 2, 0.0);
    PDA_TRY(run_sharded(parts, devices, parts, [&](int64_t r0, int64_t r1, int dev) {
        for (int64_t r = r0; r < r1; ++r) {
            const int rc = pda_permanent_range_host(A, n, total * (uint64_t)r / parts, total * (uint64_t)(r + 1) / parts,
                                                    partial.data() + 2 * r, dev);
            if (rc) return rc;
        }
        return (int)PDA_OK;
    }));
    // (hi, lo) pairs added in device order: error-free two-sum on the high parts -- the result does not depend on timing
    double hi = 0.0, lo = 0.0;
    for (int r = 0; r < parts; ++r) {
        const double h = partial[2 * (size_t)r], l = partial[2 * (size_t)r + 1];
        const double s2 = hi + h, bb = s2 - hi, e = (hi - (s2 - bb)) + (h - bb);
        hi = s2;
        lo += e + l;
    }
    *out = (double)(4 * (n & 1) - 2) * (hi + lo);  // sign and factor 2 of the NW formula (nwPerm.cpp:326)
    return PDA_OK;
}

}  // extern "C"
