// weights_kernel.cu -- the small data-parallel steps either side of the k-best kernel:
//   conditionCosts (assignment.cpp:439-525): per-column minimum, keep rows that have any
//     entry within 42 of their column minimum, shift kept entries, gate the rest to +inf,
//     compact rows (order preserved) and return the row map;
//   toProbs (assignment.cpp:527-542): exp(min - c) for entries within 42 of the global
//     minimum, 0 elsewhere.
// One warp per problem / vector; both are pure streaming passes (HBM-bound, bytes in ~= bytes out).
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <math_constants.h>

#include <algorithm>

namespace pda {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr double GATE = 42.0;  // assignment.cpp:9
constexpr int WARPS = 4;

__device__ __forceinline__ double warp_min(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { double y = __shfl_xor_sync(FULL, x, o); x = (y < x) ? y : x; }
    return x;
}

__global__ void condition_costs_kernel(const double* __restrict__ costs, const int64_t* __restrict__ costOff,
                                       const int32_t* __restrict__ numRow, const int32_t* __restrict__ numCol,
                                       const int64_t nProblems, const int64_t* __restrict__ rowOff,
                                       double* __restrict__ outCosts, int64_t* __restrict__ rowIdx,
                                       int32_t* __restrict__ goodRows, const int32_t* __restrict__ nLopt,
                                       int32_t* __restrict__ condNL, const int32_t maxRow, const int32_t maxCol) {
    __shared__ double colMinS[WARPS][PDA_MAX_DIM];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nProblems) return;
    const int nC = numCol[p];
    const int nR = nLopt ? nLopt[p] + nC : numRow[p];  // the association pipeline passes nL and lets this kernel add
    if (nC > maxCol || nR > maxRow) {  // outside the caller's scope: left alone (colMinS holds PDA_MAX_DIM columns)
        if (lane == 0) { goodRows[p] = 0; if (condNL) condNL[p] = -1; }
        return;
    }
    const double* C = costs + costOff[p];
    double* colMin = colMinS[warp];
    for (int c = 0; c < nC; ++c) {
        double m = CUDART_INF;
        for (int r = lane; r < nR; r += 32) { const double x = C[(size_t)c * nR + r]; m = (x < m) ? x : m; }
        m = warp_min(m);
        if (lane == 0) colMin[c] = m;
    }
    __syncwarp();
    // pass 1: count kept rows
    int good = 0;
    for (int r0 = 0; r0 < nR; r0 += 32) {
        const int r = r0 + lane;
        bool keep = false;
        if (r < nR)
            for (int c = 0; c < nC; ++c)
                if (C[(size_t)c * nR + r] <= colMin[c] + GATE) { keep = true; break; }
        good += __popc(__ballot_sync(FULL, keep));
    }
    // pass 2: compact
    double* out = outCosts + costOff[p];
    int64_t* idx = rowIdx + rowOff[p];
    int base = 0;
    for (int r0 = 0; r0 < nR; r0 += 32) {
        const int r = r0 + lane;
        bool keep = false;
        if (r < nR)
            for (int c = 0; c < nC; ++c)
                if (C[(size_t)c * nR + r] <= colMin[c] + GATE) { keep = true; break; }
        const unsigned m = __ballot_sync(FULL, keep);
        if (keep) {
            const int o = base + __popc(m & ((1u << lane) - 1u));
            idx[o] = r;
            for (int c = 0; c < nC; ++c) {
                const double e = C[(size_t)c * nR + r];
                out[(size_t)c * good + o] = (e <= colMin[c] + GATE) ? e - colMin[c] : CUDART_INF;
            }
        }
        base += __popc(m);
    }
    if (lane == 0) {
        goodRows[p] = good;
        if (condNL) condNL[p] = good - nC;  // condL = goodRows - nM (assignment.cpp:60)
    }
}

__global__ void to_probs_kernel(double* __restrict__ values, const int64_t* __restrict__ off,
                                const int64_t* __restrict__ len, const int64_t nVectors,
                                const int32_t* __restrict__ rows, const int32_t* __restrict__ cols) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nVectors) return;
    double* v = values + off[p];
    const int64_t n = rows ? (int64_t)rows[p] * cols[p] : len[p];
    double lo = CUDART_INF;
    for (int64_t i = lane; i < n; i += 32) { const double x = v[i]; lo = (x < lo) ? x : lo; }
    lo = warp_min(lo);
    for (int64_t i = lane; i < n; i += 32) {
        const double x = v[i];
        v[i] = (lo + GATE > x) ? exp(lo - x) : 0.0;
    }
}

}  // namespace

int launch_condition_costs(const double* costs, const int64_t* costOff, const int32_t* numRow,
                           const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                           double* outCosts, int64_t* rowIdx, int32_t* goodRows, cudaStream_t stream,
                           const int32_t* nLopt, int32_t* condNL, int32_t maxRow, int32_t maxCol) {
    const int64_t ctas = (nProblems + WARPS - 1) / WARPS;
    condition_costs_kernel<<<(unsigned)ctas, 32 * WARPS, 0, stream>>>(costs, costOff, numRow, numCol, nProblems, rowOff,
                                                                      outCosts, rowIdx, goodRows, nLopt, condNL, maxRow, maxCol);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int launch_to_probs(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, cudaStream_t stream,
                    const int32_t* rows, const int32_t* cols) {
    const int64_t ctas = (nVectors + WARPS - 1) / WARPS;
    to_probs_kernel<<<(unsigned)ctas, 32 * WARPS, 0, stream>>>(values, off, len, nVectors, rows, cols);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

}  // namespace pda

using namespace pda;

extern "C" {

int pda_condition_costs_batch(const double* costs, const int64_t* costOff, const int32_t* numRow,
                              const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                              double* outCosts, int64_t* rowIdx, int32_t* goodRows, void* stream) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "condition_costs: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !rowOff || !outCosts || !rowIdx || !goodRows)
        return fail(PDA_ERR_INVALID, "condition_costs: NULL argument");
    // the kernel keeps one column minimum per column in shared memory: a problem with more than PDA_MAX_DIM columns
    // is skipped (goodRows = 0, nothing else written), as the host form rejects it
    return launch_condition_costs(costs, costOff, numRow, numCol, nProblems, rowOff, outCosts, rowIdx, goodRows,
                                  reinterpret_cast<cudaStream_t>(stream), nullptr, nullptr, INT32_MAX, PDA_MAX_DIM);
}

int pda_condition_costs_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow,
                                   const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                                   double* outCosts, int64_t* rowIdx, int32_t* goodRows, int32_t device) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "condition_costs: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !rowOff || !outCosts || !rowIdx || !goodRows)
        return fail(PDA_ERR_INVALID, "condition_costs: NULL argument");
    size_t nCost = 0, nRows = 0;
    for (int64_t p = 0; p < nProblems; ++p) {
        const int r = numRow[p], c = numCol[p];
        if (r < 0 || c < 0 || c > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "condition_costs: problem %lld is %d x %d", (long long)p, r, c);
        nCost = std::max(nCost, (size_t)costOff[p] + (size_t)r * c);
        nRows = std::max(nRows, (size_t)rowOff[p] + r);
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const size_t n = (size_t)nProblems;
    Stage st(device);
    const size_t oC = st.reserve(nCost * 8), oCO = st.reserve(n * 8), oNR = st.reserve(n * 4), oNC = st.reserve(n * 4);
    const size_t oRO = st.reserve(n * 8), oOut = st.reserve(nCost * 8), oIdx = st.reserve(nRows * 8), oG = st.reserve(n * 4);
    PDA_TRY(st.commit());
    cudaStream_t s = 0;
    PDA_TRY(h2d(st.at<double>(oC), costs, nCost, s));
    PDA_TRY(h2d(st.at<int64_t>(oCO), costOff, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oNR), numRow, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oNC), numCol, n, s));
    PDA_TRY(h2d(st.at<int64_t>(oRO), rowOff, n, s));
    PDA_TRY(launch_condition_costs(st.at<double>(oC), st.at<int64_t>(oCO), st.at<int32_t>(oNR), st.at<int32_t>(oNC),
                                   nProblems, st.at<int64_t>(oRO), st.at<double>(oOut), st.at<int64_t>(oIdx),
                                   st.at<int32_t>(oG), s));
    PDA_TRY(d2h(outCosts, st.at<double>(oOut), nCost, s));
    PDA_TRY(d2h(rowIdx, st.at<int64_t>(oIdx), nRows, s));
    PDA_TRY(d2h(goodRows, st.at<int32_t>(oG), n, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    return PDA_OK;
}

int pda_to_probs_batch(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, void* stream) {
    if (nVectors < 0) return fail(PDA_ERR_INVALID, "to_probs: nVectors < 0");
    if (nVectors == 0) return PDA_OK;
    if (!values || !off || !len) return fail(PDA_ERR_INVALID, "to_probs: NULL argument");
    return launch_to_probs(values, off, len, nVectors, reinterpret_cast<cudaStream_t>(stream));
}

int pda_to_probs_batch_host(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, int32_t device) {
    if (nVectors < 0) return fail(PDA_ERR_INVALID, "to_probs: nVectors < 0");
    if (nVectors == 0) return PDA_OK;
    if (!values || !off || !len) return fail(PDA_ERR_INVALID, "to_probs: NULL argument");
    size_t total = 0;
    for (int64_t i = 0; i < nVectors; ++i) total = std::max(total, (size_t)(off[i] + len[i]));
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const size_t n = (size_t)nVectors;
    Stage st(device);
    const size_t oV = st.reserve(total * 8), oO = st.reserve(n * 8), oL = st.reserve(n * 8);
    PDA_TRY(st.commit());
    cudaStream_t s = 0;
    PDA_TRY(h2d(st.at<double>(oV), values, total, s));
    PDA_TRY(h2d(st.at<int64_t>(oO), off, n, s));
    PDA_TRY(h2d(st.at<int64_t>(oL), len, n, s));
    PDA_TRY(launch_to_probs(st.at<double>(oV), st.at<int64_t>(oO), st.at<int64_t>(oL), nVectors, s));
    PDA_TRY(d2h(values, st.at<double>(oV), total, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    return PDA_OK;
}

}  // extern "C"
