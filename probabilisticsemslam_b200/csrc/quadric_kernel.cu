// quadric_kernel.cu -- the step in front of the association path: cost matrices from quadric moments.
//
// Reference: computeQuadricCostMatrix (assignment.cpp:705-722) fills the (nL+nM) x nM column-major matrix with the
// squared Mahalanobis distance d^T (cov_l + cov_m)^-1 d between every landmark and every detection, solved with
// Eigen's 3x3 `ldlt().solve(d)` (:716-717), +inf elsewhere and NONASSIGN_QUADRIC on the dummy diagonal (:710, :719);
// getCovs (:693-703) takes the 3x3 shape matrix out of a 4x4 dual quadric.  Built on the device so that a batch of
// frames x window frames never ships cost matrices over PCIe: moments in, association weights out
// (pda_association_from_moments_batch_host = this kernel -> conditionCosts -> k-best weights -> un-compaction).
// The device-pointer forms pda_association_{,perm_}from_moments_batch read the frame shapes on the device instead
// (moment_shapes_kernel), so a CUDA graph captured once with fixed bounds serves frames of any shape (DESIGN.md 3.8b).
//
// Eigen is not installed in this image, so the factorisation below restates Eigen 3.4's published algorithm
// (Cholesky/LDLT.h, ldlt_inplace<Lower>::unblocked: diagonal pivoting with first-maximum ties, unit-lower L, then
// solve = P^T L^-T D^+ L^-1 P with pivots below DBL_MIN treated as zero) rather than a compiled copy of it: results
// agree with any backward-stable 3x3 solve to ~1e-15 relative on SPD input; the parity bar for this row is the
// north_star's 1e-9 relative, checked against the C restatement in oracle/ and against numpy.linalg.solve.
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <algorithm>
#include <cfloat>
#include <math_constants.h>
#include <vector>

namespace pda {
namespace {

constexpr int QWARPS = 8;

// lower-triangular in-place LDLT with diagonal pivoting of the symmetric 3x3 matrix a (a[i][j], i >= j used), then
// x = A^-1 d and the value d . x
__device__ __forceinline__ double mahalanobis3(const double* __restrict__ m1, const double* __restrict__ S1,
                                               const double* __restrict__ m2, const double* __restrict__ S2) {
    double d[3], a[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) d[i] = m1[i] - m2[i];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) a[i][j] = S1[3 * j + i] + S2[3 * j + i];  // column-major 3x3, as Eigen stores it
    int tr[3] = {0, 1, 2};
    bool zero = false;
    // ---- k = 0
    {
        int idx = 0;
        double best = fabs(a[0][0]);
        if (fabs(a[1][1]) > best) { best = fabs(a[1][1]); idx = 1; }
        if (fabs(a[2][2]) > best) { best = fabs(a[2][2]); idx = 2; }
        tr[0] = idx;
        if (idx == 1) {         // swap rows/columns 0 and 1 of the lower triangle
            double t = a[2][0]; a[2][0] = a[2][1]; a[2][1] = t;
            t = a[0][0]; a[0][0] = a[1][1]; a[1][1] = t;
        } else if (idx == 2) {  // swap 0 and 2: the element between them changes sides
            double t = a[0][0]; a[0][0] = a[2][2]; a[2][2] = t;
            t = a[1][0]; a[1][0] = a[2][1]; a[2][1] = t;
        }
        if (!(fabs(a[0][0]) > 0.0)) zero = true;  // the whole matrix is zero: Eigen stops here, D stays zero
        else { a[1][0] /= a[0][0]; a[2][0] /= a[0][0]; }
    }
    if (!zero) {
        // ---- k = 1
        if (fabs(a[2][2]) > fabs(a[1][1])) {
            tr[1] = 2;
            double t = a[1][0]; a[1][0] = a[2][0]; a[2][0] = t;
            t = a[1][1]; a[1][1] = a[2][2]; a[2][2] = t;
        }
        const double t0 = a[0][0] * a[1][0];
        a[1][1] -= a[1][0] * t0;
        a[2][1] -= a[2][0] * t0;
        if (fabs(a[1][1]) > 0.0) a[2][1] /= a[1][1];
        // ---- k = 2
        const double u0 = a[0][0] * a[2][0], u1 = a[1][1] * a[2][1];
        a[2][2] -= a[2][0] * u0 + a[2][1] * u1;
    } else {
        a[0][0] = a[1][1] = a[2][2] = 0.0;
    }
    // ---- solve: P, L^-1, D^+, L^-T, P^T   (scalars and explicit swaps: no dynamically indexed local array)
    double y0 = d[0], y1 = d[1], y2 = d[2], t;
    if (tr[0] == 1) { t = y0; y0 = y1; y1 = t; } else if (tr[0] == 2) { t = y0; y0 = y2; y2 = t; }
    if (tr[1] == 2) { t = y1; y1 = y2; y2 = t; }
    if (!zero) {
        y1 -= y0 * a[1][0];
        y2 -= y0 * a[2][0];
        y2 -= y1 * a[2][1];
    }
    y0 = (fabs(a[0][0]) > DBL_MIN) ? y0 / a[0][0] : 0.0;
    y1 = (fabs(a[1][1]) > DBL_MIN) ? y1 / a[1][1] : 0.0;
    y2 = (fabs(a[2][2]) > DBL_MIN) ? y2 / a[2][2] : 0.0;
    if (!zero) {
        y1 -= a[2][1] * y2;
        y0 -= a[1][0] * y1 + a[2][0] * y2;
    }
    if (tr[1] == 2) { t = y1; y1 = y2; y2 = t; }
    if (tr[0] == 1) { t = y0; y0 = y1; y1 = t; } else if (tr[0] == 2) { t = y0; y0 = y2; y2 = t; }
    const double y[3] = {y0, y1, y2};
    return d[0] * y[0] + (d[1] * y[1] + d[2] * y[2]);
}

// one warp per frame: every entry of the frame's cost matrix is written exactly once
__global__ void quadric_cost_kernel(const double* __restrict__ landMean, const double* __restrict__ landCov,
                                    const int64_t* __restrict__ landOff, const double* __restrict__ measMean,
                                    const double* __restrict__ measCov, const int64_t* __restrict__ measOff,
                                    const long long nFrames, const double nonassign, double* __restrict__ costs,
                                    const int64_t* __restrict__ costOff, int32_t* __restrict__ nLOut,
                                    int32_t* __restrict__ nMOut) {
    const int lane = threadIdx.x & 31;
    const long long f = (long long)blockIdx.x * QWARPS + (threadIdx.x >> 5);
    if (f >= nFrames) return;
    const long long l0 = landOff[f], m0 = measOff[f];
    const int nL = (int)(landOff[f + 1] - l0), nM = (int)(measOff[f + 1] - m0);
    if (lane == 0) {
        if (nLOut) nLOut[f] = nL;
        if (nMOut) nMOut[f] = nM;
    }
    const int nRows = nL + nM;
    double* C = costs + costOff[f];
    for (int e = lane; e < nRows * nM; e += 32) {
        const int col = e / nRows, row = e - col * nRows;
        double v = CUDART_INF;
        if (row < nL) v = mahalanobis3(landMean + 3 * (l0 + row), landCov + 9 * (l0 + row), measMean + 3 * (m0 + col), measCov + 9 * (m0 + col));
        else if (row == nL + col) v = nonassign;
        C[e] = v;
    }
}

// ---- device-pointer moments entries: frame shapes are read on the device, never on the host ----
constexpr unsigned FULL = 0xffffffffu;
constexpr int SHAPE_THREADS = 1024;  // one CTA; 32 warps, so the warp totals are scanned by one warp

struct MomentShapes {
    int32_t* nL; int32_t* nM;            // sanitised counts: 0 / 0 for a rejected frame
    int64_t* landStart; int64_t* measStart;
    int64_t* costOff; int64_t* rowOff;   // fixed strides: f * (maxNL+maxNM) * maxNM and f * (maxNL+maxNM)
    int32_t* innerStatus;                // the usePerm pipeline's status, merged into the caller's afterwards
    double* costs;
    unsigned char* inner;                // workspace of the chained pipeline
    size_t bytes;                        // everything up to `inner`
};

size_t align256(size_t x) { return (x + 255) / 256 * 256; }

MomentShapes carve_shapes(void* workspace, int64_t nFrames, int32_t maxNL, int32_t maxNM) {
    const size_t n = (size_t)std::max<int64_t>(nFrames, 1), rows = (size_t)(maxNL + maxNM);
    unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
    MomentShapes s;
    size_t o = 0;
    s.nL = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    s.nM = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    s.innerStatus = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    s.landStart = reinterpret_cast<int64_t*>(w + o); o += align256(n * 8);
    s.measStart = reinterpret_cast<int64_t*>(w + o); o += align256(n * 8);
    s.costOff = reinterpret_cast<int64_t*>(w + o); o += align256(n * 8);
    s.rowOff = reinterpret_cast<int64_t*>(w + o); o += align256(n * 8);
    s.costs = reinterpret_cast<double*>(w + o); o += align256(n * rows * (size_t)maxNM * 8);
    s.inner = w + o;
    s.bytes = o;
    return s;
}

// One CTA walks the frames in blocks of SHAPE_THREADS.  A frame passes when its offsets are non-negative and ascending,
// lie within landCap / measCap, and its counts are within maxNL / maxNM; probOff is the running sum of nM * (nL+1) over
// passing frames.  A passing non-empty frame whose span ends past probCap keeps its span but is not computed (status
// 2), so probOff stays a plain prefix sum.  Rejected frames go on as 0 x 0: the chained pipelines then touch nothing of
// theirs.
__global__ void __launch_bounds__(SHAPE_THREADS) moment_shapes_kernel(
    const int64_t* __restrict__ landOff, const int64_t landCap, const int64_t* __restrict__ measOff, const int64_t measCap,
    const long long nFrames, const int32_t maxNL, const int32_t maxNM, const int64_t probCap, const MomentShapes s,
    int64_t* __restrict__ probOff, int32_t* __restrict__ status) {
    __shared__ long long warpSum[SHAPE_THREADS / 32];
    __shared__ long long carry;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long long rows = maxNL + maxNM;
    if (t == 0) { carry = 0; probOff[0] = 0; }
    for (long long base = 0; base < nFrames; base += SHAPE_THREADS) {
        const long long f = base + t;
        int L = 0, M = 0;
        long long l0 = 0, m0 = 0;
        bool ok = false;
        if (f < nFrames) {
            l0 = landOff[f]; m0 = measOff[f];
            const long long l1 = landOff[f + 1], m1 = measOff[f + 1];
            ok = l0 >= 0 && m0 >= 0 && l1 >= l0 && m1 >= m0 && l1 <= landCap && m1 <= measCap && l1 - l0 <= maxNL &&
                 m1 - m0 <= maxNM;
            if (ok) { L = (int)(l1 - l0); M = (int)(m1 - m0); }
        }
        const long long span = (long long)M * (L + 1);
        long long x = span;  // inclusive scan: warp, then the warp totals, then the carry of earlier blocks
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(FULL, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warpSum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long w = warpSum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(FULL, w, o);
                if (lane >= o) w += y;
            }
            warpSum[lane] = w;
        }
        __syncthreads();
        const long long end = carry + (warp ? warpSum[warp - 1] : 0) + x;
        if (f < nFrames) {
            if (span > 0 && end > probCap) { ok = false; L = M = 0; }
            s.nL[f] = L; s.nM[f] = M;
            s.landStart[f] = ok ? l0 : 0; s.measStart[f] = ok ? m0 : 0;
            s.costOff[f] = f * rows * maxNM; s.rowOff[f] = f * rows;
            probOff[f + 1] = end;
            status[f] = ok ? 0 : 2;
        }
        __syncthreads();  // every thread has read carry and warpSum
        if (t == SHAPE_THREADS - 1) carry = end;
    }
}

// quadric_cost_kernel on the sanitised shapes: frame f's (nL+nM) x nM matrix at f * slot, which holds the bounds' largest
__global__ void quadric_cost_shaped_kernel(const double* __restrict__ landMean, const double* __restrict__ landCov,
                                           const double* __restrict__ measMean, const double* __restrict__ measCov,
                                           const MomentShapes s, const long long nFrames, const long long slot,
                                           const double nonassign) {
    const int lane = threadIdx.x & 31;
    const long long f = (long long)blockIdx.x * QWARPS + (threadIdx.x >> 5);
    if (f >= nFrames) return;
    const long long l0 = s.landStart[f], m0 = s.measStart[f];
    const int nL = s.nL[f], nM = s.nM[f];
    const int nRows = nL + nM;
    double* C = s.costs + f * slot;
    for (int e = lane; e < nRows * nM; e += 32) {
        const int col = e / nRows, row = e - col * nRows;
        double v = CUDART_INF;
        if (row < nL) v = mahalanobis3(landMean + 3 * (l0 + row), landCov + 9 * (l0 + row), measMean + 3 * (m0 + col), measCov + 9 * (m0 + col));
        else if (row == nL + col) v = nonassign;
        C[e] = v;
    }
}

// status 2 from the shape scan stands; every other frame takes the usePerm pipeline's status
__global__ void merge_status_kernel(const int32_t* __restrict__ inner, const long long nFrames, int32_t* __restrict__ status) {
    const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nFrames && status[f] != 2) status[f] = inner[f];
}

// getCovs (assignment.cpp:693-703): Q is a 4x4 dual quadric, 16 doubles (symmetric, so either storage order)
__global__ void quadric_covs_kernel(const double* __restrict__ Q, const long long n, double* __restrict__ cov) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const double* M = Q + 16 * q;
    double* o = cov + 9 * q;
    const double q03 = M[3], q13 = M[7], q23 = M[11];  // Q(0,3), Q(1,3), Q(2,3) in row-major; identical in column-major
    const double c00 = M[0] + q03 * q03, c01 = M[1] + q03 * q13, c02 = M[2] + q03 * q23;
    const double c11 = M[5] + q13 * q13, c12 = M[6] + q13 * q23, c22 = M[10] + q23 * q23;
    o[0] = c00; o[1] = c01; o[2] = c02;
    o[3] = c01; o[4] = c11; o[5] = c12;
    o[6] = c02; o[7] = c12; o[8] = c22;
}

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

int pda_quadric_covs_batch(const double* quadrics, int64_t n, double* covs, void* stream) {
    if (n < 0) return fail(PDA_ERR_INVALID, "quadric_covs: n < 0");
    if (n == 0) return PDA_OK;
    if (!quadrics || !covs) return fail(PDA_ERR_INVALID, "quadric_covs: NULL argument");
    quadric_covs_kernel<<<(unsigned)((n + 127) / 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(quadrics, n, covs);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int pda_quadric_covs_batch_host(const double* quadrics, int64_t n, double* covs, int32_t device) {
    if (n < 0) return fail(PDA_ERR_INVALID, "quadric_covs: n < 0");
    if (n == 0) return PDA_OK;
    if (!quadrics || !covs) return fail(PDA_ERR_INVALID, "quadric_covs: NULL argument");
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    Stage st(device);
    const size_t oQ = st.reserve((size_t)n * 16 * 8), oC = st.reserve((size_t)n * 9 * 8);
    PDA_TRY(st.commit());
    cudaStream_t s = 0;
    PDA_TRY(h2d(st.at<double>(oQ), quadrics, (size_t)n * 16, s));
    PDA_TRY(pda_quadric_covs_batch(st.at<double>(oQ), n, st.at<double>(oC), s));
    PDA_TRY(d2h(covs, st.at<double>(oC), (size_t)n * 9, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    return PDA_OK;
}

int pda_quadric_cost_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                           const double* measMean, const double* measCov, const int64_t* measOff,
                           int64_t nFrames, double nonassign, double* costs, const int64_t* costOff,
                           int32_t* nL, int32_t* nM, void* stream) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "quadric_cost: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!landOff || !measOff || !costs || !costOff) return fail(PDA_ERR_INVALID, "quadric_cost: NULL argument");
    quadric_cost_kernel<<<(unsigned)((nFrames + QWARPS - 1) / QWARPS), 32 * QWARPS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        landMean, landCov, landOff, measMean, measCov, measOff, nFrames, nonassign, costs, costOff, nL, nM);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

// host-side shape scan shared by the two *_host entry points below
static int quadric_shapes(const int64_t* landOff, const int64_t* measOff, int64_t nFrames, std::vector<int64_t>& costOff,
                          std::vector<int64_t>& probOff, std::vector<int64_t>& rowOff, size_t& nCost, size_t& nProb,
                          size_t& nRows, int& maxR, int& maxC) {
    const size_t n = (size_t)nFrames;
    costOff.resize(n); probOff.resize(n); rowOff.resize(n);
    nCost = nProb = nRows = 0; maxR = 1; maxC = 1;
    for (size_t f = 0; f < n; ++f) {
        const int64_t L = landOff[f + 1] - landOff[f], M = measOff[f + 1] - measOff[f];
        if (L < 0 || M < 0) return fail(PDA_ERR_INVALID, "quadric: offsets of frame %lld are not ascending", (long long)f);
        if (L + M > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "quadric: frame %lld has %lld landmarks + %lld detections (limit %d)",
                                             (long long)f, (long long)L, (long long)M, PDA_MAX_DIM);
        costOff[f] = (int64_t)nCost; probOff[f] = (int64_t)nProb; rowOff[f] = (int64_t)nRows;
        nCost += (size_t)((L + M) * M); nProb += (size_t)(M * (L + 1)); nRows += (size_t)(L + M);
        maxR = std::max(maxR, (int)(L + M)); maxC = std::max(maxC, (int)M);
    }
    return PDA_OK;
}

int pda_quadric_cost_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                const double* measMean, const double* measCov, const int64_t* measOff,
                                int64_t nFrames, double nonassign, double* costs, int32_t device) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "quadric_cost: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!landOff || !measOff || !costs) return fail(PDA_ERR_INVALID, "quadric_cost: NULL argument");
    std::vector<int64_t> costOff, probOff, rowOff;
    size_t nCost, nProb, nRows; int maxR, maxC;
    PDA_TRY(quadric_shapes(landOff, measOff, nFrames, costOff, probOff, rowOff, nCost, nProb, nRows, maxR, maxC));
    const size_t n = (size_t)nFrames, nLand = (size_t)landOff[n], nMeas = (size_t)measOff[n];
    if ((nLand && (!landMean || !landCov)) || (nMeas && (!measMean || !measCov))) return fail(PDA_ERR_INVALID, "quadric_cost: NULL moments");
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    Stage st(device);
    PackedIO io(st);
    const size_t oLM = io.in(landMean, nLand * 24), oLC = io.in(landCov, nLand * 72), oLO = io.in(landOff, (n + 1) * 8);
    const size_t oMM = io.in(measMean, nMeas * 24), oMC = io.in(measCov, nMeas * 72), oMO = io.in(measOff, (n + 1) * 8);
    const size_t oCO = io.in(costOff.data(), n * 8);
    const size_t oC = io.out(costs, nCost * 8);
    PDA_TRY(st.commit());
    HostStreams* hs = nullptr;
    PDA_TRY(host_streams(device, &hs));
    PDA_TRY(io.upload(hs->run));
    PDA_TRY(pda_quadric_cost_batch(st.at<double>(oLM), st.at<double>(oLC), st.at<int64_t>(oLO), st.at<double>(oMM), st.at<double>(oMC),
                                   st.at<int64_t>(oMO), nFrames, nonassign, st.at<double>(oC), st.at<int64_t>(oCO), nullptr, nullptr, hs->run));
    return io.download(hs->run);
}

// getAssignmentProbs (assignment.cpp:38-74, usePerm == 0) from the quadric moments on, one stream, no host round trip:
// cost matrices -> conditionCosts -> assignmentProb(k) -> weights at the original landmark indices.
// probs of frame f: nM x (nL+1) row-major at the prefix sum of nM*(nL+1) (frames with nM == 0 contribute nothing;
// nL == 0 gives {1} per detection, :49-53).
int pda_association_from_moments_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                            const double* measMean, const double* measCov, const int64_t* measOff,
                                            int64_t nFrames, double nonassign, int32_t k, double* probs, int32_t device) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "association_from_moments: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!landOff || !measOff || !probs) return fail(PDA_ERR_INVALID, "association_from_moments: NULL argument");
    if (k < 1) return fail(PDA_ERR_INVALID, "association_from_moments: k < 1");
    std::vector<int64_t> costOff, probOff, rowOff;
    size_t nCost, nProb, nRows; int maxR, maxC;
    PDA_TRY(quadric_shapes(landOff, measOff, nFrames, costOff, probOff, rowOff, nCost, nProb, nRows, maxR, maxC));
    const size_t n = (size_t)nFrames, nLand = (size_t)landOff[n], nMeas = (size_t)measOff[n];
    if ((nLand && (!landMean || !landCov)) || (nMeas && (!measMean || !measCov))) return fail(PDA_ERR_INVALID, "association_from_moments: NULL moments");
    if (nProb == 0) return PDA_OK;
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const int64_t wsBytes = pda_association_workspace_bytes(nFrames, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, k, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    Stage st(device);
    PackedIO io(st);
    const size_t oLM = io.in(landMean, nLand * 24), oLC = io.in(landCov, nLand * 72), oLO = io.in(landOff, (n + 1) * 8);
    const size_t oMM = io.in(measMean, nMeas * 24), oMC = io.in(measCov, nMeas * 72), oMO = io.in(measOff, (n + 1) * 8);
    const size_t oCO = io.in(costOff.data(), n * 8), oPO = io.in(probOff.data(), n * 8), oRO = io.in(rowOff.data(), n * 8);
    const size_t oP = io.out(probs, nProb * 8);
    const size_t oC = st.reserve(nCost * 8), oNL = st.reserve(n * 4), oNM = st.reserve(n * 4), oWs = st.reserve((size_t)wsBytes);
    PDA_TRY(st.commit());
    HostStreams* hs = nullptr;
    PDA_TRY(host_streams(device, &hs));
    cudaStream_t s = hs->run;
    PDA_TRY(io.upload(s));
    PDA_TRY(pda_quadric_cost_batch(st.at<double>(oLM), st.at<double>(oLC), st.at<int64_t>(oLO), st.at<double>(oMM), st.at<double>(oMC),
                                   st.at<int64_t>(oMO), nFrames, nonassign, st.at<double>(oC), st.at<int64_t>(oCO),
                                   st.at<int32_t>(oNL), st.at<int32_t>(oNM), s));
    PDA_TRY(pda_association_probs_batch(st.at<double>(oC), st.at<int64_t>(oCO), st.at<int32_t>(oNL), st.at<int32_t>(oNM),
                                        st.at<int64_t>(oRO), nFrames, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC, k,
                                        st.at<double>(oP), st.at<int64_t>(oPO), nullptr, st.at<unsigned char>(oWs), wsBytes, s));
    return io.download(s);
}

}  // extern "C"

// argument checks shared by the device-pointer moments entries
static int moments_args(const char* who, int64_t nFrames, int32_t maxNL, int32_t maxNM, int64_t probCapacity) {
    if (nFrames < 0 || maxNL < 0 || maxNM < 1 || probCapacity < 0)
        return fail(PDA_ERR_INVALID, "%s: nFrames %lld, maxNL %d, maxNM %d, probCapacity %lld", who, (long long)nFrames, maxNL,
                    maxNM, (long long)probCapacity);
    if ((int64_t)maxNL + maxNM > PDA_MAX_DIM)
        return fail(PDA_ERR_UNSUPPORTED, "%s: maxNL + maxNM = %lld above %d", who, (long long)maxNL + maxNM, PDA_MAX_DIM);
    return PDA_OK;
}

// the shape scan and the cost matrices in front of either pipeline
static int launch_moment_costs(const double* landMean, const double* landCov, const int64_t* landOff, int64_t landCapacity,
                               const double* measMean, const double* measCov, const int64_t* measOff, int64_t measCapacity,
                               int64_t nFrames, int32_t maxNL, int32_t maxNM, double nonassign, int64_t probCapacity,
                               const MomentShapes& sh, int64_t* probOff, int32_t* status, cudaStream_t s) {
    moment_shapes_kernel<<<1, SHAPE_THREADS, 0, s>>>(landOff, landCapacity, measOff, measCapacity, nFrames, maxNL, maxNM,
                                                    probCapacity, sh, probOff, status);
    PDA_CUDA_TRY(cudaGetLastError());
    if (nFrames == 0) return PDA_OK;
    quadric_cost_shaped_kernel<<<(unsigned)((nFrames + QWARPS - 1) / QWARPS), 32 * QWARPS, 0, s>>>(
        landMean, landCov, measMean, measCov, sh, nFrames, (long long)(maxNL + maxNM) * maxNM, nonassign);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

extern "C" {

int64_t pda_association_from_moments_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxNM, int64_t probCapacity,
                                                     int32_t k) {
    PDA_TRY(moments_args("association_from_moments", nFrames, maxNL, maxNM, probCapacity));
    if (k < 1) return fail(PDA_ERR_INVALID, "association_from_moments: k < 1");
    const int64_t n = std::max<int64_t>(nFrames, 1), rows = maxNL + maxNM;
    const int64_t inner = pda_association_workspace_bytes(n, n * rows * maxNM, n * rows, probCapacity, k, (int32_t)rows, maxNM);
    if (inner < 0) return inner;
    return (int64_t)carve_shapes(nullptr, nFrames, maxNL, maxNM).bytes + inner;
}

int pda_association_from_moments_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                                       int64_t landCapacity,
                                       const double* measMean, const double* measCov, const int64_t* measOff,
                                       int64_t measCapacity, int64_t nFrames, int32_t maxNL, int32_t maxNM,
                                       double nonassign, int32_t k,
                                       double* probs, int64_t probCapacity, int64_t* probOff,
                                       int32_t* status, int32_t* nFound,
                                       void* workspace, int64_t workspaceBytes, void* stream) {
    if (!landMean || !landCov || !landOff || !measMean || !measCov || !measOff || !probs || !probOff || !status || !workspace)
        return fail(PDA_ERR_INVALID, "association_from_moments: NULL argument");
    if (landCapacity < 0 || measCapacity < 0) return fail(PDA_ERR_INVALID, "association_from_moments: negative capacity");
    const int64_t wsBytes = pda_association_from_moments_workspace_bytes(nFrames, maxNL, maxNM, probCapacity, k);
    if (wsBytes < 0) return (int)wsBytes;
    if (workspaceBytes < wsBytes)
        return fail(PDA_ERR_WORKSPACE, "association_from_moments: workspace of %lld B, %lld B needed", (long long)workspaceBytes,
                    (long long)wsBytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const MomentShapes sh = carve_shapes(workspace, nFrames, maxNL, maxNM);
    PDA_TRY(launch_moment_costs(landMean, landCov, landOff, landCapacity, measMean, measCov, measOff, measCapacity, nFrames, maxNL,
                                maxNM, nonassign, probCapacity, sh, probOff, status, s));
    if (nFrames == 0) return PDA_OK;
    const int64_t rows = maxNL + maxNM;
    return pda_association_probs_batch(sh.costs, sh.costOff, sh.nL, sh.nM, sh.rowOff, nFrames, nFrames * rows * maxNM, nFrames * rows,
                                       probCapacity, (int32_t)rows, maxNM, k, probs, probOff, nFound, sh.inner,
                                       workspaceBytes - (int64_t)sh.bytes, stream);
}

int64_t pda_association_perm_from_moments_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxNM, int64_t probCapacity) {
    PDA_TRY(moments_args("association_perm_from_moments", nFrames, maxNL, maxNM, probCapacity));
    const int64_t n = std::max<int64_t>(nFrames, 1), rows = maxNL + maxNM;
    const int64_t inner = pda_association_perm_workspace_bytes(n, n * rows * maxNM, n * rows, probCapacity, (int32_t)rows, maxNM);
    if (inner < 0) return inner;
    return (int64_t)carve_shapes(nullptr, nFrames, maxNL, maxNM).bytes + inner;
}

int pda_association_perm_from_moments_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                                            int64_t landCapacity,
                                            const double* measMean, const double* measCov, const int64_t* measOff,
                                            int64_t measCapacity, int64_t nFrames, int32_t maxNL, int32_t maxNM,
                                            double nonassign,
                                            double* probs, int64_t probCapacity, int64_t* probOff, int32_t* status,
                                            void* workspace, int64_t workspaceBytes, void* stream) {
    if (!landMean || !landCov || !landOff || !measMean || !measCov || !measOff || !probs || !probOff || !status || !workspace)
        return fail(PDA_ERR_INVALID, "association_perm_from_moments: NULL argument");
    if (landCapacity < 0 || measCapacity < 0) return fail(PDA_ERR_INVALID, "association_perm_from_moments: negative capacity");
    const int64_t wsBytes = pda_association_perm_from_moments_workspace_bytes(nFrames, maxNL, maxNM, probCapacity);
    if (wsBytes < 0) return (int)wsBytes;
    if (workspaceBytes < wsBytes)
        return fail(PDA_ERR_WORKSPACE, "association_perm_from_moments: workspace of %lld B, %lld B needed",
                    (long long)workspaceBytes, (long long)wsBytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const MomentShapes sh = carve_shapes(workspace, nFrames, maxNL, maxNM);
    PDA_TRY(launch_moment_costs(landMean, landCov, landOff, landCapacity, measMean, measCov, measOff, measCapacity, nFrames, maxNL,
                                maxNM, nonassign, probCapacity, sh, probOff, status, s));
    if (nFrames == 0) return PDA_OK;
    const int64_t rows = maxNL + maxNM;
    PDA_TRY(pda_association_perm_probs_batch(sh.costs, sh.costOff, sh.nL, sh.nM, sh.rowOff, nFrames, nFrames * rows * maxNM,
                                             nFrames * rows, probCapacity, (int32_t)rows, maxNM, probs, probOff, sh.innerStatus,
                                             sh.inner, workspaceBytes - (int64_t)sh.bytes, stream));
    merge_status_kernel<<<(unsigned)((nFrames + 255) / 256), 256, 0, s>>>(sh.innerStatus, nFrames, status);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

}  // extern "C"
