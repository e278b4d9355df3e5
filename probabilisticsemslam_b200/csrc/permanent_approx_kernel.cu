// permanent_approx_kernel.cu -- Huber's randomised approximation of the permanent, batched (SURVEY.md 8f rank 4).
//
// Reference: permanentApproximation / permanentApproximationSquare / sinkhorn / hl_factor / pickRowFromProbs
// (nwPerm.cpp:36-211), reached through conditionedPermanent(.., permOpt = 0) (assignment.cpp:401) with
// apprxIter = 300 trials (assignment.cpp:10): Sinkhorn-balance the matrix, scale rows to a unit maximum, then run
// `iterations` acceptance/rejection trials that each try to draw a permutation column by column with probabilities
// built from the Huber-Law bound, and return bound * successes / iterations, un-scaled.
//
// One warp per matrix, lane j = row j (and column j where a column-wise quantity is needed); the matrix lives in
// shared memory with a leading dimension of 33 so that both row-wise and column-wise sweeps are conflict-free; the
// products over rows are shuffle trees and the row pick is a warp prefix sum + ballot.
//
// Parity.  The reference draws from glibc rand() WITHOUT seeding, one global stream consumed in call order, so its
// estimate depends on everything the process did before -- there is nothing bit-exact to match.  Here every draw is a
// counter-based splitmix64 value keyed by (seed, matrix, trial, column): results are reproducible, independent of
// batch order, and the CPU restatement in oracle/oracle_perm_approx.c uses the same stream.  What is checked: against the
// restatement (same draws; the two differ only when a pick falls within rounding of a cumulative sum), and against
// the exact permanent within the estimator's own binomial standard error.  Matrices above dimension 32 get status 1
// (the reference has no such limit; the exact path has, nwPerm.cpp:329).
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <math_constants.h>

#include <algorithm>

namespace pda {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int AW = 4;     // warps (matrices) per CTA
constexpr int LD = 33;    // leading dimension in shared memory
constexpr double EE = 2.71828182846;  // the reference's constant (nwPerm.cpp:88, 162)

__device__ __forceinline__ double warp_prod(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) x *= __shfl_xor_sync(FULL, x, o);
    return x;
}
__device__ __forceinline__ double warp_maxd(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { const double y = __shfl_xor_sync(FULL, x, o); x = (x < y) ? y : x; }
    return x;
}
// hl_factor (nwPerm.cpp:80-97)
__device__ __forceinline__ double hl(double x) { return (x > 1.0) ? x + 0.5 * log(x) + EE - 1.0 : 1.0 + (EE - 1.0) * x; }

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
// the draw of (matrix, trial, column): uniform in [0, 1)
__device__ __forceinline__ double draw01(unsigned long long seed, long long mat, int trial, int col) {
    const unsigned long long key = mix64(seed ^ (0x9E3779B97F4A7C15ULL * (unsigned long long)(mat + 1)));
    const unsigned long long x = mix64(key + 0x9E3779B97F4A7C15ULL * ((unsigned long long)trial * 64ULL + (unsigned long long)col + 1ULL));
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}

struct ApproxArgs {
    const double* mats; const int64_t* matOff; const int32_t* rows; const int32_t* cols;
    int64_t nMats;
    int32_t iterations;
    unsigned long long seed;
    double* out; int32_t* status;
};

__global__ void __launch_bounds__(32 * AW) permanent_approx_kernel(const ApproxArgs a) {
    __shared__ double sC[AW][32 * LD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long m = (long long)blockIdx.x * AW + warp;
    if (m >= a.nMats) return;
    const int rows = a.rows[m], cols = a.cols[m];
    const int n = rows > cols ? rows : cols;
    if (n > PDA_MAX_PERM_DIM || n < 0) {
        if (lane == 0) { a.out[m] = 0.0; if (a.status) a.status[m] = 1; }
        return;
    }
    if (lane == 0 && a.status) a.status[m] = 0;
    if (n == 0) { if (lane == 0) a.out[m] = 1.0; return; }
    double* C = sC[warp];
    const double* A = a.mats + a.matOff[m];
    // A_pad = Ones(dim, dim); A_pad.block(0, 0, m, n) = A  (nwPerm.cpp:135-139); entry (j, k) at C[j + k*LD]
    for (int e = lane; e < n * n; e += 32) {
        const int j = e % n, k = e / n;
        C[j + k * LD] = (j < rows && k < cols) ? A[j + (size_t)k * rows] : 1.0;
    }
    __syncwarp();
    const bool live = lane < n;

    // ---- sinkhorn(A, 1e-4) (nwPerm.cpp:36-77): lane = column for c / cinv, lane = row for r --------------
    double c = 1.0, r = 1.0;
    {
        double s = 0.0;
        if (live) for (int j = 0; j < n; ++j) s += C[j + lane * LD];
        c = live ? 1.0 / s : 1.0;
        s = 0.0;
        for (int k = 0; k < n; ++k) { const double ck = __shfl_sync(FULL, c, k); if (live) s += C[lane + k * LD] * ck; }
        r = live ? 1.0 / s : 1.0;
        for (int iter = 0; iter < 100000; ++iter) {
            double cinv = 0.0;
            for (int j = 0; j < n; ++j) { const double rj = __shfl_sync(FULL, r, j); if (live) cinv += rj * C[j + lane * LD]; }
            const double err = warp_maxd(live ? fabs(cinv * c - 1.0) : 0.0);
            if (err <= 1e-4) break;  // NaN compares false and keeps iterating, like the reference
            c = live ? 1.0 / cinv : 1.0;
            s = 0.0;
            for (int k = 0; k < n; ++k) { const double ck = __shfl_sync(FULL, c, k); if (live) s += C[lane + k * LD] * ck; }
            r = live ? 1.0 / s : 1.0;
        }
    }
    const double prodx = warp_prod(live ? r : 1.0), prody = warp_prod(live ? c : 1.0);
    // B = B .* (r c^T); row_scale = 1 / rowwise max; C = diag(row_scale) B  (nwPerm.cpp:70, 155-156)
    double rowMax = -CUDART_INF;
    for (int k = 0; k < n; ++k) {
        const double ck = __shfl_sync(FULL, c, k);
        if (live) {
            const double b = C[lane + k * LD] * (r * ck);
            C[lane + k * LD] = b;
            rowMax = (b > rowMax) ? b : rowMax;
        }
    }
    const double rowScale = live ? 1.0 / rowMax : 1.0;
    double rowSum0 = 0.0;
    for (int k = 0; k < n; ++k)
        if (live) {
            const double v = rowScale * C[lane + k * LD];
            C[lane + k * LD] = v;
            rowSum0 += v;
        }
    __syncwarp();

    // ---- the trials (nwPerm.cpp:166-201) ----------------------------------------------------------------------
    int successes = 0;
    for (int trial = 0; trial < a.iterations; ++trial) {
        double rowSum = rowSum0;
        bool alive = live;  // a picked row is zeroed for the rest of the trial
        int column = 0;
        while (column < n) {
            const double ccol = alive ? C[lane + column * LD] : 0.0;
            const double h = hl(rowSum), h2 = hl(rowSum - ccol);
            const double hlAll = warp_prod(live ? h / EE : 1.0);
            const double hl2All = warp_prod(live ? h2 / EE : 1.0);
            double p = live ? (hl2All / hlAll) * EE * (ccol / h2) : 0.0;
            // pickRowFromProbs: first row whose running sum reaches the draw
            double run = p;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const double y = __shfl_up_sync(FULL, run, o); if (lane >= o) run += y; }
            const double u = draw01(a.seed, m, trial, column);
            const unsigned hit = __ballot_sync(FULL, live && run >= u);
            if (hit == 0u) break;  // no row: the trial failed
            const int pick = __ffs(hit) - 1;
            rowSum = rowSum - ccol;
            if (lane == pick) { alive = false; rowSum = 0.0; }
            column++;
        }
        if (column == n) successes++;
    }
    const double hlC = warp_prod(live ? hl(rowSum0) / EE : 1.0);
    const double scaleProd = warp_prod(live ? rowScale : 1.0);
    if (lane == 0) {
        double est = hlC * (double)successes / (double)a.iterations;
        est = est / scaleProd / prodx / prody;
        if (rows != cols) {  // / tgamma(|m - n| + 1)
            double f = 1.0;
            const int d = rows > cols ? rows - cols : cols - rows;
            for (int i = 2; i <= d; ++i) f *= (double)i;
            est = est / f;
        }
        a.out[m] = est;
    }
}

}  // namespace

int launch_permanent_approx_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                  int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status,
                                  cudaStream_t stream) {
    if (nMats <= 0) return PDA_OK;
    ApproxArgs a = {mats, matOff, rows, cols, nMats, iterations, (unsigned long long)seed, out, status};
    permanent_approx_kernel<<<(unsigned)((nMats + AW - 1) / AW), 32 * AW, 0, stream>>>(a);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

}  // namespace pda

using namespace pda;

extern "C" {

int pda_permanent_approx_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                               int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status, void* stream) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "permanent_approx: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out) return fail(PDA_ERR_INVALID, "permanent_approx: NULL argument");
    if (iterations < 1) return fail(PDA_ERR_INVALID, "permanent_approx: iterations < 1");
    return launch_permanent_approx_batch(mats, matOff, rows, cols, nMats, iterations, seed, out, status,
                                         reinterpret_cast<cudaStream_t>(stream));
}

int pda_permanent_approx_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                    int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status,
                                    int32_t device) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "permanent_approx: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out || !status) return fail(PDA_ERR_INVALID, "permanent_approx: NULL argument");
    if (iterations < 1) return fail(PDA_ERR_INVALID, "permanent_approx: iterations < 1");
    size_t nEl = 0;
    for (int64_t i = 0; i < nMats; ++i) {
        if (rows[i] < 0 || cols[i] < 0) return fail(PDA_ERR_INVALID, "permanent_approx: negative dimension");
        nEl = std::max(nEl, (size_t)matOff[i] + (size_t)rows[i] * cols[i]);
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const size_t n = (size_t)nMats;
    HostIO io(device);
    const size_t oM = io.in(mats, nEl * 8), oOff = io.in(matOff, n * 8), oR = io.in(rows, n * 4), oC = io.in(cols, n * 4);
    const size_t oOut = io.out(out, n * 8), oSt = io.out(status, n * 4);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    PDA_TRY(launch_permanent_approx_batch(io.at<double>(oM), io.at<int64_t>(oOff), io.at<int32_t>(oR), io.at<int32_t>(oC), nMats,
                                          iterations, seed, io.at<double>(oOut), io.at<int32_t>(oSt), io.stream()));
    return io.download();
}

}  // extern "C"
