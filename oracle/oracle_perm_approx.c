/* oracle_perm_approx.c -- CPU restatement of Huber's approximate permanent.  TEST INFRASTRUCTURE ONLY.
 *
 *   orc_permanent_approx  permanentApproximation (nwPerm.cpp:126-140) -> permanentApproximationSquare (:146-211),
 *                         with sinkhorn (:36-77), hl_factor (:80-97), pickRowFromProbs (:110-120)
 *
 * Statement by statement as the reference, sequential sums and products in its order, EXCEPT the random draws: the
 * reference calls glibc rand() without ever seeding it (nwPerm.cpp:106), one process-wide stream whose position
 * depends on everything called before, so there is no reference sample to reproduce.  The draw of (matrix, trial,
 * column) is the same counter-based splitmix64 value the CUDA kernel uses (permanent_approx_kernel.cu: draw01), which
 * makes the two comparable trial for trial; agreement with the reference itself is statistical (same estimator).
 *
 * Near ties.  The kernel forms the same partial sums in another association (a warp prefix sum), and its products over
 * rows and its log() differ from these by a few ulp, so a trial can go the other way only where a draw lies within
 * rounding of a partial sum it was compared with.  Every such draw -- within NEAR_TIE of the sum that reached it or of the
 * one before it, or of the total when no row was picked -- is counted in a thread-local counter
 * (orc_approx_near_ties); a success count that differs from the kernel's by more than that count is a real difference.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "oracle_capi.h"

static const double EE = 2.71828182846;

static uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
static double draw01(uint64_t seed, int64_t mat, int trial, int col) {
    const uint64_t key = mix64(seed ^ (0x9E3779B97F4A7C15ULL * (uint64_t)(mat + 1)));
    const uint64_t x = mix64(key + 0x9E3779B97F4A7C15ULL * ((uint64_t)trial * 64ULL + (uint64_t)col + 1ULL));
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}
static const double NEAR_TIE = 1e-12;
static __thread int64_t g_nearTies = 0;
void orc_approx_near_ties_reset(void) { g_nearTies = 0; }
int64_t orc_approx_near_ties(void) { return g_nearTies; }

static double hl(double x) { return (x > 1.0) ? x + 0.5 * log(x) + EE - 1.0 : 1.0 + (EE - 1.0) * x; }

/* A: rows x cols column-major.  successesOut (optional) receives the number of accepted trials. */
double orc_permanent_approx(const double* A, int64_t rows, int64_t cols, int64_t iterations, uint64_t seed, int64_t matIndex,
                            int64_t* successesOut) {
    const int n = (int)(rows > cols ? rows : cols);
    if (n == 0) return 1.0;
#define B(j, k) Bm[(j) + (size_t)(k) * n]
    double* Bm = (double*)malloc((size_t)n * n * sizeof(double));
    double* C = (double*)malloc((size_t)n * n * sizeof(double));
    double *c = (double*)malloc(n * sizeof(double)), *r = (double*)malloc(n * sizeof(double));
    double *cinv = (double*)malloc(n * sizeof(double)), *rowScale = (double*)malloc(n * sizeof(double));
    double *rowSum0 = (double*)malloc(n * sizeof(double)), *rowSum = (double*)malloc(n * sizeof(double));
    double *h2 = (double*)malloc(n * sizeof(double)), *prob = (double*)malloc(n * sizeof(double));
    for (int k = 0; k < n; k++)
        for (int j = 0; j < n; j++) B(j, k) = (j < rows && k < cols) ? A[j + (size_t)k * rows] : 1.0;  /* ones padding (:135-139) */
    /* sinkhorn (:56-68) */
    for (int k = 0; k < n; k++) { double s = 0; for (int j = 0; j < n; j++) s += B(j, k); c[k] = 1.0 / s; }
    for (int j = 0; j < n; j++) { double s = 0; for (int k = 0; k < n; k++) s += B(j, k) * c[k]; r[j] = 1.0 / s; }
    for (int iter = 0; iter < 100000; iter++) {
        double err = 0; int ok = 1;
        for (int k = 0; k < n; k++) {
            double s = 0; for (int j = 0; j < n; j++) s += r[j] * B(j, k);
            cinv[k] = s;
            const double e = fabs(s * c[k] - 1.0);
            if (!(e <= err)) err = e;            /* maxCoeff; NaN propagates as "not converged" */
            if (e != e) ok = 0;
        }
        if (ok && err <= 1e-4) break;
        for (int k = 0; k < n; k++) c[k] = 1.0 / cinv[k];
        for (int j = 0; j < n; j++) { double s = 0; for (int k = 0; k < n; k++) s += B(j, k) * c[k]; r[j] = 1.0 / s; }
    }
    double prodx = 1, prody = 1;
    for (int j = 0; j < n; j++) prodx *= r[j];
    for (int k = 0; k < n; k++) prody *= c[k];
    for (int k = 0; k < n; k++) for (int j = 0; j < n; j++) B(j, k) = B(j, k) * (r[j] * c[k]);
    /* row scaling (:155-156) */
    for (int j = 0; j < n; j++) {
        double mx = -INFINITY; for (int k = 0; k < n; k++) if (B(j, k) > mx) mx = B(j, k);
        rowScale[j] = 1.0 / mx;
        double s = 0;
        for (int k = 0; k < n; k++) { C[j + (size_t)k * n] = rowScale[j] * B(j, k); s += C[j + (size_t)k * n]; }
        rowSum0[j] = s;
    }
    /* trials (:166-201) */
    int64_t successes = 0;
    char* alive = (char*)malloc(n);
    for (int64_t trial = 0; trial < iterations; trial++) {
        for (int j = 0; j < n; j++) { rowSum[j] = rowSum0[j]; alive[j] = 1; }
        int column = 0;
        while (column < n) {
            double hlAll = 1, hl2All = 1;
            for (int j = 0; j < n; j++) {
                const double ccol = alive[j] ? C[j + (size_t)column * n] : 0.0;
                hlAll *= hl(rowSum[j]) / EE;
                h2[j] = hl(rowSum[j] - ccol);
                hl2All *= h2[j] / EE;
            }
            for (int j = 0; j < n; j++) {
                const double ccol = alive[j] ? C[j + (size_t)column * n] : 0.0;
                prob[j] = (hl2All / hlAll) * EE * (ccol / h2[j]);
            }
            const double u = draw01(seed, matIndex, (int)trial, column);
            double sum = 0, before = 0; int pick;
            for (pick = 0; pick < n; pick++) { before = sum; sum += prob[pick]; if (sum >= u) break; }
            if (fabs(sum - u) <= NEAR_TIE || (pick < n && fabs(before - u) <= NEAR_TIE)) g_nearTies++;
            if (pick >= n) { column = n + 1; break; }
            for (int j = 0; j < n; j++) rowSum[j] = rowSum[j] - (alive[j] ? C[j + (size_t)column * n] : 0.0);
            alive[pick] = 0; rowSum[pick] = 0;
            column++;
        }
        if (column == n) successes++;
    }
    double hlC = 1, scaleProd = 1;
    for (int j = 0; j < n; j++) { hlC *= hl(rowSum0[j]) / EE; scaleProd *= rowScale[j]; }
    double est = hlC * (double)successes / (double)iterations;
    est = est / scaleProd / prodx / prody;
    if (rows != cols) est = est / tgamma(fabs((double)(rows - cols)) + 1);
    if (successesOut) *successesOut = successes;
    free(Bm); free(C); free(c); free(r); free(cinv); free(rowScale); free(rowSum0); free(rowSum); free(h2); free(prob); free(alive);
#undef B
    return est;
}
