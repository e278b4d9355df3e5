/* oracle_assign.c -- CPU parity oracle for the association-weight functions.
 * TEST INFRASTRUCTURE ONLY (see oracle_capi.h).
 *
 * Restates, on flat arrays, the numeric half of the reference's assignment.cpp:
 *   conditionCosts   :439-525      toProbs          :527-542
 *   assignmentProb   :547-683      bruteForceProb   :835-964 (+ mincConstant/mincFactor :28-36)
 *   permanentProb    :145-290      setupAssgnMatrix :292-323
 * Probability tables are returned flat, row-major [measurement][landmark 0..nL-1, non-assignment].
 */
#include "oracle_capi.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define PDA_GATE 42.0 /* assignment.cpp:9  `const static size_t cutoff = 42` */
#define PDA_TAU 6.2831853071 /* assignment.cpp:11 */

int64_t orc_condition_costs(const double* costs, int64_t nRows, int64_t nCols, double* outCosts, int64_t* rowIdx) {
    double* colMin = (double*)malloc((size_t)(nCols > 0 ? nCols : 1) * sizeof(double));
    uint8_t* keep = (uint8_t*)malloc((size_t)(nRows > 0 ? nRows : 1));
    for (int64_t c = 0; c < nCols; c++) {
        double m = INFINITY;
        for (int64_t r = 0; r < nRows; r++) if (costs[c * nRows + r] < m) m = costs[c * nRows + r];
        colMin[c] = m;
    }
    int64_t good = 0;
    for (int64_t r = 0; r < nRows; r++) {
        keep[r] = 0;
        for (int64_t c = 0; c < nCols; c++)
            if (costs[c * nRows + r] <= colMin[c] + PDA_GATE) { keep[r] = 1; good++; break; }
    }
    int64_t o = 0;
    for (int64_t r = 0; r < nRows; r++) {
        if (!keep[r]) continue;
        rowIdx[o] = r;
        for (int64_t c = 0; c < nCols; c++) {
            double e = costs[c * nRows + r];
            outCosts[c * good + o] = (e <= colMin[c] + PDA_GATE) ? e - colMin[c] : INFINITY;
        }
        o++;
    }
    free(colMin);
    free(keep);
    return good;
}

void orc_to_probs(double* v, int64_t n) {
    if (n <= 0) return;
    double lo = v[0];
    for (int64_t i = 1; i < n; i++) if (v[i] < lo) lo = v[i];
    for (int64_t i = 0; i < n; i++) v[i] = (lo + PDA_GATE > v[i]) ? exp(lo - v[i]) : 0;
}

/* single-detection shortcut shared by assignmentProb (:554-570) and bruteForceProb (:840-856) */
static void single_column(const double* costs, int64_t nL, double* probs) {
    double norm = 0;
    for (int64_t i = 0; i <= nL; i++) {
        probs[i] = 0;
        if (costs[i] < PDA_GATE) { probs[i] = exp(-costs[i]); norm += probs[i]; }
    }
    norm = 1.0 / norm;
    for (int64_t i = 0; i <= nL; i++) probs[i] = probs[i] * norm;
}

/* k-best list -> marginals (:616-648 / :912-945) */
static void marginalise(const int64_t* r4c, const double* gains, int64_t nFound, int64_t nL, int64_t nM,
                        int gate, double* probs) {
    const int64_t W = nL + 1;
    for (int64_t i = 0; i < nM * W; i++) probs[i] = 0;
    /* with nFound == 0 the reference reads an uninitialised best cost and ends up multiplying zeros by 1/0 */
    const double best = nFound > 0 ? gains[0] : 0.0;
    double total = 0;
    for (int64_t s = 0; s < nFound; s++) {
        if (gate && !(best + PDA_GATE > gains[s])) continue;
        const double w = exp(best - gains[s]);
        total += w;
        for (int64_t c = 0; c < nM; c++) {
            int64_t to = r4c[s * nM + c];
            probs[c * W + (to >= nL ? nL : to)] += w;
        }
    }
    const double norm = 1.0 / total;
    for (int64_t i = 0; i < nM * W; i++) probs[i] *= norm;
}

int orc_assignment_prob(const double* costs, int64_t nL, int64_t nM, int64_t k, double* probs) {
    if (nM == 1) { single_column(costs, nL, probs); return 0; }
    const int64_t nR = nL + nM;
    int64_t* c4r = (int64_t*)malloc((size_t)(nR * k) * sizeof(int64_t));
    int64_t* r4c = (int64_t*)malloc((size_t)(nM * k) * sizeof(int64_t));
    double* g = (double*)malloc((size_t)k * sizeof(double));
    int64_t found = orc_kbest2d_cutoff(k, nR, nM, 0, costs, c4r, r4c, g, PDA_GATE);
    marginalise(r4c, g, found, nL, nM, 1, probs);
    free(c4r); free(r4c); free(g);
    return 0;
}

static double minc_constant(int64_t ni, int64_t mi) {
    double n = (double)ni, m = (double)mi;
    return pow(PDA_TAU, (m - n) / (2 * n)) * pow(n / m, m) * exp(m / (12 * n * n) - 1 / (12 * m + 1));
}
static double minc_factor(int64_t ni) {
    double n = (double)ni;
    return pow(PDA_TAU * n, 1.0 / (2.0 * n)) * n * exp(-1 + 1.0 / (12 * n * n));
}

/* upperK = min(size_t(mincBound)+1, 20000) (:868).  Deviation, documented: the
 * reference's double->size_t cast is undefined for bounds >= 2^64 (dense problems
 * overflow it easily); here anything at or above 20000 saturates to 20000. */
static int64_t brute_force_k(const double* costs, int64_t nR, int64_t nM) {
    double bound = minc_constant(nR, nM);
    for (int64_t r = 0; r < nR; r++) {
        int64_t card = 1;
        for (int64_t c = 0; c < nM; c++) if (costs[c * nR + r] < INFINITY) card++;
        bound *= minc_factor(card);
    }
    if (!(bound < 20000.0)) return 20000;
    return (int64_t)bound + 1;
}

int orc_brute_force_prob(const double* costs, int64_t nL, int64_t nM, double* probs) {
    if (nM == 1) { single_column(costs, nL, probs); return 0; }
    const int64_t nR = nL + nM;
    const int64_t k = brute_force_k(costs, nR, nM);
    int64_t* c4r = (int64_t*)malloc((size_t)(nR * k) * sizeof(int64_t));
    int64_t* r4c = (int64_t*)malloc((size_t)(nM * k) * sizeof(int64_t));
    double* g = (double*)malloc((size_t)k * sizeof(double));
    int64_t found = orc_kbest2d(k, nR, nM, 0, costs, c4r, r4c, g);
    marginalise(r4c, g, found, nL, nM, 0, probs);
    free(c4r); free(r4c); free(g);
    return 0;
}

/* std::reduce over a random-access range sums in blocks of four (libstdc++ <numeric>:295-308);
 * permanentProb's single-column path (:168) inherits that order. */
static double reduce_by_fours(const double* v, int64_t n) {
    double acc = 0;
    int64_t i = 0;
    for (; n - i >= 4; i += 4) acc = acc + ((v[i] + v[i + 1]) + (v[i + 2] + v[i + 3]));
    for (; i < n; i++) acc = acc + v[i];
    return acc;
}

int orc_permanent_prob(const double* costsIn, int64_t nL, int64_t nM, int permOpt, double* probs) {
    const int64_t nR = nL + nM, nC = nM, W = nL + 1;
    double* P = (double*)malloc((size_t)(nR * nC) * sizeof(double)); /* fullProbs, column-major */
    memcpy(P, costsIn, (size_t)(nR * nC) * sizeof(double));
    orc_to_probs(P, nR * nC);
    if (nM == 1) {
        double norm = 1.0 / reduce_by_fours(P, nR * nC);
        for (int64_t i = 0; i < nR * nC; i++) probs[i] = P[i] * norm;
        free(P);
        return 0;
    }
    for (int64_t i = 0; i < nM * W; i++) probs[i] = 0;
    const int64_t sR = nR - 1, sC = nC - 1;
    double* S = (double*)malloc((size_t)(sR * sC) * sizeof(double)); /* subProbs */
    int64_t* others = (int64_t*)malloc((size_t)sC * sizeof(int64_t));
    double fullPerm = 0;
    int status = 0;
    for (int64_t m = 0; m < nM && !status; m++) {
        /* columns of P other than m, in order (colIdx of :204-209, :256-259) */
        for (int64_t j = 0, c = 0; c < nC; c++) if (c != m) others[j++] = c;
        /* setupAssgnMatrix (:292-323): rows 1.. of P without column m */
        for (int64_t j = 0; j < sC; j++)
            for (int64_t r = 0; r < sR; r++) S[r + j * sR] = P[(r + 1) + others[j] * nR];
        double colPerm = 0;
        for (int64_t l = 0; l < nL && !status; l++) {
            if (P[l + m * nR] != 0) {
                orc_set_approx_stream(20260217ULL, m * W + l);
                double t = P[l + m * nR] * orc_conditioned_permanent(S, sR, sC, permOpt, &status);
                colPerm += fabs(t);
                probs[m * W + l] = fabs(t);
            }
            for (int64_t j = 0; j < sC; j++) S[l + j * sR] = P[l + others[j] * nR]; /* :233 */
        }
        if (status) break;
        if (m != 0) S[(nL - 1 + m) + 0 * sR] = P[nL + 0 * nR]; /* :237-239 */
        orc_set_approx_stream(20260217ULL, m * W + nL);
        double t = P[(nL + m) + m * nR] * orc_conditioned_permanent(S, sR, sC, permOpt, &status);
        colPerm += fabs(t);
        probs[m * W + nL] = fabs(t);
        fullPerm = (fullPerm < colPerm) ? colPerm : fullPerm; /* std::max(fullPerm, colPerm) (:255) */
    }
    if (!status) {
        const double norm = 1.0 / fullPerm;
        for (int64_t i = 0; i < nM * W; i++) probs[i] *= norm;
    }
    free(P); free(S); free(others);
    return status;
}

/* The numeric body of getAssignmentProbs (assignment.cpp:57-74): condition the costs, compute the weights of the
 * conditioned problem (k-best, or permanent-based when usePerm), scatter them back through rowIdx.
 * probs is nM x (nL+1), row-major.  nL == 0 -> {1} per detection (:51-53). */
int orc_association_probs(const double* costs, int64_t nL, int64_t nM, int64_t k, int usePerm, double* probs) {
    if (nM <= 0) return 0;
    if (nL == 0) { for (int64_t m = 0; m < nM; m++) probs[m] = 1.0; return 0; }
    const int64_t nR = nL + nM, W = nL + 1;
    double* cond = (double*)malloc((size_t)(nR * nM) * sizeof(double));
    int64_t* rowIdx = (int64_t*)malloc((size_t)nR * sizeof(int64_t));
    const int64_t good = orc_condition_costs(costs, nR, nM, cond, rowIdx);
    const int64_t condL = good - nM; /* (conditionedCosts.size()/nM) - nM (:60) */
    for (int64_t i = 0; i < nM * W; i++) probs[i] = 0;
    /* fewer kept rows than detections: the reference's size_t subtraction underflows; status 3 and a zero table, as
     * the device pipelines report it */
    if (condL < 0) { free(cond); free(rowIdx); return 3; }
    double* cp = (double*)malloc((size_t)(nM * (condL + 1)) * sizeof(double));
    int status = usePerm ? orc_permanent_prob(cond, condL, nM, 1, cp) : orc_assignment_prob(cond, condL, nM, k, cp);
    if (!status)
        for (int64_t m = 0; m < nM; m++) {
            for (int64_t l = 0; l < condL; l++) probs[m * W + rowIdx[l]] = cp[m * (condL + 1) + l];
            probs[m * W + nL] = cp[m * (condL + 1) + condL];
        }
    free(cond); free(rowIdx); free(cp);
    return status;
}
