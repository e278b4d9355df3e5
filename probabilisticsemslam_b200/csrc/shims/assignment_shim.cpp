// assignment_shim.cpp -- the reference's assignment.h numeric entry points (assignment.cpp:145-290,
// 325-435, 439-525, 527-542, 547-683, 835-964) and nwPerm.h exact permanents (nwPerm.cpp:217-231,
// 251-332, 386-400) as batch-of-one calls into libpda_b200.so.  Marshalling only.
#include "assignment.h"

#include <math.h>
#include <stdint.h>

#include <limits>
#include <stdexcept>
#include <string>

#include "pda_b200.h"

void pdaCheck(int rc, const char* where);
int pdaShimDevice();

static std::vector<std::vector<double> > unflatten(const std::vector<double>& flat, size_t nM, size_t width) {
    std::vector<std::vector<double> > out(nM, std::vector<double>(width, 0.0));
    for (size_t m = 0; m < nM; m++)
        for (size_t l = 0; l < width; l++) out[m][l] = flat[m * width + l];
    return out;
}

static std::vector<std::vector<double> > murtyWeights(const std::vector<double>& costMatrix, size_t nL, size_t nM, size_t k,
                                                      int cutMode, int weightMode, const char* who) {
    const int64_t costOff = 0, probOff = 0;
    const int32_t nr = int32_t(nL + nM), nc = int32_t(nM), nl = int32_t(nL);
    int32_t nFound = 0;
    std::vector<double> probs(nM * (nL + 1), 0.0);
    pdaCheck(pda_murty_batch_host(costMatrix.data(), &costOff, &nr, &nc, 1, int32_t(k), cutMode, 42.0, 0, 0, NULL, NULL, NULL,
                                  NULL, NULL, &nFound, weightMode, probs.data(), &probOff, &nl, pdaShimDevice()),
             who);
    return unflatten(probs, nM, nL + 1);
}

std::vector<std::vector<double> > assignmentProb(const std::vector<double>& costMatrix, size_t nL, size_t nM, size_t k) {
    return murtyWeights(costMatrix, nL, nM, k, PDA_CUT_RELATIVE, PDA_WEIGHTS_GATED, "assignmentProb");
}

// upperK of bruteForceProb (assignment.cpp:28-36, 858-868).  The reference casts the Minc-type bound to
// size_t, which is undefined once the bound exceeds 2^64; here anything at or above 20000 saturates.
static size_t bruteForceK(const std::vector<double>& C, size_t nRows, size_t nCols) {
    const double tau = 6.2831853071, n = double(nRows), m = double(nCols);
    double bound = pow(tau, (m - n) / (2 * n)) * pow(n / m, m) * exp(m / (12 * n * n) - 1 / (12 * m + 1));
    for (size_t r = 0; r < nRows; r++) {
        double card = 1;
        for (size_t c = 0; c < nCols; c++)
            if (C[c * nRows + r] < std::numeric_limits<double>::infinity()) card += 1;
        bound *= pow(tau * card, 1.0 / (2.0 * card)) * card * exp(-1 + 1.0 / (12 * card * card));
    }
    if (!(bound < 20000.0)) return 20000;
    return size_t(bound) + 1;
}

std::vector<std::vector<double> > bruteForceProb(const std::vector<double>& costMatrix, size_t nL, size_t nM) {
    const size_t k = (nM == 1) ? 1 : bruteForceK(costMatrix, nL + nM, nM);
    return murtyWeights(costMatrix, nL, nM, k, PDA_CUT_NONE, PDA_WEIGHTS_UNGATED, "bruteForceProb");
}

std::vector<std::vector<double> > permanentProb(std::vector<double> costMatrix, size_t nL, size_t nM, int permOpt) {
    const int64_t costOff = 0, probOff = 0;
    const int32_t nl = int32_t(nL), nm = int32_t(nM);
    int32_t status = 0;
    std::vector<double> probs(nM * (nL + 1), 0.0);
    pdaCheck(pda_permanent_prob_batch_host(costMatrix.data(), &costOff, &nl, &nm, 1, permOpt, probs.data(), &probOff, &status,
                                           pdaShimDevice()),
             "permanentProb");
    if (status) {
        if (permOpt >= 0 && permOpt <= 2)
            throw std::runtime_error("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().");
        throw std::runtime_error("Unknown perm option in conditioned permanent!");
    }
    return unflatten(probs, nM, nL + 1);
}

// status of the usePerm pipeline -> the reference's exceptions
static void permStatusCheck(int32_t status) {
    if (status == 1) throw std::runtime_error("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().");
    if (status)
        throw std::runtime_error("getAssignmentProbs: conditionCosts kept fewer rows than there are detections, so condL "
                                 "= goodRows - nM is negative (the reference's size_t subtraction underflows)");
}

std::vector<std::vector<double> > getAssignmentProbsFromCosts(const std::vector<double>& costMatrix, size_t nL, size_t nM,
                                                              size_t k, bool usePerm) {
    if (nM == 0) return std::vector<std::vector<double> >();
    if (!usePerm) {  // one fused device pipeline
        const int64_t costOff = 0, probOff = 0;
        const int32_t nl = int32_t(nL), nm = int32_t(nM);
        std::vector<double> probs(nM * (nL + 1), 0.0);
        pdaCheck(pda_association_probs_batch_host(costMatrix.data(), &costOff, &nl, &nm, 1, int32_t(k), probs.data(), &probOff,
                                                  pdaShimDevice()),
                 "getAssignmentProbsFromCosts");
        return unflatten(probs, nM, nL + 1);
    }
    const int64_t costOff = 0, probOff = 0;  // usePerm: the fused permanent pipeline
    const int32_t nl = int32_t(nL), nm = int32_t(nM);
    int32_t status = 0;
    std::vector<double> probs(nM * (nL + 1), 0.0);
    pdaCheck(pda_association_perm_probs_batch_host(costMatrix.data(), &costOff, &nl, &nm, 1, probs.data(), &probOff, &status,
                                                   pdaShimDevice()),
             "getAssignmentProbsFromCosts");
    permStatusCheck(status);
    return unflatten(probs, nM, nL + 1);
}

std::vector<double> computeQuadricCostMatrixRaw(const std::vector<double>& landMeans, const std::vector<double>& landCovs,
                                                const std::vector<double>& measMeans, const std::vector<double>& measCovs,
                                                double nonassign) {
    const size_t nL = landMeans.size() / 3, nM = measMeans.size() / 3;
    if (landCovs.size() != 9 * nL || measCovs.size() != 9 * nM) throw std::runtime_error("computeQuadricCostMatrix: moment sizes disagree");
    const int64_t offL[2] = {0, int64_t(nL)}, offM[2] = {0, int64_t(nM)};
    std::vector<double> costs((nL + nM) * nM);
    if (nM == 0) return costs;
    pdaCheck(pda_quadric_cost_batch_host(landMeans.data(), landCovs.data(), offL, measMeans.data(), measCovs.data(), offM, 1, nonassign,
                                         costs.data(), pdaShimDevice()),
             "computeQuadricCostMatrix");
    return costs;
}

std::vector<std::vector<double> > getAssignmentProbsFromMoments(const std::vector<double>& landMeans,
                                                                const std::vector<double>& landCovs,
                                                                const std::vector<double>& measMeans,
                                                                const std::vector<double>& measCovs, double nonassign, size_t k) {
    const size_t nL = landMeans.size() / 3, nM = measMeans.size() / 3;
    if (landCovs.size() != 9 * nL || measCovs.size() != 9 * nM) throw std::runtime_error("getAssignmentProbs: moment sizes disagree");
    if (nM == 0) return std::vector<std::vector<double> >();
    const int64_t offL[2] = {0, int64_t(nL)}, offM[2] = {0, int64_t(nM)};
    std::vector<double> probs(nM * (nL + 1), 0.0);
    pdaCheck(pda_association_from_moments_batch_host(landMeans.data(), landCovs.data(), offL, measMeans.data(), measCovs.data(), offM, 1,
                                                     nonassign, int32_t(k), probs.data(), pdaShimDevice()),
             "getAssignmentProbsFromMoments");
    return unflatten(probs, nM, nL + 1);
}

std::vector<std::vector<double> > getAssignmentProbsFromMoments(const std::vector<double>& landMeans,
                                                                const std::vector<double>& landCovs,
                                                                const std::vector<double>& measMeans,
                                                                const std::vector<double>& measCovs, double nonassign, size_t k,
                                                                bool usePerm) {
    if (!usePerm) return getAssignmentProbsFromMoments(landMeans, landCovs, measMeans, measCovs, nonassign, k);
    const size_t nL = landMeans.size() / 3, nM = measMeans.size() / 3;
    if (landCovs.size() != 9 * nL || measCovs.size() != 9 * nM) throw std::runtime_error("getAssignmentProbs: moment sizes disagree");
    if (nM == 0) return std::vector<std::vector<double> >();
    const int64_t offL[2] = {0, int64_t(nL)}, offM[2] = {0, int64_t(nM)};
    std::vector<double> probs(nM * (nL + 1), 0.0);
    int32_t status = 0;
    pdaCheck(pda_association_perm_from_moments_batch_host(landMeans.data(), landCovs.data(), offL, measMeans.data(), measCovs.data(),
                                                          offM, 1, nonassign, probs.data(), &status, pdaShimDevice()),
             "getAssignmentProbsFromMoments");
    permStatusCheck(status);
    return unflatten(probs, nM, nL + 1);
}

std::vector<int> asgnBBRaw(const std::vector<double>& boxesL, const std::vector<double>& boxesR, double nonassign) {
    const int64_t offL[2] = {0, int64_t(boxesL.size() / 5)}, offR[2] = {0, int64_t(boxesR.size() / 5)};
    std::vector<int32_t> a(size_t(offL[1]) ? size_t(offL[1]) : 1, -1);
    pdaCheck(pda_asgn_bb_batch_host(boxesL.data(), offL, boxesR.data(), offR, 1, nonassign, a.data(), pdaShimDevice()), "asgnBB");
    return std::vector<int>(a.begin(), a.begin() + offL[1]);
}

std::vector<double> conditionCosts(const std::vector<double>& costs, size_t nRows, size_t nCols,
                                   std::vector<ptrdiff_t>& rowIdxOut) {
    const int64_t costOff = 0, rowOff = 0;
    const int32_t nr = int32_t(nRows), nc = int32_t(nCols);
    int32_t good = 0;
    std::vector<double> out(costs.size() ? costs.size() : 1);
    std::vector<int64_t> idx(nRows ? nRows : 1);
    pdaCheck(pda_condition_costs_batch_host(costs.data(), &costOff, &nr, &nc, 1, &rowOff, out.data(), idx.data(), &good,
                                            pdaShimDevice()),
             "conditionCosts");
    out.resize(size_t(good) * nCols);
    std::vector<ptrdiff_t> rows(idx.begin(), idx.begin() + good);
    rowIdxOut.swap(rows);
    return out;
}

void toProbs(std::vector<double>& costMatrix) {
    if (costMatrix.empty()) return;
    const int64_t off = 0, len = int64_t(costMatrix.size());
    pdaCheck(pda_to_probs_batch_host(costMatrix.data(), &off, &len, 1, pdaShimDevice()), "toProbs");
}

double conditionedPermanentRaw(const double* A, size_t rows, size_t cols, int permOpt) {
    const int64_t off = 0;
    const int32_t r = int32_t(rows), c = int32_t(cols);
    int32_t status = 0;
    double out = 0;
    pdaCheck(pda_conditioned_permanent_batch_host(A, &off, &r, &c, 1, permOpt, &out, &status, pdaShimDevice()),
             "conditionedPermanent");
    if (status) {
        if (permOpt >= 0 && permOpt <= 2)
            throw std::runtime_error("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().");
        throw std::runtime_error("Unknown perm option in conditioned permanent!");
    }
    return out;
}

double permanentApproximationRaw(const double* A, size_t rows, size_t cols, size_t iterations) {
    static uint64_t calls = 0;  // successive calls draw from successive streams, like successive rand() calls would
    const int64_t off = 0;
    const int32_t r = int32_t(rows), c = int32_t(cols);
    int32_t status = 0;
    double out = 0;
    pdaCheck(pda_permanent_approx_batch_host(A, &off, &r, &c, 1, int32_t(iterations), 20260217ULL + (calls++), &out, &status,
                                             pdaShimDevice()),
             "permanentApproximation");
    if (status) throw std::runtime_error("permanentApproximation: matrix dimension limited to 32 on the device");
    return out;
}

double permanentExactRaw(const double* A, size_t rows, size_t cols) {
    const int64_t off = 0;
    const int32_t r = int32_t(rows), c = int32_t(cols);
    int32_t status = 0;
    double out = 0;
    pdaCheck(pda_permanent_batch_host(A, &off, &r, &c, 1, &out, &status, pdaShimDevice()), "permanentExact");
    if (status) throw std::runtime_error("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().");
    return out;
}

long double permanentExactLongRaw(const double* A, size_t rows, size_t cols) { return permanentExactRaw(A, rows, cols); }

namespace {
// flat, offset-addressed form of a vector-of-problems batch (what the C ABI takes)
struct FlatBatch {
    std::vector<int64_t> costOff, probOff;
    std::vector<int32_t> nr, nc, nl;
    std::vector<double> flat, probs;
    FlatBatch(const std::vector<std::vector<double> >& costs, const std::vector<size_t>& nL, const std::vector<size_t>& nM) {
        const size_t n = costs.size();
        costOff.resize(n); probOff.resize(n); nr.resize(n); nc.resize(n); nl.resize(n);
        size_t nCost = 0, nProb = 0;
        for (size_t p = 0; p < n; p++) {
            if (costs[p].size() != (nL[p] + nM[p]) * nM[p]) throw std::invalid_argument("batch: cost matrix size does not match (nL + nM) * nM");
            costOff[p] = int64_t(nCost); probOff[p] = int64_t(nProb);
            nr[p] = int32_t(nL[p] + nM[p]); nc[p] = int32_t(nM[p]); nl[p] = int32_t(nL[p]);
            nCost += costs[p].size(); nProb += nM[p] * (nL[p] + 1);
        }
        flat.resize(nCost ? nCost : 1); probs.resize(nProb ? nProb : 1);
        for (size_t p = 0; p < n; p++) std::copy(costs[p].begin(), costs[p].end(), flat.begin() + costOff[p]);
    }
    std::vector<std::vector<std::vector<double> > > tables(const std::vector<size_t>& nL, const std::vector<size_t>& nM) const {
        std::vector<std::vector<std::vector<double> > > out(nr.size());
        for (size_t p = 0; p < nr.size(); p++) {
            std::vector<double> slice(probs.begin() + probOff[p], probs.begin() + probOff[p] + nM[p] * (nL[p] + 1));
            out[p] = unflatten(slice, nM[p], nL[p] + 1);
        }
        return out;
    }
};
std::vector<int32_t> deviceList(const std::vector<int>& devices) {
    std::vector<int32_t> d(devices.begin(), devices.end());
    if (d.empty()) d.push_back(pdaShimDevice());
    return d;
}
}  // namespace

std::vector<std::vector<std::vector<double> > > assignmentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                    const std::vector<size_t>& nL,
                                                                    const std::vector<size_t>& nM, size_t k,
                                                                    const std::vector<int>& devices) {
    FlatBatch fb(costs, nL, nM);
    const size_t n = costs.size();
    std::vector<int32_t> found(n ? n : 1);
    const std::vector<int32_t> dev = deviceList(devices);
    if (n)
        pdaCheck(pda_murty_batch_host_multi(fb.flat.data(), fb.costOff.data(), fb.nr.data(), fb.nc.data(), int64_t(n), int32_t(k),
                                            PDA_CUT_RELATIVE, 42.0, 0, 0, NULL, NULL, NULL, NULL, NULL, found.data(),
                                            PDA_WEIGHTS_GATED, fb.probs.data(), fb.probOff.data(), fb.nl.data(), dev.data(),
                                            int32_t(dev.size())),
                 "assignmentProbBatch");
    return fb.tables(nL, nM);
}

std::vector<std::vector<std::vector<double> > > assignmentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                    const std::vector<size_t>& nL,
                                                                    const std::vector<size_t>& nM, size_t k) {
    return assignmentProbBatch(costs, nL, nM, k, std::vector<int>());
}

std::vector<std::vector<std::vector<std::vector<double> > > > assignmentProbLadderBatch(
    const std::vector<std::vector<double> >& costs, const std::vector<size_t>& nL, const std::vector<size_t>& nM,
    const std::vector<size_t>& ks) {
    if (nL.size() != costs.size() || nM.size() != costs.size()) throw std::invalid_argument("assignmentProbLadder: nL / nM sizes differ from costs");
    if (ks.empty() || ks.size() > 16) throw std::invalid_argument("assignmentProbLadder: need 1 to 16 values of k");
    std::vector<int32_t> k32(ks.size());
    for (size_t j = 0; j < ks.size(); j++) {
        if (ks[j] < 1 || ks[j] > size_t(INT32_MAX)) throw std::invalid_argument("assignmentProbLadder: k out of range");
        k32[j] = int32_t(ks[j]);
    }
    const size_t n = costs.size(), nK = ks.size();
    FlatBatch fb(costs, nL, nM);
    std::vector<int64_t> probOff(n);
    size_t nProb = 0;
    for (size_t p = 0; p < n; p++) { probOff[p] = int64_t(nProb); nProb += nK * nM[p] * (nL[p] + 1); }
    std::vector<double> probs(nProb ? nProb : 1);
    std::vector<int32_t> found(n * nK + 1);
    if (n)
        pdaCheck(pda_assignment_prob_ladder_batch_host(fb.flat.data(), fb.costOff.data(), fb.nr.data(), fb.nc.data(), fb.nl.data(),
                                                       int64_t(n), k32.data(), int32_t(nK), probs.data(), probOff.data(),
                                                       found.data(), pdaShimDevice()),
                 "assignmentProbLadder");
    std::vector<std::vector<std::vector<std::vector<double> > > > out(n);
    for (size_t p = 0; p < n; p++) {
        const size_t cells = nM[p] * (nL[p] + 1);
        for (size_t j = 0; j < nK; j++) {
            const std::vector<double> slice(probs.begin() + probOff[p] + j * cells, probs.begin() + probOff[p] + (j + 1) * cells);
            out[p].push_back(unflatten(slice, nM[p], nL[p] + 1));
        }
    }
    return out;
}

std::vector<std::vector<std::vector<double> > > assignmentProbLadder(const std::vector<double>& costMatrix, size_t nL, size_t nM,
                                                                     const std::vector<size_t>& ks) {
    return assignmentProbLadderBatch(std::vector<std::vector<double> >(1, costMatrix), std::vector<size_t>(1, nL),
                                     std::vector<size_t>(1, nM), ks)[0];
}

std::vector<std::vector<std::vector<double> > > permanentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                   const std::vector<size_t>& nL,
                                                                   const std::vector<size_t>& nM, int permOpt,
                                                                   const std::vector<int>& devices) {
    FlatBatch fb(costs, nL, nM);
    const size_t n = costs.size();
    std::vector<int32_t> status(n ? n : 1, 0);
    const std::vector<int32_t> dev = deviceList(devices);
    if (n)
        pdaCheck(pda_permanent_prob_batch_host_multi(fb.flat.data(), fb.costOff.data(), fb.nl.data(), fb.nc.data(), int64_t(n), permOpt,
                                                     fb.probs.data(), fb.probOff.data(), status.data(), dev.data(), int32_t(dev.size())),
                 "permanentProbBatch");
    for (size_t p = 0; p < n; p++)
        if (status[p]) throw std::runtime_error("permanentProbBatch: the reference throws for one of these problems (dimension > 32 or bad permOpt)");
    return fb.tables(nL, nM);
}

std::vector<std::vector<std::vector<double> > > getAssignmentProbsBatch(const std::vector<std::vector<double> >& costs,
                                                                        const std::vector<size_t>& nL,
                                                                        const std::vector<size_t>& nM, size_t k, bool usePerm,
                                                                        const std::vector<int>& devices) {
    if (nL.size() != costs.size() || nM.size() != costs.size()) throw std::invalid_argument("getAssignmentProbsBatch: nL / nM sizes differ from costs");
    FlatBatch fb(costs, nL, nM);
    const size_t n = costs.size();
    const std::vector<int32_t> dev = deviceList(devices);
    if (n == 0) return fb.tables(nL, nM);
    for (size_t p = 0; p < n; p++)
        if (nM[p] == 0) throw std::invalid_argument("getAssignmentProbsBatch: a frame without detections");
    if (!usePerm) {
        pdaCheck(pda_association_probs_batch_host_multi(fb.flat.data(), fb.costOff.data(), fb.nl.data(), fb.nc.data(), int64_t(n), int32_t(k),
                                                        fb.probs.data(), fb.probOff.data(), dev.data(), int32_t(dev.size())),
                 "getAssignmentProbsBatch");
        return fb.tables(nL, nM);
    }
    std::vector<int32_t> status(n, 0);
    pdaCheck(pda_association_perm_probs_batch_host_multi(fb.flat.data(), fb.costOff.data(), fb.nl.data(), fb.nc.data(), int64_t(n),
                                                         fb.probs.data(), fb.probOff.data(), status.data(), dev.data(),
                                                         int32_t(dev.size())),
             "getAssignmentProbsBatch");
    for (size_t p = 0; p < n; p++) permStatusCheck(status[p]);
    return fb.tables(nL, nM);
}

double permanentExactShardedRaw(const double* A, size_t n, const int* devices, size_t nDevices) {
    if (n > 32) throw std::runtime_error("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().");
    std::vector<int32_t> dev(devices, devices + nDevices);
    if (dev.empty()) dev.push_back(pdaShimDevice());
    double out = 0;
    pdaCheck(pda_permanent_sharded_host(A, int32_t(n), dev.data(), int32_t(dev.size()), &out), "permanentExactSharded");
    return out;
}
