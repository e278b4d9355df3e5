/* assignment.h -- drop-in replacement for the numeric half of the reference's assignment.h
 * (reference: assignment.h:11-43; assignment.cpp:145-290 permanentProb, :325-435 conditionedPermanent,
 * :439-525 conditionCosts, :527-542 toProbs, :547-683 assignmentProb, :835-964 bruteForceProb).
 * Same names, same std::vector-based signatures, same return shapes: probs[nM][nL+1], the last entry
 * of each row being the non-assignment probability.  Everything runs as a batch of one on the B200
 * through libpda_b200.so; the *Batch forms underneath are what a multi-frame caller should use.
 *
 * Not here: the GTSAM / OpenCV typed entry points of the reference header (getAssignmentProbs, asgnBB,
 * computeBBCostMatrix, getMeans, getCovs, saveAssignmentProb).  They only unpack GTSAM / OpenCV objects and then call
 * the functions below (the *Raw / *FromMoments forms take what they unpack); keep the reference's definitions for
 * them (INTEGRATION.md).
 */
#ifndef sensSLAM_assignment
#define sensSLAM_assignment

#include <stddef.h>

#include <vector>

#include "nwPerm.h"

std::vector<std::vector<double> > assignmentProb(const std::vector<double>& costMatrix, size_t nL, size_t nM, size_t k);

/* permOpt: 0 Huber's approximation (300 trials per sub-permanent, seeded counter-based draws instead of the reference's
 * unseeded rand(): statistically equivalent, not sample for sample), 1 exact, 2 "long" (same double kernel, as in the
 * reference); anything else throws std::runtime_error. */
std::vector<std::vector<double> > permanentProb(std::vector<double> costMatrix, size_t nL, size_t nM, int permOpt);

std::vector<std::vector<double> > bruteForceProb(const std::vector<double>& costMatrix, size_t nL, size_t nM);

std::vector<double> conditionCosts(const std::vector<double>& costs, size_t nRows, size_t nCols,
                                   std::vector<ptrdiff_t>& rowIdxOut);

void toProbs(std::vector<double>& costMatrix);

/* The body of getAssignmentProbs (assignment.cpp:57-74) from the cost matrix on: conditionCosts, then
 * assignmentProb(k) or (usePerm) permanentProb(.., 1) on the conditioned problem, then the weights scattered back to
 * the original landmark indices.  costMatrix is what computeQuadricCostMatrix returns ((nL+nM) x nM, column-major).
 * In the reference's getAssignmentProbs, replace lines :57-74 by a call to this. */
std::vector<std::vector<double> > getAssignmentProbsFromCosts(const std::vector<double>& costMatrix, size_t nL, size_t nM,
                                                              size_t k, bool usePerm);

/* computeQuadricCostMatrix (reference assignment.h:31-33, assignment.cpp:705-722) and getAssignmentProbs
 * (assignment.h:11-13, assignment.cpp:38-74; usePerm == 0 unless the last argument says otherwise) on raw moments: a
 * mean is 3 doubles, a covariance 9 (column-major 3x3 -- Eigen's layout, so &cov(0,0) of an Eigen::Matrix3d can be
 * copied as is), landmarks first.
 * nonassign = runConsts.NONASSIGN_QUADRIC, k = runConsts.k.  The second form never materialises the cost matrix on the
 * host: moments go in, weights come out of one device pipeline. */
std::vector<double> computeQuadricCostMatrixRaw(const std::vector<double>& landMeans, const std::vector<double>& landCovs,
                                                const std::vector<double>& measMeans, const std::vector<double>& measCovs,
                                                double nonassign);
std::vector<std::vector<double> > getAssignmentProbsFromMoments(const std::vector<double>& landMeans,
                                                                const std::vector<double>& landCovs,
                                                                const std::vector<double>& measMeans,
                                                                const std::vector<double>& measCovs, double nonassign, size_t k);
/* ... and with the reference's runConsts.usePerm (assignment.cpp:64): true takes permanentProb(cond, condL, nM, 1) in place
 * of assignmentProb(k), as one device pipeline too (k is then unused).  Throws where the reference throws. */
std::vector<std::vector<double> > getAssignmentProbsFromMoments(const std::vector<double>& landMeans,
                                                                const std::vector<double>& landCovs,
                                                                const std::vector<double>& measMeans,
                                                                const std::vector<double>& measCovs, double nonassign, size_t k,
                                                                bool usePerm);
#ifdef PDA_HAVE_EIGEN
/* the reference's own argument types (m1/cov1 = landmarks, m2/cov2 = detections) */
inline std::vector<double> computeQuadricCostMatrix(const std::vector<Eigen::Matrix<double, 3, 1> >& m1,
                                                    const std::vector<Eigen::Matrix<double, 3, 3> >& cov1,
                                                    const std::vector<Eigen::Vector3d>& m2,
                                                    const std::vector<Eigen::Matrix<double, 3, 3> >& cov2, double nonassign) {
    std::vector<double> a(3 * m1.size()), b(9 * cov1.size()), c(3 * m2.size()), d(9 * cov2.size());
    for (size_t i = 0; i < m1.size(); i++) for (int j = 0; j < 3; j++) a[3 * i + j] = m1[i](j);
    for (size_t i = 0; i < cov1.size(); i++) for (int j = 0; j < 9; j++) b[9 * i + j] = cov1[i].data()[j];
    for (size_t i = 0; i < m2.size(); i++) for (int j = 0; j < 3; j++) c[3 * i + j] = m2[i](j);
    for (size_t i = 0; i < cov2.size(); i++) for (int j = 0; j < 9; j++) d[9 * i + j] = cov2[i].data()[j];
    return computeQuadricCostMatrixRaw(a, b, c, d, nonassign);
}
/* ... and the reference's exact signature (assignment.h:31-32): the last argument is its `const semConsts& runConsts`, of
 * which only NONASSIGN_QUADRIC is read (assignment.cpp:718).  A template, so this header does not need constsUtils.h. */
template <class Consts>
inline std::vector<double> computeQuadricCostMatrix(const std::vector<Eigen::Matrix<double, 3, 1> >& m1,
                                                    const std::vector<Eigen::Matrix<double, 3, 3> >& cov1,
                                                    const std::vector<Eigen::Vector3d>& m2,
                                                    const std::vector<Eigen::Matrix<double, 3, 3> >& cov2, const Consts& runConsts) {
    return computeQuadricCostMatrix(m1, cov1, m2, cov2, (double)runConsts.NONASSIGN_QUADRIC);
}
#endif

/* asgnBB (reference assignment.h:21, assignment.cpp:724-775) on raw boxes: five doubles per box
 * (xmin, ymin, xmax, ymax, xOffset), nonassign = runConsts.NONASSIGN_BOUNDBOX.  Returns, per left box, the index of
 * the right box it is paired with or -1.  A boundBox-typed asgnBB is a three-line wrapper over this (INTEGRATION.md). */
std::vector<int> asgnBBRaw(const std::vector<double>& boxesL, const std::vector<double>& boxesR, double nonassign);

/* raw form of conditionedPermanent: A is rows x cols, column-major */
double conditionedPermanentRaw(const double* A, size_t rows, size_t cols, int permOpt);
#ifdef PDA_HAVE_EIGEN
inline double conditionedPermanent(const Eigen::MatrixXd& A, int permOpt) {
    return conditionedPermanentRaw(A.data(), size_t(A.rows()), size_t(A.cols()), permOpt);
}
#endif

/* ---- batch forms (one call, many frames): what the GPU is built for --------------------------------
 * costs[p] is problem p's column-major (nL[p]+nM[p]) x nM[p] matrix. Returns probs[p][m][l]. */
std::vector<std::vector<std::vector<double> > > assignmentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                    const std::vector<size_t>& nL,
                                                                    const std::vector<size_t>& nM, size_t k);
/* the same batch spread over several GPUs of this process (one host thread per device, contiguous slices, no
 * collective: pda_murty_batch_host_multi); `devices` lists CUDA device ordinals */
std::vector<std::vector<std::vector<double> > > assignmentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                    const std::vector<size_t>& nL,
                                                                    const std::vector<size_t>& nM, size_t k,
                                                                    const std::vector<int>& devices);
/* assignmentProb for several k at once (compMethods' k = 1, 20, 1000, 100, 200, ... on one frame,
 * comparison.cpp:194-222) from ONE enumeration to the largest k: returns probs[j][m][l], the table of ks[j], each
 * bit-identical to assignmentProb(costMatrix, nL, nM, ks[j]).  ks: 1 to 16 values >= 1, any order, duplicates allowed.
 * The Batch form takes problems as assignmentProbBatch does and returns probs[p][j][m][l]. */
std::vector<std::vector<std::vector<double> > > assignmentProbLadder(const std::vector<double>& costMatrix, size_t nL, size_t nM,
                                                                     const std::vector<size_t>& ks);
std::vector<std::vector<std::vector<std::vector<double> > > > assignmentProbLadderBatch(
    const std::vector<std::vector<double> >& costs, const std::vector<size_t>& nL, const std::vector<size_t>& nM,
    const std::vector<size_t>& ks);
/* permanentProb (assignment.cpp:145-290) for many problems, optionally over several GPUs (empty `devices` = the shim's
 * device).  Throws where the reference throws. */
std::vector<std::vector<std::vector<double> > > permanentProbBatch(const std::vector<std::vector<double> >& costs,
                                                                   const std::vector<size_t>& nL,
                                                                   const std::vector<size_t>& nM, int permOpt,
                                                                   const std::vector<int>& devices = std::vector<int>());
/* getAssignmentProbsFromCosts for many frames at once (the probWin frames of a sliding-window update,
 * slidingWindow.cpp:339), optionally over several GPUs (contiguous slices, empty `devices` = the shim's device):
 * conditionCosts -> assignmentProb(k) or (usePerm) permanentProb(.., 1) -> scatter, per frame.  costs[p] is frame p's
 * (nL[p]+nM[p]) x nM[p] cost matrix, nM[p] >= 1.  Returns probs[p][m][l]; throws where the reference throws. */
std::vector<std::vector<std::vector<double> > > getAssignmentProbsBatch(const std::vector<std::vector<double> >& costs,
                                                                        const std::vector<size_t>& nL,
                                                                        const std::vector<size_t>& nM, size_t k, bool usePerm,
                                                                        const std::vector<int>& devices = std::vector<int>());

#endif
