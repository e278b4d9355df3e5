/* oracle_capi.h -- C entry points of the CPU parity oracle (liboracle.so).
 *
 * TEST INFRASTRUCTURE ONLY.  The oracle is a plain-C restatement of the reference's
 * algorithm for the probabilistic data-association hot path; it exists so that
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg can check (never
 * replace) the CUDA product path.  Nothing under probabilisticsemslam_b200/ or
 * include/ may include, link, load or call it.
 *
 * Pinning: the reference ships no tests or golden vectors for this path
 * (SURVEY.md section 4), so the oracle is pinned against OUTPUTS OF THE REFERENCE
 * ITSELF: oracle/_ref/libpda_ref_strict.so is the reference's own code compiled
 * here (oracle/Makefile), tests/test_oracle_vs_ref.py compares the two on seeded
 * inputs when it is present, and tests/golden/ holds vectors generated from it
 * (tests/golden/make_golden.py) that travel to the GPU box.
 *
 * Every function below has a `ref_` twin with the same signature in
 * oracle/ref_glue/ref_capi.cpp.  All matrices are column-major doubles:
 * C[row + col*numRow]; indices are int64 (the reference's ptrdiff_t).
 */
#ifndef PDA_ORACLE_CAPI_H
#define PDA_ORACLE_CAPI_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* shortestPathCPP.cpp:571-644.  Returns #hypotheses found (0 = infeasible). */
int64_t orc_kbest2d(int64_t k, int64_t numRow, int64_t numCol, int maximize, const double* C,
                    int64_t* col4row, int64_t* row4col, double* gain);
/* shortestPathCPP.cpp:646-733. */
int64_t orc_kbest2d_cutoff(int64_t k, int64_t numRow, int64_t numCol, int maximize, const double* C,
                           int64_t* col4row, int64_t* row4col, double* gain, double cutoff);
/* kBest2D on a ScratchSpace previously used by kBest2DCutoff(k=1, firstMaximize, firstC,
 * firstCutoff): toCut/cutoffGain/maximize are sticky (shortestPathCPP.hpp:84-86, cpp:650-651). */
int64_t orc_kbest2d_after_cutoff(int64_t k, int64_t numRow, int64_t numCol, int maximize, const double* C,
                                 int64_t* col4row, int64_t* row4col, double* gain,
                                 int firstMaximize, const double* firstC, double firstCutoff);
/* CPU model of the CUDA pruning kernel's decisions (bound, tightening, abandonment, tie bail-out) over the reference
 * arithmetic: returns what kBest2DCutoff returns, or -2 where the kernel would hand the problem to the exact kernel.
 * maxCol = the batch's largest numCol (sizes the open list like the kernel's geometry).  stats[6]: children, abandoned,
 * dropped when finished, kept, tightenings, slots at tightening.  No `ref_` twin: it models THIS repository's kernel. */
int64_t orc_kbest2d_cutoff_pruned(int64_t k, int64_t numRow, int64_t numCol, int maximize, const double* C,
                                  int64_t* col4row, int64_t* row4col, double* gain, double cutoff,
                                  int64_t maxCol, int64_t* stats);
/* shortestPathCPP.cpp:735-762.  Returns 1 solved / 0 infeasible. */
int orc_assign2d(int64_t numRow, int64_t numCol, int maximize, const double* C,
                 int64_t* col4row, int64_t* row4col, double* u, double* v, double* gain);
/* shortestPathCPP.cpp:119-238 on an already-safe matrix.  Returns 1 if infeasible. */
int orc_shortest_path(int64_t numRow, int64_t numCol, int64_t numCol4Gain, const double* Cprepared,
                      int64_t* col4row, int64_t* row4col, double* u, double* v, double* gain,
                      uint8_t* forbidden);

/* assignment.cpp:439-525.  outCosts has room for nRows*nCols, rowIdx for nRows. Returns goodRows. */
int64_t orc_condition_costs(const double* costs, int64_t nRows, int64_t nCols, double* outCosts, int64_t* rowIdx);
/* assignment.cpp:527-542. */
void orc_to_probs(double* v, int64_t n);
/* assignment.cpp:547-683.  probs is nM x (nL+1), row-major [m][l].  Returns 0. */
int orc_assignment_prob(const double* costs, int64_t nL, int64_t nM, int64_t k, double* probs);
/* assignment.cpp:835-964. */
int orc_brute_force_prob(const double* costs, int64_t nL, int64_t nM, double* probs);
/* assignment.cpp:145-290 (+292-323, 325-435).  Returns 0, or 1 where the reference throws. */
int orc_permanent_prob(const double* costs, int64_t nL, int64_t nM, int permOpt, double* probs);

/* assignment.cpp:57-74 (getAssignmentProbs after the cost matrix has been built). Returns 0, or 1 where the reference throws. */
int orc_association_probs(const double* costs, int64_t nL, int64_t nM, int64_t k, int usePerm, double* probs);

/* oracle_perm_approx.c: Huber's approximate permanent (nwPerm.cpp:36-211) with the CUDA kernel's counter-based draws
 * in place of the reference's unseeded rand().  No `ref_` twin. */
double orc_permanent_approx(const double* A, int64_t rows, int64_t cols, int64_t iterations, uint64_t seed, int64_t matIndex,
                            int64_t* successesOut);
/* draws of orc_permanent_approx on this thread (conditionedPermanent / permanentProb with permOpt 0 included) that lay
 * within 1e-12 of a partial sum they were compared with: where the kernel may pick differently (oracle_perm_approx.c) */
void orc_approx_near_ties_reset(void);
int64_t orc_approx_near_ties(void);
/* which stream the next conditionedPermanent(.., permOpt = 0) draws from (thread-local index) */
void orc_set_approx_stream(uint64_t seed, int64_t index);

/* oracle_quadric.c: getCovs (assignment.cpp:693-703), computeQuadricCostMatrix (:705-722, the 3x3 Eigen LDLT solve
 * restated -- parity unpinned, see that file), getAssignmentProbs from the moments on (:38-74).  No `ref_` twins. */
void orc_quadric_covs(const double* Q, int64_t n, double* covs);
void orc_quadric_cost_matrix(const double* landMean, const double* landCov, int64_t nL, const double* measMean,
                             const double* measCov, int64_t nM, double nonassign, double* costs);
int orc_association_from_moments(const double* landMean, const double* landCov, int64_t nL, const double* measMean,
                                 const double* measCov, int64_t nM, double nonassign, int64_t k, double* probs);

/* nwPerm.cpp:217-231 / 251-332 / 386-400; status 1 where the reference throws (dim > 32). */
double orc_permanent_exact(const double* A, int64_t rows, int64_t cols, int* status);
double orc_permanent_exact_square(const double* A, int64_t n, int* status);
double orc_permanent_exact_long(const double* A, int64_t rows, int64_t cols, int* status);
/* assignment.cpp:325-435; status 1 where the reference throws (bad permOpt, or permOpt 0 = Huber, out of scope). */
double orc_conditioned_permanent(const double* A, int64_t rows, int64_t cols, int permOpt, int* status);

/* Stereo box association: boundBox.h:62-75, assignment.cpp:724-797.  A box = xmin, ymin, xmax, ymax, xOffset. */
void orc_bb_cost_matrix(const double* boxesL, int64_t nL, const double* boxesR, int64_t nR, double nonassign, double* out);
void orc_asgn_bb(const double* boxesL, int64_t nL, const double* boxesR, int64_t nR, double nonassign, int32_t* out);

/* Batch drivers for CPU-baseline timing: problems [0,n) over nThreads host threads,
 * returns wall seconds.  probs != NULL -> assignmentProb per problem;
 * gain != NULL -> kBest2DCutoff lists (minimise). */
double orc_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                 int64_t n, int64_t k, double cutoff, int nThreads,
                 double* probs, const int64_t* probOff,
                 int64_t* col4row, const int64_t* c4rOff, int64_t* row4col, const int64_t* r4cOff,
                 double* gain, int32_t* nFound);
double orc_permanent_batch(const double* mats, int64_t dim, int64_t n, int nThreads, double* out);

/* Work counters of the most recent orc_kbest2d* call on this thread (SURVEY.md 8d). */
void orc_last_counters(int64_t* pops, int64_t* childSolves, int64_t* dijkstraIters, int64_t* evaluations, int64_t* maxHeap);

#ifdef __cplusplus
}
#endif
#endif
