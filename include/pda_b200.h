/* pda_b200.h -- C ABI of libpda_b200.so: the B200 (sm_100a) implementation of the
 * probabilistic data-association hot path of EladMichael/probabilisticSemSlam.
 *
 * The reference has no FFI layer of its own: its boundary for this path is three C++
 * headers (shortestPathCPP.hpp, assignment.h, nwPerm.h).  This file is the flat,
 * batch-oriented C door underneath them; include/shortestPathCPP.hpp,
 * include/assignment.h and include/nwPerm.h in this repository re-state the
 * reference's C++ signatures on top of it (batch of one), see INTEGRATION.md.
 *
 * Conventions
 *   - every matrix is column-major double, C[row + col*numRow], rows = landmarks
 *     followed by one dummy row per detection, columns = detections
 *     (reference: assignment.cpp:705-722); numRow >= numCol (shortestPathCPP.hpp:156-157).
 *   - index outputs are int64 (the reference's ptrdiff_t); -1 = unassigned.
 *   - functions without the _host suffix take DEVICE pointers, enqueue on `stream`
 *     (a cudaStream_t passed as void*, NULL = default stream) and do not synchronise.
 *   - *_host functions take HOST pointers, copy in, run, copy out and synchronise.
 *   - the caller owns every buffer, including the scratch `workspace`.
 *   - return value: PDA_OK (0) or a negative PDA_ERR_*; pda_last_error() describes it.
 *   - there is no CPU fallback: without a CUDA device every compute entry point
 *     returns PDA_ERR_CUDA.
 */
#ifndef PDA_B200_H
#define PDA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDA_OK 0
#define PDA_ERR_INVALID (-1)     /* bad argument (NULL, negative size, numRow < numCol, ...) */
#define PDA_ERR_CUDA (-2)        /* CUDA runtime error or no device */
#define PDA_ERR_UNSUPPORTED (-3) /* dimension above PDA_MAX_DIM / PDA_MAX_PERM_DIM */
#define PDA_ERR_WORKSPACE (-4)   /* workspace too small for even one resident problem */

#define PDA_MAX_DIM 128     /* largest numRow the Murty kernels take */
#define PDA_MAX_PERM_DIM 32 /* largest permanent dimension (reference: nwPerm.cpp:265, 329) */

/* cutMode of pda_murty_batch */
#define PDA_CUT_NONE 0     /* kBest2D                      (shortestPathCPP.cpp:571-644) */
#define PDA_CUT_RELATIVE 1 /* kBest2DCutoff(..., cutoff)   (shortestPathCPP.cpp:646-733) */
#define PDA_CUT_STICKY 2   /* kBest2D on a ScratchSpace whose toCut/cutoffGain/maximize were left set by
                              an earlier kBest2DCutoff (hpp:84-86, 130-132): children are still pruned
                              against the absolute, shifted `cutoff`, in the sense of `cutMaximize` */

/* weightMode of pda_murty_batch */
#define PDA_WEIGHTS_NONE 0
#define PDA_WEIGHTS_GATED 1   /* assignmentProb  (assignment.cpp:547-683): terms within 42 of the best */
#define PDA_WEIGHTS_UNGATED 2 /* bruteForceProb  (assignment.cpp:910-945): every enumerated term */

int pda_version(void);
const char* pda_last_error(void);
int pda_device_count(void);
/* Diagnostic: measured FP64 FMA throughput of the current device in TFLOP/s (a DFMA micro-benchmark;
 * the denominator of the permanent kernel's roofline). Negative on failure. */
double pda_diag_dfma_tflops(void);

/* ------------------------------------------------------------------------------------------
 * Murty k-best enumeration (+ optional fused association weights), one warp per problem.
 * Replaces kBest2D / kBest2DCutoff (shortestPathCPP.hpp:204-212, 256-265) and, with
 * weightMode != 0, the marginalisation tail of assignmentProb / bruteForceProb.
 *
 *   costs, costOff[p]   problem p's numRow[p] x numCol[p] matrix starts at costs + costOff[p]
 *   k                   hypotheses requested per problem
 *   row4colBest         problem p, hypothesis i at row4colBest + r4cOff[p] + i*numCol[p]   (may be NULL)
 *   col4rowBest         problem p, hypothesis i at col4rowBest + c4rOff[p] + i*numRow[p]   (may be NULL)
 *   gainBest            problem p, hypothesis i at gainBest[p*k + i]                       (may be NULL)
 *   nFound[p]           number of hypotheses found, 0 = infeasible (the reference's return value); -1 = the problem was
 *                       not solved because its dimensions are malformed (numCol < 1, numCol > numRow, nL + numCol !=
 *                       numRow with weights) or exceed maxNumRow / maxNumCol of this call -- only reachable through the
 *                       device-pointer entry, the *_host entries reject such batches up front
 *   probs, probOff, nL  weightMode != 0: numCol[p] x (nL[p]+1) row-major table at probs + probOff[p]
 *   workspace           >= pda_murty_workspace_bytes(...) gives full occupancy; smaller is legal
 *                       (fewer problems in flight) down to one problem's worth
 * Bit-exactness: row4col, col4row, enumeration order and gains are bit-identical to an
 * IEEE-strict build of the reference (same operand order, same tie-breaks, same heap mechanics).
 */
int64_t pda_murty_workspace_bytes(int64_t nProblems, int32_t k, int32_t maxNumRow, int32_t maxNumCol);

/* Page-locked host buffers for the k-best *_host entry points (pda_murty_batch_host, pda_assignment_prob_ladder_batch_host
 * and their shards in pda_murty_batch_host_multi).  Such a call whose declared arrays exceed 8 MB, and which finds its
 * cost matrices (in) or weight tables (out) page-locked, uses them IN PLACE: every warp reads its cost matrix and writes
 * its weight table over the bus itself, so the transfers hide under the computing instead of standing in front of and
 * behind the kernel.  Smaller calls, every other array and every other *_host entry copy, from any kind of memory.
 * Buffers from pda_host_alloc are portable: every device of the process may use them in place (the multi-device
 * entry points below).  Memory the caller pinned itself (cudaHostAlloc / cudaHostRegister) is used in place only by the
 * device whose context pinned it; pageable memory is copied.  Returns NULL on failure (pda_last_error). */
void* pda_host_alloc(int64_t bytes);
void pda_host_free(void* p);

/* Three kernels stand behind pda_murty_batch, with bit-identical results: one WARP per problem, exact (the
 * reference's heap order replayed; always right), one WARP per problem, FAST (large batches: hypotheses that provably
 * cannot be among the k best are abandoned early and the open list is a warp-parallel queue; a problem in which two
 * open hypotheses have bit-equal gains is handed to the exact kernel, which runs right behind it), and one CTA per
 * problem (latency: a node's Murty split is computed by 16 warps before the node reaches the top of the queue and
 * committed in the reference's order; taken for batches of up to 4 problems per SM with at most 16 detections each
 * -- the per-frame call of the SLAM loop, system.cpp:268).  PDA_MURTY_PATH_AUTO picks by batch size (CTA for small
 * batches, else FAST when the geometry admits it, else WARP); the other values force a kernel (tests, measurements).
 * Process-wide; returns the previous value.  Set it before sizing the workspace. */
#define PDA_MURTY_PATH_AUTO 0
#define PDA_MURTY_PATH_WARP 1
#define PDA_MURTY_PATH_CTA 2
#define PDA_MURTY_PATH_FAST 3
int pda_murty_set_path(int32_t path);

int pda_murty_batch(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                    int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                    int32_t k, int32_t cutMode, double cutoff, int32_t maximize, int32_t cutMaximize,
                    int64_t* row4colBest, const int64_t* r4cOff,
                    int64_t* col4rowBest, const int64_t* c4rOff,
                    double* gainBest, int32_t* nFound,
                    int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                    void* workspace, int64_t workspaceBytes, void* stream);

/* Same, HOST pointers; allocates and frees its own device buffers on `device`. */
int pda_murty_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                         int64_t nProblems, int32_t k, int32_t cutMode, double cutoff, int32_t maximize,
                         int32_t cutMaximize,
                         int64_t* row4colBest, const int64_t* r4cOff,
                         int64_t* col4rowBest, const int64_t* c4rOff,
                         double* gainBest, int32_t* nFound,
                         int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                         int32_t device);

/* The same over SEVERAL devices of one process (SURVEY.md 8e: "single process drives all GPUs"): the batch is cut into
 * one contiguous slice per entry of `devices`, every slice runs pda_murty_batch_host on its own host thread and device
 * (own lock, staging arena and stream), and the results land directly in the caller's arrays -- problems are
 * independent, so there is no data-path collective.  Offsets stay absolute: pass the arrays of the whole batch.
 * What a frames x probWin window batch of the SLAM loop (slidingWindow.cpp:260-339, system.cpp:268) would call. */
int pda_murty_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                               int64_t nProblems, int32_t k, int32_t cutMode, double cutoff, int32_t maximize,
                               int32_t cutMaximize,
                               int64_t* row4colBest, const int64_t* r4cOff,
                               int64_t* col4rowBest, const int64_t* c4rOff,
                               double* gainBest, int32_t* nFound,
                               int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                               const int32_t* devices, int32_t nDevices);

/* assignmentProb (assignment.cpp:547-683) for several k at once, from ONE Murty enumeration: the weight tables of
 * every k in ks[0..nK) (any order, duplicates allowed, 1 <= nK <= 16, every k >= 1).  The enumeration runs to the
 * largest k.  Exactness: kBest2DCutoff's k only bounds its sweep loop, so the list for k is the first min(k, nFound)
 * entries of the list for any larger k, and assignmentProb adds the weights in list order and normalises at the end;
 * each table is the running sum after its k-th hypothesis with that same normalisation.  Slot j is therefore
 * bit-identical to a separate pda_murty_batch(k = ks[j], PDA_CUT_RELATIVE, cutoff 42, PDA_WEIGHTS_GATED) call, nFound
 * included, on every kernel path.
 *   probs     slot j of problem p: numCol[p] x (nL[p]+1) row-major at probs + probOff[p] + j*numCol[p]*(nL[p]+1)
 *   nFound    slot j of problem p at nFound[p*nK + j]: min(ks[j], hypotheses found); 0 = infeasible (NaN tables);
 *             -1 = malformed or above maxNumRow / maxNumCol (device-pointer form only; the _host form rejects such
 *             batches up front)
 *   ks        a HOST array, in both forms
 * Workspace, kernel choice (pda_murty_set_path) and launch shape are those of pda_murty_batch at k = max(ks):
 * size the workspace with pda_murty_workspace_bytes(n, max(ks), ...).  The device-pointer form enqueues on `stream`
 * and does not synchronise.  The _host form stages as pda_murty_batch_host does, page-locked buffers from
 * pda_host_alloc used in place.  PDA_ERR_INVALID: nK outside 1..16, a k < 1, NULL ks, or what pda_murty_batch rejects. */
int pda_assignment_prob_ladder_batch(const double* costs, const int64_t* costOff, const int32_t* numRow,
                                     const int32_t* numCol, const int32_t* nL, int64_t nProblems, int32_t maxNumRow,
                                     int32_t maxNumCol, const int32_t* ks, int32_t nK, double* probs,
                                     const int64_t* probOff, int32_t* nFound, void* workspace, int64_t workspaceBytes,
                                     void* stream);
int pda_assignment_prob_ladder_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow,
                                          const int32_t* numCol, const int32_t* nL, int64_t nProblems, const int32_t* ks,
                                          int32_t nK, double* probs, const int64_t* probOff, int32_t* nFound,
                                          int32_t device);

/* Single LAP on a rectangular matrix without padding: assign2D (shortestPathCPP.hpp:144-149) when
 * makeSafe != 0, shortestPathCPP (hpp:178-182) on an already-safe matrix otherwise.
 * Per problem p: col4row[rowOff.. +numRow], row4col[colOff.. +numCol], u[colOff..], v[rowOff..],
 * forbidden[rowOff..] (bytes), gain[p], feasible[p] (1 solved, 0 infeasible).
 * rowOff/colOff are prefix sums of numRow/numCol.  Any output pointer may be NULL.
 * An n x 0 problem is feasible with gain 0.0, every col4row -1 and forbidden all 0.  In the device-pointer form a
 * problem above maxNumRow x maxNumCol (or with numCol > numRow) is not solved: feasible[p] = 0, nothing else written. */
int pda_lap_batch(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                  const int32_t* numCol4Gain, int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                  int32_t makeSafe, int32_t maximize,
                  const int64_t* rowOff, const int64_t* colOff,
                  int64_t* col4row, int64_t* row4col, double* u, double* v, uint8_t* forbidden,
                  double* gain, int32_t* feasible, void* stream);
int pda_lap_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                       const int32_t* numCol4Gain, int64_t nProblems, int32_t makeSafe, int32_t maximize,
                       const int64_t* rowOff, const int64_t* colOff,
                       int64_t* col4row, int64_t* row4col, double* u, double* v, uint8_t* forbidden,
                       double* gain, int32_t* feasible, int32_t device);

/* ------------------------------------------------------------------------------------------
 * Cost conditioning and element-wise likelihoods.
 * conditionCosts (assignment.cpp:439-525): outCosts at costOff[p] (compacted goodRows[p] x numCol[p]),
 * rowIdx at rowOff[p] (first goodRows[p] entries valid).  toProbs (assignment.cpp:527-542) in place.
 * numCol is at most PDA_MAX_DIM: the _host form rejects a larger problem (PDA_ERR_UNSUPPORTED); the device-pointer
 * form skips it (goodRows[p] = 0, its outCosts and rowIdx not written) and conditions the rest of the batch.
 */
int pda_condition_costs_batch(const double* costs, const int64_t* costOff, const int32_t* numRow,
                              const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                              double* outCosts, int64_t* rowIdx, int32_t* goodRows, void* stream);
int pda_condition_costs_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow,
                                   const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                                   double* outCosts, int64_t* rowIdx, int32_t* goodRows, int32_t device);
int pda_to_probs_batch(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, void* stream);
int pda_to_probs_batch_host(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, int32_t device);

/* ------------------------------------------------------------------------------------------
 * The numeric body of getAssignmentProbs (assignment.cpp:57-74) with usePerm == 0, fused on the device:
 * conditionCosts -> assignmentProb(k) on the conditioned problem -> weights scattered back to the original
 * landmark indices through rowIdx.  In: the raw (nL+nM) x nM cost matrices (what computeQuadricCostMatrix,
 * assignment.cpp:705-722, produces).  Out: probs[p] = nM x (nL+1) row-major at probOff[p]; nL == 0 gives {1}
 * per detection (:51-53).  rowOff = prefix sums of (nL+nM); the total* arguments size the intermediates.
 * The bounds must satisfy 1 <= maxNumCol <= maxNumRow <= PDA_MAX_DIM (else PDA_ERR_INVALID / PDA_ERR_UNSUPPORTED before
 * anything is launched); a problem with nL+nM > maxNumRow or nM > maxNumCol is skipped: nFound[p] = -1 and its table
 * is zeros (ones where nL == 0).
 */
int64_t pda_association_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                        int64_t totalProbElems, int32_t k, int32_t maxNumRow, int32_t maxNumCol);
int pda_association_probs_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                const int64_t* rowOff, int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol, int32_t k,
                                double* probs, const int64_t* probOff, int32_t* nFound,
                                void* workspace, int64_t workspaceBytes, void* stream);
int pda_association_probs_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                     int64_t nProblems, int32_t k, double* probs, const int64_t* probOff,
                                     int32_t device);

/* The same body with usePerm == 1 (assignment.cpp:64: permanentProb(cond, condL, nM, 1) in place of assignmentProb),
 * fused on the device: conditionCosts -> likelihoods -> every sub-permanent by one fused gather / condition / subset-DP
 * kernel that keeps each sub-matrix in shared memory -> column sums, normalisation and the scatter through rowIdx.
 * Tables are bit-identical to conditionCosts -> pda_permanent_prob_batch_host(.., 1) -> scatter.  Arguments as for
 * pda_association_probs_batch; status[p] = 0, 1 where the reference throws (a sub-matrix with more than 32 kept rows),
 * 2 where problem p exceeds maxNumRow / maxNumCol (not computed, table untouched -- the conditioning skips it too), 3
 * where conditioning kept fewer rows than there are detections (condL = goodRows - nM < 0, where the reference's size_t
 * subtraction underflows; table all zero).  A gated dummy row with goodRows >= nM is computed as the reference does.
 * pda_association_perm_probs_batch takes problems with nM <= 11 only (maxNumCol > 11 -> PDA_ERR_UNSUPPORTED): every
 *   sub-permanent then has a short side <= 10 and none can come out negative.  It enqueues four launches on `stream`
 *   and never synchronises, so it can be captured in a CUDA graph.  Workspace: O(sum of nM*(nL+1)) doubles.
 * pda_association_perm_probs_batch_host validates the whole batch on the host first; problems with 12+ detections take
 *   the route above (conditionCosts, pda_permanent_prob_batch_host, scatter), so their results are that route's.
 * pda_association_perm_from_moments_batch_host: pda_quadric_cost_batch followed by the pipeline (the usePerm form of
 *   pda_association_from_moments_batch_host); probs and status per frame, frames back to back.
 * The _multi forms cut the batch into contiguous slices, one per device (offsets must be non-decreasing). */
int64_t pda_association_perm_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                             int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol);
int pda_association_perm_probs_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                     const int64_t* rowOff, int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                     int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol,
                                     double* probs, const int64_t* probOff, int32_t* status,
                                     void* workspace, int64_t workspaceBytes, void* stream);
int pda_association_perm_probs_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                          int64_t nProblems, double* probs, const int64_t* probOff, int32_t* status,
                                          int32_t device);
int pda_association_probs_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                           int64_t nProblems, int32_t k, double* probs, const int64_t* probOff,
                                           const int32_t* devices, int32_t nDevices);
int pda_association_perm_probs_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL,
                                                const int32_t* nM, int64_t nProblems, double* probs, const int64_t* probOff,
                                                int32_t* status, const int32_t* devices, int32_t nDevices);

/* ------------------------------------------------------------------------------------------
 * The step in front of the path: cost matrices from quadric moments, on the device.
 * pda_quadric_covs_batch: getCovs (assignment.cpp:693-703) -- quadrics = n 4x4 dual-quadric matrices (16 doubles
 *   each; symmetric, so row- or column-major), covs = n 3x3 matrices (9 doubles each).
 * pda_quadric_cost_batch: computeQuadricCostMatrix (assignment.cpp:705-722) for a batch of frames.  Frame f owns
 *   landmarks [landOff[f], landOff[f+1]) and detections [measOff[f], measOff[f+1]) (offset arrays have nFrames+1
 *   entries); a mean is 3 doubles (what getMeans returns, :685-692), a covariance 9 (column-major 3x3).  Writes the
 *   (nL+nM) x nM column-major matrix of frame f at costs + costOff[f]: squared Mahalanobis distances
 *   d^T (cov_l + cov_m)^-1 d (pivoted 3x3 LDLT as Eigen's ldlt().solve, :716-717), +inf, and `nonassign`
 *   (NONASSIGN_QUADRIC) on the dummy diagonal.  nL / nM (may be NULL) receive the per-frame counts.
 *   The _host form lays the matrices out back to back (costOff = prefix sums of (nL+nM)*nM).
 * pda_association_from_moments_batch_host: getAssignmentProbs (assignment.cpp:38-74, usePerm == 0) from the moments
 *   on -- cost matrices, conditionCosts, assignmentProb(k), weights back at the original landmark indices -- as one
 *   device pipeline.  probs of frame f: nM x (nL+1) row-major, frames back to back.
 * Eigen is not part of this library: the 3x3 solve restates Eigen 3.4's LDLT; agreement with the reference is to
 * rounding (~1e-15 relative on SPD input), not bit-for-bit. */
int pda_quadric_covs_batch(const double* quadrics, int64_t n, double* covs, void* stream);
int pda_quadric_covs_batch_host(const double* quadrics, int64_t n, double* covs, int32_t device);
int pda_quadric_cost_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                           const double* measMean, const double* measCov, const int64_t* measOff,
                           int64_t nFrames, double nonassign, double* costs, const int64_t* costOff,
                           int32_t* nL, int32_t* nM, void* stream);
int pda_quadric_cost_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                const double* measMean, const double* measCov, const int64_t* measOff,
                                int64_t nFrames, double nonassign, double* costs, int32_t device);
int pda_association_from_moments_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                            const double* measMean, const double* measCov, const int64_t* measOff,
                                            int64_t nFrames, double nonassign, int32_t k, double* probs, int32_t device);
int pda_association_perm_from_moments_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                                 const double* measMean, const double* measCov, const int64_t* measOff,
                                                 int64_t nFrames, double nonassign, double* probs, int32_t* status,
                                                 int32_t device);

/* Device-pointer forms of the two moments entries above, with the frame shapes read on the device: every pointer is a
 * device pointer, the host reads only the scalar arguments, and the call enqueues on `stream` without a
 * synchronisation, an allocation or a copy between host and device.  One CUDA graph captured with fixed bounds
 * therefore serves frames of any shape within them (the per-frame call of the SLAM loop).
 *   maxNL, maxNM          the caller's per-frame bounds (host scalars); maxNL >= 0, maxNM >= 1
 *   landCapacity          landmarks the landMean / landCov arrays hold; measCapacity likewise for detections
 *   probs, probCapacity   the tables and the number of doubles probs holds
 *   probOff               nFrames + 1 entries, written: probOff[0] = 0, probOff[f+1] = probOff[f] + nM*(nL+1) for a
 *                         frame that passes the checks below, + 0 for one that does not
 *   status[f]             2: not computed and no table entry written -- offsets negative or descending, reaching past
 *                         landCapacity / measCapacity, nL > maxNL or nM > maxNM (all of these add nothing to probOff),
 *                         or a non-empty table that would end past probCapacity (that frame keeps its span in probOff,
 *                         so every later non-empty frame is status 2 too).  Otherwise the status of the _host form: 0,
 *                         and in the usePerm form 1 and 3 as in pda_association_perm_probs_batch.
 *   nFound[f]             (k-best form; may be NULL) as pda_association_probs_batch reports it; -1 for status 2 or nM == 0
 * Tables of frames with status 0 are bit-identical to the _host form's on the same frames, for any bounds at or above
 * the batch's real maxima.  The usePerm form takes maxNM <= 11 (PDA_ERR_UNSUPPORTED above): its _host form sends
 * frames with 12+ detections down a separate host-driven route, which this form does not have.
 * Errors: PDA_ERR_INVALID for a NULL pointer (other than nFound), nFrames < 0, maxNL < 0, maxNM < 1, a negative capacity
 * or k < 1; PDA_ERR_UNSUPPORTED for maxNL + maxNM > PDA_MAX_DIM; PDA_ERR_WORKSPACE below *_workspace_bytes.
 * Workspace (for the current device): per frame the (maxNL+maxNM) x maxNM cost matrix and 44 B of shapes, plus the
 * chained pipeline's workspace (pda_association_workspace_bytes / pda_association_perm_workspace_bytes at
 * nFrames * (maxNL+maxNM) * maxNM cost elements, nFrames * (maxNL+maxNM) rows and probCapacity table elements). */
int64_t pda_association_from_moments_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxNM, int64_t probCapacity,
                                                     int32_t k);
int pda_association_from_moments_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                                       int64_t landCapacity,
                                       const double* measMean, const double* measCov, const int64_t* measOff,
                                       int64_t measCapacity, int64_t nFrames, int32_t maxNL, int32_t maxNM,
                                       double nonassign, int32_t k,
                                       double* probs, int64_t probCapacity, int64_t* probOff,
                                       int32_t* status, int32_t* nFound,
                                       void* workspace, int64_t workspaceBytes, void* stream);
int64_t pda_association_perm_from_moments_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxNM,
                                                          int64_t probCapacity);
int pda_association_perm_from_moments_batch(const double* landMean, const double* landCov, const int64_t* landOff,
                                            int64_t landCapacity,
                                            const double* measMean, const double* measCov, const int64_t* measOff,
                                            int64_t measCapacity, int64_t nFrames, int32_t maxNL, int32_t maxNM,
                                            double nonassign,
                                            double* probs, int64_t probCapacity, int64_t* probOff, int32_t* status,
                                            void* workspace, int64_t workspaceBytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stereo bounding-box association: asgnBB (assignment.h:21, assignment.cpp:724-775) with computeBBCostMatrix
 * (:777-797) and boundBox::IoU (boundBox.h:62-75), for a batch of frames.  A box is five doubles
 * (xmin, ymin, xmax, ymax, xOffset); frame f owns left boxes [offL[f], offL[f+1]) and right boxes
 * [offR[f], offR[f+1]) (offL/offR have nFrames+1 entries).  assignment[i] = index (within its frame) of the right
 * box paired with left box i, or -1.  nonassign = NONASSIGN_BOUNDBOX.
 * pda_asgn_bb_batch_host reads, stages and writes only [offL[0], offL[nFrames]) of boxesL / assignment and
 * [offR[0], offR[nFrames]) of boxesR, so the entries of a larger batch outside that slice are left as they were.
 * pda_asgn_bb_batch_host_multi cuts the frames into contiguous slices, one per device, each run by the _host form on
 * its own host thread; the arrays are those of the whole batch.
 */
int pda_asgn_bb_batch_host(const double* boxesL, const int64_t* offL, const double* boxesR, const int64_t* offR,
                           int64_t nFrames, double nonassign, int32_t* assignment, int32_t device);
int pda_asgn_bb_batch_host_multi(const double* boxesL, const int64_t* offL, const double* boxesR, const int64_t* offR,
                                 int64_t nFrames, double nonassign, int32_t* assignment,
                                 const int32_t* devices, int32_t nDevices);

/* Device-pointer form of pda_asgn_bb_batch_host, with the frame shapes read on the device: every pointer is a device
 * pointer, the host reads only the scalar arguments, and the call enqueues on `stream` without a synchronisation, an
 * allocation or a copy between host and device.  One CUDA graph captured with fixed bounds therefore serves frames of
 * any shape within them (the per-frame stereo match of the SLAM loop, dataframe.cpp:306).
 *   maxNL, maxBoxes   the caller's per-frame bounds (host scalars): left boxes nL <= maxNL, and nL + nR <= maxBoxes
 *   capL, capR        boxes boxesL / boxesR hold; assignment holds capL entries.  boxesL (boxesR) may be NULL when capL
 *                     (capR) is 0
 *   status[f]         0: computed -- every left box of the frame gets its partner or -1 (all -1 without right boxes),
 *                     bit-identical to the _host form for any bounds at or above the batch's maxima;
 *                     2: not computed, nothing written.  A frame is status 2 when a range is negative, descending or
 *                     past capL / capR, when nL > maxNL or nL + nR > maxBoxes, or when offL[f] is below an earlier
 *                     offL[g] (g < f): then an earlier frame may own some of its left entries, and results are
 *                     addressed by offL directly.  Entries outside every computed frame are left untouched.
 * Errors: PDA_ERR_INVALID for a NULL pointer, nFrames < 0, a negative capacity, maxNL < 1 or maxBoxes < maxNL;
 * PDA_ERR_UNSUPPORTED for maxBoxes > PDA_MAX_DIM (or what pda_murty_workspace_bytes refuses at these bounds);
 * PDA_ERR_WORKSPACE below pda_asgn_bb_workspace_bytes.
 * Workspace (for the current device and Murty path): per frame a maxBoxes x maxNL cost matrix, maxNL row4col entries
 * and 48 B of shapes, plus pda_murty_workspace_bytes(nFrames, 1, maxBoxes, maxNL). */
int64_t pda_asgn_bb_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxBoxes);
int pda_asgn_bb_batch(const double* boxesL, const int64_t* offL, int64_t capL,
                      const double* boxesR, const int64_t* offR, int64_t capR,
                      int64_t nFrames, int32_t maxNL, int32_t maxBoxes, double nonassign,
                      int32_t* assignment, int32_t* status,
                      void* workspace, int64_t workspaceBytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Matrix permanent, Nijenhuis-Wilf / Ryser over Gray-code column subsets.
 * Replaces permanentExactSquare / permanentExact (nwPerm.h:22-24; nwPerm.cpp:217-231, 251-332).
 *
 * pda_permanent_batch: nMats matrices, matrix i is rows[i] x cols[i] at mats + matOff[i];
 *   rectangular ones are padded with ones to max(rows, cols) and divided by (|rows-cols|)!
 *   exactly as the reference does.  out[i] = permanent; status[i] = 0, or 1 where the
 *   reference throws (dimension > 32).  maxDim >= max(rows[i], cols[i]) over the batch
 *   (it selects the register tile; a batch is fastest when its matrices share one size).
 *   This device-pointer form walks every matrix the reference's way (NW on the ones-padded
 *   square), whatever its size; a matrix with max(rows, cols) above maxDim (but <= 32) is not
 *   computed: out[i] = 0 and status[i] = 2.  Status 1 takes precedence.
 * pda_permanent_batch_host sees the dimensions, so it sends matrices whose short side is <= 10
 *   to a cancellation-free subset dynamic programme instead; it never reports status 2.
 * pda_permanent_range: partial NW sum of ONE n x n matrix over Gray indices [begin, end)
 *   (index 0 = the empty-subset seed term), as an unevaluated double-double partial[0] + partial[1];
 *   partial sums over disjoint ranges covering [0, 2^(n-1)) add up to p, and the permanent is
 *   (4*(n&1)-2) * p.  This is the unit the multi-GPU split all-reduces.
 * Results agree with the reference to ~1e-13 relative on well-conditioned inputs (the summation
 * order differs: the walk is split into per-thread ranges and accumulated in double-double).
 */
int64_t pda_permanent_workspace_bytes(int64_t nMats);
int pda_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                        int64_t nMats, int32_t maxDim, double* out, int32_t* status,
                        void* workspace, int64_t workspaceBytes, void* stream);
int pda_permanent_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                             int64_t nMats, double* out, int32_t* status, int32_t device);
int pda_permanent_range(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial,
                        void* workspace, int64_t workspaceBytes, void* stream);
int pda_permanent_range_host(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial,
                             int32_t device);

/* Multi-device forms.  pda_permanent_batch_host_multi: independent matrices, one contiguous slice per device, no
 * collective.  pda_permanent_sharded_host: ONE matrix (BASELINE config 5, n = 28): the Gray index range [0, 2^(n-1)) of
 * the NW walk (nwPerm.cpp:294-323) is cut into a power-of-two number of equal pieces, one per device (devices beyond the
 * largest power of two <= nDevices stay idle), each device runs pda_permanent_range on its piece, and the 16-byte
 * (hi, lo) partial sums are gathered by the host and added in device order with an error-free two-sum -- the one real
 * exchange step of this path, and a deterministic one. */
int pda_permanent_batch_host_multi(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                   int64_t nMats, double* out, int32_t* status, const int32_t* devices, int32_t nDevices);
int pda_permanent_sharded_host(const double* A, int32_t n, const int32_t* devices, int32_t nDevices, double* out);

/* Huber's randomised approximation of the permanent: permanentApproximation / permanentApproximationSquare with their
 * sinkhorn / hl_factor / pickRowFromProbs helpers (nwPerm.h:27-35, nwPerm.cpp:36-211), `iterations` acceptance /
 * rejection trials per matrix (the reference uses apprxIter = 300, assignment.cpp:10).  Rectangular input is padded with
 * ones and divided by (|rows-cols|)!; status[i] = 1 above dimension 32.  The reference draws from an unseeded global
 * rand(); here every draw is a counter-based value keyed by (seed, matrix index, trial, column), so results are
 * reproducible and independent of batch order -- agreement with the reference is statistical (same estimator, same
 * trial count), not sample for sample.  pda_set_approx_seed sets the seed used where the reference signature has no
 * room for one (permOpt == 0 below). */
int pda_permanent_approx_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                               int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status, void* stream);
int pda_permanent_approx_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                    int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status,
                                    int32_t device);
void pda_set_approx_seed(uint64_t seed);

/* conditionedPermanent (assignment.cpp:325-435) for a batch of matrices: zero rows/columns dropped,
 * columns scaled, permanent of the transpose, negative-result retry.  permOpt 0 (Huber approximation, 300 trials),
 * 1 (exact) or 2 ("long": the same double kernel, as in the reference); anything else sets status (the reference throws).
 * Stages the matrices and runs pda_conditioned_permanent_batch once; a matrix with a side above 128 is status 1. */
int pda_conditioned_permanent_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows,
                                         const int32_t* cols, int64_t nMats, int32_t permOpt,
                                         double* out, int32_t* status, int32_t device);

/* permanentProb (assignment.cpp:145-290): permanent-based marginals for a batch of problems.
 * probs at probOff[p], numCol[p] x (nL[p]+1) row-major; status[p] = 1 where the reference throws.  Stages the
 * problems and runs pda_permanent_prob_batch once per chunk of at most 65 536 sub-permanents; the whole range from the
 * first table to the end of the last is written, zeros in any gaps between tables. */
int pda_permanent_prob_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL,
                                  const int32_t* nM, int64_t nProblems, int32_t permOpt,
                                  double* probs, const int64_t* probOff, int32_t* status, int32_t device);

/* Device-pointer forms of pda_conditioned_permanent_batch_host and pda_permanent_prob_batch_host: every array is a device
 * pointer, the host reads none of it, and the call is enqueued on `stream` without a synchronisation or a copy between
 * host and device, so it can follow a device producer and be captured in a CUDA graph.  The _host forms run these
 * calls, so tables, results and statuses equal theirs on any batch the _host form runs as one chunk (up to 65 536
 * sub-permanents; every conditioned_permanent batch), for every permOpt:
 *   - a sub-matrix whose short side is <= 10 runs the subset programme in shared memory, straight out of the input;
 *   - a short side of 11..31 is walked by the NW kernel with the launch shape pda_permanent_batch_host takes for the
 *     batch's sub-permanents (their count and largest dimension, counted over all problems), and an item that comes
 *     out negative is walked again untransposed with the shape of a one-matrix launch (assignment.cpp:409-419), all on
 *     the device;
 *   - permOpt == 0 runs Huber's approximation (300 trials) with the seed of pda_set_approx_seed.  Its draws are keyed by
 *     item index: for permanent_prob, the sub-permanents of the call counted from its first problem, nM * (nL+1) per
 *     problem with nM > 1, (m, l) in m-major order; for conditioned_permanent, the matrix index.
 * Status per problem / matrix: 0 computed; 1 where the reference throws (a sub-matrix keeps more than 32 rows, or
 * permOpt outside 0..2 for a problem with nM > 1 / any matrix); 2 above the call's maxNumRow / maxNumCol (maxDim), or
 * with nL < 0, nM < 1 or a negative dimension: not computed, its table (out[i]) is left untouched.  The nM * (nL+1)
 * tables must not overlap: the sub-permanents of the call must fit in totalProbElems, a problem beyond that is status 2.
 *
 * Workspace (pda_*_workspace_bytes, for the current device): a copy of the costs, per problem 12 B, and per item
 * (totalProbElems, or nMats) 20 B.  Calls that may materialise items -- permOpt == 0, or sub-matrices with a short side
 * of 11 or more (maxNumCol >= 12 and maxNumRow >= 12; maxDim >= 11) -- add per item the scaled sub-matrix, 8 B times
 * min(32, maxNumRow - 1) * min(32, maxNumCol - 1) (min(32, maxDim)^2), and 32 B of descriptors; calls that may walk
 * (permOpt 1 or 2 with such sub-matrices) add 16 B per CTA a matrix may take (twice the SM count) plus 4 B per item.
 * A smaller workspace is PDA_ERR_WORKSPACE; nothing beyond workspaceBytes is written. */
int64_t pda_permanent_prob_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalProbElems,
                                           int32_t maxNumRow, int32_t maxNumCol, int32_t permOpt);
int pda_permanent_prob_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                             int64_t nProblems, int64_t totalCostElems, int64_t totalProbElems,
                             int32_t maxNumRow, int32_t maxNumCol, int32_t permOpt,
                             double* probs, const int64_t* probOff, int32_t* status,
                             void* workspace, int64_t workspaceBytes, void* stream);
int64_t pda_conditioned_permanent_workspace_bytes(int64_t nMats, int32_t maxDim, int32_t permOpt);
int pda_conditioned_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                    int64_t nMats, int32_t maxDim, int32_t permOpt, double* out, int32_t* status,
                                    void* workspace, int64_t workspaceBytes, void* stream);

/* The same over several devices: contiguous slices of problems, one per device (the (nL+1) * nM sub-permanents of a
 * problem stay together; assignment.cpp:213-246). */
int pda_permanent_prob_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL,
                                        const int32_t* nM, int64_t nProblems, int32_t permOpt,
                                        double* probs, const int64_t* probOff, int32_t* status,
                                        const int32_t* devices, int32_t nDevices);

#ifdef __cplusplus
}
#endif
#endif /* PDA_B200_H */
