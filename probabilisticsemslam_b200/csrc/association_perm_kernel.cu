// association_perm_kernel.cu -- the numeric body of getAssignmentProbs with usePerm (assignment.cpp:57-74, :64
// permanentProb(cond, condL, nM, 1)) as one device pipeline on one stream, without a host synchronisation or a copy
// between host and device inside it:
//   1. condition_costs_kernel  conditionCosts; writes goodRows and condL = goodRows - nM (weights_kernel.cu)
//   2. to_probs_kernel         likelihoods of the conditioned goodRows x nM matrix, in place
//   3. cond_perm_kernel        blockIdx.x = problem, its warps over the problem's sub-permanents: each gathers its
//                              sub-matrix straight out of the likelihoods, conditions and scales it into shared memory
//                              and runs the subset DP there -- nothing is materialised in global memory.  A batch too
//                              small to fill the chip (a single SLAM frame) spreads each problem over blockIdx.y too
//   4. finish_scatter_kernel   one warp per problem: |P(l,m) * perm|, column sums, normalisation by the largest column
//                              sum (finish_kernel of permprob_device_kernel.cu), written straight into the caller's
//                              nM x (nL+1) table through rowIdx
// The sub-permanents live in slots sized from the UNconditioned dimensions, nM * (nL+1) per problem at probOff[p]
// (slot (m, l): landmark item l for l < condL, the non-assignment item for l == nL), so the host never needs condL.
// Scope: nM <= 11.  Every sub-permanent then has a short side <= 10, which the subset DP takes, and no permanent can
// come out negative (no retry, :409-419).  The arithmetic is permanentProb's own (perm_device.cuh), so the
// tables equal conditionCosts -> pda_permanent_prob_batch_host(.., 1) -> scatter bit for bit.  The *_host entries send
// problems with 12+ detections down exactly that route.
#include "pda_internal.h"
#include "pda_host_stage.h"
#include "perm_device.cuh"

#include <algorithm>
#include <vector>

namespace pda {
namespace {

constexpr int FUSED_MAX_COL = 11;              // detections per problem the fused kernel takes
constexpr int SUB_COLS = FUSED_MAX_COL - 1;    // kept columns of a sub-matrix (its short side)
constexpr int SUB_ROWS = PDA_MAX_PERM_DIM;     // kept rows (long side); more is where the reference throws
constexpr int PERM_WARPS = 4;
constexpr int FINISH_WARPS = 4;
constexpr int SMEM_BUDGET = 48 * 1024;         // dynamic shared memory per CTA: below the opt-in limit, so no attribute call

// shared memory of one warp of cond_perm_kernel, in doubles: DP buffers (2 cap + 16), the scaled transposed sub-matrix,
// the column scales, then the kept column (16) and row (PDA_MAX_DIM) indices as shorts
__host__ __device__ constexpr int warp_doubles(int cap) { return 2 * cap + 16 + SUB_ROWS * SUB_COLS + 16 + (16 + PDA_MAX_DIM) / 4; }

struct CondPermArgs {
    const double* P; const int64_t* costOff; const int32_t* nL; const int32_t* nM; const int32_t* condNL;
    const int64_t* probOff; double* perm; int32_t* slotStatus;
    int32_t maxRow, maxCol, cap, warps;
};

// problems the fused kernels leave alone: nM above the call's maxNumCol (or above 11), or nL + nM above maxNumRow
__device__ __forceinline__ bool out_of_scope(int L, int M, int maxRow, int maxCol) { return M > maxCol || L + M > maxRow; }

__global__ void __launch_bounds__(32 * PERM_WARPS) cond_perm_kernel(const CondPermArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = blockIdx.x;
    const int L = a.nL[p], M = a.nM[p], cL = a.condNL[p];
    if (M < 2 || L == 0 || cL < 0 || out_of_scope(L, M, a.maxRow, a.maxCol)) return;
    double* buf = smem + (size_t)warp * warp_doubles(a.cap);
    double* sub = buf + 2 * a.cap + 16;
    double* scale = sub + SUB_ROWS * SUB_COLS;
    short* keepC = reinterpret_cast<short*>(scale + 16);
    short* keepR = keepC + 16;
    const double* Pp = a.P + a.costOff[p];
    const int64_t slot0 = a.probOff[p];
    const int items = M * (cL + 1);
    for (int e = (int)blockIdx.y * a.warps + warp; e < items; e += (int)gridDim.y * a.warps) {
        const int m = e / (cL + 1), l = e % (cL + 1);
        const int64_t slot = slot0 + (int64_t)m * (L + 1) + (l < cL ? l : L);
        Gather g;
        if (!item_gather(Pp, cL, M, m, l, g)) continue;  // zero likelihood: the finish never reads this slot
        __syncwarp();  // the previous item's reads of the shared buffers are done
        int nKR, nKC;
        condition_warp(g, scale, keepC, keepR, lane, nKR, nKC);
        if ((nKR > nKC ? nKR : nKC) > PDA_MAX_PERM_DIM) {  // permanentExactSquare throws (nwPerm.cpp:327-330): 1 and
            if (lane == 0) { a.perm[slot] = 1.0; a.slotStatus[slot] = 1; }  // status 1, as permanentProb leaves them
            continue;
        }
        write_scaled(g, scale, keepC, keepR, nKR, nKC, 1, sub, lane);
        __syncwarp();
        const double r = perm_dp_subsets(sub, nKC, nKR, buf, a.cap, lane);
        if (lane == 0) { a.perm[slot] = r / scale_product(scale, nKC); a.slotStatus[slot] = 0; }
    }
}

// status: 0 ok, 1 where the reference throws (a sub-matrix with more than 32 kept rows), 2 not computed here (out of
// scope), 3 where conditioning kept fewer rows than there are detections, so that condL = goodRows - nM (:60) would be
// negative (the reference's size_t subtraction underflows).  A gated dummy row with goodRows >= nM is NOT an error: the
// reference runs permanentProb with that condL and scatters the first condL rows back, and so does this pipeline.
__global__ void finish_scatter_kernel(const double* __restrict__ P, const int64_t* __restrict__ costOff,
                                      const int32_t* __restrict__ nL, const int32_t* __restrict__ nM,
                                      const int32_t* __restrict__ condNL, const int64_t* __restrict__ rowIdx,
                                      const int64_t* __restrict__ rowOff, double* __restrict__ perm,
                                      const int32_t* __restrict__ slotStatus, int64_t nProblems, int32_t maxRow, int32_t maxCol,
                                      double* __restrict__ probs, const int64_t* __restrict__ probOff, int32_t* __restrict__ status) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * FINISH_WARPS + warp;
    if (p >= nProblems) return;
    const int L = nL[p], M = nM[p], cL = condNL[p];
    if (out_of_scope(L, M, maxRow, maxCol)) { if (lane == 0) status[p] = 2; return; }
    double* out = probs + probOff[p];
    if (L == 0) {  // :51-53
        for (int m = lane; m < M; m += 32) out[m] = 1.0;
        if (lane == 0) status[p] = 0;
        return;
    }
    for (int e = lane; e < M * (L + 1); e += 32) out[e] = 0.0;
    const int64_t* idx = rowIdx + rowOff[p];
    if (M == 0 || cL < 0) {
        if (lane == 0) status[p] = (M == 0) ? 0 : 3;
        return;
    }
    __syncwarp();
    const double* Pp = P + costOff[p];
    if (M == 1) {  // permanentProb with one detection (:166-171): normalise by std::reduce, which sums in blocks of four
        double norm = 0.0;
        if (lane == 0) {
            const int n = cL + 1;
            double acc = 0.0;
            int i = 0;
            for (; n - i >= 4; i += 4) acc = acc + ((Pp[i] + Pp[i + 1]) + (Pp[i + 2] + Pp[i + 3]));
            for (; i < n; ++i) acc = acc + Pp[i];
            norm = 1.0 / acc;
            status[p] = 0;
        }
        norm = __shfl_sync(0xffffffffu, norm, 0);
        for (int i = lane; i <= cL; i += 32) out[i < cL ? (int)idx[i] : L] = Pp[i] * norm;
        return;
    }
    // permprob_device_kernel.cu's finish_kernel on the conditioned problem (nL = cL); the terms go back into the slots
    const int good = cL + M;
    const int64_t slot0 = probOff[p];
    double best = 0.0;
    int bad = 0;
    for (int m = lane; m < M; m += 32) {
        double colPerm = 0.0;
        for (int l = 0; l <= cL; ++l) {
            const int64_t s = slot0 + (int64_t)m * (L + 1) + (l < cL ? l : L);
            const double e = (l < cL) ? Pp[l + (size_t)m * good] : Pp[(cL + m) + (size_t)m * good];
            double t = 0.0;
            if (l == cL || e != 0.0) {
                bad |= slotStatus[s];
                t = fabs(e * perm[s]);
                colPerm += t;
            }
            perm[s] = t;
        }
        best = (best < colPerm) ? colPerm : best;  // std::max over columns (:255)
    }
    best = warp_max(best);
    bad = __any_sync(0xffffffffu, bad != 0);
    __syncwarp();
    const double norm = 1.0 / best;
    for (int e = lane; e < M * (cL + 1); e += 32) {  // scatter through rowIdx (:68-74)
        const int m = e / (cL + 1), l = e % (cL + 1);
        const int dst = (l < cL) ? (int)idx[l] : L;
        out[(size_t)m * (L + 1) + dst] = perm[slot0 + (int64_t)m * (L + 1) + (l < cL ? l : L)] * norm;
    }
    if (lane == 0) status[p] = bad ? 1 : 0;
}

struct PermWorkspace {
    int32_t* goodRows; int32_t* condNL; double* condCosts; int64_t* rowIdx; double* perm; int32_t* slotStatus;
    size_t bytes;
};
PermWorkspace carve(void* workspace, int64_t nProblems, int64_t totalCostElems, int64_t totalRows, int64_t totalProbElems) {
    const size_t n = (size_t)std::max<int64_t>(nProblems, 1);
    WorkspaceLayout w(workspace);
    PermWorkspace ws;
    ws.goodRows = w.take<int32_t>(n);
    ws.condNL = w.take<int32_t>(n);
    ws.condCosts = w.take<double>((size_t)totalCostElems);
    ws.rowIdx = w.take<int64_t>((size_t)totalRows);
    ws.perm = w.take<double>((size_t)totalProbElems);
    ws.slotStatus = w.take<int32_t>((size_t)totalProbElems);
    ws.bytes = w.bytes();
    return ws;
}

// The four launches; maxCol <= FUSED_MAX_COL.  Problems out of scope get status 2 and an untouched table.
int launch_perm_pipeline(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                         const int64_t* rowOff, int64_t nProblems, const PermWorkspace& ws, int32_t maxRow, int32_t maxCol,
                         double* probs, const int64_t* probOff, int32_t* status, cudaStream_t s) {
    PDA_TRY(launch_condition_costs(costs, costOff, nullptr, nM, nProblems, rowOff, ws.condCosts, ws.rowIdx, ws.goodRows, s, nL,
                                   ws.condNL, maxRow, maxCol));  // out-of-scope problems are not even read
    // conditioned problems live at the original cost offsets (they only shrink)
    PDA_TRY(launch_to_probs(ws.condCosts, costOff, nullptr, nProblems, s, ws.goodRows, nM));
    CondPermArgs a;
    a.P = ws.condCosts; a.costOff = costOff; a.nL = nL; a.nM = nM; a.condNL = ws.condNL;
    a.probOff = probOff; a.perm = ws.perm; a.slotStatus = ws.slotStatus;
    a.maxRow = maxRow; a.maxCol = maxCol;
    a.cap = 1 << std::max(0, maxCol - 1);  // states of the largest short side, nM - 1
    const int perWarp = warp_doubles(a.cap) * (int)sizeof(double);
    a.warps = std::max(1, std::min(PERM_WARPS, SMEM_BUDGET / perWarp));
    if (maxCol >= 2) {
        // CTAs per problem: one for large batches; for small ones enough to fill every SM about eight times over, but no
        // more than the largest problem has items (nM * (condL + 1) <= maxCol * maxRow)
        DeviceInfo dev;
        PDA_TRY(current_device_info(&dev));
        const int64_t want = ((int64_t)dev.smCount * 8 + nProblems - 1) / nProblems;
        const int64_t most = ((int64_t)maxCol * maxRow + a.warps - 1) / a.warps;
        const unsigned split = (unsigned)std::max<int64_t>(1, std::min<int64_t>(std::min(want, most), 65535));
        cond_perm_kernel<<<dim3((unsigned)nProblems, split), 32 * a.warps, (size_t)a.warps * perWarp, s>>>(a);
        PDA_CUDA_TRY(cudaGetLastError());
    }
    finish_scatter_kernel<<<(unsigned)((nProblems + FINISH_WARPS - 1) / FINISH_WARPS), 32 * FINISH_WARPS, 0, s>>>(
        ws.condCosts, costOff, nL, nM, ws.condNL, ws.rowIdx, rowOff, ws.perm, ws.slotStatus, nProblems, maxRow, maxCol, probs,
        probOff, status);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

// Problems with 12+ detections, as getAssignmentProbsFromCosts(.., usePerm = true) has always run them: conditionCosts,
// then pda_permanent_prob_batch_host(.., 1) on the conditioned problems, then the scatter through rowIdx, on the host.
// Problem i of this list is costs[i] ((nL+nM) x nM, column-major); its table goes to probs + probOff[i].
int routed_perm_probs(const std::vector<std::vector<double> >& costs, const std::vector<int32_t>& nL,
                      const std::vector<int32_t>& nM, double* probs, const std::vector<int64_t>& probOff, int32_t* status,
                      const std::vector<int64_t>& statusAt, int device) {
    const size_t n = costs.size();
    std::vector<int64_t> cOff(n), rOff(n);
    std::vector<int32_t> nr(n), good(n);
    size_t nC = 0, nR = 0;
    for (size_t i = 0; i < n; ++i) {
        cOff[i] = (int64_t)nC; rOff[i] = (int64_t)nR; nr[i] = nL[i] + nM[i];
        nC += costs[i].size(); nR += (size_t)nr[i];
    }
    std::vector<double> flat(std::max<size_t>(nC, 1)), cond(std::max<size_t>(nC, 1));
    std::vector<int64_t> idx(std::max<size_t>(nR, 1));
    for (size_t i = 0; i < n; ++i) std::copy(costs[i].begin(), costs[i].end(), flat.begin() + cOff[i]);
    PDA_TRY(pda_condition_costs_batch_host(flat.data(), cOff.data(), nr.data(), nM.data(), (int64_t)n, rOff.data(), cond.data(),
                                           idx.data(), good.data(), device));
    std::vector<int64_t> pcOff, ppOff;
    std::vector<int32_t> pL, pM;
    std::vector<size_t> which;
    size_t nP = 0;
    for (size_t i = 0; i < n; ++i) {
        double* out = probs + probOff[i];
        const int L = nL[i], M = nM[i], cL = good[i] - M;
        std::fill(out, out + (size_t)M * (L + 1), 0.0);
        status[statusAt[i]] = 0;
        if (L == 0) { std::fill(out, out + M, 1.0); continue; }  // :51-53
        if (cL < 0) { status[statusAt[i]] = 3; continue; }  // goodRows < nM
        which.push_back(i); pcOff.push_back(cOff[i]); ppOff.push_back((int64_t)nP); pL.push_back(cL); pM.push_back(M);
        nP += (size_t)M * (cL + 1);
    }
    if (which.empty()) return PDA_OK;
    std::vector<double> cp(nP);
    std::vector<int32_t> st(which.size());
    PDA_TRY(pda_permanent_prob_batch_host(cond.data(), pcOff.data(), pL.data(), pM.data(), (int64_t)which.size(), 1, cp.data(),
                                          ppOff.data(), st.data(), device));
    for (size_t j = 0; j < which.size(); ++j) {
        const size_t i = which[j];
        const int L = nL[i], M = nM[i], cL = pL[j];
        double* out = probs + probOff[i];
        const double* in = cp.data() + ppOff[j];
        for (int m = 0; m < M; ++m) {
            for (int l = 0; l < cL; ++l) out[(size_t)m * (L + 1) + (size_t)idx[(size_t)rOff[i] + l]] = in[(size_t)m * (cL + 1) + l];
            out[(size_t)m * (L + 1) + L] = in[(size_t)m * (cL + 1) + cL];
        }
        status[statusAt[i]] = st[j];
    }
    return PDA_OK;
}

// ---- multi-device forms: contiguous slices of problems, one per device.  Each slice is handed to the single-device
// entry with offsets relative to its own first cost / table, so a device stages and writes back only its slice; offsets
// must therefore be non-decreasing. ----
template <class F>
int run_slices(const int64_t* costOff, const int64_t* probOff, int64_t nProblems, const int32_t* devices, int32_t nDevices,
               const char* who, F&& f) {
    for (int64_t p = 1; p < nProblems; ++p)
        if (costOff[p] < costOff[p - 1] || probOff[p] < probOff[p - 1]) return fail(PDA_ERR_INVALID, "%s: offsets must be non-decreasing", who);
    if (costOff[0] < 0 || probOff[0] < 0) return fail(PDA_ERR_INVALID, "%s: negative offset", who);
    return run_sharded(nProblems, devices, nDevices, [&](int64_t p0, int64_t p1, int dev) {
        std::vector<int64_t> co((size_t)(p1 - p0)), po((size_t)(p1 - p0));
        for (int64_t p = p0; p < p1; ++p) { co[(size_t)(p - p0)] = costOff[p] - costOff[p0]; po[(size_t)(p - p0)] = probOff[p] - probOff[p0]; }
        return f(p0, p1, dev, co.data(), po.data());
    });
}
}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

int64_t pda_association_perm_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                             int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol) {
    if (nProblems < 0 || totalCostElems < 0 || totalRows < 0 || totalProbElems < 0)
        return fail(PDA_ERR_INVALID, "association_perm: negative size");
    if (maxNumCol > FUSED_MAX_COL || maxNumRow > PDA_MAX_DIM)
        return fail(PDA_ERR_UNSUPPORTED, "association_perm: maxNumRow %d / maxNumCol %d above %d / %d", maxNumRow, maxNumCol,
                    PDA_MAX_DIM, FUSED_MAX_COL);
    return (int64_t)carve(nullptr, nProblems, totalCostElems, totalRows, totalProbElems).bytes;
}

int pda_association_perm_probs_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                     const int64_t* rowOff, int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                     int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol,
                                     double* probs, const int64_t* probOff, int32_t* status,
                                     void* workspace, int64_t workspaceBytes, void* stream) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association_perm: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !rowOff || !probs || !probOff || !status || !workspace)
        return fail(PDA_ERR_INVALID, "association_perm: NULL argument");
    if (maxNumCol > FUSED_MAX_COL)
        return fail(PDA_ERR_UNSUPPORTED, "association_perm: maxNumCol %d above %d (the *_host entry routes such problems)",
                    maxNumCol, FUSED_MAX_COL);
    if (maxNumRow > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "association_perm: maxNumRow %d above %d", maxNumRow, PDA_MAX_DIM);
    if (maxNumRow < 1 || maxNumCol < 1) return fail(PDA_ERR_INVALID, "association_perm: maxNumRow / maxNumCol < 1");
    if (totalCostElems < 0 || totalRows < 0 || totalProbElems < 0) return fail(PDA_ERR_INVALID, "association_perm: negative total");
    const PermWorkspace ws = carve(workspace, nProblems, totalCostElems, totalRows, totalProbElems);
    if ((int64_t)ws.bytes > workspaceBytes) return fail(PDA_ERR_WORKSPACE, "association_perm: workspace too small");
    return launch_perm_pipeline(costs, costOff, nL, nM, rowOff, nProblems, ws, maxNumRow, maxNumCol, probs, probOff, status,
                                reinterpret_cast<cudaStream_t>(stream));
}

int pda_association_perm_probs_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                          int64_t nProblems, double* probs, const int64_t* probOff, int32_t* status,
                                          int32_t device) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association_perm: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status) return fail(PDA_ERR_INVALID, "association_perm: NULL argument");
    const size_t n = (size_t)nProblems;
    std::vector<int64_t> rowOff(n);
    std::vector<size_t> large;
    size_t nCost = 0, nRows = 0, nProb = 0;
    int maxR = 1, maxC = 1;
    for (size_t p = 0; p < n; ++p) {
        const int L = nL[p], M = nM[p];
        if (L < 0 || M < 1) return fail(PDA_ERR_INVALID, "association_perm: problem %lld has nL=%d nM=%d", (long long)p, L, M);
        if (costOff[p] < 0 || probOff[p] < 0) return fail(PDA_ERR_INVALID, "association_perm: problem %lld has a negative offset", (long long)p);
        if (L + M > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "association_perm: problem %lld has nL + nM = %d (limit %d)", (long long)p, L + M, PDA_MAX_DIM);
        rowOff[p] = (int64_t)nRows;
        nRows += (size_t)(L + M);
        nCost = std::max(nCost, (size_t)costOff[p] + (size_t)(L + M) * M);
        nProb = std::max(nProb, (size_t)probOff[p] + (size_t)M * (L + 1));
        if (M > FUSED_MAX_COL) { large.push_back(p); continue; }
        maxR = std::max(maxR, L + M); maxC = std::max(maxC, M);
    }
    if (large.size() < n) {
        DeviceScope scope;
        PDA_TRY(scope.enter(device));
        const int64_t wsBytes = pda_association_perm_workspace_bytes(nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC);
        if (wsBytes < 0) return (int)wsBytes;
        HostIO io(device);
        const size_t oC = io.in(costs, nCost * 8), oCO = io.in(costOff, n * 8), oL = io.in(nL, n * 4), oM = io.in(nM, n * 4);
        const size_t oRO = io.in(rowOff.data(), n * 8), oPO = io.in(probOff, n * 8);
        const size_t oP = io.out(probs, nProb * 8), oS = io.out(status, n * 4), oWs = io.scratch((size_t)wsBytes);
        PDA_TRY(io.commit());
        PDA_TRY(io.upload());
        PDA_TRY(pda_association_perm_probs_batch(io.at<double>(oC), io.at<int64_t>(oCO), io.at<int32_t>(oL), io.at<int32_t>(oM),
                                                 io.at<int64_t>(oRO), nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR,
                                                 maxC, io.at<double>(oP), io.at<int64_t>(oPO), io.at<int32_t>(oS),
                                                 io.at<unsigned char>(oWs), wsBytes, io.stream()));
        PDA_TRY(io.download());
    }
    if (large.empty()) return PDA_OK;
    std::vector<std::vector<double> > lc(large.size());
    std::vector<int32_t> lL(large.size()), lM(large.size());
    std::vector<int64_t> lPO(large.size()), lSt(large.size());
    for (size_t i = 0; i < large.size(); ++i) {
        const size_t p = large[i];
        lL[i] = nL[p]; lM[i] = nM[p]; lPO[i] = probOff[p]; lSt[i] = (int64_t)p;
        lc[i].assign(costs + costOff[p], costs + costOff[p] + (size_t)(nL[p] + nM[p]) * nM[p]);
    }
    return routed_perm_probs(lc, lL, lM, probs, lPO, status, lSt, device);
}

// getAssignmentProbs (assignment.cpp:38-74, usePerm == 1) from the quadric moments on: cost matrices, then the pipeline
// above.  probs of frame f: nM x (nL+1) row-major at the prefix sum of nM*(nL+1) (frames with nM == 0 contribute
// nothing); status[f] as in pda_association_perm_probs_batch_host.
int pda_association_perm_from_moments_batch_host(const double* landMean, const double* landCov, const int64_t* landOff,
                                                 const double* measMean, const double* measCov, const int64_t* measOff,
                                                 int64_t nFrames, double nonassign, double* probs, int32_t* status,
                                                 int32_t device) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "association_perm_from_moments: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!landOff || !measOff || !probs || !status) return fail(PDA_ERR_INVALID, "association_perm_from_moments: NULL argument");
    const size_t n = (size_t)nFrames;
    std::vector<int64_t> costOff(n), probOff(n), rowOff(n);
    std::vector<size_t> large;
    size_t nCost = 0, nProb = 0, nRows = 0;
    int maxR = 1, maxC = 1;
    for (size_t f = 0; f < n; ++f) {
        const int64_t L = landOff[f + 1] - landOff[f], M = measOff[f + 1] - measOff[f];
        if (landOff[f] < 0 || measOff[f] < 0 || L < 0 || M < 0)
            return fail(PDA_ERR_INVALID, "association_perm_from_moments: offsets of frame %lld are negative or not ascending", (long long)f);
        if (L + M > PDA_MAX_DIM)
            return fail(PDA_ERR_UNSUPPORTED, "association_perm_from_moments: frame %lld has %lld landmarks + %lld detections (limit %d)",
                        (long long)f, (long long)L, (long long)M, PDA_MAX_DIM);
        costOff[f] = (int64_t)nCost; probOff[f] = (int64_t)nProb; rowOff[f] = (int64_t)nRows;
        nCost += (size_t)((L + M) * M); nProb += (size_t)(M * (L + 1)); nRows += (size_t)(L + M);
        if (M > FUSED_MAX_COL) { large.push_back(f); continue; }
        maxR = std::max(maxR, (int)(L + M)); maxC = std::max(maxC, (int)M);
    }
    const size_t nLand = (size_t)landOff[n], nMeas = (size_t)measOff[n];
    if ((nLand && (!landMean || !landCov)) || (nMeas && (!measMean || !measCov)))
        return fail(PDA_ERR_INVALID, "association_perm_from_moments: NULL moments");
    if (large.size() < n) {
        DeviceScope scope;
        PDA_TRY(scope.enter(device));
        const int64_t wsBytes = pda_association_perm_workspace_bytes(nFrames, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC);
        if (wsBytes < 0) return (int)wsBytes;
        HostIO io(device);
        const size_t oLM = io.in(landMean, nLand * 24), oLC = io.in(landCov, nLand * 72), oLO = io.in(landOff, (n + 1) * 8);
        const size_t oMM = io.in(measMean, nMeas * 24), oMC = io.in(measCov, nMeas * 72), oMO = io.in(measOff, (n + 1) * 8);
        const size_t oCO = io.in(costOff.data(), n * 8), oPO = io.in(probOff.data(), n * 8), oRO = io.in(rowOff.data(), n * 8);
        const size_t oP = io.out(probs, nProb * 8), oS = io.out(status, n * 4);
        const size_t oC = io.scratch(nCost * 8), oNL = io.scratch(n * 4), oNM = io.scratch(n * 4), oWs = io.scratch((size_t)wsBytes);
        PDA_TRY(io.commit());
        const cudaStream_t s = io.stream();
        PDA_TRY(io.upload());
        PDA_TRY(pda_quadric_cost_batch(io.at<double>(oLM), io.at<double>(oLC), io.at<int64_t>(oLO), io.at<double>(oMM), io.at<double>(oMC),
                                       io.at<int64_t>(oMO), nFrames, nonassign, io.at<double>(oC), io.at<int64_t>(oCO),
                                       io.at<int32_t>(oNL), io.at<int32_t>(oNM), s));
        PDA_TRY(pda_association_perm_probs_batch(io.at<double>(oC), io.at<int64_t>(oCO), io.at<int32_t>(oNL), io.at<int32_t>(oNM),
                                                 io.at<int64_t>(oRO), nFrames, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC,
                                                 io.at<double>(oP), io.at<int64_t>(oPO), io.at<int32_t>(oS), io.at<unsigned char>(oWs),
                                                 wsBytes, s));
        PDA_TRY(io.download());
    }
    if (large.empty()) return PDA_OK;
    // frames with 12+ detections: their cost matrices, then today's route
    std::vector<double> lm, lcov, mm, mcov;
    std::vector<int64_t> lo(1, 0), mo(1, 0);
    for (size_t f : large) {
        lm.insert(lm.end(), landMean + 3 * landOff[f], landMean + 3 * landOff[f + 1]);
        lcov.insert(lcov.end(), landCov + 9 * landOff[f], landCov + 9 * landOff[f + 1]);
        mm.insert(mm.end(), measMean + 3 * measOff[f], measMean + 3 * measOff[f + 1]);
        mcov.insert(mcov.end(), measCov + 9 * measOff[f], measCov + 9 * measOff[f + 1]);
        lo.push_back(lo.back() + landOff[f + 1] - landOff[f]);
        mo.push_back(mo.back() + measOff[f + 1] - measOff[f]);
    }
    std::vector<int32_t> lL(large.size()), lM(large.size());
    std::vector<int64_t> lPO(large.size()), lSt(large.size());
    size_t total = 0;
    for (size_t i = 0; i < large.size(); ++i) {
        lL[i] = (int32_t)(lo[i + 1] - lo[i]); lM[i] = (int32_t)(mo[i + 1] - mo[i]);
        lPO[i] = probOff[large[i]]; lSt[i] = (int64_t)large[i];
        total += (size_t)(lL[i] + lM[i]) * lM[i];
    }
    std::vector<double> flat(total);
    PDA_TRY(pda_quadric_cost_batch_host(lm.empty() ? nullptr : lm.data(), lcov.empty() ? nullptr : lcov.data(), lo.data(), mm.data(),
                                        mcov.data(), mo.data(), (int64_t)large.size(), nonassign, flat.data(), device));
    std::vector<std::vector<double> > lc(large.size());
    size_t o = 0;
    for (size_t i = 0; i < large.size(); ++i) {
        const size_t sz = (size_t)(lL[i] + lM[i]) * lM[i];
        lc[i].assign(flat.begin() + o, flat.begin() + o + sz);
        o += sz;
    }
    return routed_perm_probs(lc, lL, lM, probs, lPO, status, lSt, device);
}

int pda_association_probs_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                           int64_t nProblems, int32_t k, double* probs, const int64_t* probOff,
                                           const int32_t* devices, int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "association (multi): need at least one device");
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff) return fail(PDA_ERR_INVALID, "association: NULL argument");
    return run_slices(costOff, probOff, nProblems, devices, nDevices, "association (multi)",
                      [&](int64_t p0, int64_t p1, int dev, const int64_t* co, const int64_t* po) {
                          return association_probs_host(costs + costOff[p0], co, nL + p0, nM + p0, p1 - p0, k,
                                                        probs + probOff[p0], po, dev, p0);
                      });
}

int pda_association_perm_probs_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL,
                                                const int32_t* nM, int64_t nProblems, double* probs, const int64_t* probOff,
                                                int32_t* status, const int32_t* devices, int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "association_perm (multi): need at least one device");
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association_perm: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status) return fail(PDA_ERR_INVALID, "association_perm: NULL argument");
    return run_slices(costOff, probOff, nProblems, devices, nDevices, "association_perm (multi)",
                      [&](int64_t p0, int64_t p1, int dev, const int64_t* co, const int64_t* po) {
                          return pda_association_perm_probs_batch_host(costs + costOff[p0], co, nL + p0, nM + p0, p1 - p0,
                                                                       probs + probOff[p0], po, status + p0, dev);
                      });
}

}  // extern "C"
