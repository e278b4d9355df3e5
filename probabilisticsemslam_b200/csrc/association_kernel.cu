// association_kernel.cu -- the numeric body of getAssignmentProbs (assignment.cpp:57-74) as one device-side
// pipeline: conditionCosts -> assignmentProb on the conditioned problem -> scatter the conditioned weights back to
// the original landmark indices through rowIdx.  (The reference's first lines, :42-55, turn GTSAM quadrics into the
// cost matrix; that stays with the caller -- see INTEGRATION.md.)  No host round trip between the three stages:
// the k-best kernel reads the conditioned dimensions that the conditioning kernel just wrote.
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <algorithm>

namespace pda {
namespace {

constexpr int WARPS = 4;

// probs[m][rowIdx[l]] = cond[m][l] for l < condL; probs[m][nL] = cond[m][condL]; everything else 0 (:68-74).
// nL == 0 -> {1} per detection (:51-53).  One warp per problem.
__global__ void uncompact_probs_kernel(const double* __restrict__ cond, const int64_t* __restrict__ probOff,
                                       const int32_t* __restrict__ nL, const int32_t* __restrict__ nM,
                                       const int32_t* __restrict__ condNL, const int64_t* __restrict__ rowIdx,
                                       const int64_t* __restrict__ rowOff, int64_t nProblems, double* __restrict__ probs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nProblems) return;
    const int L = nL[p], M = nM[p], cL = condNL[p];
    double* out = probs + probOff[p];
    const double* in = cond + probOff[p];
    if (L == 0) {
        for (int m = lane; m < M; m += 32) out[m] = 1.0;
        return;
    }
    for (int e = lane; e < M * (L + 1); e += 32) out[e] = 0.0;
    __syncwarp();
    const int64_t* idx = rowIdx + rowOff[p];
    for (int e = lane; e < M * (cL + 1); e += 32) {
        const int m = e / (cL + 1), l = e % (cL + 1);
        const int dst = (l < cL) ? (int)idx[l] : L;
        out[(size_t)m * (L + 1) + dst] = in[(size_t)m * (cL + 1) + l];
    }
}

struct AssocWorkspace {
    int32_t* goodRows; int32_t* condNL; int32_t* found;
    double* condCosts; int64_t* rowIdx; double* condProbs;
    unsigned char* murty;  // workspace of pda_murty_batch
    size_t bytes;          // everything up to `murty`
};

AssocWorkspace carve(void* workspace, int64_t nProblems, int64_t totalCostElems, int64_t totalRows, int64_t totalProbElems) {
    const size_t n = (size_t)std::max<int64_t>(nProblems, 1);
    WorkspaceLayout w(workspace);
    AssocWorkspace a;
    a.goodRows = w.take<int32_t>(n);
    a.condNL = w.take<int32_t>(n);
    a.found = w.take<int32_t>(n);
    a.condCosts = w.take<double>((size_t)totalCostElems);
    a.rowIdx = w.take<int64_t>((size_t)totalRows);
    a.condProbs = w.take<double>((size_t)totalProbElems);
    a.murty = w.rest();
    a.bytes = w.bytes();
    return a;
}

}  // namespace

// The k-best _host forms size the Murty kernel once for the whole batch: the largest nL+nM and the largest nM over the
// frames that reach it (nL >= 1; frames with no landmarks are {1} per detection and never see a LAP).  When the kernel
// cannot take that geometry, the call fails with the first frame it cannot take on its own, or, when every frame fits
// alone, with the two largest dimensions that do not fit together.
int check_association_geometry(const int32_t* nL, const int32_t* nM, size_t n, int32_t k, int maxR, int maxC,
                               int64_t frameBase) {
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    MurtyGeometry g;
    const int rc = murty_geometry(k, maxR, maxC, true, dev, &g);
    if (rc != PDA_ERR_UNSUPPORTED) return rc;
    for (size_t p = 0; p < n; ++p) {
        const int L = nL[p], M = nM[p];
        if (L < 1 || M < 1) continue;
        if (murty_geometry(k, L + M, M, true, dev, &g) == PDA_ERR_UNSUPPORTED)
            return fail(PDA_ERR_UNSUPPORTED, "association: frame %lld (nL=%d, nM=%d) is beyond the Murty kernel at k=%d "
                        "(a %d x %d problem with weights)", (long long)(frameBase + (int64_t)p), L, M, k, L + M, M);
    }
    return fail(PDA_ERR_UNSUPPORTED, "association: every frame fits the Murty kernel alone, but the batch's largest nL+nM "
                "(%d) and largest nM (%d) at k=%d do not fit together; split the batch", maxR, maxC, k);
}

}  // namespace pda

using namespace pda;

extern "C" {

int64_t pda_association_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                        int64_t totalProbElems, int32_t k, int32_t maxNumRow, int32_t maxNumCol) {
    const int64_t murty = pda_murty_workspace_bytes(nProblems, k, maxNumRow, maxNumCol);
    if (murty < 0) return murty;
    return (int64_t)carve(nullptr, nProblems, totalCostElems, totalRows, totalProbElems).bytes + murty;
}

int pda_association_probs_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                const int64_t* rowOff, int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                int64_t totalProbElems, int32_t maxNumRow, int32_t maxNumCol, int32_t k,
                                double* probs, const int64_t* probOff, int32_t* nFound,
                                void* workspace, int64_t workspaceBytes, void* stream) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !rowOff || !probs || !probOff || !workspace)
        return fail(PDA_ERR_INVALID, "association: NULL argument");
    // checked before the first launch: the conditioning kernel skips the problems beyond these bounds (the k-best
    // kernel then reports nFound = -1 for them), which keeps its per-column minima inside shared memory
    if (maxNumCol < 1 || maxNumCol > maxNumRow)
        return fail(PDA_ERR_INVALID, "association: need 1 <= maxNumCol <= maxNumRow (got %d x %d)", maxNumRow, maxNumCol);
    if (maxNumRow > PDA_MAX_DIM)
        return fail(PDA_ERR_UNSUPPORTED, "association: maxNumRow %d exceeds PDA_MAX_DIM %d", maxNumRow, PDA_MAX_DIM);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const AssocWorkspace w = carve(workspace, nProblems, totalCostElems, totalRows, totalProbElems);
    if ((int64_t)w.bytes > workspaceBytes) return fail(PDA_ERR_WORKSPACE, "association: workspace too small");
    // (numRow = nL + nM and condL = goodRows - nM are formed inside the conditioning kernel: two launches fewer)
    PDA_TRY(launch_condition_costs(costs, costOff, nullptr, nM, nProblems, rowOff, w.condCosts, w.rowIdx, w.goodRows, s, nL,
                                   w.condNL, maxNumRow, maxNumCol));
    // conditioned problems live at the original cost offsets (they only shrink) and use the original probability offsets
    PDA_TRY(pda_murty_batch(w.condCosts, costOff, w.goodRows, nM, nProblems, maxNumRow, maxNumCol, k, PDA_CUT_RELATIVE, 42.0, 0, 0,
                            nullptr, nullptr, nullptr, nullptr, nullptr, nFound ? nFound : w.found, PDA_WEIGHTS_GATED, w.condProbs,
                            probOff, w.condNL, w.murty, workspaceBytes - (int64_t)w.bytes, stream));
    uncompact_probs_kernel<<<(unsigned)((nProblems + WARPS - 1) / WARPS), 32 * WARPS, 0, s>>>(
        w.condProbs, probOff, nL, nM, w.condNL, w.rowIdx, rowOff, nProblems, probs);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int pda_association_probs_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                     int64_t nProblems, int32_t k, double* probs, const int64_t* probOff,
                                     int32_t device) {
    return association_probs_host(costs, costOff, nL, nM, nProblems, k, probs, probOff, device, 0);
}

}  // extern "C"

// pda_association_probs_batch_host on a slice of a caller's batch that starts at frame frameBase (the _multi form):
// errors name frames by their index in the caller's batch
int pda::association_probs_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                int64_t nProblems, int32_t k, double* probs, const int64_t* probOff, int32_t device,
                                int64_t frameBase) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "association: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff) return fail(PDA_ERR_INVALID, "association: NULL argument");
    if (k < 1) return fail(PDA_ERR_INVALID, "association: k < 1");
    const size_t n = (size_t)nProblems;
    std::vector<int64_t> rowOff(n);
    size_t nCost = 0, nRows = 0, nProb = 0;
    int maxR = 1, maxC = 1;
    for (size_t p = 0; p < n; ++p) {
        const int L = nL[p], M = nM[p];
        if (L < 0 || M < 1) return fail(PDA_ERR_INVALID, "association: problem %lld has nL=%d nM=%d", (long long)p, L, M);
        rowOff[p] = (int64_t)nRows;
        nRows += (size_t)(L + M);
        nCost = std::max(nCost, (size_t)costOff[p] + (size_t)(L + M) * M);
        nProb = std::max(nProb, (size_t)probOff[p] + (size_t)M * (L + 1));
        if (L > 0) { maxR = std::max(maxR, L + M); maxC = std::max(maxC, M); }
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    PDA_TRY(check_association_geometry(nL, nM, n, k, maxR, maxC, frameBase));
    const int64_t wsBytes = pda_association_workspace_bytes(nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, k, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    HostIO io(device);
    const size_t oC = io.in(costs, nCost * 8), oCO = io.in(costOff, n * 8), oL = io.in(nL, n * 4), oM = io.in(nM, n * 4);
    const size_t oRO = io.in(rowOff.data(), n * 8), oPO = io.in(probOff, n * 8);
    const size_t oP = io.out(probs, nProb * 8), oWs = io.scratch((size_t)wsBytes);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    PDA_TRY(pda_association_probs_batch(io.at<double>(oC), io.at<int64_t>(oCO), io.at<int32_t>(oL), io.at<int32_t>(oM),
                                        io.at<int64_t>(oRO), nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC, k,
                                        io.at<double>(oP), io.at<int64_t>(oPO), nullptr, io.at<unsigned char>(oWs), wsBytes,
                                        io.stream()));
    return io.download();
}
