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

size_t align256(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

int64_t pda_association_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalRows,
                                        int64_t totalProbElems, int32_t k, int32_t maxNumRow, int32_t maxNumCol) {
    const int64_t murty = pda_murty_workspace_bytes(nProblems, k, maxNumRow, maxNumCol);
    if (murty < 0) return murty;
    const size_t n = (size_t)std::max<int64_t>(nProblems, 1);
    return (int64_t)(4 * align256(n * 4) + align256((size_t)totalCostElems * 8) + align256((size_t)totalRows * 8) +
                     align256((size_t)totalProbElems * 8) + 256) + murty;
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
    const size_t n = (size_t)nProblems;
    unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
    size_t o = 0;
    int32_t* numRow = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    int32_t* goodRows = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    int32_t* condNL = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    int32_t* found = reinterpret_cast<int32_t*>(w + o); o += align256(n * 4);
    double* condCosts = reinterpret_cast<double*>(w + o); o += align256((size_t)totalCostElems * 8);
    int64_t* rowIdx = reinterpret_cast<int64_t*>(w + o); o += align256((size_t)totalRows * 8);
    double* condProbs = reinterpret_cast<double*>(w + o); o += align256((size_t)totalProbElems * 8);
    if ((int64_t)o + 256 > workspaceBytes) return fail(PDA_ERR_WORKSPACE, "association: workspace too small");
    // (numRow = nL + nM and condL = goodRows - nM are formed inside the conditioning kernel: two launches fewer)
    (void)numRow;
    PDA_TRY(launch_condition_costs(costs, costOff, nullptr, nM, nProblems, rowOff, condCosts, rowIdx, goodRows, s, nL, condNL,
                                   maxNumRow, maxNumCol));
    // conditioned problems live at the original cost offsets (they only shrink) and use the original probability offsets
    PDA_TRY(pda_murty_batch(condCosts, costOff, goodRows, nM, nProblems, maxNumRow, maxNumCol, k, PDA_CUT_RELATIVE, 42.0, 0, 0,
                            nullptr, nullptr, nullptr, nullptr, nullptr, nFound ? nFound : found, PDA_WEIGHTS_GATED, condProbs,
                            probOff, condNL, w + o, workspaceBytes - (int64_t)o, stream));
    uncompact_probs_kernel<<<(unsigned)((n + WARPS - 1) / WARPS), 32 * WARPS, 0, s>>>(condProbs, probOff, nL, nM, condNL, rowIdx,
                                                                                   rowOff, nProblems, probs);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int pda_association_probs_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                                     int64_t nProblems, int32_t k, double* probs, const int64_t* probOff,
                                     int32_t device) {
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
        maxR = std::max(maxR, L + M); maxC = std::max(maxC, M);
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const int64_t wsBytes = pda_association_workspace_bytes(nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, k, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    if (8 * (nCost + nProb + 3 * n) + 8 * n <= PDA_PACKED_LIMIT) {  // small call (the per-frame SLAM shape): one pinned copy each way
        Stage st(device);
        PackedIO io(st);
        const size_t oC = io.in(costs, nCost * 8), oCO = io.in(costOff, n * 8), oL = io.in(nL, n * 4), oM = io.in(nM, n * 4);
        const size_t oRO = io.in(rowOff.data(), n * 8), oPO = io.in(probOff, n * 8);
        const size_t oP = io.out(probs, nProb * 8), oWs = st.reserve((size_t)wsBytes);
        PDA_TRY(st.commit());
        HostStreams* hs = nullptr;
        PDA_TRY(host_streams(device, &hs));
        PDA_TRY(io.upload(hs->run));
        PDA_TRY(pda_association_probs_batch(st.at<double>(oC), st.at<int64_t>(oCO), st.at<int32_t>(oL), st.at<int32_t>(oM),
                                            st.at<int64_t>(oRO), nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC, k,
                                            st.at<double>(oP), st.at<int64_t>(oPO), nullptr, st.at<unsigned char>(oWs), wsBytes, hs->run));
        return io.download(hs->run);
    }
    Stage st(device);
    const size_t oC = st.reserve(nCost * 8), oCO = st.reserve(n * 8), oL = st.reserve(n * 4), oM = st.reserve(n * 4);
    const size_t oRO = st.reserve(n * 8), oP = st.reserve(nProb * 8), oPO = st.reserve(n * 8), oWs = st.reserve((size_t)wsBytes);
    PDA_TRY(st.commit());
    cudaStream_t s = 0;
    PDA_TRY(h2d(st.at<double>(oC), costs, nCost, s));
    PDA_TRY(h2d(st.at<int64_t>(oCO), costOff, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oL), nL, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oM), nM, n, s));
    PDA_TRY(h2d(st.at<int64_t>(oRO), rowOff.data(), n, s));
    PDA_TRY(h2d(st.at<int64_t>(oPO), probOff, n, s));
    PDA_TRY(pda_association_probs_batch(st.at<double>(oC), st.at<int64_t>(oCO), st.at<int32_t>(oL), st.at<int32_t>(oM),
                                        st.at<int64_t>(oRO), nProblems, (int64_t)nCost, (int64_t)nRows, (int64_t)nProb, maxR, maxC, k,
                                        st.at<double>(oP), st.at<int64_t>(oPO), nullptr, st.at<unsigned char>(oWs), wsBytes, s));
    PDA_TRY(d2h(probs, st.at<double>(oP), nProb, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    return PDA_OK;
}

}  // extern "C"
