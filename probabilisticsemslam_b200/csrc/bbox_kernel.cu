// bbox_kernel.cu -- stereo bounding-box association (SURVEY.md 8f rank 4): the second caller of the LAP solver.
//   boundBox::IoU        boundBox.h:62-75
//   computeBBCostMatrix  assignment.cpp:777-797   (nR+nL) x nL scores: -inf background, min of the two IoUs
//                                                 (the x offset shifts only the box IoU is called on), dummy diagonal
//   asgnBB               assignment.cpp:724-775   kBest2D(k = 1, maximize = true); dummy pairing -> -1
// Pipeline on one stream: bb_costs_kernel (one warp per frame) -> murty_kernel (k = 1, maximise) -> bb_finish_kernel.
// A box is five doubles: xmin, ymin, xmax, ymax, xOffset.
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <math_constants.h>

#include <algorithm>
#include <vector>

namespace pda {
namespace {

constexpr int WARPS = 4;

__device__ __forceinline__ double box_area(const double* b) { return (b[2] - b[0]) * (b[3] - b[1]); }

__device__ __forceinline__ double box_iou(const double* self, const double* other) {
    const double l = fmax(self[0] + self[4], other[0]);
    const double r = fmin(self[2] + self[4], other[2]);
    const double t = fmax(self[1], other[1]);
    const double b = fmin(self[3], other[3]);
    if (l >= r || t >= b) return 0.0;
    const double inter = (r - l) * (b - t);
    return inter / (box_area(self) + box_area(other) - inter);
}

// problems here are the frames that have boxes on both sides; frameL/frameR give their first box
__global__ void bb_costs_kernel(const double* __restrict__ boxesL, const double* __restrict__ boxesR,
                                const int64_t* __restrict__ firstL, const int64_t* __restrict__ firstR,
                                const int32_t* __restrict__ numRow, const int32_t* __restrict__ numCol,
                                const int64_t* __restrict__ costOff, const int64_t nProblems, const double nonassign,
                                double* __restrict__ costs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nProblems) return;
    const int nL = numCol[p], nRows = numRow[p], nR = nRows - nL;
    const double* L = boxesL + 5 * firstL[p];
    const double* R = boxesR + 5 * firstR[p];
    double* C = costs + costOff[p];
    for (int e = lane; e < nRows * nL; e += 32) {
        const int c = e / nRows, r = e % nRows;
        double val = -CUDART_INF;
        if (r < nR) {
            const double i1 = box_iou(R + 5 * r, L + 5 * c), i2 = box_iou(L + 5 * c, R + 5 * r);
            val = (i2 < i1) ? i2 : i1;
        } else if (r == nR + c) {
            val = nonassign;
        }
        C[e] = val;
    }
}

__global__ void bb_finish_kernel(const int64_t* __restrict__ row4col, const int64_t* __restrict__ r4cOff,
                                 const int32_t* __restrict__ nFound, const int32_t* __restrict__ numRow,
                                 const int32_t* __restrict__ numCol, const int64_t* __restrict__ firstL,
                                 const int64_t nProblems, int32_t* __restrict__ assignment) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nProblems) return;
    const int nL = numCol[p], nR = numRow[p] - nL;
    for (int c = lane; c < nL; c += 32) {
        int a = -1;
        if (nFound[p] > 0) {
            const int64_t r = row4col[r4cOff[p] + c];
            if (r < nR) a = (int)r;  // assignment.cpp:769-773
        }
        assignment[firstL[p] + c] = a;
    }
}

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" int pda_asgn_bb_batch_host(const double* boxesL, const int64_t* offL, const double* boxesR, const int64_t* offR,
                                      int64_t nFrames, double nonassign, int32_t* assignment, int32_t device) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "asgn_bb: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!offL || !offR || !assignment) return fail(PDA_ERR_INVALID, "asgn_bb: NULL argument");
    const int64_t totalL = offL[nFrames], totalR = offR[nFrames];
    for (int64_t i = 0; i < totalL; ++i) assignment[i] = -1;  // frames with an empty side: every left box unmatched (:730-732)
    std::vector<int64_t> firstL, firstR, costOff, r4cOff;
    std::vector<int32_t> numRow, numCol;
    size_t nCost = 0, nR4c = 0;
    int maxR = 1, maxC = 1;
    for (int64_t f = 0; f < nFrames; ++f) {
        const int64_t nL = offL[f + 1] - offL[f], nR = offR[f + 1] - offR[f];
        if (nL < 0 || nR < 0) return fail(PDA_ERR_INVALID, "asgn_bb: offsets must be non-decreasing");
        if (nL == 0 || nR == 0) continue;
        if (nL + nR > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "asgn_bb: frame %lld has %lld boxes (limit %d)", (long long)f, (long long)(nL + nR), PDA_MAX_DIM);
        firstL.push_back(offL[f]); firstR.push_back(offR[f]);
        numRow.push_back((int32_t)(nL + nR)); numCol.push_back((int32_t)nL);
        costOff.push_back((int64_t)nCost); r4cOff.push_back((int64_t)nR4c);
        nCost += (size_t)((nL + nR) * nL); nR4c += (size_t)nL;
        maxR = std::max<int>(maxR, (int)(nL + nR)); maxC = std::max<int>(maxC, (int)nL);
    }
    const size_t n = numRow.size();
    if (n == 0) return PDA_OK;
    if (!boxesL || !boxesR) return fail(PDA_ERR_INVALID, "asgn_bb: NULL boxes");
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const int64_t wsBytes = pda_murty_workspace_bytes((int64_t)n, 1, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    HostIO io(device);
    const size_t oBL = io.in(boxesL, (size_t)totalL * 40), oBR = io.in(boxesR, (size_t)totalR * 40);
    const size_t oFL = io.in(firstL.data(), n * 8), oFR = io.in(firstR.data(), n * 8), oNR = io.in(numRow.data(), n * 4);
    const size_t oNC = io.in(numCol.data(), n * 4), oCO = io.in(costOff.data(), n * 8), oRO = io.in(r4cOff.data(), n * 8);
    const size_t oAsg = io.inout(assignment, (size_t)totalL * 4);
    const size_t oC = io.scratch(nCost * 8), oR4c = io.scratch(nR4c * 8), oFound = io.scratch(n * 4), oWs = io.scratch((size_t)wsBytes);
    PDA_TRY(io.commit());
    const cudaStream_t s = io.stream();
    PDA_TRY(io.upload());
    const unsigned blocks = (unsigned)((n + WARPS - 1) / WARPS);
    bb_costs_kernel<<<blocks, 32 * WARPS, 0, s>>>(io.at<double>(oBL), io.at<double>(oBR), io.at<int64_t>(oFL), io.at<int64_t>(oFR),
                                                  io.at<int32_t>(oNR), io.at<int32_t>(oNC), io.at<int64_t>(oCO), (int64_t)n, nonassign,
                                                  io.at<double>(oC));
    PDA_CUDA_TRY(cudaGetLastError());
    PDA_TRY(pda_murty_batch(io.at<double>(oC), io.at<int64_t>(oCO), io.at<int32_t>(oNR), io.at<int32_t>(oNC), (int64_t)n, maxR, maxC,
                            1, PDA_CUT_NONE, 0.0, 1 /* maximize */, 0, io.at<int64_t>(oR4c), io.at<int64_t>(oRO), nullptr, nullptr,
                            nullptr, io.at<int32_t>(oFound), PDA_WEIGHTS_NONE, nullptr, nullptr, nullptr,
                            io.at<unsigned char>(oWs), wsBytes, s));
    bb_finish_kernel<<<blocks, 32 * WARPS, 0, s>>>(io.at<int64_t>(oR4c), io.at<int64_t>(oRO), io.at<int32_t>(oFound), io.at<int32_t>(oNR),
                                                   io.at<int32_t>(oNC), io.at<int64_t>(oFL), (int64_t)n, io.at<int32_t>(oAsg));
    PDA_CUDA_TRY(cudaGetLastError());
    return io.download();
}
