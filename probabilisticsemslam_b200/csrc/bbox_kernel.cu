// bbox_kernel.cu -- stereo bounding-box association (SURVEY.md 8f rank 4): the second caller of the LAP solver.
//   boundBox::IoU        boundBox.h:62-75
//   computeBBCostMatrix  assignment.cpp:777-797   (nR+nL) x nL scores: -inf background, min of the two IoUs
//                                                 (the x offset shifts only the box IoU is called on), dummy diagonal
//   asgnBB               assignment.cpp:724-775   kBest2D(k = 1, maximize = true); dummy pairing -> -1
// Pipeline on one stream: bb_costs_kernel (one warp per frame) -> murty_kernel (k = 1, maximise) -> bb_finish_kernel.
// A box is five doubles: xmin, ymin, xmax, ymax, xOffset.
// The device-pointer form pda_asgn_bb_batch reads the frame shapes on the device (bb_shapes_kernel) instead of on the
// host, so a CUDA graph captured once with fixed bounds serves frames of any shape (DESIGN.md 3.6b).
#include "pda_internal.h"
#include "pda_host_stage.h"
#include "cta_scan.cuh"

#include <math_constants.h>

#include <algorithm>
#include <climits>
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

// nLeft[p] left boxes of problem p get their partner or -1: numCol[p] of them, or all of a frame that went to the
// solver as 0 x 0 because it has no right box (the solver then reports nFound -1)
__global__ void bb_finish_kernel(const int64_t* __restrict__ row4col, const int64_t* __restrict__ r4cOff,
                                 const int32_t* __restrict__ nFound, const int32_t* __restrict__ numRow,
                                 const int32_t* __restrict__ numCol, const int32_t* __restrict__ nLeft,
                                 const int64_t* __restrict__ firstL, const int64_t nProblems, int32_t* __restrict__ assignment) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * WARPS + warp;
    if (p >= nProblems) return;
    const int nL = nLeft[p], nR = numRow[p] - numCol[p];
    for (int c = lane; c < nL; c += 32) {
        int a = -1;
        if (nFound[p] > 0) {
            const int64_t r = row4col[r4cOff[p] + c];
            if (r < nR) a = (int)r;  // assignment.cpp:769-773
        }
        assignment[firstL[p] + c] = a;
    }
}

// ---- device-pointer form: frame shapes are read on the device, never on the host ----
struct BBShapes {
    int32_t* numRow; int32_t* numCol;  // nL + nR and nL; 0 x 0 for a frame with an empty side or a rejected one
    int32_t* nLeft;                    // left boxes the finish step writes: nL of a computed frame, else 0
    int32_t* nFound;
    int64_t* firstL; int64_t* firstR;
    int64_t* costOff; int64_t* r4cOff;  // fixed strides: f * maxBoxes * maxNL and f * maxNL
    double* costs;
    int64_t* r4c;
    unsigned char* murty;              // workspace of pda_murty_batch
    size_t bytes;                      // everything up to `murty`
};

BBShapes carve_bb(void* workspace, int64_t nFrames, int32_t maxNL, int32_t maxBoxes) {
    const size_t n = (size_t)std::max<int64_t>(nFrames, 1);
    WorkspaceLayout w(workspace);
    BBShapes s;
    s.numRow = w.take<int32_t>(n);
    s.numCol = w.take<int32_t>(n);
    s.nLeft = w.take<int32_t>(n);
    s.nFound = w.take<int32_t>(n);
    s.firstL = w.take<int64_t>(n);
    s.firstR = w.take<int64_t>(n);
    s.costOff = w.take<int64_t>(n);
    s.r4cOff = w.take<int64_t>(n);
    s.costs = w.take<double>(n * (size_t)maxBoxes * (size_t)maxNL);
    s.r4c = w.take<int64_t>(n * (size_t)maxNL);
    s.murty = w.rest();
    s.bytes = w.bytes();
    return s;
}

// One CTA walks the frames in blocks of CTA_SCAN_THREADS.  Results are addressed by offL directly, so a frame is computed
// only if no other computed frame can write its left entries: offL[f] must be the largest of offL[0..f] (a running
// maximum carried across blocks) and its own ranges must ascend.  Then every earlier frame ends at some offL[g+1] <=
// offL[f] and every later computed frame starts at or after offL[f+1].  Both ranges must also lie within capL / capR,
// and nL <= maxNL, nL + nR <= maxBoxes.  Right boxes are only read, so they need the bounds checks alone.  Frames with
// an empty side go on as 0 x 0 (the solver reports nFound -1 and touches nothing), with their nL left boxes still
// written -1 by the finish step when computed; status 2 frames write nothing.
__global__ void __launch_bounds__(CTA_SCAN_THREADS) bb_shapes_kernel(
    const int64_t* __restrict__ offL, const int64_t capL, const int64_t* __restrict__ offR, const int64_t capR,
    const long long nFrames, const int32_t maxNL, const int32_t maxBoxes, const BBShapes s, int32_t* __restrict__ status) {
    __shared__ long long warpMax[32];
    long long carry = LLONG_MIN;
    for (long long base = 0; base < nFrames; base += CTA_SCAN_THREADS) {
        const long long f = base + threadIdx.x;
        const long long l0 = f < nFrames ? offL[f] : LLONG_MIN;
        const long long runMax = cta_scan(l0, carry, warpMax, ScanMax());
        if (f < nFrames) {
            const long long l1 = offL[f + 1], r0 = offR[f], r1 = offR[f + 1];
            const bool ok = l0 == runMax && l0 >= 0 && l1 >= l0 && l1 <= capL && r0 >= 0 && r1 >= r0 && r1 <= capR &&
                            l1 - l0 <= maxNL && (l1 - l0) + (r1 - r0) <= maxBoxes;
            const int nL = ok ? (int)(l1 - l0) : 0, nR = ok ? (int)(r1 - r0) : 0;
            const bool solve = nL > 0 && nR > 0;
            s.numRow[f] = solve ? nL + nR : 0; s.numCol[f] = solve ? nL : 0;
            s.nLeft[f] = nL;
            s.firstL[f] = ok ? l0 : 0; s.firstR[f] = ok ? r0 : 0;
            s.costOff[f] = f * maxBoxes * maxNL; s.r4cOff[f] = f * maxNL;
            status[f] = ok ? 0 : 2;
        }
    }
}

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

// Frame f owns [offL[f], offL[f+1]) of boxesL / assignment and [offR[f], offR[f+1]) of boxesR: only [offL[0], offL[n])
// and [offR[0], offR[n]) are read, staged and written back, so a call on a slice of a larger batch (a shard of
// pda_asgn_bb_batch_host_multi) leaves the other frames' entries alone.
int pda_asgn_bb_batch_host(const double* boxesL, const int64_t* offL, const double* boxesR, const int64_t* offR,
                           int64_t nFrames, double nonassign, int32_t* assignment, int32_t device) {
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "asgn_bb: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!offL || !offR || !assignment) return fail(PDA_ERR_INVALID, "asgn_bb: NULL argument");
    if (offL[0] < 0 || offR[0] < 0) return fail(PDA_ERR_INVALID, "asgn_bb: negative offset");
    const int64_t baseL = offL[0], baseR = offR[0];
    std::vector<int64_t> firstL, firstR, costOff, r4cOff;
    std::vector<int32_t> numRow, numCol;
    size_t nCost = 0, nR4c = 0;
    int maxR = 1, maxC = 1;
    for (int64_t f = 0; f < nFrames; ++f) {
        const int64_t nL = offL[f + 1] - offL[f], nR = offR[f + 1] - offR[f];
        if (nL < 0 || nR < 0) return fail(PDA_ERR_INVALID, "asgn_bb: offsets must be non-decreasing");
        if (nL == 0 || nR == 0) continue;
        if (nL + nR > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "asgn_bb: frame %lld has %lld boxes (limit %d)", (long long)f, (long long)(nL + nR), PDA_MAX_DIM);
        firstL.push_back(offL[f] - baseL); firstR.push_back(offR[f] - baseR);
        numRow.push_back((int32_t)(nL + nR)); numCol.push_back((int32_t)nL);
        costOff.push_back((int64_t)nCost); r4cOff.push_back((int64_t)nR4c);
        nCost += (size_t)((nL + nR) * nL); nR4c += (size_t)nL;
        maxR = std::max<int>(maxR, (int)(nL + nR)); maxC = std::max<int>(maxC, (int)nL);
    }
    const int64_t totalL = offL[nFrames] - baseL, totalR = offR[nFrames] - baseR;
    int32_t* const asg = assignment + baseL;
    for (int64_t i = 0; i < totalL; ++i) asg[i] = -1;  // frames with an empty side: every left box unmatched (:730-732)
    const size_t n = numRow.size();
    if (n == 0) return PDA_OK;
    if (!boxesL || !boxesR) return fail(PDA_ERR_INVALID, "asgn_bb: NULL boxes");
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const int64_t wsBytes = pda_murty_workspace_bytes((int64_t)n, 1, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    HostIO io(device);
    const size_t oBL = io.in(boxesL + 5 * baseL, (size_t)totalL * 40), oBR = io.in(boxesR + 5 * baseR, (size_t)totalR * 40);
    const size_t oFL = io.in(firstL.data(), n * 8), oFR = io.in(firstR.data(), n * 8), oNR = io.in(numRow.data(), n * 4);
    const size_t oNC = io.in(numCol.data(), n * 4), oCO = io.in(costOff.data(), n * 8), oRO = io.in(r4cOff.data(), n * 8);
    const size_t oAsg = io.inout(asg, (size_t)totalL * 4);
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
                                                   io.at<int32_t>(oNC), io.at<int32_t>(oNC), io.at<int64_t>(oFL), (int64_t)n,
                                                   io.at<int32_t>(oAsg));
    PDA_CUDA_TRY(cudaGetLastError());
    return io.download();
}

int64_t pda_asgn_bb_workspace_bytes(int64_t nFrames, int32_t maxNL, int32_t maxBoxes) {
    if (nFrames < 0 || maxNL < 1 || maxBoxes < maxNL)
        return fail(PDA_ERR_INVALID, "asgn_bb: nFrames %lld, maxNL %d, maxBoxes %d", (long long)nFrames, maxNL, maxBoxes);
    if (maxBoxes > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "asgn_bb: maxBoxes %d above %d", maxBoxes, PDA_MAX_DIM);
    const int64_t murty = pda_murty_workspace_bytes(std::max<int64_t>(nFrames, 1), 1, maxBoxes, maxNL);
    if (murty < 0) return murty;
    return (int64_t)carve_bb(nullptr, nFrames, maxNL, maxBoxes).bytes + murty;
}

int pda_asgn_bb_batch(const double* boxesL, const int64_t* offL, int64_t capL, const double* boxesR, const int64_t* offR,
                      int64_t capR, int64_t nFrames, int32_t maxNL, int32_t maxBoxes, double nonassign, int32_t* assignment,
                      int32_t* status, void* workspace, int64_t workspaceBytes, void* stream) {
    if (!offL || !offR || !assignment || !status || !workspace || (capL > 0 && !boxesL) || (capR > 0 && !boxesR))
        return fail(PDA_ERR_INVALID, "asgn_bb: NULL argument");
    if (capL < 0 || capR < 0) return fail(PDA_ERR_INVALID, "asgn_bb: negative capacity");
    const int64_t wsBytes = pda_asgn_bb_workspace_bytes(nFrames, maxNL, maxBoxes);
    if (wsBytes < 0) return (int)wsBytes;
    PDA_TRY(check_workspace("asgn_bb", workspaceBytes, wsBytes));
    if (nFrames == 0) return PDA_OK;
    const cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const BBShapes sh = carve_bb(workspace, nFrames, maxNL, maxBoxes);
    bb_shapes_kernel<<<1, CTA_SCAN_THREADS, 0, s>>>(offL, capL, offR, capR, nFrames, maxNL, maxBoxes, sh, status);
    PDA_CUDA_TRY(cudaGetLastError());
    const unsigned blocks = (unsigned)((nFrames + WARPS - 1) / WARPS);
    bb_costs_kernel<<<blocks, 32 * WARPS, 0, s>>>(boxesL, boxesR, sh.firstL, sh.firstR, sh.numRow, sh.numCol, sh.costOff, nFrames,
                                                  nonassign, sh.costs);
    PDA_CUDA_TRY(cudaGetLastError());
    PDA_TRY(pda_murty_batch(sh.costs, sh.costOff, sh.numRow, sh.numCol, nFrames, maxBoxes, maxNL, 1, PDA_CUT_NONE, 0.0,
                            1 /* maximize */, 0, sh.r4c, sh.r4cOff, nullptr, nullptr, nullptr, sh.nFound, PDA_WEIGHTS_NONE, nullptr,
                            nullptr, nullptr, sh.murty, workspaceBytes - (int64_t)sh.bytes, stream));
    bb_finish_kernel<<<blocks, 32 * WARPS, 0, s>>>(sh.r4c, sh.r4cOff, sh.nFound, sh.numRow, sh.numCol, sh.nLeft, sh.firstL, nFrames,
                                                   assignment);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

// contiguous slices of frames, one per device, each a pda_asgn_bb_batch_host call on the whole arrays and its own
// offsets: the slices' ranges of boxesL / assignment do not overlap
int pda_asgn_bb_batch_host_multi(const double* boxesL, const int64_t* offL, const double* boxesR, const int64_t* offR,
                                 int64_t nFrames, double nonassign, int32_t* assignment, const int32_t* devices,
                                 int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "asgn_bb (multi): need at least one device");
    if (nFrames < 0) return fail(PDA_ERR_INVALID, "asgn_bb: nFrames < 0");
    if (nFrames == 0) return PDA_OK;
    if (!offL || !offR || !assignment) return fail(PDA_ERR_INVALID, "asgn_bb: NULL argument");
    return run_sharded(nFrames, devices, nDevices, [&](int64_t p0, int64_t p1, int dev) {
        return pda_asgn_bb_batch_host(boxesL, offL + p0, boxesR, offR + p0, p1 - p0, nonassign, assignment, dev);
    });
}

}  // extern "C"
