// permprob_kernel.cu -- permanent-based association weights on the device.
//
//   permanentProb        assignment.cpp:145-290   (+ setupAssgnMatrix :292-323)
//   conditionedPermanent assignment.cpp:325-435
//
// The reference computes, for every detection m and every landmark l (plus the
// non-assignment row), P(l,m) * perm(P without row l and column m) one after the other,
// each time conditioning the sub-matrix (drop all-zero rows/columns, scale columns by
// 1/sqrt(max * smallest non-zero), transpose, pad with ones).  All (nL+1)*nM sub-permanents
// of a problem are independent, so here they become ITEMS of one batch:
//   1. to_probs            element-wise likelihoods of every problem (weights_kernel.cu)
//   2. build_items_kernel  one warp per item: gathers its sub-matrix straight out of P
//                          through row/column maps, conditions it, writes the scaled,
//                          transposed matrix + its scale factor
//   3. perm_kernel         the batched NW permanent over all items (permanent_kernel.cu)
//   4. finish_probs_kernel one warp per problem: |P(l,m) * perm / scale|, column sums in
//                          the reference's order, normalise by the largest column sum
// Items whose permanent comes out negative are rebuilt untransposed and recomputed, as the
// reference does (:409-419).
#include "pda_internal.h"
#include "pda_host_stage.h"
#include "perm_device.cuh"

#include <algorithm>
#include <vector>

namespace pda {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int BUILD_WARPS = 4;
constexpr int SLOT = PDA_MAX_PERM_DIM * PDA_MAX_PERM_DIM;  // doubles per item matrix

struct BuildArgs {
    // mode 0: items are (problem, m, l) triples of permanentProb; mode 1: items are plain matrices
    int mode;
    const double* P; const int64_t* pOff; const int32_t* nL; const int32_t* nM;  // mode 0 (P = likelihoods)
    const int64_t* itemOff;                                                      // mode 0: first item of problem
    const int32_t* itemProblem;                                                  // mode 0: problem of each item
    const int32_t* rows; const int32_t* cols;                                    // mode 1
    const int32_t* subset;      // optional: only these item indices (retry pass), else NULL
    int64_t nWork;              // number of items to build in this launch
    int transpose;              // 1 = write the transposed matrix (first attempt), 0 = untransposed (retry)
    double* mats;               // [item * SLOT]
    int32_t* outRows; int32_t* outCols; double* scale; int32_t* itemStatus;
};

__global__ void build_items_kernel(const BuildArgs a) {
    __shared__ double sScale[BUILD_WARPS][PDA_MAX_DIM];
    __shared__ short sKeepC[BUILD_WARPS][PDA_MAX_DIM];
    __shared__ short sKeepR[BUILD_WARPS][PDA_MAX_DIM];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t w = (int64_t)blockIdx.x * BUILD_WARPS + warp;
    if (w >= a.nWork) return;
    const int64_t item = a.subset ? a.subset[w] : w;
    Gather g;
    bool active = true;
    if (a.mode == 0) {
        const int p = a.itemProblem[item];
        const int nL = a.nL[p], nM = a.nM[p];
        const int64_t local = item - a.itemOff[p];
        active = item_gather(a.P + a.pOff[p], nL, nM, (int)(local / (nL + 1)), (int)(local % (nL + 1)), g);
        if (nM < 2) active = false;
    } else {
        g.base = a.P + a.pOff[item]; g.ld = a.rows[item]; g.sR = a.rows[item]; g.sC = a.cols[item];
        g.skipRow = -1; g.skipCol = -1; g.patchRow = -1; g.patchVal = 0.0;
    }
    double* M = a.mats + (size_t)item * SLOT;
    if (!active || g.sR > PDA_MAX_DIM || g.sC > PDA_MAX_DIM) {
        if (lane == 0) {
            a.outRows[item] = 0; a.outCols[item] = 0; a.scale[item] = 1.0;
            a.itemStatus[item] = active ? 1 : 0;
        }
        return;
    }
    int nKR, nKC;
    condition_warp(g, sScale[warp], sKeepC[warp], sKeepR[warp], lane, nKR, nKC);
    const int n = nKR > nKC ? nKR : nKC;
    if (n > PDA_MAX_PERM_DIM) {  // permanentExactSquare throws (nwPerm.cpp:327-330)
        if (lane == 0) { a.outRows[item] = 0; a.outCols[item] = 0; a.scale[item] = 1.0; a.itemStatus[item] = 1; }
        return;
    }
    write_scaled(g, sScale[warp], sKeepC[warp], sKeepR[warp], nKR, nKC, a.transpose, M, lane);
    if (lane == 0) {
        a.scale[item] = scale_product(sScale[warp], nKC);
        a.outRows[item] = a.transpose ? nKC : nKR;
        a.outCols[item] = a.transpose ? nKR : nKC;
        a.itemStatus[item] = 0;
    }
}

// result = permanent / scaleFactor (:402); collects the items that came out negative
__global__ void unscale_kernel(double* __restrict__ perm, const double* __restrict__ scale, const int32_t* __restrict__ subset,
                               int64_t nWork, int32_t* __restrict__ negList, int32_t* __restrict__ negCount) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nWork) return;
    const int64_t item = subset ? subset[w] : w;
    const double r = perm[item] / scale[item];
    perm[item] = r;
    if (negList && r < 0.0) negList[atomicAdd(negCount, 1)] = (int32_t)item;
}

__global__ void single_column_kernel(const double* __restrict__ P, const int64_t* __restrict__ pOff,
                                     const int32_t* __restrict__ nL, const int32_t* __restrict__ nM, int64_t nProblems,
                                     double* __restrict__ probs, const int64_t* __restrict__ probOff) {
    // permanentProb with one detection (:166-171): normalise by std::reduce, which sums in blocks of four
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nProblems || nM[p] != 1) return;
    const double* v = P + pOff[p];
    const int n = nL[p] + 1;
    double acc = 0.0;
    int i = 0;
    for (; n - i >= 4; i += 4) acc = acc + ((v[i] + v[i + 1]) + (v[i + 2] + v[i + 3]));
    for (; i < n; ++i) acc = acc + v[i];
    const double norm = 1.0 / acc;
    double* out = probs + probOff[p];
    for (i = 0; i < n; ++i) out[i] = v[i] * norm;
}

__global__ void finish_probs_kernel(const double* __restrict__ P, const int64_t* __restrict__ pOff,
                                    const int32_t* __restrict__ nL, const int32_t* __restrict__ nM,
                                    const int64_t* __restrict__ itemOff, const double* __restrict__ perm,
                                    const int32_t* __restrict__ itemStatus, int64_t nProblems,
                                    double* __restrict__ probs, const int64_t* __restrict__ probOff,
                                    int32_t* __restrict__ status) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * BUILD_WARPS + warp;
    if (p >= nProblems) return;
    const int L = nL[p], M = nM[p], nR = L + M;
    if (M < 2) { if (lane == 0) status[p] = 0; return; }
    const double* Pp = P + pOff[p];
    double* out = probs + probOff[p];
    const int64_t it0 = itemOff[p];
    double best = 0.0;
    int bad = 0;
    for (int m = lane; m < M; m += 32) {
        double colPerm = 0.0;
        for (int l = 0; l <= L; ++l) {
            const int64_t it = it0 + (int64_t)m * (L + 1) + l;
            const double e = (l < L) ? Pp[l + (size_t)m * nR] : Pp[(L + m) + (size_t)m * nR];
            double t = 0.0;
            if (l == L || e != 0.0) {
                bad |= itemStatus[it];
                t = fabs(e * perm[it]);
                colPerm += t;
            }
            out[(size_t)m * (L + 1) + l] = t;
        }
        best = (best < colPerm) ? colPerm : best;  // std::max over columns (:255)
    }
    best = warp_max(best);
    bad = __any_sync(FULL, bad != 0);
    __syncwarp();
    const double norm = 1.0 / best;
    for (int e = lane; e < M * (L + 1); e += 32) out[e] *= norm;
    if (lane == 0) status[p] = bad ? 1 : 0;
}

// Runs build -> permanent -> unscale (-> retry of negatives) over `nItems` items living in a Stage.
struct ItemBuffers {
    double* mats; int64_t* matOff; int32_t* rows; int32_t* cols; double* scale; int32_t* status;
    double* perm; int32_t* permStatus; int32_t* negList; int32_t* negCount; void* ws; int64_t wsBytes;
};

int run_items(BuildArgs b, const ItemBuffers& ib, int64_t nItems, int maxDim, int permOpt, cudaStream_t s, int maxSmall) {
    b.subset = nullptr; b.nWork = nItems; b.transpose = 1;
    b.mats = ib.mats; b.outRows = ib.rows; b.outCols = ib.cols; b.scale = ib.scale; b.itemStatus = ib.status;
    build_items_kernel<<<(unsigned)((nItems + BUILD_WARPS - 1) / BUILD_WARPS), 32 * BUILD_WARPS, 0, s>>>(b);
    PDA_CUDA_TRY(cudaGetLastError());
    if (permOpt == 0)  // Huber's approximation, apprxIter = 300 trials (assignment.cpp:10, :401); never negative, so no retry
        PDA_TRY(launch_permanent_approx_batch(ib.mats, ib.matOff, ib.rows, ib.cols, nItems, 300, approx_seed(), ib.perm,
                                              ib.permStatus, s));
    else
        PDA_TRY(launch_permanent_batch(ib.mats, ib.matOff, ib.rows, ib.cols, nItems, maxDim, ib.perm, ib.permStatus, ib.ws,
                                       ib.wsBytes, s, maxSmall));
    PDA_CUDA_TRY(cudaMemsetAsync(ib.negCount, 0, 4, s));
    unscale_kernel<<<(unsigned)((nItems + 255) / 256), 256, 0, s>>>(ib.perm, ib.scale, nullptr, nItems, ib.negList, ib.negCount);
    PDA_CUDA_TRY(cudaGetLastError());
    int32_t nNeg = 0;
    PDA_CUDA_TRY(cudaMemcpyAsync(&nNeg, ib.negCount, 4, cudaMemcpyDeviceToHost, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    if (nNeg > 0) {
        // recompute the negative ones untransposed (:409-419).  The permanent launch below works on a
        // compacted copy of the item descriptors so only those items are walked again.
        std::vector<int32_t> neg((size_t)nNeg);
        PDA_CUDA_TRY(cudaMemcpy(neg.data(), ib.negList, (size_t)nNeg * 4, cudaMemcpyDeviceToHost));
        std::sort(neg.begin(), neg.end());
        PDA_CUDA_TRY(cudaMemcpyAsync(ib.negList, neg.data(), (size_t)nNeg * 4, cudaMemcpyHostToDevice, s));
        b.subset = ib.negList; b.nWork = nNeg; b.transpose = 0;
        build_items_kernel<<<(unsigned)((nNeg + BUILD_WARPS - 1) / BUILD_WARPS), 32 * BUILD_WARPS, 0, s>>>(b);
        PDA_CUDA_TRY(cudaGetLastError());
        for (int32_t i = 0; i < nNeg; ++i) {
            const int64_t it = neg[(size_t)i];
            PDA_TRY(launch_permanent_batch(ib.mats, ib.matOff + it, ib.rows + it, ib.cols + it, 1, maxDim, ib.perm + it,
                                           ib.permStatus + it, ib.ws, ib.wsBytes, s, maxSmall));
        }
        unscale_kernel<<<(unsigned)((nNeg + 255) / 256), 256, 0, s>>>(ib.perm, ib.scale, ib.negList, nNeg, nullptr, nullptr);
        PDA_CUDA_TRY(cudaGetLastError());
    }
    return PDA_OK;
}

size_t reserve_items(Stage& st, size_t nItems, size_t off[12], size_t wsBytes) {
    off[0] = st.reserve(nItems * SLOT * 8);  // mats
    off[1] = st.reserve(nItems * 8);         // matOff
    off[2] = st.reserve(nItems * 4);         // rows
    off[3] = st.reserve(nItems * 4);         // cols
    off[4] = st.reserve(nItems * 8);         // scale
    off[5] = st.reserve(nItems * 4);         // status
    off[6] = st.reserve(nItems * 8);         // perm
    off[7] = st.reserve(nItems * 4);         // permStatus
    off[8] = st.reserve(nItems * 4);         // negList
    off[9] = st.reserve(256);                // negCount
    off[10] = st.reserve(wsBytes);           // permanent workspace
    return st.used();
}

ItemBuffers bind_items(const Stage& st, const size_t off[12], size_t wsBytes) {
    ItemBuffers ib;
    ib.mats = st.at<double>(off[0]); ib.matOff = st.at<int64_t>(off[1]); ib.rows = st.at<int32_t>(off[2]);
    ib.cols = st.at<int32_t>(off[3]); ib.scale = st.at<double>(off[4]); ib.status = st.at<int32_t>(off[5]);
    ib.perm = st.at<double>(off[6]); ib.permStatus = st.at<int32_t>(off[7]); ib.negList = st.at<int32_t>(off[8]);
    ib.negCount = st.at<int32_t>(off[9]); ib.ws = st.at<unsigned char>(off[10]); ib.wsBytes = (int64_t)wsBytes;
    return ib;
}

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

int pda_conditioned_permanent_batch_host(const double* mats, const int64_t* matOff, const int32_t* rows,
                                         const int32_t* cols, int64_t nMats, int32_t permOpt,
                                         double* out, int32_t* status, int32_t device) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out || !status) return fail(PDA_ERR_INVALID, "conditioned_permanent: NULL argument");
    if (permOpt < 0 || permOpt > 2) {  // 0 = Huber approximation, 1 = exact, 2 = "long"; anything else throws (assignment.cpp:406)
        for (int64_t i = 0; i < nMats; ++i) { out[i] = 0.0; status[i] = 1; }
        return PDA_OK;
    }
    size_t nEl = 0;
    int maxDim = 1;
    for (int64_t i = 0; i < nMats; ++i) {
        if (rows[i] < 0 || cols[i] < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: negative dimension");
        nEl = std::max(nEl, (size_t)matOff[i] + (size_t)rows[i] * cols[i]);
        maxDim = std::max(maxDim, std::min(PDA_MAX_PERM_DIM, std::max(rows[i], cols[i])));
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const size_t n = (size_t)nMats;
    const size_t wsBytes = (size_t)pda_permanent_workspace_bytes(nMats);
    Stage st(device);
    const size_t oA = st.reserve(nEl * 8), oOff = st.reserve(n * 8), oR = st.reserve(n * 4), oC = st.reserve(n * 4);
    size_t off[12];
    reserve_items(st, n, off, wsBytes);
    PDA_TRY(st.commit());
    ItemBuffers ib = bind_items(st, off, wsBytes);
    cudaStream_t s = 0;
    PDA_TRY(h2d(st.at<double>(oA), mats, nEl, s));
    PDA_TRY(h2d(st.at<int64_t>(oOff), matOff, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oR), rows, n, s));
    PDA_TRY(h2d(st.at<int32_t>(oC), cols, n, s));
    std::vector<int64_t> slotOff(n);
    for (size_t i = 0; i < n; ++i) slotOff[i] = (int64_t)i * SLOT;
    PDA_TRY(h2d(ib.matOff, slotOff.data(), n, s));
    BuildArgs b = {};
    b.mode = 1; b.P = st.at<double>(oA); b.pOff = st.at<int64_t>(oOff); b.rows = st.at<int32_t>(oR); b.cols = st.at<int32_t>(oC);
    int maxSmall = 0;
    for (int64_t i = 0; i < nMats; ++i) maxSmall = std::max(maxSmall, std::min(rows[i], cols[i]));
    PDA_TRY(run_items(b, ib, nMats, maxDim, permOpt, s, maxSmall));
    PDA_TRY(d2h(out, ib.perm, n, s));
    PDA_TRY(d2h(status, ib.status, n, s));
    PDA_CUDA_TRY(cudaStreamSynchronize(s));
    return PDA_OK;
}

int pda_permanent_prob_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL,
                                  const int32_t* nM, int64_t nProblems, int32_t permOpt,
                                  double* probs, const int64_t* probOff, int32_t* status, int32_t device) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status) return fail(PDA_ERR_INVALID, "permanent_prob: NULL argument");
    const bool throws = (permOpt < 0 || permOpt > 2);
    // chunk the batch so that one chunk's items fit a bounded staging area
    const int64_t maxItemsPerChunk = 1 << 16;
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    int64_t p0 = 0;
    while (p0 < nProblems) {
        int64_t p1 = p0, items = 0;
        size_t nCost = 0, nProb = 0;
        int maxDim = 1, maxSmall = 0;
        size_t c0 = (size_t)costOff[p0];
        std::vector<int64_t> itemOff, locCostOff, locProbOff;
        std::vector<int32_t> itemProblem;
        size_t pr0 = (size_t)probOff[p0];
        // problems of a chunk must be addressable relative to the chunk's first cost/prob offset
        while (p1 < nProblems) {
            const int64_t L = nL[p1], M = nM[p1];
            if (L < 0 || M < 1 || L + M > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_prob: problem %lld is nL=%lld nM=%lld", (long long)p1, (long long)L, (long long)M);
            const int64_t add = (M > 1) ? M * (L + 1) : 0;
            if (p1 > p0 && items + add > maxItemsPerChunk) break;
            if ((size_t)costOff[p1] < c0 || (size_t)probOff[p1] < pr0) return fail(PDA_ERR_INVALID, "permanent_prob: offsets must be non-decreasing");
            itemOff.push_back(items);
            for (int64_t i = 0; i < add; ++i) itemProblem.push_back((int32_t)(p1 - p0));
            items += add;
            locCostOff.push_back((int64_t)((size_t)costOff[p1] - c0));
            locProbOff.push_back((int64_t)((size_t)probOff[p1] - pr0));
            nCost = std::max(nCost, (size_t)costOff[p1] - c0 + (size_t)((L + M) * M));
            nProb = std::max(nProb, (size_t)probOff[p1] - pr0 + (size_t)(M * (L + 1)));
            if (M > 1) maxDim = std::max<int>(maxDim, (int)std::min<int64_t>(PDA_MAX_PERM_DIM, std::max(L + M - 1, M - 1)));
            if (M > 1) maxSmall = std::max<int>(maxSmall, (int)std::min<int64_t>(M - 1, L + M - 1));
            ++p1;
        }
        const size_t n = (size_t)(p1 - p0), nIt = (size_t)std::max<int64_t>(items, 1);
        if (throws) {
            for (int64_t p = p0; p < p1; ++p) status[p] = (nM[p] == 1) ? 0 : 1;
        }
        const size_t wsBytes = (size_t)pda_permanent_workspace_bytes((int64_t)nIt);
        Stage st(device);
        const size_t oP = st.reserve(nCost * 8), oOff = st.reserve(n * 8), oLen = st.reserve(n * 8), oL = st.reserve(n * 4), oM = st.reserve(n * 4);
        const size_t oItemOff = st.reserve(n * 8), oItemProb = st.reserve(nIt * 4), oProbs = st.reserve(nProb * 8), oProbOff = st.reserve(n * 8), oStatus = st.reserve(n * 4);
        size_t off[12];
        reserve_items(st, nIt, off, wsBytes);
        PDA_TRY(st.commit());
        ItemBuffers ib = bind_items(st, off, wsBytes);
        cudaStream_t s = 0;
        std::vector<int64_t> len(n), slotOff(nIt);
        for (size_t i = 0; i < n; ++i) len[i] = (int64_t)(nL[p0 + (int64_t)i] + nM[p0 + (int64_t)i]) * nM[p0 + (int64_t)i];
        for (size_t i = 0; i < nIt; ++i) slotOff[i] = (int64_t)i * SLOT;
        PDA_TRY(h2d(st.at<double>(oP), costs + c0, nCost, s));
        PDA_TRY(h2d(st.at<int64_t>(oOff), locCostOff.data(), n, s));
        PDA_TRY(h2d(st.at<int64_t>(oLen), len.data(), n, s));
        PDA_TRY(h2d(st.at<int32_t>(oL), nL + p0, n, s));
        PDA_TRY(h2d(st.at<int32_t>(oM), nM + p0, n, s));
        PDA_TRY(h2d(st.at<int64_t>(oItemOff), itemOff.data(), n, s));
        if (items > 0) PDA_TRY(h2d(st.at<int32_t>(oItemProb), itemProblem.data(), (size_t)items, s));
        PDA_TRY(h2d(st.at<int64_t>(oProbOff), locProbOff.data(), n, s));
        PDA_TRY(h2d(ib.matOff, slotOff.data(), nIt, s));
        PDA_CUDA_TRY(cudaMemsetAsync(st.at<double>(oProbs), 0, nProb * 8, s));
        // 1. likelihoods (toProbs, :164), in place on the staged costs
        PDA_TRY(launch_to_probs(st.at<double>(oP), st.at<int64_t>(oOff), st.at<int64_t>(oLen), (int64_t)n, s));
        single_column_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(st.at<double>(oP), st.at<int64_t>(oOff), st.at<int32_t>(oL),
                                                                      st.at<int32_t>(oM), (int64_t)n, st.at<double>(oProbs),
                                                                      st.at<int64_t>(oProbOff));
        PDA_CUDA_TRY(cudaGetLastError());
        if (!throws) {
            if (items > 0) {
                BuildArgs b = {};
                b.mode = 0; b.P = st.at<double>(oP); b.pOff = st.at<int64_t>(oOff); b.nL = st.at<int32_t>(oL); b.nM = st.at<int32_t>(oM);
                b.itemOff = st.at<int64_t>(oItemOff); b.itemProblem = st.at<int32_t>(oItemProb);
                PDA_TRY(run_items(b, ib, items, maxDim, permOpt, s, maxSmall));
            }
            finish_probs_kernel<<<(unsigned)((n + BUILD_WARPS - 1) / BUILD_WARPS), 32 * BUILD_WARPS, 0, s>>>(
                st.at<double>(oP), st.at<int64_t>(oOff), st.at<int32_t>(oL), st.at<int32_t>(oM), st.at<int64_t>(oItemOff), ib.perm,
                ib.status, (int64_t)n, st.at<double>(oProbs), st.at<int64_t>(oProbOff), st.at<int32_t>(oStatus));
            PDA_CUDA_TRY(cudaGetLastError());
            PDA_TRY(d2h(status + p0, st.at<int32_t>(oStatus), n, s));
        }
        PDA_TRY(d2h(probs + pr0, st.at<double>(oProbs), nProb, s));
        PDA_CUDA_TRY(cudaStreamSynchronize(s));
        p0 = p1;
    }
    return PDA_OK;
}

int pda_permanent_prob_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* nL,
                                        const int32_t* nM, int64_t nProblems, int32_t permOpt,
                                        double* probs, const int64_t* probOff, int32_t* status,
                                        const int32_t* devices, int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "permanent_prob (multi): need at least one device");
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status) return fail(PDA_ERR_INVALID, "permanent_prob: NULL argument");
    // the (nL+1) * nM sub-permanents of a problem are independent (assignment.cpp:213-246), and so are the problems:
    // contiguous slices of problems, one per device
    return run_sharded(nProblems, devices, nDevices, [&](int64_t p0, int64_t p1, int dev) {
        return pda_permanent_prob_batch_host(costs, costOff + p0, nL + p0, nM + p0, p1 - p0, permOpt, probs, probOff + p0,
                                             status + p0, dev);
    });
}

}  // extern "C"
