// permprob_device_kernel.cu -- permanentProb (assignment.cpp:145-290) and conditionedPermanent (:325-435), the one
// implementation of both the device-pointer and the *_host entries.  The device-pointer forms take device arrays only:
// the host reads none of them, and the whole call is enqueued on the caller's stream without a synchronisation, so it can
// follow a device producer or be captured in a CUDA graph.  The *_host forms (at the end) stage their inputs and make
// one such call per chunk.
//
// Items are the sub-permanents, numbered m-major per problem:
//   1. prep_kernel      one CTA: the item index of every problem's first sub-permanent (a scan over the problems), the
//                       batch's item count and largest dimension, and from those the NW launch shapes (perm_shape for
//                       the whole batch, cut to the partials of pda_permanent_workspace_bytes(items), and that of a
//                       one-matrix launch for the retry)
//   2. to_probs         the likelihoods, on a copy of the costs (weights_kernel.cu)
//   3. gather_kernel    one warp per sub-permanent: gathers it straight out of the likelihoods and conditions it
//                       (perm_device.cuh).  A short side <= 10 runs the subset DP in shared memory -- nothing is
//                       materialised.  A short side of 11..31 (and every item under permOpt 0) is written, scaled and
//                       transposed, into its slot of the workspace and appended to a device list
//   4. walk_list_kernel the NW walk (perm_walk.cuh) of the listed items: a persistent grid takes (item group, CTA)
//                       units one after another, with perm_kernel's per-CTA range split and reduction order
//      or Huber's approximation (permanent_approx_kernel.cu) on the slots under permOpt 0
//   5. unscale          perm / scale; a negative result is appended to a second device list
//   6. the retry (:409-419): regather_kernel writes those items untransposed, walk_list_kernel walks them with the
//      shape of a single-matrix launch (the reference recomputes each one alone), unscale once more
//   7. finish           |P(l,m) * perm|, column sums, normalisation by the largest column sum
#include "pda_internal.h"
#include "pda_host_stage.h"
#include "perm_device.cuh"
#include "perm_walk.cuh"
#include "cta_scan.cuh"

#include <algorithm>
#include <vector>

namespace pda {
namespace {

constexpr int SUB_DOUBLES = PDA_MAX_PERM_DIM * PERM_DP_MAX;
constexpr int GATHER_WARPS = 4;
constexpr int FINISH_WARPS = 4;
constexpr int SMEM_BUDGET = 48 * 1024;
constexpr int APPROX_TRIALS = 300;    // apprxIter (assignment.cpp:10)

// Written by prep_kernel at the head of the workspace; the host never reads it.
struct Ctrl {
    long long nItems;       // sub-permanents of the call
    int effDim;             // largest min(32, kept-rows bound) over the call
    unsigned nList, nNeg;   // materialised items, items that came out negative
    PermShape mainShape, retryShape;
};

struct Work {
    Ctrl* ctrl;
    double* P; int32_t* rowsLen; int64_t* itemOff;              // mode 0
    double* perm; double* scale; int32_t* istat;
    int32_t* mRows; int32_t* mCols; int64_t* matOff; int32_t* owner; int32_t* list; int32_t* negList; int32_t* apStat;
    double* mats;
    dd* partial; unsigned* done;
    int64_t cap;            // items the workspace has room for
    int slotDoubles, cpmCap;
    bool materialise, nw;
    size_t bytes;
};

// mode 0: problems (nL, nM); mode 1: matrices (rows, cols).  maxA / maxB: maxNumRow / maxNumCol, or maxDim / maxDim.
Work carve(void* workspace, int mode, int64_t nUnits, int64_t totalCostElems, int64_t cap, int32_t maxA, int32_t maxB,
           int32_t permOpt, int smCount) {
    const bool valid = permOpt >= 0 && permOpt <= 2;
    const int keptA = std::max(1, std::min(PDA_MAX_PERM_DIM, mode == 0 ? maxA - 1 : maxA));  // kept rows
    const int keptB = std::max(1, std::min(PDA_MAX_PERM_DIM, mode == 0 ? maxB - 1 : maxB));  // kept columns
    Work w{};
    w.cap = cap;
    w.nw = valid && permOpt != 0 && std::min(keptA, keptB) > PERM_DP_MAX;
    w.materialise = valid && (permOpt == 0 || w.nw);
    w.slotDoubles = keptA * keptB;
    w.cpmCap = perm_shape(1, PDA_MAX_PERM_DIM, smCount, 0).ctasPerMat;  // no launch shape has more CTAs per matrix
    const size_t n = (size_t)std::max<int64_t>(nUnits, 1), c = (size_t)std::max<int64_t>(cap, 1);
    WorkspaceLayout L(workspace);
    w.ctrl = L.take<Ctrl>(1);
    if (mode == 0) {
        w.P = L.take<double>((size_t)totalCostElems);
        w.rowsLen = L.take<int32_t>(n);
        w.itemOff = L.take<int64_t>(n);
    }
    w.perm = L.take<double>(c);
    w.scale = L.take<double>(c);
    w.istat = L.take<int32_t>(c);
    if (w.materialise) {
        w.mRows = L.take<int32_t>(c);
        w.mCols = L.take<int32_t>(c);
        w.matOff = L.take<int64_t>(c);
        w.owner = L.take<int32_t>(c);
        w.list = L.take<int32_t>(c);
        w.negList = L.take<int32_t>(c);
        w.apStat = L.take<int32_t>(c);
        w.mats = L.take<double>(c * (size_t)w.slotDoubles);
    }
    if (w.nw) {
        w.partial = L.take<dd>(c * (size_t)w.cpmCap);
        w.done = L.take<unsigned>(c);
    }
    w.bytes = L.bytes();
    return w;
}

__device__ __forceinline__ bool out_of_scope0(int L, int M, int maxRow, int maxCol) {
    return L < 0 || M < 1 || M > maxCol || L + M > maxRow;
}
__device__ __forceinline__ bool out_of_scope1(int r, int c, int maxDim) { return r < 0 || c < 0 || r > maxDim || c > maxDim; }

// The NW launch shapes for a batch of nItems items of largest dimension effDim: the shape launch_permanent_batch
// picks, with the CTA count cut to its workspace (pda_permanent_workspace_bytes(nItems)); and that of a one-matrix
// launch, which recomputes a negative item.
__device__ void plan_shapes(Ctrl* c, long long nItems, int effDim, int smCount) {
    const long long nIt = nItems > 1 ? nItems : 1;  // a call without items walks nothing
    PermShape sh = perm_shape(nIt, effDim, smCount, 0);
    const long long partBytes = perm_partial_bytes(nIt);
    while (sh.ctasPerMat > 1 && (long long)sh.ctasPerMat * nIt * (long long)sizeof(dd) > partBytes) sh.ctasPerMat >>= 1;
    c->mainShape = sh;
    c->retryShape = perm_shape(1, effDim, smCount, 0);
    c->nItems = nItems;
    c->effDim = effDim;
    c->nList = 0;
    c->nNeg = 0;
}

// mode 0: itemOff[p] = sub-permanents of the problems before p (nM * (nL + 1) for nM > 1, counted for every problem in
// scope or not), rowsLen[p] = nL + nM (0 out of scope: to_probs leaves it alone).  mode 1: only the largest dimension.
__global__ void __launch_bounds__(CTA_SCAN_THREADS) prep_kernel(int mode, const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                                                               int64_t n, int32_t maxA, int32_t maxB, int32_t* __restrict__ rowsLen,
                                                               int64_t* __restrict__ itemOff, Ctrl* ctrl, int smCount) {
    __shared__ long long sWarp[32];
    long long carry = 0, eff = 1;
    for (int64_t base = 0; base < n; base += CTA_SCAN_THREADS) {
        const int64_t p = base + threadIdx.x;
        long long add = 0;
        if (p < n) {
            const int x = a[p], y = b[p];
            if (mode == 0) {  // x = nL, y = nM
                rowsLen[p] = out_of_scope0(x, y, maxA, maxB) ? 0 : x + y;
                if (y > 1 && x >= 0) { add = (long long)y * (x + 1); eff = max(eff, (long long)min(PDA_MAX_PERM_DIM, x + y - 1)); }
            } else {          // x = rows, y = cols
                add = 1;
                eff = max(eff, (long long)min(PDA_MAX_PERM_DIM, max(max(x, y), 0)));
            }
        }
        const long long before = cta_scan(add, carry, sWarp, ScanSum()) - add;
        if (mode == 0 && p < n) itemOff[p] = before;
    }
    long long effMax = 1;
    cta_scan(eff, effMax, sWarp, ScanMax());
    if (threadIdx.x == 0) plan_shapes(ctrl, carry, (int)effMax, smCount);
}

struct GatherArgs {
    int mode, permOpt;
    const double* P; const int64_t* pOff;
    const int32_t* a; const int32_t* b;   // mode 0: nL, nM; mode 1: rows, cols
    const int64_t* itemOff;
    int64_t nUnits;
    int32_t maxA, maxB;
    int cap, warps;                       // DP states of the largest short side, warps per CTA
    Work w;
};

// shared memory of one gather warp, in doubles: DP buffers (2 cap + 16), the scaled sub-matrix of a DP item, the column
// scales, then the kept column and row indices as shorts
__host__ __device__ constexpr int gather_doubles(int cap) { return 2 * cap + 16 + SUB_DOUBLES + PDA_MAX_DIM + 2 * PDA_MAX_DIM / 4; }

// One sub-permanent by one warp: conditioned, then either the subset DP and perm / scale (perm_item_warp), or written
// to its slot
__device__ __forceinline__ void gather_item(const GatherArgs& a, const Gather& g, const int64_t it, const int32_t owner,
                                            double* buf, const int lane) {
    double* sub = buf + 2 * a.cap + 16;
    double* scale = sub + SUB_DOUBLES;
    short* keepC = reinterpret_cast<short*>(scale + PDA_MAX_DIM);
    short* keepR = keepC + PDA_MAX_DIM;
    const Work& w = a.w;
    int nKR, nKC;
    if (perm_item_warp(g, a.permOpt != 0, buf, a.cap, sub, scale, keepC, keepR, lane, nKR, nKC,
                       [&](double v, int st) { w.perm[it] = v; w.istat[it] = st; }))
        return;
    double* M = w.mats + (size_t)it * w.slotDoubles;
    write_scaled(g, scale, keepC, keepR, nKR, nKC, 1, M, lane);
    if (lane == 0) {
        w.scale[it] = scale_product(scale, nKC);
        w.mRows[it] = nKC; w.mCols[it] = nKR;
        w.matOff[it] = it * w.slotDoubles;
        w.owner[it] = owner;
        w.istat[it] = 0;
        w.list[atomicAdd(&w.ctrl->nList, 1u)] = (int32_t)it;
    }
}

__global__ void __launch_bounds__(32 * GATHER_WARPS) gather_kernel(const GatherArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* buf = smem + (size_t)warp * gather_doubles(a.cap);
    if (a.mode == 0) {
        const int64_t p = blockIdx.x;
        const int L = a.a[p], M = a.b[p];
        if (M < 2 || out_of_scope0(L, M, a.maxA, a.maxB)) return;
        const int items = M * (L + 1);
        const int64_t base = a.itemOff[p];
        if (base + items > a.w.cap) return;  // finish reports status 2
        const double* Pp = a.w.P + a.pOff[p];
        for (int e = (int)blockIdx.y * a.warps + warp; e < items; e += (int)gridDim.y * a.warps) {
            Gather g;
            if (!item_gather(Pp, L, M, e / (L + 1), e % (L + 1), g)) continue;  // zero likelihood: never read (:217)
            gather_item(a, g, base + e, (int32_t)p, buf, lane);
        }
    } else {
        const int64_t it = (int64_t)blockIdx.x * a.warps + warp;
        if (warp >= a.warps || it >= a.nUnits) return;
        const int r = a.a[it], c = a.b[it];
        if (out_of_scope1(r, c, a.maxA)) return;
        Gather g;
        g.base = a.P + a.pOff[it]; g.ld = r; g.sR = r; g.sC = c;
        g.skipRow = -1; g.skipCol = -1; g.patchRow = -1; g.patchVal = 0.0;
        gather_item(a, g, it, (int32_t)it, buf, lane);
    }
}

// the retry's build: a listed item once more, untransposed (:409-419)
__global__ void __launch_bounds__(32 * GATHER_WARPS) regather_kernel(const GatherArgs a) {
    __shared__ double sScale[GATHER_WARPS][PDA_MAX_DIM];
    __shared__ short sKeepC[GATHER_WARPS][PDA_MAX_DIM];
    __shared__ short sKeepR[GATHER_WARPS][PDA_MAX_DIM];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Work& w = a.w;
    const unsigned nNeg = w.ctrl->nNeg;
    for (unsigned k = blockIdx.x * GATHER_WARPS + warp; k < nNeg; k += gridDim.x * GATHER_WARPS) {
        const int64_t it = w.negList[k];
        Gather g;
        if (a.mode == 0) {
            const int p = w.owner[it];
            const int L = a.a[p], M = a.b[p];
            const int e = (int)(it - a.itemOff[p]);
            item_gather(w.P + a.pOff[p], L, M, e / (L + 1), e % (L + 1), g);
        } else {
            g.base = a.P + a.pOff[it]; g.ld = a.a[it]; g.sR = a.a[it]; g.sC = a.b[it];
            g.skipRow = -1; g.skipCol = -1; g.patchRow = -1; g.patchVal = 0.0;
        }
        __syncwarp();
        int nKR, nKC;
        condition_warp(g, sScale[warp], sKeepC[warp], sKeepR[warp], lane, nKR, nKC);
        write_scaled(g, sScale[warp], sKeepC[warp], sKeepR[warp], nKR, nKC, 0, w.mats + (size_t)it * w.slotDoubles, lane);
        if (lane == 0) { w.scale[it] = scale_product(sScale[warp], nKC); w.mRows[it] = nKR; w.mCols[it] = nKC; }
    }
}

struct WalkArgs {
    const double* mats; int slotDoubles;
    const int32_t* rows; const int32_t* cols;
    const int32_t* list; const unsigned* count; const PermShape* shape;
    dd* partial; int cpmCap; unsigned* done; double* out;
};

// perm_kernel's unit of the NW walk (nw_unit) for the listed items.  The grid is persistent: unit u is (item group
// u / cpm, CTA u % cpm) of the launch perm_kernel would be, so every item gets the same per-thread ranges and the same
// reduction order as in a perm_kernel launch of that shape.  The shape and the item count are read on the device.
template <int NP>
__global__ void __launch_bounds__(PERM_THREADS, perm_min_blocks(NP)) walk_list_kernel(const WalkArgs a) {
    extern __shared__ __align__(16) double smemD[];
    const PermShape sh = *a.shape;
    const unsigned count = *a.count;
    const int tid = threadIdx.x, tpm = sh.threadsPerMat, cpm = sh.ctasPerMat;
    const int slot = tid / tpm, t = tid % tpm, slots = PERM_THREADS / tpm;
    double* sA = smemD + (size_t)slot * (perm_ld(NP) * NP + NP);
    const long long units = (long long)((count + slots - 1) / slots) * cpm;
    for (long long u = blockIdx.x; u < units; u += gridDim.x) {
        const long long k = (u / cpm) * slots + slot;
        const int cta = (int)(u % cpm);
        const bool live = k < count;
        const int64_t m = live ? a.list[k] : 0;
        const int rows = live ? a.rows[m] : 0, cols = live ? a.cols[m] : 0;
        const int n = rows > cols ? rows : cols;
        const bool last = nw_unit<NP>(a.mats + (size_t)m * a.slotDoubles, rows, cols, live, live && n >= 1 && n <= NP, false, 0,
                                      0, sh.chunk, tpm, cpm, cta, sA, sA + perm_ld(NP) * NP, m, a.partial, a.cpmCap, a.done);
        if (last) {
            const dd s = nw_partials_sum(a.partial + (size_t)m * a.cpmCap, cpm, t);
            if (t == 0) {
                a.out[m] = nw_value(s, rows, cols);
                if (cpm > 1) a.done[m] = 0u;
            }
        }
        __syncthreads();  // the next unit reuses the shared slots
    }
}

template <int NP>
int launch_walk_np(const WalkArgs& a, int smCount, cudaStream_t s) {
    const size_t smem = (size_t)(PERM_THREADS / 32) * (perm_ld(NP) * NP + NP) * sizeof(double);  // up to 8 slots
    PDA_CUDA_TRY(cudaFuncSetAttribute(walk_list_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    walk_list_kernel<NP><<<(unsigned)(smCount * perm_min_blocks(NP)), PERM_THREADS, smem, s>>>(a);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int launch_walk(const WalkArgs& a, int maxN, int smCount, cudaStream_t s) {
    return nw_dispatch<12>(maxN, [&](auto np) { return launch_walk_np<decltype(np)::value>(a, smCount, s); });
}

// perm[it] /= scale[it] over a device list (:402); negatives go to negList when it is given
__global__ void unscale_list_kernel(double* __restrict__ perm, const double* __restrict__ scale, const int32_t* __restrict__ list,
                                    const unsigned* __restrict__ count, int32_t* __restrict__ negList, unsigned* negCount) {
    const unsigned n = *count;
    for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const int32_t it = list[k];
        const double r = perm[it] / scale[it];
        perm[it] = r;
        if (negList && r < 0.0) negList[atomicAdd(negCount, 1u)] = it;
    }
}

// permanentProb's tables, one warp per problem: |P(l,m) * perm|, column sums, normalisation; one detection: :166-171
__global__ void finish_kernel(const double* __restrict__ P, const int64_t* __restrict__ pOff, const int32_t* __restrict__ nL,
                              const int32_t* __restrict__ nM, const int64_t* __restrict__ itemOff, const double* __restrict__ perm,
                              const int32_t* __restrict__ istat, int64_t nProblems, int32_t maxRow, int32_t maxCol, int64_t cap,
                              int valid, double* __restrict__ probs, const int64_t* __restrict__ probOff, int32_t* __restrict__ status) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = (int64_t)blockIdx.x * FINISH_WARPS + warp;
    if (p >= nProblems) return;
    const int L = nL[p], M = nM[p];
    if (out_of_scope0(L, M, maxRow, maxCol)) { if (lane == 0) status[p] = 2; return; }
    const double* Pp = P + pOff[p];
    double* out = probs + probOff[p];
    const auto entry = [&](int, int, int e) -> double& { return out[e]; };
    const auto put = [&](int, int, int e, double v) { out[e] = v; };
    if (M == 1) {
        perm_prob_one(Pp, L, put, lane);
        if (lane == 0) status[p] = 0;
        return;
    }
    const int64_t it0 = itemOff[p];
    if (!valid) {  // the reference throws (assignment.cpp:406)
        for (int e = lane; e < M * (L + 1); e += 32) out[e] = 0.0;
        if (lane == 0) status[p] = 1;
        return;
    }
    if (it0 + (int64_t)M * (L + 1) > cap) { if (lane == 0) status[p] = 2; return; }
    const bool bad = perm_prob_table(Pp, L, M, perm, istat, [&](int, int, int e) { return it0 + e; }, entry, put, lane);
    if (lane == 0) status[p] = bad ? 1 : 0;
}

__global__ void finish_mats_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ cols, int64_t nMats, int32_t maxDim,
                                   int valid, const double* __restrict__ perm, const int32_t* __restrict__ istat,
                                   double* __restrict__ out, int32_t* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMats) return;
    if (out_of_scope1(rows[i], cols[i], maxDim)) { status[i] = 2; return; }
    if (!valid) { out[i] = 0.0; status[i] = 1; return; }
    out[i] = perm[i];
    status[i] = istat[i];
}

// Both entries: mode 0 = permanentProb over problems, mode 1 = conditionedPermanent over matrices.
int run(int mode, const double* src, const int64_t* srcOff, const int32_t* a, const int32_t* b, int64_t nUnits,
        int64_t totalCostElems, int64_t cap, int32_t maxA, int32_t maxB, int32_t permOpt, void* workspace, int64_t workspaceBytes,
        cudaStream_t s, const char* who, Work* out) {
    // the size with one SM is a lower bound on every device's (exact without the NW walk): checked before the device
    if ((int64_t)carve(nullptr, mode, nUnits, totalCostElems, cap, maxA, maxB, permOpt, 1).bytes > workspaceBytes)
        return fail(PDA_ERR_WORKSPACE, "%s: workspace of %lld B too small", who, (long long)workspaceBytes);
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    const Work w = carve(workspace, mode, nUnits, totalCostElems, cap, maxA, maxB, permOpt, dev.smCount);
    if ((int64_t)w.bytes > workspaceBytes)
        return fail(PDA_ERR_WORKSPACE, "%s: workspace of %lld B too small (need %lld)", who, (long long)workspaceBytes, (long long)w.bytes);
    *out = w;
    const bool valid = permOpt >= 0 && permOpt <= 2;
    prep_kernel<<<1, CTA_SCAN_THREADS, 0, s>>>(mode, a, b, nUnits, maxA, maxB, w.rowsLen, w.itemOff, w.ctrl, dev.smCount);
    PDA_CUDA_TRY(cudaGetLastError());
    GatherArgs g;
    g.mode = mode; g.permOpt = permOpt; g.a = a; g.b = b; g.itemOff = w.itemOff; g.nUnits = nUnits; g.maxA = maxA; g.maxB = maxB;
    g.w = w;
    if (mode == 0) {
        if (totalCostElems > 0) PDA_CUDA_TRY(cudaMemcpyAsync(w.P, src, (size_t)totalCostElems * 8, cudaMemcpyDeviceToDevice, s));
        PDA_TRY(launch_to_probs(w.P, srcOff, nullptr, nUnits, s, w.rowsLen, b));  // toProbs (:164)
        g.P = w.P; g.pOff = srcOff;
    } else {
        g.P = src; g.pOff = srcOff;
    }
    if (!valid) return PDA_OK;
    const int shortMax = std::max(0, std::min(PERM_DP_MAX, mode == 0 ? maxB - 1 : maxA));
    g.cap = 1 << shortMax;
    const int perWarp = gather_doubles(g.cap) * (int)sizeof(double);
    g.warps = std::max(1, std::min(GATHER_WARPS, SMEM_BUDGET / perWarp));
    if (w.materialise) {
        PDA_CUDA_TRY(cudaMemsetAsync(w.mRows, 0, (size_t)std::max<int64_t>(cap, 1) * 4, s));
        PDA_CUDA_TRY(cudaMemsetAsync(w.mCols, 0, (size_t)std::max<int64_t>(cap, 1) * 4, s));
    }
    if (w.nw) PDA_CUDA_TRY(cudaMemsetAsync(w.done, 0, (size_t)std::max<int64_t>(cap, 1) * 4, s));
    if (mode == 0) {
        if (maxB >= 2) {  // CTAs per problem: up to 64 per SM in all, several waves, so that batches of a few hundred to
                          // a few thousand problems with uneven item counts keep every SM busy (B200, 1200 G2 problems:
                          // more than twice as fast as 8 per SM); one CTA per problem from 64 problems per SM on
            const int64_t want = ((int64_t)dev.smCount * 64 + nUnits - 1) / nUnits;
            const int64_t most = ((int64_t)maxB * maxA + g.warps - 1) / g.warps;
            const unsigned split = (unsigned)std::max<int64_t>(1, std::min<int64_t>(std::min(want, most), 65535));
            gather_kernel<<<dim3((unsigned)nUnits, split), 32 * g.warps, (size_t)g.warps * perWarp, s>>>(g);
        }
    } else {
        gather_kernel<<<(unsigned)((nUnits + g.warps - 1) / g.warps), 32 * g.warps, (size_t)g.warps * perWarp, s>>>(g);
    }
    PDA_CUDA_TRY(cudaGetLastError());
    if (!w.materialise) return PDA_OK;
    const unsigned listGrid = (unsigned)std::min<int64_t>((cap + 255) / 256 + 1, (int64_t)dev.smCount * 8);
    if (permOpt == 0) {  // Huber's approximation on every item, keyed by its item index; never negative, so no retry
        PDA_TRY(launch_permanent_approx_batch(w.mats, w.matOff, w.mRows, w.mCols, cap, APPROX_TRIALS, approx_seed(), w.perm, w.apStat, s));
        unscale_list_kernel<<<listGrid, 256, 0, s>>>(w.perm, w.scale, w.list, &w.ctrl->nList, nullptr, nullptr);
        PDA_CUDA_TRY(cudaGetLastError());
        return PDA_OK;
    }
    const int maxN = std::min(PDA_MAX_PERM_DIM, mode == 0 ? maxA - 1 : maxA);
    WalkArgs wa = {w.mats, w.slotDoubles, w.mRows, w.mCols, w.list, &w.ctrl->nList, &w.ctrl->mainShape, w.partial, w.cpmCap, w.done, w.perm};
    PDA_TRY(launch_walk(wa, maxN, dev.smCount, s));
    unscale_list_kernel<<<listGrid, 256, 0, s>>>(w.perm, w.scale, w.list, &w.ctrl->nList, w.negList, &w.ctrl->nNeg);
    PDA_CUDA_TRY(cudaGetLastError());
    // the retry (:409-419): whatever came out negative, untransposed, each item with a one-matrix launch's shape
    regather_kernel<<<(unsigned)dev.smCount, 32 * GATHER_WARPS, 0, s>>>(g);
    PDA_CUDA_TRY(cudaGetLastError());
    wa.list = w.negList; wa.count = &w.ctrl->nNeg; wa.shape = &w.ctrl->retryShape;
    PDA_TRY(launch_walk(wa, maxN, dev.smCount, s));
    unscale_list_kernel<<<listGrid, 256, 0, s>>>(w.perm, w.scale, w.negList, &w.ctrl->nNeg, nullptr, nullptr);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

}  // namespace
}  // namespace pda

using namespace pda;

extern "C" {

int64_t pda_permanent_prob_workspace_bytes(int64_t nProblems, int64_t totalCostElems, int64_t totalProbElems,
                                           int32_t maxNumRow, int32_t maxNumCol, int32_t permOpt) {
    if (nProblems < 0 || totalCostElems < 0 || totalProbElems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: negative size");
    if (maxNumRow > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_prob: maxNumRow %d above %d", maxNumRow, PDA_MAX_DIM);
    if (maxNumRow < 1 || maxNumCol < 1) return fail(PDA_ERR_INVALID, "permanent_prob: maxNumRow / maxNumCol < 1");
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    return (int64_t)carve(nullptr, 0, nProblems, totalCostElems, totalProbElems, maxNumRow, maxNumCol, permOpt, dev.smCount).bytes;
}

int pda_permanent_prob_batch(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                             int64_t nProblems, int64_t totalCostElems, int64_t totalProbElems,
                             int32_t maxNumRow, int32_t maxNumCol, int32_t permOpt,
                             double* probs, const int64_t* probOff, int32_t* status,
                             void* workspace, int64_t workspaceBytes, void* stream) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status || !workspace)
        return fail(PDA_ERR_INVALID, "permanent_prob: NULL argument");
    if (totalCostElems < 0 || totalProbElems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: negative total");
    if (maxNumRow > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_prob: maxNumRow %d above %d", maxNumRow, PDA_MAX_DIM);
    if (maxNumRow < 1 || maxNumCol < 1) return fail(PDA_ERR_INVALID, "permanent_prob: maxNumRow / maxNumCol < 1");
    if (nProblems > INT32_MAX) return fail(PDA_ERR_UNSUPPORTED, "permanent_prob: more than %d problems", INT32_MAX);
    const cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    Work w;
    PDA_TRY(run(0, costs, costOff, nL, nM, nProblems, totalCostElems, totalProbElems, maxNumRow, maxNumCol, permOpt, workspace,
                workspaceBytes, s, "permanent_prob", &w));
    finish_kernel<<<(unsigned)((nProblems + FINISH_WARPS - 1) / FINISH_WARPS), 32 * FINISH_WARPS, 0, s>>>(
        w.P, costOff, nL, nM, w.itemOff, w.perm, w.istat, nProblems, maxNumRow, maxNumCol, w.cap, permOpt >= 0 && permOpt <= 2,
        probs, probOff, status);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int64_t pda_conditioned_permanent_workspace_bytes(int64_t nMats, int32_t maxDim, int32_t permOpt) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: nMats < 0");
    if (maxDim > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "conditioned_permanent: maxDim %d above %d", maxDim, PDA_MAX_DIM);
    if (maxDim < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: maxDim < 0");
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    return (int64_t)carve(nullptr, 1, nMats, 0, nMats, maxDim, maxDim, permOpt, dev.smCount).bytes;
}

int pda_conditioned_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                    int64_t nMats, int32_t maxDim, int32_t permOpt, double* out, int32_t* status,
                                    void* workspace, int64_t workspaceBytes, void* stream) {
    if (nMats < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: nMats < 0");
    if (nMats == 0) return PDA_OK;
    if (!mats || !matOff || !rows || !cols || !out || !status || !workspace)
        return fail(PDA_ERR_INVALID, "conditioned_permanent: NULL argument");
    if (maxDim > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "conditioned_permanent: maxDim %d above %d", maxDim, PDA_MAX_DIM);
    if (maxDim < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: maxDim < 0");
    if (nMats > INT32_MAX) return fail(PDA_ERR_UNSUPPORTED, "conditioned_permanent: more than %d matrices", INT32_MAX);
    const cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    Work w;
    PDA_TRY(run(1, mats, matOff, rows, cols, nMats, 0, nMats, maxDim, maxDim, permOpt, workspace, workspaceBytes, s,
                "conditioned_permanent", &w));
    finish_mats_kernel<<<(unsigned)((nMats + 255) / 256), 256, 0, s>>>(rows, cols, nMats, maxDim, permOpt >= 0 && permOpt <= 2,
                                                                      w.perm, w.istat, out, status);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

// The *_host forms: the inputs are staged on `device` and the device-pointer form runs on them.

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
    // A matrix with a side above PDA_MAX_DIM is staged as 0 x 32: an empty permanent over scale 1, reported as status 1
    // below.  Its 32 columns keep the batch's largest dimension, which the NW launch shape of the other matrices follows.
    const size_t n = (size_t)nMats;
    std::vector<int32_t> r(rows, rows + n), c(cols, cols + n);
    size_t nEl = 0;
    int32_t maxDim = 0;
    for (size_t i = 0; i < n; ++i) {
        if (rows[i] < 0 || cols[i] < 0) return fail(PDA_ERR_INVALID, "conditioned_permanent: negative dimension");
        nEl = std::max(nEl, (size_t)matOff[i] + (size_t)rows[i] * cols[i]);
        if (std::max(rows[i], cols[i]) > PDA_MAX_DIM) { r[i] = 0; c[i] = PDA_MAX_PERM_DIM; }
        maxDim = std::max(maxDim, std::max(r[i], c[i]));
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    const size_t wsBytes = carve(nullptr, 1, nMats, 0, nMats, maxDim, maxDim, permOpt, dev.smCount).bytes;
    HostIO io(device);
    const size_t oA = io.in(mats, nEl * 8), oOff = io.in(matOff, n * 8), oR = io.in(r.data(), n * 4), oC = io.in(c.data(), n * 4);
    const size_t oOut = io.out(out, n * 8), oSt = io.out(status, n * 4), oWs = io.scratch(wsBytes);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    PDA_TRY(pda_conditioned_permanent_batch(io.at<double>(oA), io.at<int64_t>(oOff), io.at<int32_t>(oR), io.at<int32_t>(oC), nMats,
                                            maxDim, permOpt, io.at<double>(oOut), io.at<int32_t>(oSt), io.at<unsigned char>(oWs),
                                            (int64_t)wsBytes, io.stream()));
    PDA_TRY(io.download());
    for (size_t i = 0; i < n; ++i)
        if (std::max(rows[i], cols[i]) > PDA_MAX_DIM) status[i] = 1;
    return PDA_OK;
}

int pda_permanent_prob_batch_host(const double* costs, const int64_t* costOff, const int32_t* nL,
                                  const int32_t* nM, int64_t nProblems, int32_t permOpt,
                                  double* probs, const int64_t* probOff, int32_t* status, int32_t device) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "permanent_prob: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !nL || !nM || !probs || !probOff || !status) return fail(PDA_ERR_INVALID, "permanent_prob: NULL argument");
    // One device call per chunk of at most 1 << 16 sub-permanents, which bounds the staging area.  The chunks are part of
    // the results: under permOpt 0 the draws are keyed by the item index within the call, and the NW launch shape follows
    // the call's item count.
    const int64_t maxItemsPerChunk = 1 << 16;
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    int64_t p0 = 0;
    while (p0 < nProblems) {
        int64_t p1 = p0, items = 0;
        size_t nCost = 0, nProb = 0;
        int32_t maxRow = 1, maxCol = 1;
        const size_t c0 = (size_t)costOff[p0], pr0 = (size_t)probOff[p0];
        std::vector<int64_t> locCostOff, locProbOff;
        // problems of a chunk are addressed relative to the chunk's first cost / table offset
        while (p1 < nProblems) {
            const int64_t L = nL[p1], M = nM[p1];
            if (L < 0 || M < 1 || L + M > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "permanent_prob: problem %lld is nL=%lld nM=%lld", (long long)p1, (long long)L, (long long)M);
            const int64_t add = (M > 1) ? M * (L + 1) : 0;
            if (p1 > p0 && items + add > maxItemsPerChunk) break;
            if ((size_t)costOff[p1] < c0 || (size_t)probOff[p1] < pr0) return fail(PDA_ERR_INVALID, "permanent_prob: offsets must be non-decreasing");
            items += add;
            locCostOff.push_back((int64_t)((size_t)costOff[p1] - c0));
            locProbOff.push_back((int64_t)((size_t)probOff[p1] - pr0));
            nCost = std::max(nCost, (size_t)costOff[p1] - c0 + (size_t)((L + M) * M));
            nProb = std::max(nProb, (size_t)probOff[p1] - pr0 + (size_t)(M * (L + 1)));
            maxRow = std::max(maxRow, (int32_t)(L + M));
            maxCol = std::max(maxCol, (int32_t)M);
            ++p1;
        }
        const size_t n = (size_t)(p1 - p0);
        // the capacity is the chunk's item count: callers may leave gaps between their tables
        const size_t wsBytes = carve(nullptr, 0, (int64_t)n, (int64_t)nCost, items, maxRow, maxCol, permOpt, dev.smCount).bytes;
        HostIO io(device);
        const size_t oP = io.in(costs + c0, nCost * 8), oOff = io.in(locCostOff.data(), n * 8), oL = io.in(nL + p0, n * 4);
        const size_t oM = io.in(nM + p0, n * 4), oProbOff = io.in(locProbOff.data(), n * 8);
        const size_t oStatus = io.out(status + p0, n * 4), oProbs = io.out(probs + pr0, nProb * 8), oWs = io.scratch(wsBytes);
        PDA_TRY(io.commit());
        const cudaStream_t s = io.stream();
        PDA_TRY(io.upload());
        // the whole staged range goes back: gaps between the caller's tables come back as zeros
        PDA_CUDA_TRY(cudaMemsetAsync(io.at<double>(oProbs), 0, nProb * 8, s));
        PDA_TRY(pda_permanent_prob_batch(io.at<double>(oP), io.at<int64_t>(oOff), io.at<int32_t>(oL), io.at<int32_t>(oM), (int64_t)n,
                                         (int64_t)nCost, items, maxRow, maxCol, permOpt, io.at<double>(oProbs),
                                         io.at<int64_t>(oProbOff), io.at<int32_t>(oStatus), io.at<unsigned char>(oWs),
                                         (int64_t)wsBytes, s));
        PDA_TRY(io.download());
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
