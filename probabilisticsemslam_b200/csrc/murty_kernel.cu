// murty_kernel.cu -- batched Murty k-best assignment enumeration for sm_100a.
//
// One warp owns one association problem at a time (persistent warps, atomic work
// cursor).  The algorithm is the reference's (shortestPathCPP.cpp): a shortest-
// augmenting-path LAP on the zero-padded square matrix for the root, then Murty's
// partition where every child inherits the parent's duals and needs ONE Dijkstra
// from the freed column (Miller-Stone-Cox).  What is different is where things live:
//
//   lane l owns rows  l, l+32, ...   (v, col4row, shortestPathCost, pred  in registers)
//   lane l owns cols  l, l+32, ...   (u, row4col                            in registers)
//   shared memory per warp: the shifted cost matrix (real columns only -- the
//     reference's padding columns are exactly 0.0 and are never stored), a mirror of
//     u / row4col for the data-dependent lookups, and the weight accumulators
//   global memory per warp: a node arena (bump allocated, written once, read once)
//     and the binary heap that orders the nodes
//
// The row scan of one Dijkstra step is a single pass over the lane's R rows; the
// "closest row" is a warp arg-min done with three REDUX.MIN on an order-preserving
// 64-bit key, lowest row index winning ties -- exactly the reference's first-minimum-
// in-list-order rule because its Row2Scan lists are always ascending
// (shortestPathCPP.cpp:155-157, 486, 215/345).  Every FP64 expression keeps the
// reference's operand order (this file is compiled with -fmad=false; there is no
// multiply on the path except CDelta*numCol), so row4col, col4row, gains and the
// enumeration order are bit-identical to an IEEE-strict build of the reference.
// The heap replays libstdc++'s __push_heap / __adjust_heap so that exact gain ties
// pop in the same order as std::priority_queue<pMurtyHyp> (shortestPathCPP.cpp:30-42).
//
// Two instantiations of the same enumeration:
//   FAST = false  the exact kernel: the open list is the libstdc++ heap replay, every child is solved and kept.  Always
//                 right, including the order of hypotheses with bit-equal gains.
//   FAST = true   the pruning kernel, tried first on large batches.  (1) The open list is the warp-parallel FastPQ.
//                 (2) Once `k` hypotheses are known to exist at or below a bound T (those already emitted plus open ones),
//                 a child whose search distance pushes it past T is abandoned after its first arg-min and a finished
//                 child above T is not stored: such hypotheses can never be emitted, and on the benchmark shape they are
//                 a third of all children.  Both shortcuts are invisible in the output as long as the hypothesis chosen
//                 next is unique; the moment it is not (two open entries with the same gain bits) the problem is
//                 appended to a fallback list and redone from scratch by the exact kernel, which runs right behind on
//                 the same stream over that list.  Continuous costs never tie; integer or 6-decimal costs do, and simply
//                 take the exact kernel.
#include "murty_device.cuh"

namespace pda {
namespace {

#ifdef PDA_FAST_STATS
__device__ unsigned long long g_fastStats[8];  // children, abandoned, dropped at the end, kept, tighten calls, slots at tighten, pops
#define PDA_STAT(i, v) do { if (lane == 0) atomicAdd(&g_fastStats[i], (unsigned long long)(v)); } while (0)
#else
#define PDA_STAT(i, v) do { } while (0)
#endif

// LADDER: the k-ladder form (MurtyLadder): weights only, k = the largest rung, tables stored at every rung.
template <int R, bool FAST, bool LADDER = false>
__device__ void solve_problem(const MurtyArgs& a, const long long p, const WarpSmem& sm, const Heap& heap,
                              const FastPQ& pq, unsigned char* nodes, const int lane, const MurtyLadder* L = nullptr) {
    const int n = a.numRow[p], nc = a.numCol[p];
    const int D = a.geo.nodeDim;
    const bool wantW = a.weightMode != PDA_WEIGHTS_NONE;
    const int nL = wantW ? a.nL[p] : 0;
    // malformed, or larger than the maxima this launch was sized for (shared-memory matrix, node slots, arena): not
    // solved; reported as -1, which no reference call can return (0 = infeasible)
    if (nc < 1 || nc > n || n > 32 * R || n > a.geo.nodeDim || n * nc > a.geo.cCap || nc > a.geo.maxCol || (wantW && nL + nc != n)) {
        if constexpr (LADDER) ladder_found(a, *L, p, -1, lane);
        else if (lane == 0) a.nFound[p] = -1;
        return;
    }
    const double* Cg = a.costs + a.costOff[p];

    // single-detection shortcut of assignmentProb / bruteForceProb (assignment.cpp:554-570, 840-856)
    if (wantW && nc == 1) {
        for (int i = lane; i <= nL; i += 32) sm.acc[i] = (Cg[i] < a.weightGate) ? exp(-Cg[i]) : 0.0;
        __syncwarp();
        double norm = 0.0;
        for (int i = 0; i <= nL; ++i) if (Cg[i] < a.weightGate) norm += sm.acc[i];
        norm = 1.0 / norm;
        if constexpr (LADDER) {  // the same table for every k
            for (int i = lane; i <= nL; i += 32) ladder_put(a, *L, p, 0, PDA_LADDER_MAX, nL + 1, i, sm.acc[i] * norm);
        } else {
            double* out = a.probs + a.probOff[p];
            for (int i = lane; i <= nL; i += 32) out[i] = sm.acc[i] * norm;
        }
        __syncwarp();
    }

    const bool maximize = a.maximize != 0;
    double CDelta = stage_safe_matrix(Cg, sm.C, n * nc, maximize, true, lane);
    CDelta = CDelta * (double)nc;  // (:583, :664) a separately rounded product
    if (wantW && nc > 1) {
        for (int i = lane; i < nc * (nL + 1); i += 32) sm.acc[i] = 0.0;
    }

    // ---- root: shortestPathCPP on the zero-padded n x n matrix (:119-238) --------------------
    Node<R> nd;
#pragma unroll
    for (int s = 0; s < R; ++s) { nd.v[s] = 0.0; nd.u[s] = 0.0; nd.c4r[s] = -1; nd.r4c[s] = -1; }
    publish_cols<R>(sm, nd, lane);
    unsigned allRows = 0u;
#pragma unroll
    for (int s = 0; s < R; ++s) if (lane + 32 * s < n) allRows |= 1u << s;
    for (int c = 0; c < n; ++c) {
#ifndef PDA_ROOT_FF
#define PDA_ROOT_FF 1
#endif
        const bool stuck = augment_from<R, false, PDA_ROOT_FF != 0>(c, nc, n, sm, nd, allRows, 0u, lane);
        publish_cols<R>(sm, nd, lane);  // the next column starts from this solution
        if (stuck) {
            if constexpr (LADDER) ladder_found(a, *L, p, 0, lane);
            else if (lane == 0) a.nFound[p] = 0;
            if (wantW && nc > 1) {  // the reference ends up scaling zeros by 1/0 here
                double* out = a.probs + a.probOff[p];
                const int len = (LADDER ? L->nSlots : 1) * nc * (nL + 1);  // ladder: the slots lie back to back
                for (int i = lane; i < len; i += 32) out[i] = CUDART_NAN;
            }
            return;
        }
    }
    double gain = path_gain(sm, n, nc);
    unsigned forb = 0u;
    {
        const int r0 = sm.r4c[0];
#pragma unroll
        for (int s = 0; s < R; ++s) if (lane + 32 * s == r0) forb |= 1u << s;
    }
    int activeCol = 0;

    double gain0Out, cutoffGain = a.cutoff;
    bool cutMax = a.cutMaximize != 0;
    if (!maximize) {
        if (a.cutMode == PDA_CUT_RELATIVE) { cutoffGain = gain + a.cutoff; cutMax = false; }
        gain0Out = gain + CDelta;
    } else {
        if (a.cutMode == PDA_CUT_RELATIVE) { cutoffGain = gain - a.cutoff; cutMax = true; }
        gain0Out = -gain + CDelta;
    }
    const bool cutting = a.cutMode != PDA_CUT_NONE;
    const EmitPtrs ep = emit_ptrs(a, p);  // per-problem output bases, fetched once
    emit<R>(ep, 0, n, nc, nd, gain0Out, lane);
    double total = 0.0;
    if (wantW && nc > 1) add_weight<R>(a, sm, nd, nc, nL, gain0Out, gain0Out, total, lane);
    int rungAt = 0, rungK = 0;  // ladder: the next rung to store and its k
    if constexpr (LADDER) {
        rungK = L->rung[0];
        if (nc > 1) ladder_step(a, *L, p, sm, 0, nc * (nL + 1), total, rungAt, rungK, lane);
    }

    int heapLen = FAST ? 0 : 1;   // exact: the root is the heap's only entry (its state is live in registers, slot 0 of
                                  // the arena stays unused); fast: slots in use, the root never enters the list
    int nNodes = 1;
    int sweep = 1;
    int live = 0;                 // fast: open entries (heapLen counts the removed slots as well until a compaction)
    double T = CUDART_INF;        // fast: no hypothesis above T can be among the k best
    int trig = 0;                 // fast: surplus of open entries over hypotheses still wanted that triggers pq_tighten
    bool bail = false;
    for (; sweep < a.k; ++sweep) {
        double limit = CUDART_INF;
        if (FAST) {
            const int m = a.k - sweep;  // hypotheses still to be emitted: sweep .. k-1
            if ((T == CUDART_INF) ? (live >= m) : (live - m >= trig)) {
                PDA_STAT(4, 1); PDA_STAT(5, heapLen);
                pq_tighten(pq, heapLen, live, T, m, lane);
                trig = live - m + PQ_SLACK;
            }
            if (heapLen + nc > pq.cap) { bail = true; break; }
            // children are compared with T through parent gain + search distance: 1e-7 relative is ~1e6 times the
            // rounding that separates that sum from the child's calcGain value
            limit = (T - gain) + 1e-7 * (T + 1.0);
        } else {
            // ---- pop the node whose state we hold (it is the heap top) -----------------------
            if (lane == 0) heap_pop(heap, heapLen);
            heapLen--;
            __syncwarp();
        }

        // ---- split (:455-532) --------------------------------------------------------------
        Node<R> par = nd;
        const unsigned parForb = forb;
        const int a0 = activeCol;
        publish_cols<R>(sm, par, lane);  // the mirrors hold the parent for the whole split
        unsigned inPar = 0u;  // Row2ScanParent: rows paired with columns >= a0
        double uRowPar[R];    // u of the column each row is paired with (fast_forward), the same for every child
#pragma unroll
        for (int s = 0; s < R; ++s) {
            if (lane + 32 * s < n && par.c4r[s] >= a0) inPar |= 1u << s;
            uRowPar[s] = (par.c4r[s] >= 0) ? sm.u[par.c4r[s]] : 0.0;
        }
        for (int c = a0; c < nc; ++c) {
            nd = par;
            unsigned hideFirst = 0u, mine = 0u;  // mine: this lane owns the row that column c gives up
#pragma unroll
            for (int s = 0; s < R; ++s) {
                if (par.c4r[s] == c) {
                    nd.c4r[s] = -1; mine |= 1u << s;
                    sm.c4r[lane + 32 * s] = 0xffffu;  // the freed row is the only sink of this search
                }
                if (lane + 32 * s == c) nd.r4c[s] = -1;
            }
            hideFirst = (c == a0) ? parForb : mine;  // first child inherits every constraint on the active column (:490)
            __syncwarp();
            const int stuck = augment_from<R, FAST>(c, nc, n, sm, nd, inPar, hideFirst, lane, uRowPar, limit);
            if (FAST) { PDA_STAT(0, 1); if (stuck == 2) PDA_STAT(1, 1); }
#pragma unroll
            for (int s = 0; s < R; ++s) if ((mine >> s) & 1u) sm.c4r[lane + 32 * s] = (unsigned short)c;  // the parent's pairing again
            if (!stuck) {
                const double g = path_gain_reg<R>(sm, nd, n, nc, lane);
                bool cut = cutting && (cutMax ? (g < cutoffGain) : (g > cutoffGain));
                if (FAST) { if (!cut && g > T) PDA_STAT(2, 1); cut = cut || (g > T); }
                if (!cut) {
                    if (FAST) PDA_STAT(3, 1);
                    unsigned childForb = hideFirst;
#pragma unroll
                    for (int s = 0; s < R; ++s) if (nd.c4r[s] == c) childForb |= 1u << s;  // the row column c ended up with (:362)
                    node_store<R>(nodes + (size_t)nNodes * a.geo.nodeStride, D, n, nd, childForb, c, lane);
                    if (FAST) {
                        pq_push(pq, heapLen, g, nNodes, lane);
                        live++;
                    } else {
                        if (lane == 0) {
                            HeapEntry e;
                            e.gain = g; e.node = nNodes; e.pad = 0;
                            heap_sift_up(heap, heapLen, e);
                        }
                        heapLen++;
                    }
                    nNodes++;
                }
            }
            inPar &= ~mine;  // column c is fixed from here on
        }
        __syncwarp();
        // ---- the new top is hypothesis number `sweep` (:703-719) ---------------------------
        int topNode;
        if (FAST) {
            if (live == 0) break;
            unsigned long long kb;
            const bool tie = pq_take_min(pq, heapLen, kb, topNode, lane);
            PDA_STAT(6, 1);
            live--;
            if (tie) { bail = true; break; }
            gain = __longlong_as_double((long long)kb);
        } else {
            if (heapLen == 0) break;
            const HeapEntry top = heap.get(0);
            __syncwarp();  // every lane has read the top before lane 0 starts the next pop
            gain = top.gain;
            topNode = top.node;
        }
        node_load<R>(nodes + (size_t)topNode * a.geo.nodeStride, D, n, nd, forb, activeCol, lane);
        double gainOut;
        bool stop = false;
        if (!maximize) {
            gainOut = gain + CDelta;
            if (a.cutMode == PDA_CUT_RELATIVE && gainOut > gain0Out + a.cutoff) stop = true;
        } else {
            gainOut = -gain + CDelta;
            if (a.cutMode == PDA_CUT_RELATIVE && gainOut < gain0Out - a.cutoff) stop = true;
        }
        emit<R>(ep, sweep, n, nc, nd, gainOut, lane);
        if (stop) break;
        if (wantW && nc > 1) add_weight<R>(a, sm, nd, nc, nL, gain0Out, gainOut, total, lane);
        if constexpr (LADDER) {
            if (nc > 1) ladder_step(a, *L, p, sm, sweep, nc * (nL + 1), total, rungAt, rungK, lane);
        }
    }
    if (FAST && bail) {  // not decidable without the reference's heap order (or the list is full): the exact kernel redoes it
        if (lane == 0) a.fallbackList[atomicAdd(a.fallbackCount, 1u)] = (int32_t)p;
        return;
    }
    if constexpr (LADDER) ladder_found(a, *L, p, sweep, lane);
    else if (lane == 0) a.nFound[p] = sweep;
    if (wantW && nc > 1) {
        __syncwarp();
        const double norm = 1.0 / total;
        if constexpr (LADDER) {  // the loop ended (cutoff, empty queue, k): every rung not stored yet gets the final table
            for (int i = lane; i < nc * (nL + 1); i += 32) ladder_put(a, *L, p, rungAt, PDA_LADDER_MAX, nc * (nL + 1), i, sm.acc[i] * norm);
        } else {
            double* out = a.probs + a.probOff[p];
            for (int i = lane; i < nc * (nL + 1); i += 32) out[i] = sm.acc[i] * norm;
        }
        __syncwarp();
    }
}

// Per-warp shared memory: the mirrors first, at offsets that depend only on R (so every access is base + immediate and
// one register carries them all), then the cost matrix and the weight accumulators.
template <int R>
__device__ __forceinline__ WarpSmem carve(unsigned char* base, const MurtyGeometry& g) {
    WarpSmem sm;
    constexpr int D = 32 * R;
    sm.u = reinterpret_cast<double*>(base);
    sm.spc = sm.u + D;
    sm.r4c = reinterpret_cast<short*>(base + 16 * D);
    sm.pred = sm.r4c + D;
    sm.c4r = reinterpret_cast<unsigned short*>(base + 20 * D);
    sm.C = reinterpret_cast<double*>(base + 22 * D);  // 704 R bytes: a multiple of 16
    sm.acc = sm.C + g.cCap;
    return sm;
}

#ifndef PDA_MURTY_LADDER_TU  // murty_ladder_kernel.cu compiles this file for the ladder kernels alone
template <int R, bool FAST>
__global__ void __launch_bounds__(32 * PDA_MURTY_WPC, FAST ? PDA_FAST_MINB : PDA_MURTY_MINB) murty_kernel(const MurtyArgs a) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * (blockDim.x >> 5) + warp;
    if (gw >= a.nWarps) return;
    const int smemPerWarp = FAST ? a.geo.fastSmemPerWarp : a.geo.smemPerWarp;
    unsigned char* mySmem = smemRaw + (size_t)warp * smemPerWarp;
    const WarpSmem sm = carve<R>(mySmem, a.geo);
    unsigned char* arena = a.arena + (size_t)gw * a.geo.arenaStride;
    Heap heap;
    heap.deep = reinterpret_cast<HeapEntry*>(arena);
    heap.top = reinterpret_cast<HeapEntry*>(mySmem + a.geo.heapTopOff);
    heap.topCap = a.geo.heapTopCap;
    FastPQ pq;
    pq.cap = a.geo.pqCap;
    pq.gmin = reinterpret_cast<unsigned long long*>(mySmem + a.geo.heapTopOff);
    if (a.geo.pqInSmem) {
        pq.key = pq.gmin + (a.geo.pqCap >> 5);
        pq.node = reinterpret_cast<int*>(pq.key + a.geo.pqCap);
    } else {  // the arena's heap region is free in this kernel
        pq.key = reinterpret_cast<unsigned long long*>(arena);
        pq.node = reinterpret_cast<int*>(pq.key + a.geo.pqCap);
    }
    pq.hist = reinterpret_cast<unsigned*>(sm.spc);
    unsigned char* nodes = arena + a.geo.heapBytes;
    // the exact kernel, when it runs behind the fast one, takes its problem count from the fallback counter
    const long long nProblems = a.nProblemsDev ? (long long)*a.nProblemsDev : a.nProblems;
    for (;;) {
        unsigned long long p = 0;
        if (lane == 0) p = atomicAdd(a.cursor, 1ULL);
        p = __shfl_sync(FULL, p, 0);
        if ((long long)p >= nProblems) break;
        if (a.order) p = (unsigned long long)a.order[p];  // most expensive problems first: a short tail
        solve_problem<R, FAST>(a, (long long)p, sm, heap, pq, nodes, lane);
        __syncwarp();
    }
}

// Longest-processing-time-first order for the work cursor.  A problem's cost grows with its number of detections
// (children per pop), so a counting sort by numCol, descending, is enough: the persistent warps then finish on the
// cheapest problems and run dry almost together.  One CTA; ~30 us for 100 000 problems.
__global__ void order_by_cost_kernel(const int32_t* __restrict__ numCol, const long long n, int32_t* __restrict__ order) {
    __shared__ unsigned bucket[PDA_MAX_DIM + 2];
    for (int i = threadIdx.x; i < PDA_MAX_DIM + 2; i += blockDim.x) bucket[i] = 0u;
    __syncthreads();
    for (long long p = threadIdx.x; p < n; p += blockDim.x) {
        int key = numCol[p];
        key = key < 0 ? 0 : (key > PDA_MAX_DIM ? PDA_MAX_DIM : key);
        atomicAdd(&bucket[key], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // exclusive prefix over keys in DESCENDING order
        unsigned run = 0;
        for (int key = PDA_MAX_DIM; key >= 0; --key) { const unsigned c = bucket[key]; bucket[key] = run; run += c; }
    }
    __syncthreads();
    for (long long p = threadIdx.x; p < n; p += blockDim.x) {
        int key = numCol[p];
        key = key < 0 ? 0 : (key > PDA_MAX_DIM ? PDA_MAX_DIM : key);
        order[atomicAdd(&bucket[key], 1u)] = (int32_t)p;
    }
}

// ---- plain LAP (assign2D / shortestPathCPP on a rectangular matrix, no padding) ---------------------
template <int R>
__global__ void lap_kernel(const LapArgs a, const int smemPerWarp, const int cCap) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long p = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (p >= a.nProblems) return;
    MurtyGeometry g;
    g.R = R; g.cCap = cCap; g.pCap = 0;
    const WarpSmem sm = carve<R>(smemRaw + (size_t)warp * smemPerWarp, g);
    const int n = a.numRow[p], nc = a.numCol[p];
    const int ncGain = a.numCol4Gain ? a.numCol4Gain[p] : nc;
    if (nc < 0 || nc > n || n > a.maxNumRow || nc > a.maxNumCol || n > 32 * R || n * nc > cCap) {  // malformed or beyond the declared maxima
        if (lane == 0 && a.feasible) a.feasible[p] = 0;
        return;
    }
    double CDelta = stage_safe_matrix(a.costs + a.costOff[p], sm.C, n * nc, a.maximize != 0, a.makeSafe != 0, lane);
    // n x 0: the extremum of no entries is +-inf, and inf * 0 would turn the gain (a sum of no terms) into NaN
    CDelta = nc > 0 ? CDelta * (double)nc : 0.0;
    Node<R> nd;
#pragma unroll
    for (int s = 0; s < R; ++s) { nd.v[s] = 0.0; nd.u[s] = 0.0; nd.c4r[s] = -1; nd.r4c[s] = -1; }
    publish_cols<R>(sm, nd, lane);
    unsigned allRows = 0u;
#pragma unroll
    for (int s = 0; s < R; ++s) if (lane + 32 * s < n) allRows |= 1u << s;
    bool infeasible = false;
    for (int c = 0; c < nc && !infeasible; ++c) {
        infeasible = augment_from<R>(c, nc, n, sm, nd, allRows, 0u, lane);
        publish_cols<R>(sm, nd, lane);
    }
    double gain = -1.0;
    int r0 = -1;
    if (!infeasible) {
        gain = path_gain(sm, n, ncGain);
        if (a.makeSafe) gain = a.maximize ? (-gain + CDelta) : (gain + CDelta);
        if (nc > 0) r0 = sm.r4c[0];
    }
    const int64_t ro = a.rowOff[p], co = a.colOff[p];
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int i = lane + 32 * s;
        if (i < n) {
            if (a.col4row) a.col4row[ro + i] = nd.c4r[s];
            if (a.v) a.v[ro + i] = nd.v[s];
            if (a.forbidden) a.forbidden[ro + i] = (i == r0) ? 1 : 0;
        }
        if (i < nc) {
            if (a.row4col) a.row4col[co + i] = nd.r4c[s];
            if (a.u) a.u[co + i] = nd.u[s];
        }
    }
    if (lane == 0) {
        if (a.gain) a.gain[p] = gain;
        if (a.feasible) a.feasible[p] = infeasible ? 0 : 1;
    }
}

}  // namespace

// ---- host side ------------------------------------------------------------------------------------
static int round_up(int x, int m) { return (x + m - 1) / m * m; }

template <int R, bool FAST>
static int occupancy_one(int smemPerWarp, const DeviceInfo& dev, int* wpcOut, int* occOut) {
    int wpc = PDA_MURTY_WPC;
    while (wpc > 1 && wpc * smemPerWarp > dev.maxSmemOptin) wpc >>= 1;
    const size_t smem = (size_t)wpc * smemPerWarp;
    int occ = 0;
    cudaError_t e = cudaFuncSetAttribute(murty_kernel<R, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, murty_kernel<R, FAST>, 32 * wpc, smem);
    if (e != cudaSuccess) return cuda_fail(e, "occupancy query for murty_kernel");
    *wpcOut = wpc;
    *occOut = occ < 1 ? 1 : occ;
    return PDA_OK;
}
template <int R>
static int occupancy_r(MurtyGeometry* g, const DeviceInfo& dev) {
    int rc = occupancy_one<R, false>(g->smemPerWarp, dev, &g->warpsPerCta, &g->ctasPerSm);
    if (rc) return rc;
    g->fastWarpsPerCta = g->warpsPerCta;
    g->fastCtasPerSm = g->ctasPerSm;
    if (g->fastOk) rc = occupancy_one<R, true>(g->fastSmemPerWarp, dev, &g->fastWarpsPerCta, &g->fastCtasPerSm);
    return rc;
}

int murty_geometry(int32_t k, int32_t maxNumRow, int32_t maxNumCol, bool weights, const DeviceInfo& dev,
                   MurtyGeometry* g) {
    if (k < 1 || maxNumRow < 1 || maxNumCol < 1 || maxNumCol > maxNumRow)
        return fail(PDA_ERR_INVALID, "murty: need k >= 1 and 1 <= maxNumCol <= maxNumRow (got k=%d, %d x %d)", k, maxNumRow, maxNumCol);
    if (maxNumRow > PDA_MAX_DIM)
        return fail(PDA_ERR_UNSUPPORTED, "murty: numRow %d exceeds PDA_MAX_DIM %d", maxNumRow, PDA_MAX_DIM);
    g->R = (maxNumRow + 31) / 32;
    if (g->R == 3) g->R = 4;
    g->maxCol = maxNumCol;
    const int D = 32 * g->R;
    g->nodeDim = round_up(maxNumRow, 8);
    g->nodeStride = round_up(18 * g->nodeDim + 4 * (g->R + 1), 16);
    const int64_t nodes = 1 + (int64_t)(k - 1) * maxNumCol;  // every pop creates at most numCol children
    if (nodes > (int64_t)1 << 30) return fail(PDA_ERR_UNSUPPORTED, "murty: k * numCol too large");
    g->maxNodes = (int)nodes;
    g->heapBytes = (int64_t)round_up((int)nodes, 8) * (int64_t)sizeof(HeapEntry);
    g->arenaStride = (g->heapBytes + nodes * g->nodeStride + 255) / 256 * 256;
    g->cCap = round_up(maxNumRow * maxNumCol, 2);
    g->pCap = weights ? round_up(maxNumCol * maxNumRow, 2) : 0;
    const int baseSmem = round_up(8 * (g->cCap + g->pCap + 2 * D) + 3 * 2 * D, 16);
    // leftover shared memory (at the warps per SM the register budget allows) holds the top of the heap
    const int budget = (227 * 1024 - PDA_MURTY_MINB * 1024) / (PDA_MURTY_WPC * PDA_MURTY_MINB);
    int topCap = budget > baseSmem ? (budget - baseSmem) / (int)sizeof(HeapEntry) : 0;
    if (topCap > g->maxNodes) topCap = g->maxNodes;
    if (topCap < 3) topCap = 0;
    g->heapTopOff = baseSmem;
    g->heapTopCap = topCap;
    g->smemPerWarp = baseSmem + topCap * (int)sizeof(HeapEntry);
    // the pruning fast path (murty_kernel<R, true>): its open list never holds more than k + slack entries, so it lives
    // in shared memory when that fits the same per-warp budget, else in the arena's heap region (group minima stay in
    // shared memory either way).  Not offered for k <= 2 (nothing to prune) or lists beyond 64 groups.
    g->pqCap = round_up(k + 2 * maxNumCol + PQ_SLACK + 32, 32);
    g->fastOk = (k > 2 && g->pqCap <= 64 * 32 && (int64_t)g->pqCap * 12 <= g->heapBytes) ? 1 : 0;
    const int fastBudget = (227 * 1024 - PDA_FAST_MINB * 1024) / (PDA_MURTY_WPC * PDA_FAST_MINB);
    g->pqInSmem = (baseSmem + g->pqCap * 12 + (g->pqCap >> 5) * 8 <= fastBudget) ? 1 : 0;
    g->fastSmemPerWarp = round_up(baseSmem + (g->pqCap >> 5) * 8 + (g->pqInSmem ? g->pqCap * 12 : 0), 16);
    if (g->smemPerWarp > dev.maxSmemOptin)
        return fail(PDA_ERR_UNSUPPORTED, "murty: a %d x %d problem needs %d B of shared memory per warp (limit %d)",
                    maxNumRow, maxNumCol, g->smemPerWarp, dev.maxSmemOptin);
    if (g->fastSmemPerWarp > dev.maxSmemOptin) g->fastOk = 0;
    // resident CTAs per SM, as the occupancy calculator sees each instantiation (registers, shared memory)
    int rc = PDA_OK;
    switch (g->R) {
        case 1: rc = occupancy_r<1>(g, dev); break;
        case 2: rc = occupancy_r<2>(g, dev); break;
        default: rc = occupancy_r<4>(g, dev); break;
    }
    return rc;
}

template <int R, bool FAST>
static int launch_murty_r(const MurtyArgs& a, cudaStream_t stream, const MurtyLadder* ladder) {
    const int wpc = FAST ? a.geo.fastWarpsPerCta : a.geo.warpsPerCta;
    const int threads = 32 * wpc;
    const int smem = wpc * (FAST ? a.geo.fastSmemPerWarp : a.geo.smemPerWarp);
    if (ladder) return launch_murty_ladder(a, FAST, *ladder, wpc, smem, stream);
    PDA_CUDA_TRY(cudaFuncSetAttribute(murty_kernel<R, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int ctas = (a.nWarps + wpc - 1) / wpc;
    murty_kernel<R, FAST><<<ctas, threads, smem, stream>>>(a);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

template <bool FAST>
static int launch_murty_any(const MurtyArgs& a, cudaStream_t stream, const MurtyLadder* ladder) {
    switch (a.geo.R) {
        case 1: return launch_murty_r<1, FAST>(a, stream, ladder);
        case 2: return launch_murty_r<2, FAST>(a, stream, ladder);
        case 4: return launch_murty_r<4, FAST>(a, stream, ladder);
    }
    return fail(PDA_ERR_UNSUPPORTED, "murty: unsupported row-slot count %d", a.geo.R);
}

#ifdef PDA_FAST_STATS
extern "C" void pda_debug_fast_stats(unsigned long long* out, int reset) {
    cudaMemcpyFromSymbol(out, g_fastStats, sizeof(unsigned long long) * 8);
    cudaMemcpyFromSymbol(out + 8, g_augStats, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_fastStats, z, sizeof(z)); cudaMemcpyToSymbol(g_augStats, z, sizeof(z)); }
}
#endif

int launch_murty(const MurtyArgs& a, cudaStream_t stream, const MurtyLadder* ladder) {
    // header of the workspace: cursor (8 B) | fallback count (4 B, +4 pad) | cursor of the fallback pass (8 B)
    PDA_CUDA_TRY(cudaMemsetAsync(a.cursor, 0, 32, stream));
    if (a.order) {
        order_by_cost_kernel<<<1, 1024, 0, stream>>>(a.numCol, a.nProblems, a.order);
        PDA_CUDA_TRY(cudaGetLastError());
    }
    if (!a.useFast) return launch_murty_any<false>(a, stream, ladder);
    int rc = launch_murty_any<true>(a, stream, ladder);
    if (rc) return rc;
    // the exact kernel over whatever the fast one could not decide (usually nothing: it then finds a count of zero); a
    // ladder problem it redoes gets every rung rewritten, with the same bits where the fast kernel had stored one
    MurtyArgs b = a;
    b.useFast = 0;
    b.cursor = a.cursor2;
    b.order = a.fallbackList;
    b.nProblemsDev = a.fallbackCount;
    return launch_murty_any<false>(b, stream, ladder);
}

template <int R>
static int launch_lap_r(const LapArgs& a, cudaStream_t stream, const DeviceInfo& dev) {
    const int D = 32 * R;
    const int cCap = round_up(a.maxNumRow * a.maxNumCol, 2);
    const int smemPerWarp = round_up(8 * (cCap + 2 * D) + 6 * D, 16);
    if (smemPerWarp > dev.maxSmemOptin) return fail(PDA_ERR_UNSUPPORTED, "lap: matrix too large for shared memory");
    int wpc = 4;
    while (wpc > 1 && wpc * smemPerWarp > dev.maxSmemOptin) wpc >>= 1;
    const int smem = wpc * smemPerWarp;
    PDA_CUDA_TRY(cudaFuncSetAttribute(lap_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const long long ctas = (a.nProblems + wpc - 1) / wpc;
    lap_kernel<R><<<(unsigned)ctas, 32 * wpc, smem, stream>>>(a, smemPerWarp, cCap);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int launch_lap(const LapArgs& a, cudaStream_t stream) {
    DeviceInfo dev;
    int rc = current_device_info(&dev);
    if (rc) return rc;
    if (a.maxNumRow > PDA_MAX_DIM) return fail(PDA_ERR_UNSUPPORTED, "lap: numRow %d exceeds PDA_MAX_DIM", a.maxNumRow);
    const int R = (a.maxNumRow + 31) / 32;
    if (R <= 1) return launch_lap_r<1>(a, stream, dev);
    if (R == 2) return launch_lap_r<2>(a, stream, dev);
    return launch_lap_r<4>(a, stream, dev);
}

#else
// The k-ladder form: same geometry, same launch shape, the same loop over problems as murty_kernel.  (The loop is
// written out twice rather than shared through an inlined helper: with the helper, the code of murty_kernel<4, *> moves.)
template <int R, bool FAST>
__global__ void __launch_bounds__(32 * PDA_MURTY_WPC, FAST ? PDA_FAST_MINB : PDA_MURTY_MINB)
    murty_ladder_kernel(const MurtyArgs a, const __grid_constant__ MurtyLadder L) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * (blockDim.x >> 5) + warp;
    if (gw >= a.nWarps) return;
    const int smemPerWarp = FAST ? a.geo.fastSmemPerWarp : a.geo.smemPerWarp;
    unsigned char* mySmem = smemRaw + (size_t)warp * smemPerWarp;
    const WarpSmem sm = carve<R>(mySmem, a.geo);
    unsigned char* arena = a.arena + (size_t)gw * a.geo.arenaStride;
    Heap heap;
    heap.deep = reinterpret_cast<HeapEntry*>(arena);
    heap.top = reinterpret_cast<HeapEntry*>(mySmem + a.geo.heapTopOff);
    heap.topCap = a.geo.heapTopCap;
    FastPQ pq;
    pq.cap = a.geo.pqCap;
    pq.gmin = reinterpret_cast<unsigned long long*>(mySmem + a.geo.heapTopOff);
    if (a.geo.pqInSmem) {
        pq.key = pq.gmin + (a.geo.pqCap >> 5);
        pq.node = reinterpret_cast<int*>(pq.key + a.geo.pqCap);
    } else {  // the arena's heap region is free in this kernel
        pq.key = reinterpret_cast<unsigned long long*>(arena);
        pq.node = reinterpret_cast<int*>(pq.key + a.geo.pqCap);
    }
    pq.hist = reinterpret_cast<unsigned*>(sm.spc);
    unsigned char* nodes = arena + a.geo.heapBytes;
    // the exact kernel, when it runs behind the fast one, takes its problem count from the fallback counter
    const long long nProblems = a.nProblemsDev ? (long long)*a.nProblemsDev : a.nProblems;
    for (;;) {
        unsigned long long p = 0;
        if (lane == 0) p = atomicAdd(a.cursor, 1ULL);
        p = __shfl_sync(FULL, p, 0);
        if ((long long)p >= nProblems) break;
        if (a.order) p = (unsigned long long)a.order[p];  // most expensive problems first: a short tail
        solve_problem<R, FAST, true>(a, (long long)p, sm, heap, pq, nodes, lane, &L);
        __syncwarp();
    }
}

}  // namespace

int launch_murty_ladder(const MurtyArgs& a, const bool fast, const MurtyLadder& ladder, const int wpc, const int smem,
                        cudaStream_t stream) {
    const int ctas = (a.nWarps + wpc - 1) / wpc;
    void (*k)(const MurtyArgs, const MurtyLadder) = nullptr;
    switch (a.geo.R * 2 + (fast ? 1 : 0)) {
        case 2: k = murty_ladder_kernel<1, false>; break;
        case 3: k = murty_ladder_kernel<1, true>; break;
        case 4: k = murty_ladder_kernel<2, false>; break;
        case 5: k = murty_ladder_kernel<2, true>; break;
        case 8: k = murty_ladder_kernel<4, false>; break;
        case 9: k = murty_ladder_kernel<4, true>; break;
        default: return fail(PDA_ERR_UNSUPPORTED, "murty: unsupported row-slot count %d", a.geo.R);
    }
    PDA_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k<<<ctas, 32 * wpc, smem, stream>>>(a, ladder);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}
#endif  // PDA_MURTY_LADDER_TU

}  // namespace pda
