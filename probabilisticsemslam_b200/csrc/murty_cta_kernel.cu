// murty_cta_kernel.cu -- Murty k-best for FEW problems: one CTA (16 warps) per problem.
//
// The throughput kernel (murty_kernel.cu) gives a problem to a single warp; that is the right shape
// for 100 000 problems, but a single problem -- what the SLAM loop submits once per frame
// (system.cpp:268, slidingWindow.cpp:339) and what compMethods times (comparison.cpp:194-222) --
// then runs at the latency of one warp: ~5 us per sweep, ~1 ms at k = 200.  This kernel keeps the
// same arithmetic (the same augment_from / heap / node format from murty_device.cuh, so results are
// bit-identical to the warp kernel and to the reference) but runs the k-best loop as
// out-of-order execution with in-order commit:
//
//   * a node's split (shortestPathCPP.cpp:455-532) depends only on the node itself, so it can be done
//     BEFORE the node reaches the top of the queue.  Warp 0 picks the cheapest not-yet-split nodes among
//     the first 32 heap entries (the top itself first) and turns each (node, child column) pair into a
//     task; warps 1-15 solve the tasks (one Dijkstra each) in the NEXT round and leave the children's
//     gains in a split record in shared memory;
//   * warp 0 replays the reference's loop strictly in order -- pop, push the popped node's children in
//     column order, read the new top -- for as long as the top's split record exists and is not being
//     solved in the current round.  The heap therefore sees exactly the reference's sequence of push/pop
//     operations, including the order among exactly equal gains.  Commit and child solves overlap: task
//     lists, done flags and in-flight masks are double-buffered by round parity, one barrier per round.
//   On the KITTI-shaped problems ~97 % of the speculated splits are consumed (a node close to the top
//   is almost always popped within the next few sweeps): 199 sweeps are committed in ~23 bursts, each
//   ended by a freshly created child becoming the top (its split cannot have been computed ahead).
//   * lists and weights are written at the end, by all warps, from the recorded pop order; weights are
//     accumulated per table entry in hypothesis order, i.e. in the reference's order (assignment.cpp:620-640).
#include "murty_device.cuh"

namespace pda {
#ifdef PDA_CTA_PROFILE
__device__ long long g_prof[16];
__device__ long long g_trace[64 * 4];  // per round: warp-0 cycles, warp-1 task cycles, tasks, sweep after the round
#endif
namespace {

constexpr int CTA_WARPS = 16;
constexpr int CTA_RECORDS = 64;             // split records (splits done but not yet committed)
#ifndef PDA_CTA_MAXTASKS
#define PDA_CTA_MAXTASKS 48
#endif
#ifndef PDA_CTA_SPEC
#define PDA_CTA_SPEC 16
#endif
#ifndef PDA_CTA_AHEAD
#define PDA_CTA_AHEAD 8
#endif
constexpr int CTA_MAXTASKS = PDA_CTA_MAXTASKS;  // child solves per round
constexpr int CTA_SPEC = PDA_CTA_SPEC;         // nodes split per round, at most
constexpr int CTA_AHEAD = PDA_CTA_AHEAD;       // no new picks while this many splits are waiting to be committed and the top is one of them

struct Task {
    int parent;  // node whose split this child belongs to
    int child;   // arena slot for the child
    short c;     // the child's active column
    short rec;   // split record
};

struct CtaCtl {
    double CDelta, gain0Out, cutoffGain;
    unsigned long long freeRec;  // bit r set = record r is free
    long long problem;
    int heapLen, sweep, nNodes, nFound, nEmit, uncommitted, cutMax, cutting, feasible;
    int nTasks[2];  // task list r&1 is executed in round r and was filled by warp 0 during round r-1
    int done[2];    // done[r&1] is written by warp 0 during round r and read by everybody after that round's barrier
    unsigned long long flight[2];  // flight[r&1]: records whose children are being solved during round r
#ifdef PDA_CTA_PROFILE
    long long tCommit, tSelect, tTasks, tRoot, tFinal, t0, ns0, tPop, tPush;
    int rounds, tasksTotal, commits;
#endif
};
#ifdef PDA_CTA_PROFILE
#define PROF_T() clock64()
#else
#define PROF_T() 0LL
#endif

// HeapEntry::pad of this kernel: bits 0-7 activeCol, bits 8-23 split record + 1 (0 = not split yet)
__device__ __forceinline__ int pad_active(int pad) { return pad & 0xff; }
__device__ __forceinline__ int pad_record(int pad) { return (pad >> 8) & 0xffff; }

struct CtaSmem {
    double* C;
    double* acc;
    unsigned char* mirrors;  // CTA_WARPS x mirrorBytes
    double* recGain;         // [CTA_RECORDS][PDA_CTA_MAX_COL]
    int* recBase;            // [CTA_RECORDS]
    Task* tasks;             // [2][CTA_MAXTASKS]
    CtaCtl* ctl;
    HeapEntry* heapTop;
};

__device__ __forceinline__ CtaSmem carve_cta(unsigned char* base, const MurtyGeometry& g, const CtaGeometry& cg) {
    CtaSmem s;
    s.C = reinterpret_cast<double*>(base);
    s.acc = s.C + g.cCap;
    s.mirrors = reinterpret_cast<unsigned char*>(s.acc + g.pCap);
    s.recGain = reinterpret_cast<double*>(s.mirrors + (size_t)CTA_WARPS * cg.mirrorBytes);
    s.recBase = reinterpret_cast<int*>(s.recGain + CTA_RECORDS * PDA_CTA_MAX_COL);
    s.tasks = reinterpret_cast<Task*>(s.recBase + CTA_RECORDS);
    s.ctl = reinterpret_cast<CtaCtl*>(base + cg.ctlOff);
    s.heapTop = reinterpret_cast<HeapEntry*>(base + cg.heapTopOff);
    return s;
}

__device__ __forceinline__ WarpSmem warp_view(const CtaSmem& s, const CtaGeometry& cg, const int R, const int warp) {
    WarpSmem sm;
    const int D = 32 * R;
    unsigned char* m = s.mirrors + (size_t)warp * cg.mirrorBytes;
    sm.C = s.C;
    sm.acc = s.acc;
    sm.u = reinterpret_cast<double*>(m);
    sm.spc = sm.u + D;
    sm.r4c = reinterpret_cast<short*>(sm.spc + D);
    sm.pred = sm.r4c + D;
    sm.c4r = reinterpret_cast<unsigned short*>(sm.pred + D);
    return sm;
}

// per-problem global scratch behind the heap
struct CtaArena {
    HeapEntry* heapDeep;
    double* orderGain;     // [k] reported gain of hypothesis i
    double* orderW;        // [k] its weight
    int* orderNode;        // [k] arena slot holding hypothesis i
    unsigned char* hypRows;  // [k][PDA_CTA_MAX_COL] row4col of hypothesis i, one byte each
    unsigned char* nodes;
};
__device__ __forceinline__ CtaArena carve_arena(unsigned char* base, const CtaGeometry& cg, const int k) {
    CtaArena A;
    A.heapDeep = reinterpret_cast<HeapEntry*>(base);
    A.orderGain = reinterpret_cast<double*>(base + cg.heapBytes);
    A.orderW = A.orderGain + k;
    A.orderNode = reinterpret_cast<int*>(A.orderW + k);
    A.hypRows = reinterpret_cast<unsigned char*>(A.orderNode + ((k + 3) & ~3));
    A.nodes = base + cg.nodesOff;
    return A;
}

// ---- the commit lane's heap ---------------------------------------------------------------------------
// Same array, same libstdc++ moves as heap_pop / heap_sift_up in murty_device.cuh, tuned for ONE lane whose every
// dependent load is exposed latency (the other 15 warps wait for it): entries move as one 128-bit access, gains
// compare as integers (they are sums of entries of the shifted matrix, hence >= +0.0, where the bit pattern orders
// like the value), and the sift-down looks two levels ahead -- the children and the four grandchildren come back
// from one round trip to shared memory, which halves the chain of dependent loads of a pop.
struct FastHeap {
    int4* top;
    int4* deep;
    int topCap;
    __device__ __forceinline__ int4 get(int i) const { return (i < topCap) ? top[i] : deep[i]; }
    __device__ __forceinline__ void put(int i, const int4 e) const { if (i < topCap) top[i] = e; else deep[i] = e; }
};
__device__ __forceinline__ long long ekey(const int4 e) { return ((long long)e.y << 32) | (unsigned)e.x; }
__device__ __forceinline__ int4 make_entry(double gain, int node, int pad) {
    return make_int4(__double2loint(gain), __double2hiint(gain), node, pad);
}
__device__ __forceinline__ double entry_gain(const int4 e) { return __hiloint2double(e.y, e.x); }

__device__ __forceinline__ void fast_sift_up(const FastHeap& h, int hole, const int4 val) {
    const long long kv = ekey(val);
    while (hole > 0) {
        const int p1 = (hole - 1) / 2, p2 = (p1 - 1) / 2;  // p2 == 0 when p1 == 0 (C++ division truncates)
        const int4 e1 = h.get(p1), e2 = h.get(p2);
        if (!(ekey(e1) > kv)) break;
        h.put(hole, e1);
        hole = p1;
        if (p1 == 0 || !(ekey(e2) > kv)) break;
        h.put(hole, e2);
        hole = p2;
    }
    h.put(hole, val);
}
__device__ __forceinline__ void fast_pop(const FastHeap& h, const int lenBefore) {
    if (lenBefore <= 1) return;
    const int len = lenBefore - 1;
    const int4 val = h.get(len);
    int hole = 0, child = 0;
    while (4 * child + 6 < len) {  // both children of `child` have two children of their own: two levels per round trip
        const int a = 2 * child + 1;
        const int4 ea = h.get(a), eb = h.get(a + 1);
        const int4 e0 = h.get(2 * a + 1), e1 = h.get(2 * a + 2), e2 = h.get(2 * a + 3), e3 = h.get(2 * a + 4);
        const bool left1 = ekey(eb) > ekey(ea);  // the right child wins an exact tie
        const int n1 = left1 ? a : a + 1;
        const int4 gl = left1 ? e0 : e2, gr = left1 ? e1 : e3;
        const bool left2 = ekey(gr) > ekey(gl);
        const int n2 = 2 * n1 + (left2 ? 1 : 2);
        h.put(hole, left1 ? ea : eb);
        h.put(n1, left2 ? gl : gr);
        hole = n2;
        child = n2;
    }
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        const int4 right = h.get(child), left = h.get(child - 1);
        const bool takeLeft = ekey(right) > ekey(left);
        if (takeLeft) child--;
        h.put(hole, takeLeft ? left : right);
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        h.put(hole, h.get(child - 1));
        hole = child - 1;
    }
    fast_sift_up(h, hole, val);
}

// The same two routines when the whole heap fits in shared memory (k = 200 and k = 1000 at 8 detections do): keys
// are read as 64-bit loads, only indices are selected on, and an entry moves with one LDS.128 + STS.128 off the
// dependent chain -- ~30 instructions per two levels instead of ~70, and the lane pays ~3.6 cycles per instruction.
__device__ __forceinline__ long long skey(const int4* top, int i) { return reinterpret_cast<const long long*>(top)[2 * i]; }
__device__ __forceinline__ void smem_sift_up(int4* top, int hole, const int4 val) {
    const long long kv = ekey(val);
    while (hole > 0) {
        const int p1 = (hole - 1) / 2, p2 = (p1 - 1) / 2;
        const long long k1 = skey(top, p1), k2 = skey(top, p2);
        if (!(k1 > kv)) break;
        top[hole] = top[p1];
        hole = p1;
        if (p1 == 0 || !(k2 > kv)) break;
        top[hole] = top[p2];
        hole = p2;
    }
    top[hole] = val;
}
__device__ __forceinline__ void smem_pop(int4* top, const int lenBefore) {
    if (lenBefore <= 1) return;
    const int len = lenBefore - 1;
    const int4 val = top[len];
    int hole = 0, child = 0;
    while (4 * child + 6 < len) {
        const int a = 2 * child + 1;
        const long long ka = skey(top, a), kb = skey(top, a + 1);
        const long long k0 = skey(top, 2 * a + 1), k1 = skey(top, 2 * a + 2), k2 = skey(top, 2 * a + 3), k3 = skey(top, 2 * a + 4);
        const bool left1 = kb > ka;  // the right child wins an exact tie
        const int n1 = left1 ? a : a + 1;
        const long long gl = left1 ? k0 : k2, gr = left1 ? k1 : k3;
        const int n2 = 2 * n1 + ((gr > gl) ? 1 : 2);
        top[hole] = top[n1];
        top[n1] = top[n2];
        hole = n2;
        child = n2;
    }
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (skey(top, child) > skey(top, child - 1)) child--;
        top[hole] = top[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        top[hole] = top[child - 1];
        hole = child - 1;
    }
    smem_sift_up(top, hole, val);
}

// ---- warp 0: staging, single-detection shortcut, root LAP (shortestPathCPP.cpp:119-238) ---------------
template <int R, bool LADDER, class... Ladder>  // the ladder as in solve_problem_cta
__device__ void root_phase(const MurtyArgs& a, const long long p, const CtaSmem& S, const WarpSmem& sm, const Heap& heap,
                           const CtaArena& A, const int lane, const Ladder*... ladder) {
    const MurtyLadder* L = nullptr;
    if constexpr (LADDER) ((L = ladder), ...);
    CtaCtl* ctl = S.ctl;
    const int n = a.numRow[p], nc = a.numCol[p];
    const int D = a.geo.nodeDim;
    const bool wantW = a.weightMode != PDA_WEIGHTS_NONE;
    const int nL = wantW ? a.nL[p] : 0;
    const double* Cg = a.costs + a.costOff[p];
    if (wantW && nc == 1) {  // assignment.cpp:554-570, 840-856
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
    CDelta = CDelta * (double)nc;
    Node<R> nd;
#pragma unroll
    for (int s = 0; s < R; ++s) { nd.v[s] = 0.0; nd.u[s] = 0.0; nd.c4r[s] = -1; nd.r4c[s] = -1; }
    publish_cols<R>(sm, nd, lane);
    unsigned allRows = 0u;
#pragma unroll
    for (int s = 0; s < R; ++s) if (lane + 32 * s < n) allRows |= 1u << s;
    for (int c = 0; c < n; ++c) {
        const bool stuck = augment_from<R>(c, nc, n, sm, nd, allRows, 0u, lane);
        publish_cols<R>(sm, nd, lane);  // the next column starts from this solution
        if (stuck) {
            if constexpr (LADDER) {
                ladder_found(a, *L, p, 0, lane);
                if (lane == 0) { ctl->feasible = 0; ctl->done[0] = ctl->done[1] = 1; ctl->nFound = 0; ctl->nEmit = 0; }
            } else {
                if (lane == 0) { a.nFound[p] = 0; ctl->feasible = 0; ctl->done[0] = ctl->done[1] = 1; ctl->nFound = 0; ctl->nEmit = 0; }
            }
            if (wantW && nc > 1) {
                double* out = a.probs + a.probOff[p];
                const int len = (LADDER ? L->nSlots : 1) * nc * (nL + 1);  // ladder: the slots lie back to back
                for (int i = lane; i < len; i += 32) out[i] = CUDART_NAN;
            }
            return;
        }
    }
    const double gain = path_gain(sm, n, nc);
    unsigned forb = 0u;
    {
        const int r0 = sm.r4c[0];
#pragma unroll
        for (int s = 0; s < R; ++s) if (lane + 32 * s == r0) forb |= 1u << s;
    }
    double gain0Out, cutoffGain = a.cutoff;
    bool cutMax = a.cutMaximize != 0;
    if (!maximize) {
        if (a.cutMode == PDA_CUT_RELATIVE) { cutoffGain = gain + a.cutoff; cutMax = false; }
        gain0Out = gain + CDelta;
    } else {
        if (a.cutMode == PDA_CUT_RELATIVE) { cutoffGain = gain - a.cutoff; cutMax = true; }
        gain0Out = -gain + CDelta;
    }
    node_store<R>(A.nodes, D, n, nd, forb, 0, lane);
    if (lane == 0) {
        HeapEntry e;
        e.gain = gain; e.node = 0; e.pad = 0;
        heap.put(0, e);
        A.orderNode[0] = 0;
        A.orderGain[0] = gain0Out;
        ctl->CDelta = CDelta; ctl->gain0Out = gain0Out; ctl->cutoffGain = cutoffGain;
        ctl->cutMax = cutMax ? 1 : 0; ctl->cutting = a.cutMode != PDA_CUT_NONE;
        ctl->freeRec = ~0ULL;
        ctl->heapLen = 1; ctl->sweep = 1; ctl->nNodes = 1; ctl->nTasks[0] = ctl->nTasks[1] = 0; ctl->uncommitted = 0; ctl->flight[0] = ctl->flight[1] = 0ULL;
        ctl->feasible = 1;
        ctl->done[0] = ctl->done[1] = (a.k <= 1) ? 1 : 0;
        ctl->nFound = 1; ctl->nEmit = 1;
    }
}

// ---- warp 0, every round: commit in order, then choose the next splits -------------------------------
__device__ void serial_phase(const MurtyArgs& a, const CtaGeometry& cg, const CtaSmem& S, const Heap& heap,
                             const CtaArena& A, const int nc, const int round, const int lane) {
    CtaCtl* ctl = S.ctl;
    const long long tc0 = PROF_T();
    FastHeap fh;
    fh.top = reinterpret_cast<int4*>(heap.top); fh.deep = reinterpret_cast<int4*>(heap.deep); fh.topCap = heap.topCap;
    const bool allTop = cg.heapTopCap >= cg.maxNodes;
    if (lane == 0) {
        int heapLen = ctl->heapLen, sweep = ctl->sweep, uncommitted = ctl->uncommitted;
        unsigned long long freeRec = ctl->freeRec;
        const bool maximize = a.maximize != 0;
        const double CDelta = ctl->CDelta, gain0Out = ctl->gain0Out;
        const unsigned long long flight = ctl->flight[round & 1];
        int done = 0;
        int4 top = fh.get(0);
        while (sweep < a.k) {
            const int rec = pad_record(top.w);
            if (rec == 0 || ((flight >> (rec - 1)) & 1ULL)) break;  // the top is not split yet, or its children are being solved right now
            const int a0 = pad_active(top.w), cnt = nc - a0;
#ifdef PDA_CTA_PROFILE
            const long long tp0 = PROF_T();
#endif
            if (allTop) smem_pop(fh.top, heapLen); else fast_pop(fh, heapLen);
            heapLen--;
#ifdef PDA_CTA_PROFILE
            const long long tp1 = PROF_T();
            ctl->tPop += tp1 - tp0;
#endif
            const int base = S.recBase[rec - 1];
            for (int j = 0; j < cnt; ++j) {  // children in column order (:493-522)
                const double g = S.recGain[(rec - 1) * PDA_CTA_MAX_COL + j];
                if (g == g) {
                    if (allTop) smem_sift_up(fh.top, heapLen, make_entry(g, base + j, a0 + j));
                    else fast_sift_up(fh, heapLen, make_entry(g, base + j, a0 + j));
                    heapLen++;
                }
            }
#ifdef PDA_CTA_PROFILE
            ctl->tPush += PROF_T() - tp1;
#endif
            freeRec |= 1ULL << (rec - 1);
            uncommitted -= cnt;
#ifdef PDA_CTA_PROFILE
            ctl->commits++;
#endif
            if (heapLen == 0) { done = 1; ctl->nFound = sweep; ctl->nEmit = sweep; break; }
            const int4 nt = fh.get(0);  // hypothesis number `sweep` (:703-719)
            const double ntGain = entry_gain(nt);
            double gainOut;
            bool stop = false;
            if (!maximize) {
                gainOut = ntGain + CDelta;
                if (a.cutMode == PDA_CUT_RELATIVE && gainOut > gain0Out + a.cutoff) stop = true;
            } else {
                gainOut = -ntGain + CDelta;
                if (a.cutMode == PDA_CUT_RELATIVE && gainOut < gain0Out - a.cutoff) stop = true;
            }
            A.orderNode[sweep] = nt.z;
            A.orderGain[sweep] = gainOut;
            if (stop) { done = 1; ctl->nFound = sweep; ctl->nEmit = sweep + 1; break; }
            sweep++;
            top = nt;
        }
        if (!done && sweep >= a.k) { done = 1; ctl->nFound = sweep; ctl->nEmit = sweep; }
        ctl->heapLen = heapLen; ctl->sweep = sweep; ctl->uncommitted = uncommitted; ctl->freeRec = freeRec;
        ctl->done[round & 1] = done;
    }
    __syncwarp();
#ifdef PDA_CTA_PROFILE
    const long long tc1 = PROF_T();
    if (lane == 0) ctl->tCommit += tc1 - tc0;
#endif
    if (ctl->done[round & 1]) return;

    // Picking costs this warp ~3 000 cycles and it is the critical path, so it is skipped while enough splits are
    // already waiting (done or in flight) and the top of the heap is among them.  (Picking again while the top's
    // children are being solved finds almost nothing new among the first 32 entries: measured, no gain.)
    if (pad_record(heap.get(0).pad) != 0 && 64 - __popcll(ctl->freeRec) >= CTA_AHEAD) {
        if (lane == 0) { ctl->flight[(round + 1) & 1] = 0ULL; ctl->nTasks[(round + 1) & 1] = 0; }
        return;
    }
    // ---- choose what the workers split NEXT round: the cheapest unsplit entries among the first 32 of the heap.
    // All lanes at once: every lane ranks its entry against the other 31 (gains order like their bit patterns), the
    // lane of rank q then decides for the q-th cheapest; the limits are monotone in q, so "admitted" is a prefix.
    const int heapLen = ctl->heapLen;
    const int m = heapLen < 32 ? heapLen : 32;
    HeapEntry e;
    e.gain = CUDART_INF; e.node = 0; e.pad = 0;
    if (lane < m) e = heap.get(lane);
    const bool unsplit = lane < m && pad_record(e.pad) == 0;
    const long long kk = unsplit ? __double_as_longlong(e.gain) : 0x7fffffffffffffffLL;
    int rank = 0;
#pragma unroll
    for (int o = 0; o < 32; ++o) {
        const long long ko = __shfl_sync(FULL, kk, o);
        rank += (ko < kk || (ko == kk && o < lane)) ? 1 : 0;
    }
    unsigned char* inv = reinterpret_cast<unsigned char*>(S.tasks + 2 * CTA_MAXTASKS);  // 32 bytes of scratch behind the task lists
    inv[rank] = (unsigned char)lane;
    __syncwarp();
    const int src = inv[lane];  // this lane now speaks for the entry of rank `lane`
    const bool valid = __shfl_sync(FULL, unsplit ? 1 : 0, src) != 0;
    const int a0 = __shfl_sync(FULL, pad_active(e.pad), src);
    const int parent = __shfl_sync(FULL, e.node, src);
    const int cnt = valid ? nc - a0 : 0;
    int pre = cnt;  // inclusive prefix of children counts in rank order
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(FULL, pre, o);
        if (lane >= o) pre += y;
    }
    const unsigned long long freeRec0 = ctl->freeRec;
    const int nNodes0 = ctl->nNodes, uncommitted0 = ctl->uncommitted;
    const bool mandatory = lane == 0 && src == 0;  // the heap top itself: always split (one record is kept back for it)
    const bool admitted = valid && lane < CTA_SPEC &&
                          (mandatory || (pre <= CTA_MAXTASKS && __popcll(freeRec0) - lane >= 2 && uncommitted0 + pre <= cg.specSlack));
    const unsigned admMask = __ballot_sync(FULL, admitted);
    // monotone limits => admMask is a run of low bits, except that a failed rank 0 blocks everything behind it
    const int nAdm = (admMask & 1u) ? __ffs(~admMask) - 1 : 0;
    unsigned long long fr = freeRec0;
    for (int i = 0; i < lane && i < nAdm; ++i) fr &= fr - 1;  // drop the records taken by cheaper ranks
    const int rec = __ffsll((long long)fr) - 1;
    if (lane < nAdm) {
        const int childBase = nNodes0 + pre - cnt;
        if (src < heap.topCap) heap.top[src].pad |= (rec + 1) << 8; else heap.deep[src].pad |= (rec + 1) << 8;
        S.recBase[rec] = childBase;
        Task* list = S.tasks + ((round + 1) & 1) * CTA_MAXTASKS + (pre - cnt);
        for (int c = 0; c < cnt; ++c) {
            Task t;
            t.parent = parent; t.child = childBase + c; t.c = (short)(a0 + c); t.rec = (short)rec;
            list[c] = t;
        }
    }
    const int total = nAdm > 0 ? __shfl_sync(FULL, pre, nAdm - 1) : 0;
    const unsigned long long frAfter = __shfl_sync(FULL, fr & (fr - 1), nAdm > 0 ? nAdm - 1 : 0);
    __syncwarp();  // every lane has read the counters before lane 0 replaces them
    if (lane == 0) {
        const unsigned long long freeRec = nAdm > 0 ? frAfter : freeRec0;
        ctl->flight[(round + 1) & 1] = freeRec0 & ~freeRec;
        ctl->freeRec = freeRec; ctl->nNodes = nNodes0 + total; ctl->uncommitted = uncommitted0 + total;
        ctl->nTasks[(round + 1) & 1] = total;
    }
#ifdef PDA_CTA_PROFILE
    const int nTasks = total;
#endif
#ifdef PDA_CTA_PROFILE
    if (lane == 0) { ctl->tSelect += PROF_T() - tc1; ctl->rounds++; ctl->tasksTotal += nTasks; }
#endif
}

// ---- any warp: one child of one split (shortestPathUpdateCPP, shortestPathCPP.cpp:240-365) -----------
template <int R>
__device__ void run_task(const MurtyArgs& a, const CtaSmem& S, const WarpSmem& sm, const CtaArena& A, const Task t,
                         const int n, const int nc, const int lane) {
    const int D = a.geo.nodeDim;
    Node<R> nd;
    unsigned parForb;
    int a0;
    node_load<R>(A.nodes + (size_t)t.parent * a.geo.nodeStride, D, n, nd, parForb, a0, lane);
    const int c = t.c;
    unsigned inPar = 0u;  // rows paired with columns >= c: columns a0..c-1 are fixed for this child (:506-508, 525-527)
#pragma unroll
    for (int s = 0; s < R; ++s) if (lane + 32 * s < n && nd.c4r[s] >= c) inPar |= 1u << s;
    publish_cols<R>(sm, nd, lane);  // the parent's mirrors; the child solve leaves them alone
    unsigned hideFirst = 0u;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        if (nd.c4r[s] == c) {
            nd.c4r[s] = -1; hideFirst |= 1u << s;
            sm.c4r[lane + 32 * s] = 0xffffu;  // the freed row is the only sink of this search
        }
        if (lane + 32 * s == c) nd.r4c[s] = -1;
    }
    if (c == a0) hideFirst = parForb;
    __syncwarp();
    double result = CUDART_NAN;  // NaN = no child (infeasible or cut)
    const bool infeasible = augment_from<R>(c, nc, n, sm, nd, inPar, hideFirst, lane);
    if (!infeasible) {
        const double g = path_gain_reg<R>(sm, nd, n, nc, lane);
        const double cutoffGain = S.ctl->cutoffGain;
        const bool cut = S.ctl->cutting && (S.ctl->cutMax ? (g < cutoffGain) : (g > cutoffGain));
        if (!cut) {
            unsigned childForb = hideFirst;
#pragma unroll
            for (int s = 0; s < R; ++s) if (nd.c4r[s] == c) childForb |= 1u << s;
            node_store<R>(A.nodes + (size_t)t.child * a.geo.nodeStride, D, n, nd, childForb, c, lane);
            result = g;
        }
    }
    if (lane == 0) S.recGain[t.rec * PDA_CTA_MAX_COL + (c - a0)] = result;
    __syncwarp();
}

// LADDER: the k-ladder form (MurtyLadder): weights only, k = the largest rung, a table stored at every rung.  The ladder
// comes in through the pack, which is empty for the plain kernel: its calls keep the signature they have without the
// ladder, and with it the compiler's inlining decisions.
template <int R, bool LADDER, class... Ladder>
__device__ void solve_problem_cta(const MurtyArgs& a, const CtaGeometry& cg, const long long p, const CtaSmem& S,
                                  unsigned char* arenaBase, const Ladder*... ladder) {
    const MurtyLadder* L = nullptr;
    if constexpr (LADDER) ((L = ladder), ...);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = a.numRow[p], nc = a.numCol[p];
    const bool wantW = a.weightMode != PDA_WEIGHTS_NONE;
    const int nL = wantW ? a.nL[p] : 0;
    if (nc < 1 || nc > n || n > 32 * R || nc > PDA_CTA_MAX_COL || n > a.geo.nodeDim || n * nc > a.geo.cCap || nc > a.geo.maxCol ||
        (wantW && nL + nc != n)) {
        // malformed or beyond the launch's maxima: not solved (0 would mean infeasible)
        if constexpr (LADDER) ladder_found(a, *L, p, -1, threadIdx.x);
        else if (threadIdx.x == 0) a.nFound[p] = -1;
        return;
    }
    const WarpSmem sm = warp_view(S, cg, R, warp);
    const CtaArena A = carve_arena(arenaBase, cg, a.k);
    Heap heap;
    heap.top = S.heapTop;
    heap.deep = A.heapDeep;
    heap.topCap = cg.heapTopCap;
    CtaCtl* ctl = S.ctl;

#ifdef PDA_CTA_PROFILE
    if (threadIdx.x == 0) { ctl->tCommit = ctl->tSelect = ctl->tTasks = ctl->tPop = ctl->tPush = 0; ctl->rounds = ctl->tasksTotal = ctl->commits = 0; ctl->t0 = PROF_T(); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ctl->ns0)); }
#endif
    if (warp == 0) root_phase<R, LADDER>(a, p, S, sm, heap, A, lane, ladder...);
    __syncthreads();
#ifdef PDA_CTA_PROFILE
    if (threadIdx.x == 0) ctl->tRoot = PROF_T() - ctl->t0;
#endif
    const bool feasible = ctl->feasible != 0, doneAtRoot = ctl->done[0] != 0;
    __syncthreads();  // everyone has read the root's verdict before warp 0 may change it
    if (!feasible) return;

    // Rounds: warp 0 commits what earlier rounds solved and picks the next splits WHILE warps 1..15 solve the splits
    // picked one round earlier; one barrier per round.  Round 0 only picks (the root's split).
    for (int round = 0; !doneAtRoot; ++round) {
        if (warp == 0) {
#ifdef PDA_CTA_PROFILE
            const long long tw0 = PROF_T();
#endif
            serial_phase(a, cg, S, heap, A, nc, round, lane);
#ifdef PDA_CTA_PROFILE
            if (lane == 0 && round < 64) { g_trace[4 * round] = PROF_T() - tw0; g_trace[4 * round + 3] = ctl->sweep; }
#endif
        } else {
            const int nT = ctl->nTasks[round & 1];
            const long long tt0 = PROF_T();
            for (int t = warp - 1; t < nT; t += CTA_WARPS - 1)
                run_task<R>(a, S, sm, A, S.tasks[(round & 1) * CTA_MAXTASKS + t], n, nc, lane);
#ifdef PDA_CTA_PROFILE
            if (threadIdx.x == 32) { ctl->tTasks += PROF_T() - tt0; if (round < 64) { g_trace[4 * round + 1] = PROF_T() - tt0; g_trace[4 * round + 2] = nT; } }
#endif
        }
        __syncthreads();
        if (ctl->done[round & 1]) break;
    }
    const long long tf0 = PROF_T();

    // ---- lists (hpp:226-231) from the recorded pop order --------------------------------------------
    const int nFound = ctl->nFound, nEmit = ctl->nEmit;
    const int D = a.geo.nodeDim;
    for (int i = warp; i < nEmit; i += CTA_WARPS) {
        const unsigned char* nb = A.nodes + (size_t)A.orderNode[i] * a.geo.nodeStride + 16 * D;
        if (a.c4rBest) {
            int64_t* o = a.c4rBest + a.c4rOff[p] + (int64_t)i * n;
            for (int r = lane; r < n; r += 32) o[r] = (int64_t)(signed char)nb[r];
        }
        if (a.r4cBest) {
            int64_t* o = a.r4cBest + a.r4cOff[p] + (int64_t)i * nc;
            for (int c = lane; c < nc; c += 32) o[c] = (int64_t)(signed char)nb[D + c];
        }
        if (lane < nc) A.hypRows[(size_t)i * PDA_CTA_MAX_COL + lane] = nb[D + lane];
        if (a.gainBest && lane == 0) a.gainBest[p * (long long)a.k + i] = A.orderGain[i];
    }
    if constexpr (LADDER) ladder_found(a, *L, p, nFound, threadIdx.x);
    else if (threadIdx.x == 0) a.nFound[p] = nFound;

    // ---- weights (assignment.cpp:616-648, 910-945): every table entry adds its terms in hypothesis order ---
    if (wantW && nc > 1) {
        const double best = ctl->gain0Out;
        for (int i = threadIdx.x; i < nFound; i += blockDim.x) {
            const double g = A.orderGain[i];
            const bool gatedOut = a.weightMode == PDA_WEIGHTS_GATED && !(best + a.weightGate > g);
            A.orderW[i] = gatedOut ? 0.0 : exp(best - g);
        }
        __syncthreads();
        const int cells = nc * (nL + 1);
        for (int t = threadIdx.x; t < cells; t += blockDim.x) {
            const int c = t / (nL + 1), to = t - c * (nL + 1);
            double acc = 0.0, total = 0.0;
            int rungAt = 0;  // ladder: the next rung to store (nFound <= its k for the last rung)
            for (int i = 0; i < nFound; ++i) {
                const double w = A.orderW[i];
                int r = (int)(signed char)A.hypRows[(size_t)i * PDA_CTA_MAX_COL + c];
                r = r >= nL ? nL : r;
                total += w;
                if (r == to) acc += w;
                if constexpr (LADDER) {
                    if (i + 1 == L->rung[rungAt]) { ladder_put(a, *L, p, rungAt, rungAt, cells, t, acc * (1.0 / total)); ++rungAt; }
                }
            }
            if constexpr (LADDER) ladder_put(a, *L, p, rungAt, PDA_LADDER_MAX, cells, t, acc * (1.0 / total));  // rungs past the end
            else a.probs[a.probOff[p] + t] = acc * (1.0 / total);
        }
    }
#ifdef PDA_CTA_PROFILE
    __syncthreads();
    long long ns1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
    if (threadIdx.x == 0) {
        g_prof[0] = ns1 - ctl->ns0; g_prof[1] = ctl->tRoot; g_prof[2] = ctl->tCommit; g_prof[3] = ctl->tSelect;
        g_prof[4] = ctl->tTasks; g_prof[5] = PROF_T() - tf0; g_prof[6] = PROF_T() - ctl->t0; g_prof[7] = ctl->rounds;
        g_prof[8] = ctl->tasksTotal; g_prof[9] = ctl->commits; g_prof[10] = ctl->tPop; g_prof[11] = ctl->tPush;
    }
#endif
}

#ifndef PDA_MURTY_LADDER_TU  // murty_ladder_kernel.cu compiles this file for the ladder kernels alone
template <int R>
__global__ void __launch_bounds__(32 * CTA_WARPS, 1) murty_cta_kernel(const MurtyArgs a, const CtaGeometry cg) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    if ((int)blockIdx.x >= a.nWarps) return;  // nWarps = arenas available = CTAs allowed to run
    const CtaSmem S = carve_cta(smemRaw, a.geo, cg);
    unsigned char* arena = a.arena + (size_t)blockIdx.x * cg.arenaStride;
    if (a.cursor == nullptr) {  // one CTA per problem and enough arenas for all of them: no work queue
        solve_problem_cta<R, false>(a, cg, (long long)blockIdx.x, S, arena);
        return;
    }
    for (;;) {
        __syncthreads();  // the previous problem's readers of ctl are done
        if (threadIdx.x == 0) S.ctl->problem = (long long)atomicAdd(a.cursor, 1ULL);
        __syncthreads();
        const long long p = S.ctl->problem;
        if (p >= a.nProblems) break;
        solve_problem_cta<R, false>(a, cg, p, S, arena);
    }
}

}  // namespace

// ---- host side ------------------------------------------------------------------------------------
static int round_up_i(int x, int m) { return (x + m - 1) / m * m; }

int murty_cta_geometry(int32_t k, int32_t maxNumRow, int32_t maxNumCol, bool weights, const DeviceInfo& dev,
                       MurtyGeometry* g, CtaGeometry* cg) {
    int rc = murty_geometry(k, maxNumRow, maxNumCol, weights, dev, g);
    if (rc) return rc;
    if (maxNumCol > PDA_CTA_MAX_COL)
        return fail(PDA_ERR_UNSUPPORTED, "murty (CTA path): numCol %d exceeds %d", maxNumCol, PDA_CTA_MAX_COL);
    const int D = 32 * g->R;
    cg->mirrorBytes = round_up_i(22 * D, 16);
    cg->specSlack = 16 * maxNumCol;
    const int64_t nodes = 1 + (int64_t)k * maxNumCol + cg->specSlack;
    if (nodes > (int64_t)1 << 30) return fail(PDA_ERR_UNSUPPORTED, "murty: k * numCol too large");
    cg->maxNodes = (int)nodes;
    cg->heapBytes = (int64_t)round_up_i((int)nodes, 8) * (int64_t)sizeof(HeapEntry);
    const int64_t orderBytes = (int64_t)k * 8 * 2 + (int64_t)((k + 3) & ~3) * 4 + (int64_t)k * PDA_CTA_MAX_COL;
    cg->nodesOff = (cg->heapBytes + orderBytes + 255) / 256 * 256;
    cg->arenaStride = (cg->nodesOff + nodes * g->nodeStride + 255) / 256 * 256;
    int off = 8 * (g->cCap + g->pCap) + CTA_WARPS * cg->mirrorBytes + 8 * CTA_RECORDS * PDA_CTA_MAX_COL +
              4 * CTA_RECORDS + 2 * (int)sizeof(Task) * CTA_MAXTASKS + 32;
    off = round_up_i(off, 16);
    cg->ctlOff = off;
    off = round_up_i(off + (int)sizeof(CtaCtl), 16);
    cg->heapTopOff = off;
    int topCap = (dev.maxSmemOptin - off) / (int)sizeof(HeapEntry);
    if (topCap < 32) return fail(PDA_ERR_UNSUPPORTED, "murty (CTA path): problem too large for shared memory");
    if (topCap > cg->maxNodes) topCap = cg->maxNodes;
    cg->heapTopCap = topCap;
    cg->smemBytes = off + topCap * (int)sizeof(HeapEntry);
    return PDA_OK;
}

template <int R>
static int launch_murty_cta_r(const MurtyArgs& a, const CtaGeometry& cg, cudaStream_t stream) {
    PDA_CUDA_TRY(cudaFuncSetAttribute(murty_cta_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, cg.smemBytes));
    const int ctas = (int)(a.nProblems < a.nWarps ? a.nProblems : a.nWarps);
    murty_cta_kernel<R><<<ctas, 32 * CTA_WARPS, cg.smemBytes, stream>>>(a, cg);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}

int launch_murty_cta(const MurtyArgs& args, const CtaGeometry& cg, cudaStream_t stream, const MurtyLadder* ladder) {
    MurtyArgs a = args;
    if (a.nProblems <= a.nWarps) a.cursor = nullptr;  // every problem has its own CTA: skip the queue and its memset
    else PDA_CUDA_TRY(cudaMemsetAsync(a.cursor, 0, sizeof(unsigned long long), stream));
    if (ladder) return launch_murty_cta_ladder(a, cg, *ladder, stream);
    switch (a.geo.R) {
        case 1: return launch_murty_cta_r<1>(a, cg, stream);
        case 2: return launch_murty_cta_r<2>(a, cg, stream);
        case 4: return launch_murty_cta_r<4>(a, cg, stream);
    }
    return fail(PDA_ERR_UNSUPPORTED, "murty: unsupported row-slot count %d", a.geo.R);
}

#else
// The k-ladder form (written out apart from murty_cta_kernel for the reason given at murty_ladder_kernel)
template <int R>
__global__ void __launch_bounds__(32 * CTA_WARPS, 1)
    murty_cta_ladder_kernel(const MurtyArgs a, const CtaGeometry cg, const __grid_constant__ MurtyLadder L) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    if ((int)blockIdx.x >= a.nWarps) return;  // nWarps = arenas available = CTAs allowed to run
    const CtaSmem S = carve_cta(smemRaw, a.geo, cg);
    unsigned char* arena = a.arena + (size_t)blockIdx.x * cg.arenaStride;
    if (a.cursor == nullptr) {
        solve_problem_cta<R, true>(a, cg, (long long)blockIdx.x, S, arena, &L);
        return;
    }
    for (;;) {
        __syncthreads();  // the previous problem's readers of ctl are done
        if (threadIdx.x == 0) S.ctl->problem = (long long)atomicAdd(a.cursor, 1ULL);
        __syncthreads();
        const long long p = S.ctl->problem;
        if (p >= a.nProblems) break;
        solve_problem_cta<R, true>(a, cg, p, S, arena, &L);
    }
}

}  // namespace

int launch_murty_cta_ladder(const MurtyArgs& a, const CtaGeometry& cg, const MurtyLadder& ladder, cudaStream_t stream) {
    void (*k)(const MurtyArgs, const CtaGeometry, const MurtyLadder) = nullptr;
    switch (a.geo.R) {
        case 1: k = murty_cta_ladder_kernel<1>; break;
        case 2: k = murty_cta_ladder_kernel<2>; break;
        case 4: k = murty_cta_ladder_kernel<4>; break;
        default: return fail(PDA_ERR_UNSUPPORTED, "murty: unsupported row-slot count %d", a.geo.R);
    }
    PDA_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, cg.smemBytes));
    const int ctas = (int)(a.nProblems < a.nWarps ? a.nProblems : a.nWarps);
    k<<<ctas, 32 * CTA_WARPS, cg.smemBytes, stream>>>(a, cg, ladder);
    PDA_CUDA_TRY(cudaGetLastError());
    return PDA_OK;
}
#endif  // PDA_MURTY_LADDER_TU

}  // namespace pda

#ifdef PDA_CTA_PROFILE
extern "C" int pda_debug_read_prof(long long* out) {
    return (int)cudaMemcpyFromSymbol(out, pda::g_prof, sizeof(long long) * 16);
}
extern "C" int pda_debug_read_trace(long long* out) {
    return (int)cudaMemcpyFromSymbol(out, pda::g_trace, sizeof(long long) * 256);
}
#endif
