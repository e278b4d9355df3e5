// murty_device.cuh -- device building blocks shared by the two Murty kernels (murty_kernel.cu: one warp per
// problem, throughput; murty_cta_kernel.cu: one CTA per problem, latency): the warp-wide shortest augmenting
// path with the reference's arithmetic order and tie-breaks (shortestPathCPP.cpp:119-365), the libstdc++-
// compatible binary heap, the node arena format, matrix staging, list emission and weight accumulation.
#ifndef PDA_MURTY_DEVICE_CUH
#define PDA_MURTY_DEVICE_CUH
#include "pda_internal.h"

#include <math_constants.h>

namespace pda {
namespace {

constexpr unsigned FULL = 0xffffffffu;

// resident CTAs per SM the register allocator must leave room for (4 warps each)
#ifndef PDA_MURTY_MINB
#define PDA_MURTY_MINB 6
#endif
// the same for the pruning kernel (murty_kernel<R, true>): measured 6 -> 5 CTAs per SM (102 registers instead of 80)
// +9 %: at 80 registers the compiler re-derives the masked row duals and the shared-memory addresses in every Dijkstra step
#ifndef PDA_FAST_MINB
#define PDA_FAST_MINB 5
#endif
// warps per CTA of the throughput kernel (resident warps per SM = PDA_MURTY_MINB * PDA_MURTY_WPC)
#ifndef PDA_MURTY_WPC
#define PDA_MURTY_WPC 4
#endif

struct __align__(16) HeapEntry {
    double gain;
    int node;
    int pad;
};

// ---- order-preserving 64-bit key for doubles ----------------------------------------------------
__device__ __forceinline__ void to_key(double d, unsigned& khi, unsigned& klo) {
    const unsigned hi = (unsigned)__double2hiint(d), lo = (unsigned)__double2loint(d);
    const unsigned m = (unsigned)((int)hi >> 31);  // all ones for negatives
    khi = hi ^ (m | 0x80000000u);
    klo = lo ^ m;
}
__device__ __forceinline__ double from_key(unsigned khi, unsigned klo) {
    const unsigned m = (khi & 0x80000000u) ? 0u : 0xffffffffu;
    return __hiloint2double((int)(khi ^ (m | 0x80000000u)), (int)(klo ^ m));
}
constexpr unsigned KEY_INF_HI = 0xFFF00000u;  // key of +inf is (0xFFF00000, 0)
constexpr int HI_INF = 0x7ff00000;            // high word of +inf (and the NaN marker's 0x7ff80000 lies above it)

// Warp arg-min of doubles that are almost always >= +0.0 (reduced costs: tiny negatives appear only through rounding).
// For non-negative doubles -- +inf and the positive NaN marker included -- (high word as a signed int, low word as
// unsigned) orders like the numbers, so the common case needs no key conversion: REDUX.MIN.S32 on the high words,
// REDUX.MIN.U32 on the low words of the lanes that tie, REDUX.MIN on the row index of the lanes that tie again.  A
// negative minimum shows up as mhi < 0 and takes the order-preserving keys instead.
// Returns the high word of the minimum in mhiOut (>= HI_INF: nothing finite), its value in `val`, its lowest row in `row`.
__device__ __forceinline__ void warp_argmin(const double x, const int myRow, int& mhiOut, double& val, int& row) {
    const int hi = __double2hiint(x);
    const unsigned lo = (unsigned)__double2loint(x);
    const int mhi = __reduce_min_sync(FULL, hi);
    if (mhi >= 0) {
        const unsigned mlo = __reduce_min_sync(FULL, (hi == mhi) ? lo : 0xffffffffu);
        const bool win = (hi == mhi) && (lo == mlo);
        row = (int)__reduce_min_sync(FULL, win ? (unsigned)myRow : 0xffffu);
        val = __hiloint2double(mhi, (int)mlo);
        mhiOut = mhi;
    } else {
        unsigned khi, klo;
        to_key(x, khi, klo);
        const unsigned kmhi = __reduce_min_sync(FULL, khi);
        const unsigned kmlo = __reduce_min_sync(FULL, (khi == kmhi) ? klo : 0xffffffffu);
        const bool win = (khi == kmhi) && (klo == kmlo);
        row = (int)__reduce_min_sync(FULL, win ? (unsigned)myRow : 0xffffu);
        val = from_key(kmhi, kmlo);
        mhiOut = -1;  // a negative number: finite
    }
}
__device__ __forceinline__ double warp_min_val(const double x) {
    const int hi = __double2hiint(x);
    const unsigned lo = (unsigned)__double2loint(x);
    const int mhi = __reduce_min_sync(FULL, hi);
    if (mhi >= 0) {
        const unsigned mlo = __reduce_min_sync(FULL, (hi == mhi) ? lo : 0xffffffffu);
        return __hiloint2double(mhi, (int)mlo);
    }
    unsigned khi, klo;
    to_key(x, khi, klo);
    const unsigned kmhi = __reduce_min_sync(FULL, khi);
    const unsigned kmlo = __reduce_min_sync(FULL, (khi == kmhi) ? klo : 0xffffffffu);
    return from_key(kmhi, kmlo);
}

__device__ __forceinline__ double warp_min(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { double y = __shfl_xor_sync(FULL, x, o); x = (y < x) ? y : x; }
    return x;
}
__device__ __forceinline__ double warp_max(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { double y = __shfl_xor_sync(FULL, x, o); x = (x < y) ? y : x; }
    return x;
}

// Per-warp view of shared memory.
struct WarpSmem {
    double* C;       // [ld * numCol] shifted cost matrix, real columns only
    double* u;       // [32R] mirror of the working node's column duals
    double* spc;     // [32R] shortestPathCost, published after a scan for the dual update
    double* acc;     // [numCol * (nL+1)] weight accumulators
    short* r4c;      // [32R] mirror of the working node's row4col
    short* pred;     // [32R] predecessor column per row
    unsigned short* c4r;  // [32R] mirror of the working node's col4row (0xffff = free)
};

// The working node, distributed over the warp.
template <int R>
struct Node {
    double v[R];   // row duals           (lane owns rows  lane + 32 s)
    double u[R];   // column duals        (lane owns cols  lane + 32 s)
    int c4r[R];    // column of each owned row (-1 = free)
    int r4c[R];    // row of each owned column (-1 = free)
};

// One relaxation pass of the row scan from column `cur` (shortestPathCPP.cpp:179-195 / 307-325).
// Rows that must not take part carry v == -inf, which makes their reduced cost +inf, so no row mask is
// needed: `t < cand` is simply never true for them.  REAL = the column exists in sm.C; otherwise it is
// one of the reference's zero padding columns, C == +0.0 and delta + 0.0 == delta (delta is never -0.0:
// the staged matrix holds no -0.0 and x - x rounds to +0.0).
template <int R, bool REAL>
__device__ __forceinline__ void relax(const double* __restrict__ Ccol, const int n, const double delta,
                                      const double ucur, const double (&v)[R], const int cur,
                                      double (&cand)[R], int (&pred)[R], const int lane) {
    const double du = delta - ucur;  // used by the padding-column form only
#pragma unroll
    for (int s = 0; s < R; ++s) {
        double t;
        if (REAL) {
            const double c = (lane + 32 * s < n) ? Ccol[lane + 32 * s] : 0.0;
            t = ((delta + c) - ucur) - v[s];
        } else {
            t = du - v[s];
        }
        const bool better = t < cand[s];
        cand[s] = better ? t : cand[s];
        pred[s] = better ? cur : pred[s];
    }
}

constexpr int NAN_HI = 0x7ff80000;  // high word of the NaN that marks a scanned row's candidate

#ifdef PDA_FAST_STATS
__device__ unsigned long long g_augStats[8];  // argmins, ff tried, ff applied, loop trips, flip hops, searches, real relax, pad relax
#define PDA_ASTAT(i) do { if (lane == 0) atomicAdd(&g_augStats[i], 1ULL); } while (0)
#else
#define PDA_ASTAT(i) do { } while (0)
#endif

// Fast-forward over the reference's no-op hops.
//
// Most Dijkstra steps of a child solve (93 % on the benchmark shapes) go through rows that are paired with
// zero-cost PADDING columns and change nothing: scanning such a column p from row r offers every other row
// t = (cand[r] - u[p]) - v[row], which is not below what the row already holds, so the reference merely retires
// r and moves to the next-closest row.  This routine proves that for a whole run of such rows at once and
// retires them together, with results bit-identical to stepping through them:
//   stopper  = the closest live row that is NOT paired with a padding column (a free row -- the sink -- or a row
//              whose column has real costs); key order is (cand, row), the reference's first-minimum order
//   F        = live rows paired with padding columns that come before the stopper in that order
//   W        = min over F of fl(cand[r] - u[col(r)])   (what each of those hops would offer, before the row dual)
//   test     : fl(W - v[row]) >= cand[row] for EVERY live row.  Rounding is monotone, so fl(W - v) is the smallest
//              offer any hop of F could make to that row; if even that does not beat its candidate, no hop of F
//              updates anything, in any order (a sufficient condition -- it also covers offers from hops that
//              come after the row, which the reference never makes).
// If the test passes every row of F is scanned at its current candidate (parked in sm.spc), predecessors stay as
// they are, and the stopper is the next row to scan: (closest, delta) are returned so the caller skips its own
// arg-min.  If it fails nothing is changed and the caller steps normally.  With fewer than two rows in F there is
// nothing to batch, but the work done so far already identifies the next row to scan (the stopper itself, or the one row
// of F), so the caller's arg-min is saved all the same.  Returns 0 = nothing known, 1 = (closest, delta) is the
// stopper and everything before it is retired, 2 = the same and nothing finite is left (infeasible), 3 = (closest,
// delta) is the plain arg-min, nothing retired.
template <int R>
__device__ __forceinline__ int fast_forward(const int numColReal, const WarpSmem& sm, const Node<R>& nd,
                                            const double (&vEff)[R], const double (&uRow)[R], double (&cand)[R],
                                            int& closest, double& delta, const int lane) {
    // the stopper
    double sb = CUDART_INF;
    int sbs = 0;
#pragma unroll
    for (int s = 0; s < R; ++s)
        if (nd.c4r[s] < numColReal && cand[s] < sb) { sb = cand[s]; sbs = s; }
    int mhi, rT;
    double kT;
    warp_argmin(sb, lane + 32 * sbs, mhi, kT, rT);
    // F and what its hops would offer
    unsigned inF = 0u, fMask[R];
    double wmin = CUDART_INF;
    int nF = 0;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const bool f = nd.c4r[s] >= numColReal && cand[s] < CUDART_INF &&
                       (cand[s] < kT || (cand[s] == kT && lane + 32 * s < rT));
        if (f) {
            inF |= 1u << s;
            const double w = cand[s] - uRow[s];
            wmin = (w < wmin) ? w : wmin;
        }
        fMask[s] = __ballot_sync(FULL, f);
        nF += __popc(fMask[s]);
    }
    if (nF == 0) {  // no padding-paired row comes before the stopper: the stopper IS the arg-min
        closest = rT;
        delta = kT;
        return (mhi >= HI_INF) ? 2 : 1;
    }
    if (nF == 1) {  // the one row of F is the arg-min; it is scanned the ordinary way
        int slot = 0;
#pragma unroll
        for (int s = 1; s < R; ++s) if (fMask[s]) slot = s;
        unsigned msk = fMask[0];
        double cv = cand[0];
#pragma unroll
        for (int s = 1; s < R; ++s) if (slot == s) { msk = fMask[s]; cv = cand[s]; }
        const int src = __ffs(msk) - 1;
        closest = src + 32 * slot;
        delta = __shfl_sync(FULL, cv, src);
        return 3;
    }
    const double W = warp_min_val(wmin);
    bool beats = false;
#pragma unroll
    for (int s = 0; s < R; ++s) beats = beats || ((W - vEff[s]) < cand[s]);
    if (__any_sync(FULL, beats)) return 0;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        if ((inF >> s) & 1u) {
            sm.spc[lane + 32 * s] = cand[s];
            cand[s] = __hiloint2double(NAN_HI, __double2loint(cand[s]));
        }
    }
    closest = rT;
    delta = kT;
    return (mhi >= HI_INF) ? 2 : 1;
}

// One shortest augmenting path from `startCol` over the rows flagged in scanBits
// (bit s = row lane+32s), then the dual update and the flip along the path.
//   shortestPathCPP.cpp:168-226 / 297-356 (scan), :92-106 (duals), :108-116 (flip).
// forbBits hides rows on the first hop only (:310).  numColReal = columns that exist in
// sm.C; columns beyond are the reference's zero padding.  Returns true if infeasible.
//
// cand[s] is the reference's shortestPathCost of a row that is still to be scanned.  Rows outside the
// scan set keep cand == +inf (their v is -inf, so they never relax); a row that HAS been scanned gets
// its cand poisoned to NaN (one high-word write): `t < NaN` is false, so it never relaxes again, the
// arg-min skips it, and "scanned" can be read back from it afterwards.  The cost at which a row was
// scanned (== delta at that moment) is parked in sm.spc by lane 0, where the dual update reads it.
//
// The mirrors in shared memory (u / row4col / col4row of the node the search STARTS from) are read, never written:
// the dual update and the flip touch the registers only.  A Murty split publishes the parent once and solves all its
// children against it; the root LAP republishes after every column.  uRowPar, when given, is the start node's "u of the
// column each row is paired with", computed once per split (the freed row's entry is stale there, but a free row is a
// stopper and never consulted).
//
// LIMIT (the pruning fast path, murty_kernel.cu): the search is abandoned -- return 2, working node untouched -- as
// soon as the distance of the row about to be scanned exceeds `limit`.  Distances only grow along a Dijkstra search
// and the finished child's gain is the parent's gain plus the final distance (up to rounding, which the caller's
// margin absorbs), so such a child cannot be among the hypotheses still wanted.
// Returns 0 = augmented, 1 = infeasible, 2 = abandoned.
// FF = false leaves fast_forward out (the root LAP: 3 % of the work, and one inlined copy less of the largest routine
// keeps the kernel inside the instruction cache); the search then simply takes the reference's steps one by one.
template <int R, bool LIMIT = false, bool FF = true>
__device__ __forceinline__ int augment_from(const int startCol, const int numColReal, const int ld,
                                            const WarpSmem& sm, Node<R>& nd, const unsigned scanBits,
                                            const unsigned forbBits, const int lane, const double* uRowPar = nullptr,
                                            const double limit = __builtin_huge_val()) {
    double cand[R], vEff[R];
    int pred[R];
#pragma unroll
    for (int s = 0; s < R; ++s) {
        cand[s] = CUDART_INF;
        pred[s] = 0;
        vEff[s] = ((scanBits >> s) & 1u) ? nd.v[s] : -CUDART_INF;
    }
    int cur = startCol, sink;
    double delta = 0.0;
    {   // first hop: the forbidden rows sit this one out (:310)
        double vHop[R];
#pragma unroll
        for (int s = 0; s < R; ++s) vHop[s] = ((forbBits >> s) & 1u) ? -CUDART_INF : vEff[s];
        const double ucur = sm.u[cur];
        if (cur < numColReal) relax<R, true>(sm.C + cur * ld, ld, delta, ucur, vHop, cur, cand, pred, lane);
        else relax<R, false>(nullptr, ld, delta, ucur, vHop, cur, cand, pred, lane);
    }
    // u of the column each owned row is paired with (only rows paired with padding columns use it)
    double uRow[R];
#pragma unroll
    for (int s = 0; s < R; ++s) uRow[s] = !FF ? 0.0 : (uRowPar ? uRowPar[s] : ((nd.c4r[s] >= 0) ? sm.u[nd.c4r[s]] : 0.0));
    bool padPrev = cur >= numColReal;  // the last relaxation came from a padding column
    for (;;) {
        int closest = 0;
        int ff = 0;
        PDA_ASTAT(3);
        if (FF && padPrev) { PDA_ASTAT(1); ff = fast_forward<R>(numColReal, sm, nd, vEff, uRow, cand, closest, delta, lane); if (ff) PDA_ASTAT(2); }
        if (ff == 2) { __syncwarp(); return 1; }
        if (ff == 0) {
            PDA_ASTAT(0);
            // lane-local first minimum (lower slot = lower row wins ties; NaN = already scanned), then the warp arg-min
            double best = cand[0];
            int bs = 0;
#pragma unroll
            for (int s = 1; s < R; ++s) if (cand[s] < best || best != best) { best = cand[s]; bs = s; }
            int mhi;
            warp_argmin(best, lane + 32 * bs, mhi, delta, closest);
            if (mhi >= HI_INF) { __syncwarp(); return 1; }  // minVal == +inf (:197, :327): nothing finite is left
        }
        if (LIMIT && delta > limit) { __syncwarp(); return 2; }  // (sync: the caller rewrites sm.c4r next; all lanes have read it)
        if (lane == 0) sm.spc[closest] = delta;
#pragma unroll
        for (int s = 0; s < R; ++s)
            if (lane + 32 * s == closest) cand[s] = __hiloint2double(NAN_HI, __double2loint(cand[s]));
        const unsigned next = sm.c4r[closest];
        if (next == 0xffffu) { sink = closest; break; }
        cur = (int)next;
        padPrev = cur >= numColReal;
        const double ucur = sm.u[cur];
        if (padPrev) { PDA_ASTAT(7); relax<R, false>(nullptr, ld, delta, ucur, vEff, cur, cand, pred, lane); }
        else { PDA_ASTAT(6); relax<R, true>(sm.C + cur * ld, ld, delta, ucur, vEff, cur, cand, pred, lane); }
    }
    PDA_ASTAT(5);

    // duals, using row4col as it was before the flip (:92-106).  A column other than startCol was scanned
    // exactly when the row it is paired with was scanned (the sink row is unpaired).
    unsigned rowsDone[R];
#pragma unroll
    for (int s = 0; s < R; ++s) {
        rowsDone[s] = __ballot_sync(FULL, __double2hiint(cand[s]) == NAN_HI);
        sm.pred[lane + 32 * s] = (short)pred[s];
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < R; ++s) {
        if ((rowsDone[s] >> lane) & 1u) nd.v[s] = (nd.v[s] - delta) + sm.spc[lane + 32 * s];
        const int c = lane + 32 * s, r = nd.r4c[s];
        bool seen = false;
        if (r >= 0) {
            unsigned w = rowsDone[0];
#pragma unroll
            for (int q = 1; q < R; ++q) if ((r >> 5) == q) w = rowsDone[q];
            seen = (w >> (r & 31)) & 1u;
        }
        if (c == startCol) nd.u[s] = nd.u[s] + delta;
        else if (seen) nd.u[s] = (nd.u[s] + delta) - sm.spc[r];
    }
    // flip along the predecessor chain (:108-116); sm.r4c still holds the pre-flip pairing
    int r = sink, c;
    do {
        PDA_ASTAT(4);
        c = sm.pred[r];
        const int h = sm.r4c[c];
#pragma unroll
        for (int s = 0; s < R; ++s) {
            if (lane + 32 * s == r) nd.c4r[s] = c;
            if (lane + 32 * s == c) nd.r4c[s] = r;
        }
        r = h;
    } while (c != startCol);
    __syncwarp();  // the chain walk has read sm.pred / sm.r4c before anybody rewrites them
    return 0;
}

// calcGain (:59-80): ascending column order, starting from 0.0.
__device__ __forceinline__ double path_gain(const WarpSmem& sm, const int ld, const int numColGain) {
    double g = 0.0;
#pragma unroll 4
    for (int c = 0; c < numColGain; ++c) g = g + sm.C[c * ld + sm.r4c[c]];
    return g;
}
// More than 32 columns: column lane + 32 s pays the cost in row nd.r4c[s]; the terms in ascending column order.
template <int R>
__device__ __forceinline__ double path_gain_wide(const WarpSmem& sm, const Node<R>& nd, const int ld, const int numColGain,
                                                 const int lane) {
    double g = 0.0;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int c = lane + 32 * s;
        const double x = (c < numColGain) ? sm.C[c * ld + nd.r4c[s]] : 0.0;
        for (int j = 0; j < 32 && 32 * s + j < numColGain; ++j) g = g + __shfl_sync(FULL, x, j);
    }
    return g;
}
// The same sum from the working node's registers: lane c fetches the one cost its column pays, then the terms are
// added in the reference's order.  Lanes past the last column contribute +0.0, and g + 0.0 == g (g is a sum of
// entries of the shifted matrix, never -0.0), so the chain runs over a fixed eight columns at a time with no
// per-column branch: ~3 instructions per column instead of a dependent shared-memory walk by every lane.  (Not
// path_gain: sm.r4c mirrors the node the search started from, not the child it produced.)
template <int R>
__device__ __forceinline__ double path_gain_reg(const WarpSmem& sm, const Node<R>& nd, const int ld, const int numColGain,
                                                const int lane) {
    if (numColGain > 32) return path_gain_wide<R>(sm, nd, ld, numColGain, lane);
    double x = 0.0;
    if (lane < numColGain) x = sm.C[lane * ld + nd.r4c[0]];
    double g = 0.0;
#pragma unroll
    for (int c = 0; c < 8; ++c) g = g + __shfl_sync(FULL, x, c);  // constant source lanes: SHFL with an immediate
    for (int c0 = 8; c0 < numColGain; c0 += 8) {
#pragma unroll
        for (int c = 0; c < 8; ++c) g = g + __shfl_sync(FULL, x, (c0 + c) & 31);
    }
    return g;
}

// ---- the heap: lane 0 only ----------------------------------------------------------------------------
// Entries are 16 bytes and move as one 128-bit access.  The first `topCap` entries (the top levels, which every
// pop walks through) live in the warp's shared memory, the rest in its global arena: a pop's sift-down is a chain
// of dependent loads, and this turns most of its ~10 L2 round trips into shared-memory reads.  Gains are compared
// through their bit patterns: a gain is a sum of entries of the shifted matrix, i.e. >= +0.0 (never -0.0, never NaN),
// and for such doubles the 64-bit integer order IS the numeric order -- two integer compares instead of an FP64 one.
struct Heap {
    HeapEntry* top;   // shared memory, entries [0, topCap)
    HeapEntry* deep;  // global arena, entry i at deep[i] (slots below topCap unused)
    int topCap;
    __device__ __forceinline__ int4 get4(int i) const {
        return (i < topCap) ? reinterpret_cast<const int4*>(top)[i] : reinterpret_cast<const int4*>(deep)[i];
    }
    __device__ __forceinline__ void put4(int i, const int4 e) const {
        if (i < topCap) reinterpret_cast<int4*>(top)[i] = e; else reinterpret_cast<int4*>(deep)[i] = e;
    }
    __device__ __forceinline__ HeapEntry get(int i) const {
        const int4 v = get4(i);
        HeapEntry e;
        e.gain = __hiloint2double(v.y, v.x); e.node = v.z; e.pad = v.w;
        return e;
    }
    __device__ __forceinline__ void put(int i, const HeapEntry& e) const {
        put4(i, make_int4(__double2loint(e.gain), __double2hiint(e.gain), e.node, e.pad));
    }
};
__device__ __forceinline__ long long heap_key(const int4 e) { return ((long long)e.y << 32) | (unsigned)e.x; }

__device__ __forceinline__ void heap_sift_up4(const Heap& h, int hole, const int4 val) {
    const long long kv = heap_key(val);
    while (hole > 0) {
        const int parent = (hole - 1) / 2;
        const int4 par = h.get4(parent);
        if (!(heap_key(par) > kv)) break;
        h.put4(hole, par);
        hole = parent;
    }
    h.put4(hole, val);
}
__device__ __forceinline__ void heap_sift_up(const Heap& h, int hole, const HeapEntry val) {
    heap_sift_up4(h, hole, make_int4(__double2loint(val.gain), __double2hiint(val.gain), val.node, val.pad));
}
__device__ __forceinline__ void heap_pop(const Heap& h, const int lenBefore) {
    if (lenBefore > 1) {
        const int len = lenBefore - 1;
        const int4 val = h.get4(len);
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            const int4 right = h.get4(child), left = h.get4(child - 1);  // both children in one round trip
            const bool takeLeft = heap_key(right) > heap_key(left);      // right child wins an exact tie
            if (takeLeft) child--;
            h.put4(hole, takeLeft ? left : right);
            hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) {
            child = 2 * (child + 1);
            h.put4(hole, h.get4(child - 1));
            hole = child - 1;
        }
        heap_sift_up4(h, hole, val);
    }
}

// ---- the open list of the pruning fast path ---------------------------------------------------------------
// Used only while no two gains that matter are bit-equal (the caller hands the problem to the exact kernel the moment
// a selection is not unique), so ANY correct priority queue pops in the reference's order and the libstdc++ layout
// above is not needed.  That buys a structure a warp can work on with all its lanes:
//   key[] / node[]  unsorted slots; a removed slot holds PQ_EMPTY until the next compaction
//   gmin[g]         smallest key among slots 32g .. 32g+31
// push   = append + one compare (lane 0);   take-min = arg-min over gmin, one 32-wide look at that group, new group
// minimum from the keys already in registers: ~40 warp instructions whatever the size, against ~130 for a binary-heap
// pop by a single lane.  Gains are >= +0.0, so their bit patterns order like the numbers.
#ifndef PDA_PQ_UNROLL1
#define PDA_PQ_UNROLL1 1
#endif
#if PDA_PQ_UNROLL1
#define PDA_PQ_LOOP _Pragma("unroll 1")
#else
#define PDA_PQ_LOOP
#endif
#ifndef PDA_TIGHTEN_NOINLINE
#define PDA_TIGHTEN_NOINLINE 0   // measured: a real call costs 13 % (reference parameters and caller-saved registers go through local memory)
#endif
#if PDA_TIGHTEN_NOINLINE
#define PDA_TIGHTEN_INLINE __noinline__
#else
#define PDA_TIGHTEN_INLINE __forceinline__
#endif
constexpr unsigned long long PQ_EMPTY = ~0ULL;
constexpr int PQ_SLACK = 8;  // surplus candidates that trigger the next tightening of the bound
struct FastPQ {
    unsigned long long* key;   // [cap]
    int* node;                 // [cap]
    unsigned long long* gmin;  // [cap / 32], shared memory
    unsigned* hist;            // [32] scratch for pq_tighten (aliases sm.spc: never live during a search)
    int cap;
};
__device__ __forceinline__ unsigned long long warp_min_u64(const unsigned long long x) {
    const unsigned hi = (unsigned)(x >> 32), lo = (unsigned)x;
    const unsigned mhi = __reduce_min_sync(FULL, hi);
    const unsigned mlo = __reduce_min_sync(FULL, (hi == mhi) ? lo : 0xffffffffu);
    return ((unsigned long long)mhi << 32) | mlo;
}
__device__ __forceinline__ unsigned long long warp_max_u64(const unsigned long long x) {
    const unsigned hi = (unsigned)(x >> 32), lo = (unsigned)x;
    const unsigned mhi = __reduce_max_sync(FULL, hi);
    const unsigned mlo = __reduce_max_sync(FULL, (hi == mhi) ? lo : 0u);
    return ((unsigned long long)mhi << 32) | mlo;
}
__device__ __forceinline__ void pq_push(const FastPQ& q, int& len, const double gain, const int node, const int lane) {
    if (lane == 0) {
        const unsigned long long kb = (unsigned long long)__double_as_longlong(gain);
        q.key[len] = kb;
        q.node[len] = node;
        const int g = len >> 5;
        if ((len & 31) == 0 || kb < q.gmin[g]) q.gmin[g] = kb;
    }
    len++;
}
// Removes the smallest entry (len > 0 and at least one live slot).  Returns true when that choice was NOT unique: some
// other live entry has the same gain bits, and only the reference's heap mechanics can say which one goes first.
__device__ __forceinline__ bool pq_take_min(const FastPQ& q, const int len, unsigned long long& keyOut, int& nodeOut,
                                            const int lane) {
    __syncwarp();
    const int G = (len + 31) >> 5;
    unsigned long long m = PQ_EMPTY;
    int mg = 0;
    bool dup = false;
PDA_PQ_LOOP
    for (int g = lane; g < G; g += 32) {
        const unsigned long long x = q.gmin[g];
        dup = dup || (x == m && x != PQ_EMPTY);
        if (x < m) { m = x; mg = g; dup = false; }
    }
    const unsigned long long kmin = warp_min_u64(m);
    const unsigned eq = __ballot_sync(FULL, m == kmin);
    const int grp = __shfl_sync(FULL, mg, __ffs(eq) - 1);
    bool tie = (__popc(eq) > 1) || (G > 32 && __any_sync(FULL, dup && m == kmin));
    const int i = 32 * grp + lane;
    const unsigned long long kk = (i < len) ? q.key[i] : PQ_EMPTY;
    const unsigned eqi = __ballot_sync(FULL, kk == kmin);
    tie = tie || (__popc(eqi) > 1);
    const int w = __ffs(eqi) - 1;
    nodeOut = q.node[32 * grp + w];
    const unsigned long long rest = warp_min_u64((lane == w) ? PQ_EMPTY : kk);
    __syncwarp();  // every lane has read the group minima and this group's keys before lane 0 rewrites them (racecheck)
    if (lane == 0) { q.key[32 * grp + w] = PQ_EMPTY; q.gmin[grp] = rest; }
    keyOut = kmin;
    return tie;
}
// Lowers the pruning bound T and drops what it rules out.  Precondition: at least `m` live entries, m >= 1 = the
// number of hypotheses still to be emitted; every live entry is <= T.  Afterwards T is (close to) the m-th smallest live
// gain: the hypotheses already emitted plus m open ones at or below T exist, so nothing above T can be among the k
// best.  One histogram pass over 32 equal buckets between the smallest and the largest live gain picks the bucket that
// holds the m-th entry; its upper edge is the new bound (the count is re-checked with plain comparisons, so rounding
// in the bucket arithmetic can only make the bound looser, never wrong).  Survivors are compacted to the front.
__device__ PDA_TIGHTEN_INLINE void pq_tighten(const FastPQ& q, int& len, int& live, double& T, const int m, const int lane) {
    __syncwarp();
    const int S = (len + 31) >> 5;
    unsigned long long lo = PQ_EMPTY, hi = 0ULL;
PDA_PQ_LOOP
    for (int s = 0; s < S; ++s) {
        const int i = 32 * s + lane;
        const unsigned long long kk = (i < len) ? q.key[i] : PQ_EMPTY;
        if (kk != PQ_EMPTY) { lo = (kk < lo) ? kk : lo; hi = (kk > hi) ? kk : hi; }
    }
    lo = warp_min_u64(lo);
    hi = warp_max_u64(hi);
    const double dlo = __longlong_as_double((long long)lo), dhi = __longlong_as_double((long long)hi);
    double Tn = dhi;
    if (dhi > dlo) {
        const double width = (dhi - dlo) * 0.03125;
        const double inv = 1.0 / width;
        q.hist[lane] = 0u;
        __syncwarp();
    PDA_PQ_LOOP
    for (int s = 0; s < S; ++s) {
            const int i = 32 * s + lane;
            const unsigned long long kk = (i < len) ? q.key[i] : PQ_EMPTY;
            if (kk != PQ_EMPTY) {
                int b = (int)((__longlong_as_double((long long)kk) - dlo) * inv);
                b = b > 31 ? 31 : (b < 0 ? 0 : b);
                atomicAdd(&q.hist[b], 1u);
            }
        }
        __syncwarp();
        unsigned c = q.hist[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(FULL, c, o); if (lane >= o) c += y; }
        const unsigned reach = __ballot_sync(FULL, c >= (unsigned)m);
        const int bstar = __ffs(reach) - 1;
        if (bstar >= 0 && bstar < 31) { Tn = dlo + (double)(bstar + 1) * width; Tn = (Tn > dhi) ? dhi : Tn; }
        __syncwarp();  // hist is scratch of the next search from here on
    }
    unsigned long long tb = (unsigned long long)__double_as_longlong(Tn);
    int cnt = 0;
PDA_PQ_LOOP
    for (int s = 0; s < S; ++s) {
        const int i = 32 * s + lane;
        const unsigned long long kk = (i < len) ? q.key[i] : PQ_EMPTY;
        cnt += __popc(__ballot_sync(FULL, kk <= tb));
    }
    if (cnt < m) { tb = hi; Tn = dhi; }  // a bucket edge rounded the wrong way: keep every live entry
    const unsigned below = (1u << lane) - 1u;
    int out = 0;
PDA_PQ_LOOP
    for (int s = 0; s < S; ++s) {
        const int i = 32 * s + lane;
        const unsigned long long kk = (i < len) ? q.key[i] : PQ_EMPTY;
        const int nn = (i < len) ? q.node[i] : 0;
        const bool keep = kk <= tb;
        const unsigned km = __ballot_sync(FULL, keep);
        __syncwarp();  // every lane has read this slot before a survivor may be moved into it
        if (keep) { const int d = out + __popc(km & below); q.key[d] = kk; q.node[d] = nn; }
        out += __popc(km);
    }
    __syncwarp();
    len = out;
    live = out;
    T = Tn;
PDA_PQ_LOOP
    for (int g = 0; 32 * g < out; ++g) {
        const int i = 32 * g + lane;
        const unsigned long long mn = warp_min_u64((i < out) ? q.key[i] : PQ_EMPTY);
        if (lane == 0) q.gmin[g] = mn;
    }
    __syncwarp();
}

// ---- node arena -------------------------------------------------------------------------------------
// layout of one stored node (D = geo.nodeDim):  v[D] | u[D] | c4r bytes[D] | r4c bytes[D] | forb words[R] | activeCol
template <int R>
__device__ __forceinline__ void node_store(unsigned char* base, const int D, const int n, const Node<R>& nd,
                                           const unsigned forbBits, const int activeCol, const int lane) {
    double* dv = reinterpret_cast<double*>(base);
    unsigned char* bi = base + 16 * D;
    unsigned* meta = reinterpret_cast<unsigned*>(base + 18 * D);
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int i = lane + 32 * s;
        if (i < n) {
            dv[i] = nd.v[s];
            dv[D + i] = nd.u[s];
            bi[i] = (unsigned char)nd.c4r[s];
            bi[D + i] = (unsigned char)nd.r4c[s];
        }
        const unsigned w = __ballot_sync(FULL, (forbBits >> s) & 1u);
        if (lane == 0) meta[s] = w;
    }
    if (lane == 0) meta[R] = (unsigned)activeCol;
}
template <int R>
__device__ __forceinline__ void node_load(const unsigned char* base, const int D, const int n, Node<R>& nd,
                                          unsigned& forbBits, int& activeCol, const int lane) {
    const double* dv = reinterpret_cast<const double*>(base);
    const unsigned char* bi = base + 16 * D;
    const unsigned* meta = reinterpret_cast<const unsigned*>(base + 18 * D);
    forbBits = 0u;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int i = lane + 32 * s;
        if (i < n) {
            nd.v[s] = dv[i];
            nd.u[s] = dv[D + i];
            nd.c4r[s] = (int)(signed char)bi[i];
            nd.r4c[s] = (int)(signed char)bi[D + i];
        } else {
            nd.v[s] = 0.0; nd.u[s] = 0.0; nd.c4r[s] = -1; nd.r4c[s] = -1;
        }
        forbBits |= ((meta[s] >> lane) & 1u) << s;
    }
    activeCol = (int)meta[R];
}

template <int R>
__device__ __forceinline__ void publish_cols(const WarpSmem& sm, const Node<R>& nd, const int lane) {
    __syncwarp();  // earlier readers of the mirrors (gain, new row) are done before they are overwritten
#pragma unroll
    for (int s = 0; s < R; ++s) {
        sm.u[lane + 32 * s] = nd.u[s];
        sm.r4c[lane + 32 * s] = (short)nd.r4c[s];
        sm.c4r[lane + 32 * s] = (unsigned short)nd.c4r[s];
    }
    __syncwarp();
}

// makeCostMatrixSafe (:534-569): shift so every entry is >= 0; returns the shift.
__device__ __forceinline__ double stage_safe_matrix(const double* Cg, double* Cs, const int numEl,
                                                    const bool maximize, const bool makeSafe, const int lane) {
    if (!makeSafe) {
        for (int i = lane; i < numEl; i += 32) Cs[i] = Cg[i] + 0.0;  // + 0.0: no -0.0 in the staged matrix
        __syncwarp();
        return 0.0;
    }
    double d;
    if (!maximize) {
        d = CUDART_INF;
        for (int i = lane; i < numEl; i += 32) { const double x = Cg[i]; d = (x < d) ? x : d; }
        d = warp_min(d);
        for (int i = lane; i < numEl; i += 32) Cs[i] = (Cg[i] - d) + 0.0;
    } else {
        d = -CUDART_INF;
        for (int i = lane; i < numEl; i += 32) { const double x = Cg[i]; d = (d < x) ? x : d; }
        d = warp_max(d);
        for (int i = lane; i < numEl; i += 32) Cs[i] = (-Cg[i] + d) + 0.0;
    }
    __syncwarp();
    return d;
}

struct EmitPtrs { int64_t* c4r; int64_t* r4c; double* gain; };
__device__ __forceinline__ EmitPtrs emit_ptrs(const MurtyArgs& a, const long long p) {
    EmitPtrs e;
    e.c4r = a.c4rBest ? a.c4rBest + a.c4rOff[p] : nullptr;
    e.r4c = a.r4cBest ? a.r4cBest + a.r4cOff[p] : nullptr;
    e.gain = a.gainBest ? a.gainBest + p * (long long)a.k : nullptr;
    return e;
}
template <int R>
__device__ __forceinline__ void emit(const EmitPtrs& e, const int slot, const int n, const int nc, const Node<R>& nd,
                                     const double gainOut, const int lane) {
    if (e.c4r) {
        int64_t* o = e.c4r + (int64_t)slot * n;
#pragma unroll
        for (int s = 0; s < R; ++s) if (lane + 32 * s < n) o[lane + 32 * s] = (int64_t)nd.c4r[s];
    }
    if (e.r4c) {
        int64_t* o = e.r4c + (int64_t)slot * nc;
#pragma unroll
        for (int s = 0; s < R; ++s) if (lane + 32 * s < nc) o[lane + 32 * s] = (int64_t)nd.r4c[s];
    }
    if (e.gain && lane == 0) e.gain[slot] = gainOut;
}
template <int R>
__device__ __forceinline__ void emit(const MurtyArgs& a, const long long p, const int slot, const int n, const int nc,
                                     const Node<R>& nd, const double gainOut, const int lane) {
    emit<R>(emit_ptrs(a, p), slot, n, nc, nd, gainOut, lane);
}

// assignmentProb / bruteForceProb accumulation of one hypothesis (assignment.cpp:620-640, 916-937)
template <int R>
__device__ __forceinline__ void add_weight(const MurtyArgs& a, const WarpSmem& sm, const Node<R>& nd, const int nc,
                                           const int nL, const double best, const double gainOut, double& total,
                                           const int lane) {
    if (a.weightMode == PDA_WEIGHTS_GATED && !(best + a.weightGate > gainOut)) return;
    const double w = exp(best - gainOut);
    total += w;
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int c = lane + 32 * s;
        if (c < nc) {
            const int to = nd.r4c[s] >= nL ? nL : nd.r4c[s];
            sm.acc[c * (nL + 1) + to] += w;
        }
    }
}

// ---- k ladder (MurtyLadder, pda_internal.h) -----------------------------------------------------------
// nFound of every slot of problem p from the count reached by the enumeration to the largest rung; thread t < nSlots
// writes slot t.  min(k, count) keeps -1 (malformed) and 0 (infeasible) as they are.
__device__ __forceinline__ void ladder_found(const MurtyArgs& a, const MurtyLadder& L, const long long p, const int count,
                                             const int t) {
    if (t < L.nSlots) {
        const int k = L.rung[L.slotRung[t]];
        a.nFound[p * L.nSlots + t] = count < k ? count : k;
    }
}
// v into cell `cell` of every slot of problem p whose rung lies in [rLo, rHi]
__device__ __forceinline__ void ladder_put(const MurtyArgs& a, const MurtyLadder& L, const long long p, const int rLo,
                                           const int rHi, const int cells, const int cell, const double v) {
    double* out = a.probs + a.probOff[p] + cell;
    for (int j = 0; j < L.nSlots; ++j)
        if (L.slotRung[j] >= rLo && L.slotRung[j] <= rHi) out[(long long)j * cells] = v;
}
// Warp kernel: hypothesis h has just been added to the accumulators.  If it is the last one of rung `rungAt`
// (rungK == h + 1), that rung's tables are stored with the end-of-problem expression and the next rung comes up.
__device__ __forceinline__ void ladder_step(const MurtyArgs& a, const MurtyLadder& L, const long long p, const WarpSmem& sm,
                                            const int h, const int cells, const double total, int& rungAt, int& rungK,
                                            const int lane) {
    if (h + 1 != rungK) return;
    __syncwarp();  // lanes own different columns of acc
    const double norm = 1.0 / total;
    for (int i = lane; i < cells; i += 32) ladder_put(a, L, p, rungAt, rungAt, cells, i, sm.acc[i] * norm);
    __syncwarp();  // read before the next hypothesis is added
    ++rungAt;
    rungK = rungAt < L.nRungs ? L.rung[rungAt] : 0;
}

}  // namespace
}  // namespace pda
#endif
