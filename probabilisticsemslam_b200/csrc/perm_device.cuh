// perm_device.cuh -- device pieces of permanentProb shared by permanentProb / conditionedPermanent
// (permprob_device_kernel.cu), the permanent kernel's subset DP (permanent_kernel.cu) and the fused conditioned-permanent
// pipeline (association_perm_kernel.cu).  All of them run the SAME code here, so their results agree bit for bit.
#ifndef PDA_PERM_DEVICE_CUH
#define PDA_PERM_DEVICE_CUH

#include <math_constants.h>

#include "pda_internal.h"

namespace pda {

__device__ __forceinline__ double warp_max(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { double y = __shfl_xor_sync(0xffffffffu, x, o); x = (x < y) ? y : x; }
    return x;
}
__device__ __forceinline__ double warp_min(double x) {
#pragma unroll
    for (int o = 16; o; o >>= 1) { double y = __shfl_xor_sync(0xffffffffu, x, o); x = (y < x) ? y : x; }
    return x;
}

// The sub-matrix of one permanentProb item, read in place: `base` (ld rows) without row skipRow and column skipCol, with
// S(patchRow, 0) overridden (assignment.cpp:237-239).
struct Gather {
    const double* base; int ld, sR, sC;
    int skipRow, skipCol;        // row / column of `base` that is left out (-1 = none)
    int patchRow; double patchVal;  // S(patchRow, 0) is overridden (assignment.cpp:237-239), -1 = none
    __device__ __forceinline__ double at(int i, int j) const {
        if (i == patchRow && j == 0) return patchVal;
        const int r = (skipRow >= 0 && i >= skipRow) ? i + 1 : i;
        const int c = (skipCol >= 0 && j >= skipCol) ? j + 1 : j;
        return base[r + (size_t)c * ld];
    }
};

// Item (m, l) of permanentProb on the nR x nM likelihood matrix P with nL landmark rows (assignment.cpp:213-246):
// l < nL drops landmark row l, l == nL the dummy row of detection m (with the patch of :233-239).  Returns whether the
// item contributes at all (:217: a zero likelihood skips the sub-permanent).
__device__ __forceinline__ bool item_gather(const double* P, int nL, int nM, int m, int l, Gather& g) {
    const int nR = nL + nM;
    g.base = P; g.ld = nR; g.sR = nR - 1; g.sC = nM - 1;
    g.skipCol = m; g.patchRow = -1; g.patchVal = 0.0;
    bool active = true;
    if (l < nL) {
        g.skipRow = l;
        active = g.base[l + (size_t)m * nR] != 0.0;  // assignment.cpp:217
    } else {
        g.skipRow = nL;  // after the l-loop every landmark row is back; dummy row 0 is the one missing
        if (m != 0) { g.patchRow = nL - 1 + m; g.patchVal = g.base[nL]; }
    }
    return active;
}

// conditionedPermanent's conditioning (assignment.cpp:355-379) by one warp: the columns with a positive entry and their
// scale 1/sqrt(max * smallest positive entry), then the rows with a positive entry, both in order.  keepR needs room
// for g.sR entries, keepC and scale for g.sC.
__device__ __forceinline__ void condition_warp(const Gather& g, double* scale, short* keepC, short* keepR, const int lane,
                                               int& nKR, int& nKC) {
    nKC = 0;
    for (int j = 0; j < g.sC; ++j) {  // column statistics (:355-370)
        double mx = -CUDART_INF, mn = 1.0;
        for (int i = lane; i < g.sR; i += 32) {
            const double e = g.at(i, j);
            mx = (mx < e) ? e : mx;
            if (e > 0.0 && e < mn) mn = e;
        }
        mx = warp_max(mx);
        mn = warp_min(mn);
        if (mx > 0.0) {
            if (lane == 0) { keepC[nKC] = (short)j; scale[nKC] = 1.0 / sqrt(mx * mn); }
            nKC++;
        }
    }
    nKR = 0;
    for (int i0 = 0; i0 < g.sR; i0 += 32) {  // rows with any positive entry (:372-379), order preserved
        const int i = i0 + lane;
        bool keep = false;
        if (i < g.sR)
            for (int j = 0; j < g.sC; ++j) if (g.at(i, j) > 0.0) { keep = true; break; }
        const unsigned mk = __ballot_sync(0xffffffffu, keep);
        if (keep) keepR[nKR + __popc(mk & ((1u << lane) - 1u))] = (short)i;
        nKR += __popc(mk);
    }
    __syncwarp();
}

// The scaled kept sub-matrix (:381-395): transposed (nKC x nKR, the first attempt) or as is (nKR x nKC, the retry).
__device__ __forceinline__ void write_scaled(const Gather& g, const double* scale, const short* keepC, const short* keepR,
                                             const int nKR, const int nKC, const int transpose, double* M, const int lane) {
    for (int e = lane; e < nKR * nKC; e += 32) {
        const int ii = e / nKC, jj = e % nKC;
        const double val = scale[jj] * g.at(keepR[ii], keepC[jj]);
        if (transpose) M[jj + (size_t)ii * nKC] = val;  // Ascaled^T is nKC x nKR
        else M[ii + (size_t)jj * nKR] = val;
    }
}

// scaleFactor of :396-400: the product of the column scales, in column order
__device__ __forceinline__ double scale_product(const double* scale, const int nKC) {
    double sf = 1.0;
    for (int jj = 0; jj < nKC; ++jj) sf *= scale[jj];
    return sf;
}

// Sum over injective maps of the short side of the rows x cols matrix A (column-major) into its long side, by the subset
// dynamic programme over the short side (see perm_dp_warp in permanent_kernel.cu):
//     f_j[S] = f_{j-1}[S] + sum_{i in S} B[i, j] * f_{j-1}[S \ {i}],        perm = f_n[all].
// One warp; f double-buffered at buf[0, cap) and buf[cap, 2 cap), the current long-side line at buf[2 cap, 2 cap + 16);
// the short side must be <= min(log2(cap), 16).  Every lane returns the result.
__device__ __forceinline__ double perm_dp_subsets(const double* A, const int rows, const int cols, double* buf, const int cap,
                                                  const int lane) {
    const int m = rows < cols ? rows : cols, n = rows < cols ? cols : rows;
    const int states = 1 << m;
    double* cur = buf;
    double* nxt = cur + cap;
    double* sb = cur + 2 * cap;
    for (int S = lane; S < states; S += 32) cur[S] = (S == 0) ? 1.0 : 0.0;
    const bool shortRows = rows <= cols;
    for (int j = 0; j < n; ++j) {
        __syncwarp();
        if (lane < m) sb[lane] = shortRows ? A[lane + (size_t)j * rows] : A[j + (size_t)lane * rows];
        __syncwarp();
        for (int S = lane; S < states; S += 32) {
            double acc = cur[S];
            unsigned bits = (unsigned)S;
            while (bits) {
                const int i = __ffs(bits) - 1;
                bits &= bits - 1u;
                acc = fma(sb[i], cur[S ^ (1 << i)], acc);
            }
            nxt[S] = acc;
        }
        double* t = cur; cur = nxt; nxt = t;
    }
    __syncwarp();
    return cur[states - 1];
}

}  // namespace pda
#endif
