// perm_walk.cuh -- the Nijenhuis-Wilf walk of permanent_kernel.cu (see there): error-free double-double sums, the
// three walk variants, the shared-memory layout, the register budget and the launch shape.  permprob_device_kernel.cu
// walks its materialised sub-permanents with the same code and the same shape, so both give the same bits.
#ifndef PDA_PERM_WALK_CUH
#define PDA_PERM_WALK_CUH

#include "pda_internal.h"

namespace pda {
namespace {

constexpr int PERM_THREADS = 256;

struct dd { double hi, lo; };

__device__ __forceinline__ void two_sum(double a, double b, double& s, double& e) {
    s = a + b;
    const double bb = s - a;
    e = (a - (s - bb)) + (b - bb);
}
__device__ __forceinline__ dd dd_add(dd a, dd b) {
    double s, e;
    two_sum(a.hi, b.hi, s, e);
    e += a.lo + b.lo;
    dd r;
    r.hi = s + e;
    r.lo = e - (r.hi - s);
    return r;
}

// n! for n = 0..32, correctly rounded (tgamma(n+1) of nwPerm.cpp:223)
__constant__ double kFactorial[33] = {
    1.0, 1.0, 2.0, 6.0, 24.0, 120.0, 720.0, 5040.0, 40320.0, 362880.0, 3628800.0, 39916800.0, 479001600.0,
    6227020800.0, 87178291200.0, 1307674368000.0, 20922789888000.0, 355687428096000.0, 6402373705728000.0,
    121645100408832000.0, 2432902008176640000.0, 51090942171709440000.0, 1124000727777607680000.0,
    25852016738884976640000.0, 620448401733239439360000.0, 15511210043330985984000000.0,
    403291461126605635584000000.0, 10888869450418352160768000000.0, 304888344611713860501504000000.0,
    8841761993739701954543616000000.0, 265252859812191058636308480000000.0,
    8222838654177922817725562880000000.0, 263130836933693530167218012160000000.0};

#ifndef PERM_CHAINS
#define PERM_CHAINS 4
#endif
#ifndef PERM_UNROLL
#define PERM_UNROLL 1
#endif
constexpr int kPermUnroll = PERM_UNROLL;  // subsets per loop trip

// Leading dimension of the matrix in shared memory.  When the threads of a warp flip DIFFERENT columns (the first
// index of every aligned chunk) each lane reads column k at k*LD + j; with LD == NP the columns of a 24-row matrix
// start only two distinct 128-byte phases apart and those reads serialise (ncu: a third of all shared-memory
// wavefronts of the kernel were bank conflicts).  LD*8 bytes == an odd multiple of 16 modulo 128 spreads eight
// consecutive columns over all eight 16-byte slots of a 128-byte line.
__host__ __device__ constexpr int perm_ld(int np) { return ((np + 2) / 2) % 2 ? np + 2 : np + 4; }

// Walks Gray indices [i0, i1) of the NW sum: seeds x for the subset gray(i0), adds its term, then steps.
// Correct for ANY i0, i1; the column index ctz(i) is warp-uniform whenever it is below log2(chunk).
template <int NP>
__device__ __forceinline__ dd walk_range(const double* __restrict__ sA, const double* __restrict__ sBase,
                                         const unsigned long long i0, const unsigned long long i1) {
    double x[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) x[j] = sBase[j];
    unsigned long long g = i0 ^ (i0 >> 1);
    while (g) {
        const int b = __ffsll((long long)g) - 1;
        g &= g - 1;
        const double* col = sA + b * perm_ld(NP);
#pragma unroll
        for (int j = 0; j < NP; j += 2) {
            const double2 a = *reinterpret_cast<const double2*>(col + j);
            x[j] += a.x;
            x[j + 1] += a.y;
        }
    }
    double hi, lo = 0.0;
    {
        double p0 = 1.0, p1 = 1.0, p2 = 1.0, p3 = 1.0;
#pragma unroll
        for (int j = 0; j < NP; ++j) {
            if ((j & 3) == 0) p0 *= x[j];
            else if ((j & 3) == 1) p1 *= x[j];
            else if ((j & 3) == 2) p2 *= x[j];
            else p3 *= x[j];
        }
        const double prod = (p0 * p1) * (p2 * p3);
        hi = (i0 & 1ULL) ? -prod : prod;
    }
#pragma unroll kPermUnroll
    for (unsigned long long i = i0 + 1; i < i1; ++i) {
        const int k = __ffsll((long long)i) - 1;  // the bit in which gray(i) and gray(i-1) differ
        const unsigned long long gray = i ^ (i >> 1);
        const double s = ((gray >> k) & 1ULL) ? 1.0 : -1.0;
        const double* col = sA + k * perm_ld(NP);
        double p[PERM_CHAINS];
#pragma unroll
        for (int c = 0; c < PERM_CHAINS; ++c) p[c] = 1.0;
#pragma unroll
        for (int j = 0; j < NP; j += 2) {
            const double2 a = *reinterpret_cast<const double2*>(col + j);
            x[j] = fma(s, a.x, x[j]);
            x[j + 1] = fma(s, a.y, x[j + 1]);
            p[j % PERM_CHAINS] *= x[j];
            p[(j + 1) % PERM_CHAINS] *= x[j + 1];
        }
#pragma unroll
        for (int w = PERM_CHAINS / 2; w >= 1; w >>= 1)
#pragma unroll
            for (int c = 0; c < w; ++c) p[c] *= p[c + w];
        const double prod = p[0];
        const double term = (i & 1ULL) ? -prod : prod;
        double s2, e;
        two_sum(hi, term, s2, e);
        hi = s2;
        lo += e;
    }
    dd r;
    r.hi = hi;
    r.lo = lo;
    return r;
}

// Variant of walk_range that keeps column 0 in registers.  In Gray-code order every ODD index flips column 0,
// so half of all steps then need no shared-memory read at all.  That matters because a broadcast LDS.128 still
// writes 512 B into the register file: at one column read per subset the kernel is bound by that return path,
// not by the FP64 pipe.  Requires i0 even (ranges are chunk aligned) -- the loop alternates odd / even indices.
template <int NP>
__device__ __forceinline__ dd walk_range_c0(const double* __restrict__ sA, const double* __restrict__ sBase,
                                            const unsigned long long i0, const unsigned long long i1) {
    double x[NP], c0[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) { x[j] = sBase[j]; c0[j] = sA[j]; }
    unsigned long long g = i0 ^ (i0 >> 1);
    while (g) {
        const int b = __ffsll((long long)g) - 1;
        g &= g - 1;
        const double* col = sA + b * perm_ld(NP);
#pragma unroll
        for (int j = 0; j < NP; j += 2) {
            const double2 a = *reinterpret_cast<const double2*>(col + j);
            x[j] += a.x;
            x[j + 1] += a.y;
        }
    }
    double hi, lo = 0.0;
    {
        double p[PERM_CHAINS];
#pragma unroll
        for (int c = 0; c < PERM_CHAINS; ++c) p[c] = 1.0;
#pragma unroll
        for (int j = 0; j < NP; ++j) p[j % PERM_CHAINS] *= x[j];
#pragma unroll
        for (int w = PERM_CHAINS / 2; w >= 1; w >>= 1)
#pragma unroll
            for (int c = 0; c < w; ++c) p[c] *= p[c + w];
        hi = p[0];  // i0 is even: sign +
    }
    for (unsigned long long i = i0 + 1; i < i1; i += 2) {
        {   // odd index i: column 0 from registers; gray bit 0 of an odd i is 1 ^ bit1(i)
            const double s = ((i >> 1) & 1ULL) ? -1.0 : 1.0;
            double p[PERM_CHAINS];
#pragma unroll
            for (int c = 0; c < PERM_CHAINS; ++c) p[c] = 1.0;
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                x[j] = fma(s, c0[j], x[j]);
                p[j % PERM_CHAINS] *= x[j];
            }
#pragma unroll
            for (int w = PERM_CHAINS / 2; w >= 1; w >>= 1)
#pragma unroll
                for (int c = 0; c < w; ++c) p[c] *= p[c + w];
            double s2, e;
            two_sum(hi, -p[0], s2, e);  // odd index: sign -
            hi = s2;
            lo += e;
        }
        const unsigned long long ie = i + 1;
        if (ie < i1) {  // even index: column ctz(ie) >= 1 from shared memory
            const int k = __ffsll((long long)ie) - 1;
            const double s = (((ie ^ (ie >> 1)) >> k) & 1ULL) ? 1.0 : -1.0;
            const double* col = sA + k * perm_ld(NP);
            double p[PERM_CHAINS];
#pragma unroll
            for (int c = 0; c < PERM_CHAINS; ++c) p[c] = 1.0;
#pragma unroll
            for (int j = 0; j < NP; j += 2) {
                const double2 a = *reinterpret_cast<const double2*>(col + j);
                x[j] = fma(s, a.x, x[j]);
                x[j + 1] = fma(s, a.y, x[j + 1]);
                p[j % PERM_CHAINS] *= x[j];
                p[(j + 1) % PERM_CHAINS] *= x[j + 1];
            }
#pragma unroll
            for (int w = PERM_CHAINS / 2; w >= 1; w >>= 1)
#pragma unroll
                for (int c = 0; c < w; ++c) p[c] *= p[c + w];
            double s2, e;
            two_sum(hi, p[0], s2, e);  // even index: sign +
            hi = s2;
            lo += e;
        }
    }
    dd r;
    r.hi = hi;
    r.lo = lo;
    return r;
}

// Small matrices: columns 0 AND 1 in registers.  Column 1 flips at every index == 2 (mod 4), so three steps out of
// four then need no shared-memory read.  Requires i0 == 0 (mod 4) and i1 - i0 a multiple of 4 (ranges are chunk aligned
// with chunk >= 4 whenever this variant is selected).
template <int NP>
__device__ __forceinline__ dd walk_range_c01(const double* __restrict__ sA, const double* __restrict__ sBase,
                                             const unsigned long long i0, const unsigned long long i1) {
    double x[NP], c0[NP], c1[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) { x[j] = sBase[j]; c0[j] = sA[j]; c1[j] = sA[perm_ld(NP) + j]; }
    unsigned long long g = i0 ^ (i0 >> 1);
    while (g) {
        const int b = __ffsll((long long)g) - 1;
        g &= g - 1;
        const double* col = sA + b * perm_ld(NP);
#pragma unroll
        for (int j = 0; j < NP; j += 2) {
            const double2 a = *reinterpret_cast<const double2*>(col + j);
            x[j] += a.x;
            x[j + 1] += a.y;
        }
    }
    auto product = [&]() {
        double p[PERM_CHAINS];
#pragma unroll
        for (int c = 0; c < PERM_CHAINS; ++c) p[c] = 1.0;
#pragma unroll
        for (int j = 0; j < NP; ++j) p[j % PERM_CHAINS] *= x[j];
#pragma unroll
        for (int w = PERM_CHAINS / 2; w >= 1; w >>= 1)
#pragma unroll
            for (int c = 0; c < w; ++c) p[c] *= p[c + w];
        return p[0];
    };
    double hi = product(), lo = 0.0;  // i0 is even: sign +
    auto add = [&](double term) {
        double s2, e;
        two_sum(hi, term, s2, e);
        hi = s2;
        lo += e;
    };
    for (unsigned long long i = i0; i < i1; i += 4) {
        if (i != i0) {  // index i == 0 (mod 4): column ctz(i) >= 2 from shared memory
            const int k = __ffsll((long long)i) - 1;
            const double s = (((i ^ (i >> 1)) >> k) & 1ULL) ? 1.0 : -1.0;
            const double* col = sA + k * perm_ld(NP);
#pragma unroll
            for (int j = 0; j < NP; j += 2) {
                const double2 a = *reinterpret_cast<const double2*>(col + j);
                x[j] = fma(s, a.x, x[j]);
                x[j + 1] = fma(s, a.y, x[j + 1]);
            }
            add(product());
        }
        {   // i + 1 (odd): column 0; gray bit 0 = 1 ^ bit 1 of the index = 1  -> +
#pragma unroll
            for (int j = 0; j < NP; ++j) x[j] += c0[j];
            add(-product());
        }
        {   // i + 2: column 1; gray bit 1 = 1 ^ bit 2 of the index
            const double s = ((i >> 2) & 1ULL) ? -1.0 : 1.0;
#pragma unroll
            for (int j = 0; j < NP; ++j) x[j] = fma(s, c1[j], x[j]);
            add(product());
        }
        {   // i + 3 (odd): column 0; gray bit 0 = 1 ^ bit 1 = 0  -> -
#pragma unroll
            for (int j = 0; j < NP; ++j) x[j] -= c0[j];
            add(-product());
        }
    }
    dd r;
    r.hi = hi;
    r.lo = lo;
    return r;
}

#ifndef PERM_C0_MAX
#define PERM_C0_MAX 32
#endif
#ifndef PERM_C01_MAX
#define PERM_C01_MAX 16
#endif
__host__ __device__ constexpr bool perm_cache01(int np) { return np <= PERM_C01_MAX; }
__host__ __device__ constexpr bool perm_cache0(int np) { return np <= PERM_C0_MAX; }
// resident CTAs per SM the register allocator must leave room for
__host__ __device__ constexpr int perm_min_blocks(int np) {
    if (perm_cache01(np)) return np <= 8 ? 4 : 2;
    return perm_cache0(np) ? (np <= 12 ? 4 : (np <= 16 ? 3 : 2)) : (np <= 16 ? 4 : (np <= 24 ? 3 : 2));
}

}  // namespace

// Launch shape for a batch whose largest dimension is maxDim: threads that share a matrix (small matrices get
// one warp each, eight to a CTA), CTAs per matrix (a few large matrices are spread over the whole chip, in
// multiples that fill 2 CTAs per SM evenly), and the alignment of the per-thread index ranges.
struct PermShape { int threadsPerMat, ctasPerMat, chunk; };
__host__ __device__ inline PermShape perm_shape(int64_t nMats, int maxDim, int smCount, unsigned long long rangeLen) {
    const int n = maxDim < 1 ? 1 : (maxDim > PDA_MAX_PERM_DIM ? PDA_MAX_PERM_DIM : maxDim);
    const unsigned long long steps = rangeLen ? rangeLen : (1ULL << (n - 1));
    PermShape sh;
    int tpm = 32;
    while (tpm < PERM_THREADS && (unsigned long long)tpm * 64 < steps) tpm *= 2;
    sh.threadsPerMat = tpm;
    const long long slots = PERM_THREADS / tpm;
    const long long ctasForBatch = (nMats + slots - 1) / slots;
    long long cpm = 1;
    if (tpm == PERM_THREADS) {
        // few large matrices: spread each over the chip.  Prefer a CTA count that fills every SM evenly
        // (a multiple of the SM count) while leaving >= 96 subsets per thread; otherwise as many as the work allows.
        const int np = (n + 1) / 2 * 2 < 2 ? 2 : (n + 1) / 2 * 2;
        const unsigned long long w = steps / ((unsigned long long)PERM_THREADS * 96);
        const long long byWork = (long long)(w < 1 ? 1 : w);
        const long long perSmMax = perm_min_blocks(np);
        long long total = byWork * ctasForBatch < perSmMax * smCount ? byWork * ctasForBatch : perSmMax * smCount;  // CTAs for the whole batch
        if (total >= smCount) total = total / smCount * smCount;
        const long long c = total / ctasForBatch < 4096LL ? total / ctasForBatch : 4096LL;
        cpm = c < 1 ? 1 : c;
    }
    sh.ctasPerMat = (int)cpm;
    const unsigned long long q = steps / ((unsigned long long)cpm * tpm);
    const unsigned long long perThread = q < 1 ? 1 : q;
    int chunk = 1;
    while (chunk < 32 && (unsigned long long)chunk * 2 * 6 <= perThread) chunk *= 2;  // >= 6 chunks per thread keeps the shares even
    sh.chunk = chunk;
    return sh;
}

}  // namespace pda
#endif
