// pda_capi.cu -- the extern "C" surface of libpda_b200.so (include/pda_b200.h):
// argument checking, workspace geometry, kernel launches, and the *_host convenience
// entry points that stage host buffers through a cached, grow-only device arena.
// There is deliberately no CPU path in here: without a CUDA device every compute
// call fails with PDA_ERR_CUDA.
#include "pda_internal.h"
#include "pda_host_stage.h"

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

namespace pda {

static thread_local char g_err[512] = "";
static thread_local unsigned long long g_failures = 0;
unsigned long long failure_count() { return g_failures; }

int fail(int code, const char* fmt, ...) {
    ++g_failures;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    ++g_failures;
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    (void)cudaGetLastError();
    return PDA_ERR_CUDA;
}

int current_device_info(DeviceInfo* out) {
    int dev = 0;
    PDA_CUDA_TRY(cudaGetDevice(&dev));
    static std::mutex mu;
    static std::vector<DeviceInfo> cache;
    std::lock_guard<std::mutex> lk(mu);
    for (const DeviceInfo& d : cache)
        if (d.device == dev) { *out = d; return PDA_OK; }
    DeviceInfo d;
    d.device = dev;
    PDA_CUDA_TRY(cudaDeviceGetAttribute(&d.smCount, cudaDevAttrMultiProcessorCount, dev));
    PDA_CUDA_TRY(cudaDeviceGetAttribute(&d.maxSmemOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cache.push_back(d);
    *out = d;
    return PDA_OK;
}

static std::atomic<uint64_t> g_approxSeed{20260217ULL};
uint64_t approx_seed() { return g_approxSeed.load(); }

DeviceCtx g_dev[PDA_MAX_DEVICES];

static std::mutex g_pinMu;
static std::vector<std::pair<const unsigned char*, size_t> > g_pinRanges;  // pda_host_alloc's buffers
bool in_portable_range(const void* p) {
    std::lock_guard<std::mutex> lk(g_pinMu);
    for (const auto& r : g_pinRanges)
        if ((const unsigned char*)p >= r.first && (const unsigned char*)p < r.first + r.second) return true;
    return false;
}

}  // namespace pda

using namespace pda;

// FP64 pipe micro-benchmark: 8 independent DFMA chains per thread (diagnostic; gives the measured
// denominator for the permanent kernel's roofline, which MEASURED_PEAKS.json does not carry).
__global__ void dfma_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
    double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double b = 0.999999, c = 1e-7;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" {

double pda_diag_dfma_tflops(void) {
    DeviceInfo dev;
    if (current_device_info(&dev)) return -1.0;
    const int ctas = dev.smCount * 8, threads = 256, iters = 8192;
    double* out = nullptr;
    if (cudaMalloc(&out, (size_t)ctas * threads * 8) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    dfma_peak_kernel<<<ctas, threads>>>(out, iters);
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        dfma_peak_kernel<<<ctas, threads>>>(out, iters);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double tf = 2.0 * 8.0 * iters * (double)ctas * threads / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    return cudaGetLastError() == cudaSuccess ? best : -1.0;
}

int pda_version(void) { return 100; }
void pda_set_approx_seed(uint64_t seed) { g_approxSeed.store(seed); }
const char* pda_last_error(void) { return g_err; }
int pda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}

void* pda_host_alloc(int64_t bytes) {
    if (bytes <= 0) { fail(PDA_ERR_INVALID, "pda_host_alloc: bytes <= 0"); return nullptr; }
    void* p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocPortable | cudaHostAllocMapped);
    if (e != cudaSuccess) { cuda_fail(e, "cudaHostAlloc(pda_host_alloc)"); return nullptr; }
    std::lock_guard<std::mutex> lk(g_pinMu);
    g_pinRanges.push_back(std::make_pair((const unsigned char*)p, (size_t)bytes));
    return p;
}
void pda_host_free(void* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_pinMu);
        for (size_t i = 0; i < g_pinRanges.size(); ++i)
            if (g_pinRanges[i].first == (const unsigned char*)p) { g_pinRanges.erase(g_pinRanges.begin() + (long)i); break; }
    }
    cudaFreeHost(p);
}

// ---------------------------------------------------------------------------------------- Murty
// room for the cost-ordered problem list at the tail of the workspace (only worth it when warps take several problems)
static int64_t order_bytes(int64_t nProblems) { return (nProblems + 63) / 64 * 256; }

static int64_t murty_full_warps(const MurtyGeometry& g, const DeviceInfo& dev) {
    const int64_t exact = (int64_t)dev.smCount * g.ctasPerSm * g.warpsPerCta;
    const int64_t fast = g.fastOk ? (int64_t)dev.smCount * g.fastCtasPerSm * g.fastWarpsPerCta : 0;
    return std::max(exact, fast);  // one arena per warp of whichever kernel keeps more of them resident
}

// Which kernel a batch goes to.  One CTA per problem (murty_cta_kernel.cu) is the latency path: it wins while the batch
// is too small to give every SM ~4 problems' worth of warps, and loses beyond (it spends 16 warps on one problem).
static std::atomic<int> g_murtyPath{PDA_MURTY_PATH_AUTO};
static bool cta_eligible(int64_t nProblems, int32_t maxNumCol, const DeviceInfo& dev) {
    const int path = g_murtyPath.load();
    if (path == PDA_MURTY_PATH_WARP || path == PDA_MURTY_PATH_FAST || maxNumCol > PDA_CTA_MAX_COL) return false;
    return path == PDA_MURTY_PATH_CTA || nProblems <= 4LL * dev.smCount;
}

int64_t pda_murty_workspace_bytes(int64_t nProblems, int32_t k, int32_t maxNumRow, int32_t maxNumCol) {
    DeviceInfo dev;
    int rc = current_device_info(&dev);
    if (rc) return rc;
    MurtyGeometry g;
    rc = murty_geometry(k, maxNumRow, maxNumCol, false, dev, &g);
    if (rc) return rc;
    int64_t warps = std::min<int64_t>(std::max<int64_t>(nProblems, 1), murty_full_warps(g, dev));
    int64_t bytes = 256 + warps * g.arenaStride + 2 * order_bytes(nProblems);  // cost order + fallback list
    if (cta_eligible(nProblems, maxNumCol, dev)) {
        CtaGeometry cg;
        if (murty_cta_geometry(k, maxNumRow, maxNumCol, false, dev, &g, &cg) == PDA_OK) {
            const int64_t ctas = std::min<int64_t>(std::max<int64_t>(nProblems, 1), dev.smCount);
            bytes = std::max<int64_t>(bytes, 256 + ctas * cg.arenaStride);
        }
    }
    return bytes;
}

int pda_murty_set_path(int32_t path) {
    if (path < PDA_MURTY_PATH_AUTO || path > PDA_MURTY_PATH_FAST) return fail(PDA_ERR_INVALID, "murty: bad path %d", path);
    return g_murtyPath.exchange(path);
}

}  // extern "C"

// pda_murty_batch, and with `ladder` the k-ladder form behind pda_assignment_prob_ladder_batch (k = its largest rung;
// nFound and the weight tables then have ladder->nSlots entries per problem).  Path choice and geometry are the same.
static int murty_batch_dev(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                           int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                           int32_t k, int32_t cutMode, double cutoff, int32_t maximize, int32_t cutMaximize,
                           int64_t* row4colBest, const int64_t* r4cOff,
                           int64_t* col4rowBest, const int64_t* c4rOff,
                           double* gainBest, int32_t* nFound,
                           int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                           void* workspace, int64_t workspaceBytes, void* stream, const MurtyLadder* ladder) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "murty: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !nFound) return fail(PDA_ERR_INVALID, "murty: NULL input");
    if ((row4colBest && !r4cOff) || (col4rowBest && !c4rOff)) return fail(PDA_ERR_INVALID, "murty: output given without offsets");
    if (cutMode < PDA_CUT_NONE || cutMode > PDA_CUT_STICKY) return fail(PDA_ERR_INVALID, "murty: bad cutMode %d", cutMode);
    if (weightMode < PDA_WEIGHTS_NONE || weightMode > PDA_WEIGHTS_UNGATED) return fail(PDA_ERR_INVALID, "murty: bad weightMode %d", weightMode);
    if (weightMode && (!probs || !probOff || !nL)) return fail(PDA_ERR_INVALID, "murty: weights requested without probs/probOff/nL");
    if (!workspace) return fail(PDA_ERR_WORKSPACE, "murty: NULL workspace");
    DeviceInfo dev;
    PDA_TRY(current_device_info(&dev));
    MurtyArgs a;
    a.costs = costs; a.costOff = costOff; a.numRow = numRow; a.numCol = numCol; a.nProblems = nProblems;
    a.k = k; a.cutMode = cutMode; a.maximize = maximize; a.cutMaximize = cutMaximize; a.cutoff = cutoff;
    a.r4cBest = row4colBest; a.r4cOff = r4cOff; a.c4rBest = col4rowBest; a.c4rOff = c4rOff;
    a.gainBest = gainBest; a.nFound = nFound;
    a.weightMode = weightMode; a.weightGate = 42.0;  // assignment.cpp:9
    a.probs = probs; a.probOff = probOff; a.nL = nL;
    a.cursor = reinterpret_cast<unsigned long long*>(workspace);
    a.arena = reinterpret_cast<unsigned char*>(workspace) + 256;
    a.order = nullptr;
    a.fallbackCount = reinterpret_cast<unsigned*>(workspace) + 2;
    a.cursor2 = reinterpret_cast<unsigned long long*>(workspace) + 2;
    a.fallbackList = nullptr; a.nProblemsDev = nullptr; a.useFast = 0;
    if (cta_eligible(nProblems, maxNumCol, dev)) {
        const bool forced = g_murtyPath.load() == PDA_MURTY_PATH_CTA;
        CtaGeometry cg;
        int rc = murty_cta_geometry(k, maxNumRow, maxNumCol, weightMode != 0, dev, &a.geo, &cg);
        const int64_t ctas = rc ? 0 : std::min<int64_t>(std::min<int64_t>(nProblems, dev.smCount), (workspaceBytes - 256) / cg.arenaStride);
        if (rc == PDA_OK && ctas >= 1) {
            a.nWarps = (int32_t)ctas;  // arenas == CTAs allowed to run
            return launch_murty_cta(a, cg, reinterpret_cast<cudaStream_t>(stream), ladder);
        }
        if (forced) return rc ? rc : fail(PDA_ERR_WORKSPACE, "murty (CTA path): workspace of %lld B holds no arena (%lld B each)",
                                          (long long)workspaceBytes, (long long)cg.arenaStride);
    }
    PDA_TRY(murty_geometry(k, maxNumRow, maxNumCol, weightMode != 0, dev, &a.geo));
    int64_t warps = std::min<int64_t>(nProblems, murty_full_warps(a.geo, dev));
    // the cost-ordered list goes behind the arenas when the workspace has room for it and there is a tail to shorten
    const bool ordered = nProblems > 2 * warps && nProblems < (1LL << 31) &&
                         workspaceBytes >= 256 + warps * a.geo.arenaStride + order_bytes(nProblems);
    warps = std::min<int64_t>(warps, (workspaceBytes - 256 - (ordered ? order_bytes(nProblems) : 0)) / a.geo.arenaStride);
    if (warps < 1) return fail(PDA_ERR_WORKSPACE, "murty: workspace of %lld B holds no arena (%lld B each)",
                               (long long)workspaceBytes, (long long)a.geo.arenaStride);
    a.nWarps = (int32_t)warps;
    a.order = ordered ? reinterpret_cast<int32_t*>(a.arena + warps * a.geo.arenaStride) : nullptr;
    // The pruning kernel first, the exact kernel behind it for the problems with exact gain ties -- when the geometry
    // admits it, the fallback list fits behind the arenas and the caller has not pinned the exact kernel.
    const int64_t used = 256 + warps * a.geo.arenaStride + (ordered ? order_bytes(nProblems) : 0);
    const int path = g_murtyPath.load();
    if (a.geo.fastOk && path != PDA_MURTY_PATH_WARP && nProblems < (1LL << 31) && workspaceBytes >= used + order_bytes(nProblems)) {
        a.useFast = 1;
        a.fallbackList = reinterpret_cast<int32_t*>(reinterpret_cast<unsigned char*>(workspace) + used);
    }  // else (k <= 2, a list too long for shared-memory group minima, a tight workspace): the exact kernel alone
    return launch_murty(a, reinterpret_cast<cudaStream_t>(stream), ladder);
}

// pda_murty_batch_host, and with `ladder` the staging of pda_assignment_prob_ladder_batch_host (S = ladder->nSlots
// tables and counts per problem).
static int murty_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                            int64_t nProblems, int32_t k, int32_t cutMode, double cutoff, int32_t maximize,
                            int32_t cutMaximize,
                            int64_t* row4colBest, const int64_t* r4cOff,
                            int64_t* col4rowBest, const int64_t* c4rOff,
                            double* gainBest, int32_t* nFound,
                            int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                            int32_t device, const MurtyLadder* ladder) {
    const size_t S = ladder ? (size_t)ladder->nSlots : 1;
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "murty: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !nFound) return fail(PDA_ERR_INVALID, "murty: NULL input");
    if (k < 1) return fail(PDA_ERR_INVALID, "murty: k < 1");
    if (weightMode && (!probs || !probOff || !nL)) return fail(PDA_ERR_INVALID, "murty: weights requested without probs/probOff/nL");
    // Every array is addressed through per-problem offsets; only the range [lo, hi) this batch touches is staged (a
    // shard of a larger batch -- pda_murty_batch_host_multi -- passes the whole arrays and its own slice of offsets).
    int maxR = 0, maxC = 0;
    struct Range { size_t lo = ~(size_t)0, hi = 0; void add(size_t o, size_t n) { lo = std::min(lo, o); hi = std::max(hi, o + n); } size_t len() const { return hi > lo ? hi - lo : 0; } };
    Range rCost, rR4c, rC4r, rProb;
    for (int64_t p = 0; p < nProblems; ++p) {
        const int r = numRow[p], c = numCol[p];
        if (r < 1 || c < 1 || c > r) return fail(PDA_ERR_INVALID, "murty: problem %lld is %d x %d (need numRow >= numCol >= 1)", (long long)p, r, c);
        if (costOff[p] < 0 || (row4colBest && r4cOff[p] < 0) || (col4rowBest && c4rOff[p] < 0) || (weightMode && probOff[p] < 0))
            return fail(PDA_ERR_INVALID, "murty: negative offset at problem %lld", (long long)p);
        maxR = std::max(maxR, r); maxC = std::max(maxC, c);
        rCost.add((size_t)costOff[p], (size_t)r * c);
        if (row4colBest) rR4c.add((size_t)r4cOff[p], (size_t)k * c);
        if (col4rowBest) rC4r.add((size_t)c4rOff[p], (size_t)k * r);
        if (weightMode) {
            if (nL[p] + c != r) return fail(PDA_ERR_INVALID, "murty: problem %lld has nL + numCol != numRow", (long long)p);
            rProb.add((size_t)probOff[p], S * c * (nL[p] + 1));
        }
    }
    const size_t nCost = rCost.len(), nR4c = rR4c.len(), nC4r = rC4r.len(), nProb = rProb.len();
    const size_t loCost = rCost.lo, loR4c = nR4c ? rR4c.lo : 0, loC4r = nC4r ? rC4r.lo : 0, loProb = nProb ? rProb.lo : 0;
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const int64_t wsBytes = pda_murty_workspace_bytes(nProblems, k, maxR, maxC);
    if (wsBytes < 0) return (int)wsBytes;
    const size_t n = (size_t)nProblems;
    // The cost matrices and the weight tables may be used in place (beyond the packed limit, from page-locked memory): a
    // warp reads its 2.4 KB cost matrix over PCIe once when it takes the problem and writes the weight table when it is
    // done, so both transfers hide under ~1.6 ms of computing per problem instead of standing in front of and behind the
    // kernel (161 MB in + 136 MB out per 100 000 problems).
    HostIO io(device);
    const size_t oCost = io.in(costs + loCost, nCost * 8, HostIO::IN_PLACE), oCostOff = io.in(costOff, n * 8);
    const size_t oNR = io.in(numRow, n * 4), oNC = io.in(numCol, n * 4);
    const size_t oR4cOff = io.in(row4colBest ? r4cOff : nullptr, n * 8), oC4rOff = io.in(col4rowBest ? c4rOff : nullptr, n * 8);
    const size_t oProbOff = io.in(weightMode ? probOff : nullptr, n * 8), oNL = io.in(weightMode ? nL : nullptr, n * 4);
    const size_t oFound = io.out(nFound, n * 4 * S), oGain = io.out(gainBest, gainBest ? n * (size_t)k * 8 : 0);
    const size_t oProb = io.out(weightMode ? probs + loProb : nullptr, nProb * 8, HostIO::IN_PLACE);
    const size_t oR4c = io.out(row4colBest ? row4colBest + loR4c : nullptr, nR4c * 8), oC4r = io.out(col4rowBest ? col4rowBest + loC4r : nullptr, nC4r * 8);
    const size_t oWs = io.scratch((size_t)wsBytes);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    // device-side bases such that base + offset[p] lands inside the staged range
    PDA_TRY(murty_batch_dev(io.at<double>(oCost) - loCost, io.at<int64_t>(oCostOff), io.at<int32_t>(oNR), io.at<int32_t>(oNC), nProblems,
                            maxR, maxC, k, cutMode, cutoff, maximize, cutMaximize,
                            row4colBest ? io.at<int64_t>(oR4c) - loR4c : nullptr, io.at<int64_t>(oR4cOff),
                            col4rowBest ? io.at<int64_t>(oC4r) - loC4r : nullptr, io.at<int64_t>(oC4rOff),
                            gainBest ? io.at<double>(oGain) : nullptr, io.at<int32_t>(oFound),
                            weightMode, weightMode ? io.at<double>(oProb) - loProb : nullptr, io.at<int64_t>(oProbOff),
                            io.at<int32_t>(oNL), io.at<unsigned char>(oWs), wsBytes, io.stream(), ladder));
    return io.download();
}

// ks (host) -> the ladder: rungs = the sorted distinct ks, slot j -> the rung equal to ks[j]
static int make_ladder(const int32_t* ks, int32_t nK, MurtyLadder* L) {
    if (!ks) return fail(PDA_ERR_INVALID, "ladder: NULL ks");
    if (nK < 1 || nK > PDA_LADDER_MAX) return fail(PDA_ERR_INVALID, "ladder: need 1 <= nK <= %d (got %d)", PDA_LADDER_MAX, nK);
    for (int j = 0; j < nK; ++j)
        if (ks[j] < 1) return fail(PDA_ERR_INVALID, "ladder: ks[%d] = %d (need k >= 1)", j, ks[j]);
    std::vector<int32_t> r(ks, ks + nK);
    std::sort(r.begin(), r.end());
    r.erase(std::unique(r.begin(), r.end()), r.end());
    memset(L, 0, sizeof(*L));
    L->nRungs = (int32_t)r.size();
    L->nSlots = nK;
    for (size_t i = 0; i < r.size(); ++i) L->rung[i] = r[i];
    for (int j = 0; j < nK; ++j) L->slotRung[j] = (int32_t)(std::lower_bound(r.begin(), r.end(), ks[j]) - r.begin());
    return PDA_OK;
}

extern "C" {

int pda_murty_batch(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                    int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                    int32_t k, int32_t cutMode, double cutoff, int32_t maximize, int32_t cutMaximize,
                    int64_t* row4colBest, const int64_t* r4cOff,
                    int64_t* col4rowBest, const int64_t* c4rOff,
                    double* gainBest, int32_t* nFound,
                    int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                    void* workspace, int64_t workspaceBytes, void* stream) {
    return murty_batch_dev(costs, costOff, numRow, numCol, nProblems, maxNumRow, maxNumCol, k, cutMode, cutoff, maximize,
                           cutMaximize, row4colBest, r4cOff, col4rowBest, c4rOff, gainBest, nFound, weightMode, probs, probOff,
                           nL, workspace, workspaceBytes, stream, nullptr);
}

int pda_murty_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                         int64_t nProblems, int32_t k, int32_t cutMode, double cutoff, int32_t maximize,
                         int32_t cutMaximize,
                         int64_t* row4colBest, const int64_t* r4cOff,
                         int64_t* col4rowBest, const int64_t* c4rOff,
                         double* gainBest, int32_t* nFound,
                         int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                         int32_t device) {
    return murty_batch_host(costs, costOff, numRow, numCol, nProblems, k, cutMode, cutoff, maximize, cutMaximize, row4colBest,
                            r4cOff, col4rowBest, c4rOff, gainBest, nFound, weightMode, probs, probOff, nL, device, nullptr);
}

// assignmentProb's settings (assignment.cpp:547-683, as in the assignmentProb shim): kBest2DCutoff with cutoff 42, gated
// weights, no lists
int pda_assignment_prob_ladder_batch(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                                     const int32_t* nL, int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                                     const int32_t* ks, int32_t nK, double* probs, const int64_t* probOff, int32_t* nFound,
                                     void* workspace, int64_t workspaceBytes, void* stream) {
    MurtyLadder L;
    PDA_TRY(make_ladder(ks, nK, &L));
    return murty_batch_dev(costs, costOff, numRow, numCol, nProblems, maxNumRow, maxNumCol, L.rung[L.nRungs - 1], PDA_CUT_RELATIVE,
                           42.0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nFound, PDA_WEIGHTS_GATED, probs, probOff, nL,
                           workspace, workspaceBytes, stream, &L);
}

int pda_assignment_prob_ladder_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow,
                                          const int32_t* numCol, const int32_t* nL, int64_t nProblems, const int32_t* ks,
                                          int32_t nK, double* probs, const int64_t* probOff, int32_t* nFound, int32_t device) {
    MurtyLadder L;
    PDA_TRY(make_ladder(ks, nK, &L));
    return murty_batch_host(costs, costOff, numRow, numCol, nProblems, L.rung[L.nRungs - 1], PDA_CUT_RELATIVE, 42.0, 0, 0,
                            nullptr, nullptr, nullptr, nullptr, nullptr, nFound, PDA_WEIGHTS_GATED, probs, probOff, nL, device, &L);
}

// One host thread per device, each running the single-device call on a contiguous slice of the batch (SURVEY.md 8e:
// independent problems, no data-path collective, results land directly in the caller's arrays).
int pda_murty_batch_host_multi(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                               int64_t nProblems, int32_t k, int32_t cutMode, double cutoff, int32_t maximize,
                               int32_t cutMaximize,
                               int64_t* row4colBest, const int64_t* r4cOff,
                               int64_t* col4rowBest, const int64_t* c4rOff,
                               double* gainBest, int32_t* nFound,
                               int32_t weightMode, double* probs, const int64_t* probOff, const int32_t* nL,
                               const int32_t* devices, int32_t nDevices) {
    if (!devices || nDevices < 1) return fail(PDA_ERR_INVALID, "murty (multi): need at least one device");
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "murty: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !nFound) return fail(PDA_ERR_INVALID, "murty: NULL input");
    return run_sharded(nProblems, devices, nDevices, [&](int64_t p0, int64_t p1, int dev) {
        return pda_murty_batch_host(costs, costOff + p0, numRow + p0, numCol + p0, p1 - p0, k, cutMode, cutoff, maximize, cutMaximize,
                                    row4colBest, r4cOff ? r4cOff + p0 : nullptr, col4rowBest, c4rOff ? c4rOff + p0 : nullptr,
                                    gainBest ? gainBest + p0 * (int64_t)k : nullptr, nFound + p0,
                                    weightMode, probs, probOff ? probOff + p0 : nullptr, nL ? nL + p0 : nullptr, dev);
    });
}

// ------------------------------------------------------------------------------------------- LAP
int pda_lap_batch(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                  const int32_t* numCol4Gain, int64_t nProblems, int32_t maxNumRow, int32_t maxNumCol,
                  int32_t makeSafe, int32_t maximize,
                  const int64_t* rowOff, const int64_t* colOff,
                  int64_t* col4row, int64_t* row4col, double* u, double* v, uint8_t* forbidden,
                  double* gain, int32_t* feasible, void* stream) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "lap: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !rowOff || !colOff) return fail(PDA_ERR_INVALID, "lap: NULL input");
    if (maxNumRow < 1 || maxNumCol < 0 || maxNumCol > maxNumRow) return fail(PDA_ERR_INVALID, "lap: bad maximal dimensions");
    LapArgs a = {costs, costOff, numRow, numCol, numCol4Gain, nProblems, makeSafe, maximize, rowOff, colOff,
                 col4row, row4col, u, v, forbidden, gain, feasible, maxNumRow, std::max(maxNumCol, 1)};
    return launch_lap(a, reinterpret_cast<cudaStream_t>(stream));
}

int pda_lap_batch_host(const double* costs, const int64_t* costOff, const int32_t* numRow, const int32_t* numCol,
                       const int32_t* numCol4Gain, int64_t nProblems, int32_t makeSafe, int32_t maximize,
                       const int64_t* rowOff, const int64_t* colOff,
                       int64_t* col4row, int64_t* row4col, double* u, double* v, uint8_t* forbidden,
                       double* gain, int32_t* feasible, int32_t device) {
    if (nProblems < 0) return fail(PDA_ERR_INVALID, "lap: nProblems < 0");
    if (nProblems == 0) return PDA_OK;
    if (!costs || !costOff || !numRow || !numCol || !rowOff || !colOff) return fail(PDA_ERR_INVALID, "lap: NULL input");
    int maxR = 0, maxC = 0;
    size_t nCost = 0, nRows = 0, nCols = 0;
    for (int64_t p = 0; p < nProblems; ++p) {
        const int r = numRow[p], c = numCol[p];
        if (r < 1 || c < 0 || c > r) return fail(PDA_ERR_INVALID, "lap: problem %lld is %d x %d", (long long)p, r, c);
        maxR = std::max(maxR, r); maxC = std::max(maxC, c);
        nCost = std::max(nCost, (size_t)costOff[p] + (size_t)r * c);
        nRows = std::max(nRows, (size_t)rowOff[p] + r);
        nCols = std::max(nCols, (size_t)colOff[p] + c);
    }
    DeviceScope scope;
    PDA_TRY(scope.enter(device));
    const size_t n = (size_t)nProblems;
    HostIO io(device);
    const size_t oCost = io.in(costs, nCost * 8), oCostOff = io.in(costOff, n * 8), oNR = io.in(numRow, n * 4), oNC = io.in(numCol, n * 4);
    const size_t oNG = io.in(numCol4Gain, n * 4), oRO = io.in(rowOff, n * 8), oCO = io.in(colOff, n * 8);
    const size_t oC4r = io.out(col4row, nRows * 8), oR4c = io.out(row4col, nCols * 8), oU = io.out(u, nCols * 8), oV = io.out(v, nRows * 8);
    const size_t oF = io.out(forbidden, nRows), oG = io.out(gain, n * 8), oFe = io.out(feasible, n * 4);
    PDA_TRY(io.commit());
    PDA_TRY(io.upload());
    PDA_TRY(pda_lap_batch(io.at<double>(oCost), io.at<int64_t>(oCostOff), io.at<int32_t>(oNR), io.at<int32_t>(oNC),
                          numCol4Gain ? io.at<int32_t>(oNG) : nullptr, nProblems, maxR, maxC, makeSafe, maximize,
                          io.at<int64_t>(oRO), io.at<int64_t>(oCO), io.at<int64_t>(oC4r), io.at<int64_t>(oR4c),
                          io.at<double>(oU), io.at<double>(oV), io.at<uint8_t>(oF), io.at<double>(oG),
                          io.at<int32_t>(oFe), io.stream()));
    return io.download();
}

}  // extern "C"
