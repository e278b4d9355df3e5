// pda_internal.h -- declarations shared by the .cu files of libpda_b200.so.
#ifndef PDA_INTERNAL_H
#define PDA_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>

#include "pda_b200.h"

namespace pda {

// ---- error plumbing (pda_capi.cu) -------------------------------------------------------
int fail(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
unsigned long long failure_count();  // number of fail()/cuda_fail() calls made by this thread
#define PDA_CUDA_TRY(expr)                                           \
    do {                                                             \
        cudaError_t _e = (expr);                                     \
        if (_e != cudaSuccess) return ::pda::cuda_fail(_e, #expr);   \
    } while (0)

struct DeviceInfo {
    int device;
    int smCount;
    int maxSmemOptin;  // bytes per block, opt-in
};
int current_device_info(DeviceInfo* out);

// ---- device workspaces -------------------------------------------------------------------------
// A workspace is laid out as consecutive regions, each starting on a 256-byte boundary.  Every pipeline writes its
// layout once, as a function that takes its regions in order from one of these: over the caller's workspace it hands out
// the pointers, over a null base it only counts, and that count is what the pipeline's *_workspace_bytes returns.
class WorkspaceLayout {
public:
    explicit WorkspaceLayout(void* base) : base_(reinterpret_cast<uintptr_t>(base)) {}
    static size_t round(size_t bytes) { return (bytes + 255) / 256 * 256; }
    template <class T> T* take(size_t count) {
        T* const p = reinterpret_cast<T*>(at());
        off_ += round(count * sizeof(T));
        return p;
    }
    unsigned char* rest() const { return reinterpret_cast<unsigned char*>(at()); }  // where a chained pipeline's workspace starts
    size_t bytes() const { return off_; }
private:
    uintptr_t at() const { return base_ ? base_ + off_ : 0; }
    uintptr_t base_;
    size_t off_ = 0;
};

inline int check_workspace(const char* who, int64_t have, int64_t need) {
    if (have >= need) return PDA_OK;
    return fail(PDA_ERR_WORKSPACE, "%s: workspace of %lld B, %lld B needed", who, (long long)have, (long long)need);
}

// ---- Murty k-best (murty_kernel.cu) ----------------------------------------------------------
struct MurtyGeometry {
    int R;              // row slots per lane: numRow <= 32*R
    int maxCol;         // largest numCol the node slots were counted for
    int nodeDim;        // padded per-node array length
    int nodeStride;     // bytes per stored node
    int maxNodes;       // node slots per warp arena
    int64_t heapBytes;  // bytes of the heap region at the head of each arena
    int64_t arenaStride;
    int smemPerWarp;
    int heapTopOff;     // byte offset of the shared-memory heap top inside a warp's shared region
    int heapTopCap;     // heap entries kept in shared memory
    int cCap;           // doubles reserved for the cost matrix per warp
    int pCap;           // doubles reserved for the weight accumulators per warp
    int warpsPerCta;
    int ctasPerSm;
    // pruning fast path (murty_kernel<R, true>)
    int fastOk;           // geometry admits the fast path
    int pqCap;            // slots of its open list (multiple of 32)
    int pqInSmem;         // list in shared memory (else in the arena's heap region)
    int fastSmemPerWarp;
    int fastWarpsPerCta;
    int fastCtasPerSm;
};
int murty_geometry(int32_t k, int32_t maxNumRow, int32_t maxNumCol, bool weights, const DeviceInfo& dev,
                   MurtyGeometry* g);
// PDA_OK when the k-best association pipeline can run frames nL[0..n) x nM[0..n) at the bounds maxR x maxC (taken over
// the frames with nL >= 1); otherwise PDA_ERR_UNSUPPORTED naming a frame, numbered from frameBase (association_kernel.cu)
int check_association_geometry(const int32_t* nL, const int32_t* nM, size_t n, int32_t k, int maxR, int maxC,
                               int64_t frameBase);
// pda_association_probs_batch_host on frames numbered from frameBase in its error messages (the _multi form's slices)
int association_probs_host(const double* costs, const int64_t* costOff, const int32_t* nL, const int32_t* nM,
                           int64_t nProblems, int32_t k, double* probs, const int64_t* probOff, int32_t device,
                           int64_t frameBase);

struct MurtyArgs {
    const double* costs; const int64_t* costOff; const int32_t* numRow; const int32_t* numCol;
    int64_t nProblems;
    int32_t k, cutMode, maximize, cutMaximize;
    double cutoff;
    int64_t* r4cBest; const int64_t* r4cOff;
    int64_t* c4rBest; const int64_t* c4rOff;
    double* gainBest; int32_t* nFound;
    int32_t weightMode; double weightGate;
    double* probs; const int64_t* probOff; const int32_t* nL;
    unsigned char* arena;
    unsigned long long* cursor;  // work-queue cursor (zeroed before launch)
    int32_t* order;              // optional: problem indices, most expensive first (NULL = index order)
    int32_t nWarps;              // arenas available == warps allowed to run
    MurtyGeometry geo;
    // pruning fast path: problems it cannot decide (exact gain ties) are appended here and redone by the exact kernel
    unsigned* fallbackCount;           // zeroed by launch_murty
    int32_t* fallbackList;             // [nProblems]
    const unsigned* nProblemsDev;      // when set, the kernel takes its problem count from here (the fallback pass)
    unsigned long long* cursor2;       // work cursor of the fallback pass
    int32_t useFast;
};
// The k ladder of pda_assignment_prob_ladder_batch: ONE enumeration to k = rung[nRungs - 1] gives the weight tables of
// every rung.  The list for k is the first min(k, nFound) entries of the list for any larger k (k only bounds the sweep
// loop), and the tables add their terms in list order, so the table of rung r is the running sum after hypothesis
// rung[r] - 1 with the end-of-problem normalisation.  Slot j of problem p -- the numCol x (nL+1) table at
// probs + probOff[p] + j*numCol*(nL+1) and nFound[p*nSlots + j] -- takes rung slotRung[j].  The ladder kernels are
// separate instantiations; the plain ones do not see this struct.
#define PDA_LADDER_MAX 16
struct MurtyLadder {
    int32_t nRungs, nSlots;
    int32_t rung[PDA_LADDER_MAX];      // ascending, distinct, >= 1
    int32_t slotRung[PDA_LADDER_MAX];  // rung of each requested slot
};
int launch_murty(const MurtyArgs& a, cudaStream_t stream, const MurtyLadder* ladder = nullptr);
// the ladder launches, compiled apart in murty_ladder_kernel.cu (wpc, smem: the launch shape launch_murty chose)
int launch_murty_ladder(const MurtyArgs& a, bool fast, const MurtyLadder& ladder, int wpc, int smem, cudaStream_t stream);

// ---- Murty k-best, one CTA per problem (murty_cta_kernel.cu): the latency path for small batches ----
#define PDA_CTA_MAX_COL 16  // detections per problem the CTA path takes (children per split record)
struct CtaGeometry {
    int mirrorBytes;     // per-warp shared-memory mirrors (u, spc, r4c, pred, c4r)
    int specSlack;       // arena slots that splits done ahead of their pop may hold
    int maxNodes;
    int64_t heapBytes;   // global part of the heap at the head of the arena
    int64_t nodesOff;    // byte offset of the node slots inside the arena
    int64_t arenaStride;
    int ctlOff, heapTopOff, heapTopCap, smemBytes;
};
int murty_cta_geometry(int32_t k, int32_t maxNumRow, int32_t maxNumCol, bool weights, const DeviceInfo& dev,
                       MurtyGeometry* g, CtaGeometry* cg);
int launch_murty_cta(const MurtyArgs& a, const CtaGeometry& cg, cudaStream_t stream, const MurtyLadder* ladder = nullptr);
int launch_murty_cta_ladder(const MurtyArgs& a, const CtaGeometry& cg, const MurtyLadder& ladder, cudaStream_t stream);

struct LapArgs {
    const double* costs; const int64_t* costOff; const int32_t* numRow; const int32_t* numCol;
    const int32_t* numCol4Gain;
    int64_t nProblems;
    int32_t makeSafe, maximize;
    const int64_t* rowOff; const int64_t* colOff;
    int64_t* col4row; int64_t* row4col; double* u; double* v; uint8_t* forbidden;
    double* gain; int32_t* feasible;
    int32_t maxNumRow, maxNumCol;
};
int launch_lap(const LapArgs& a, cudaStream_t stream);

// ---- conditioning / likelihoods (weights_kernel.cu) --------------------------------------------
int launch_condition_costs(const double* costs, const int64_t* costOff, const int32_t* numRow,
                           const int32_t* numCol, int64_t nProblems, const int64_t* rowOff,
                           double* outCosts, int64_t* rowIdx, int32_t* goodRows, cudaStream_t stream,
                           const int32_t* nLopt = nullptr, int32_t* condNL = nullptr,  // nLopt: numRow = nLopt + numCol
                           int32_t maxRow = INT32_MAX, int32_t maxCol = INT32_MAX);    // larger problems are skipped
// rows / cols (device, optional): vector p is the rows[p] x cols[p] matrix at off[p] (len is not read) -- the
// conditioned matrices, whose size only the device knows
int launch_to_probs(double* values, const int64_t* off, const int64_t* len, int64_t nVectors, cudaStream_t stream,
                    const int32_t* rows = nullptr, const int32_t* cols = nullptr);

// ---- permanents (permanent_kernel.cu) ------------------------------------------------------------
int launch_permanent_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                           int64_t nMats, int32_t maxDim, double* out, int32_t* status, void* workspace,
                           int64_t workspaceBytes, cudaStream_t stream, int32_t maxSmall, int32_t minSmall);
int launch_permanent_range(const double* A, int32_t n, uint64_t begin, uint64_t end, double* partial,
                           void* workspace, int64_t workspaceBytes, cudaStream_t stream);

// ---- Huber's approximate permanent (permanent_approx_kernel.cu) -------------------------------------------------
int launch_permanent_approx_batch(const double* mats, const int64_t* matOff, const int32_t* rows, const int32_t* cols,
                                  int64_t nMats, int32_t iterations, uint64_t seed, double* out, int32_t* status,
                                  cudaStream_t stream);
uint64_t approx_seed();  // seed of the draws behind permOpt == 0 (pda_set_approx_seed)

}  // namespace pda
#endif
