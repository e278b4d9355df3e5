// moments_graph_driver.cpp -- the per-frame call of a SLAM loop through one CUDA graph per weighting: the device-pointer
// forms pda_association_from_moments_batch (k-best, k = 200) and pda_association_perm_from_moments_batch (usePerm),
// each captured once with fixed bounds (one frame, at most 40 landmarks and 8 detections) together with the upload of
// the moments and offsets from page-locked buffers and the download of the table and status.  Every frame then only
// fills the page-locked buffers and launches the graph, whatever its shape.  Reads "nFrames nonassign" and then, per
// frame, "nL nM" and the flattened moments (landmark means, landmark covariances, detection means, detection
// covariances; covariances column-major) from stdin; prints every table row at full precision and each frame's status
// (and nFound); tests/test_gpu_moments_device.py compares them with the Python face of the library.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>

#include "pda_b200.h"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { std::fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)
#define PK(x) do { int rc = (x); if (rc != PDA_OK) { std::fprintf(stderr, "%s: %d %s\n", #x, rc, pda_last_error()); return 1; } } while (0)

namespace {

constexpr int MAX_NL = 40, MAX_NM = 8, K = 200;
constexpr int64_t PROB_CAP = (int64_t)MAX_NM * (MAX_NL + 1);

// the upload, one contiguous block: moments at their capacities, then the two offset pairs
struct Inputs {
    double landMean[3 * MAX_NL], landCov[9 * MAX_NL], measMean[3 * MAX_NM], measCov[9 * MAX_NM];
    int64_t landOff[2], measOff[2];
};
struct Outputs {
    double probs[PROB_CAP];
    int64_t probOff[2];
    int32_t status[1], nFound[1];
};

struct Form {
    const char* name;
    bool perm;
    Outputs* dOut;
    void* ws;
    int64_t wsBytes;
    cudaGraphExec_t exec;
};

int call(const Form& f, const Inputs* dIn, cudaStream_t s) {
    if (f.perm)
        return pda_association_perm_from_moments_batch(dIn->landMean, dIn->landCov, dIn->landOff, MAX_NL, dIn->measMean, dIn->measCov,
                                                       dIn->measOff, MAX_NM, 1, MAX_NL, MAX_NM, 10.0, f.dOut->probs, PROB_CAP,
                                                       f.dOut->probOff, f.dOut->status, f.ws, f.wsBytes, s);
    return pda_association_from_moments_batch(dIn->landMean, dIn->landCov, dIn->landOff, MAX_NL, dIn->measMean, dIn->measCov,
                                              dIn->measOff, MAX_NM, 1, MAX_NL, MAX_NM, 10.0, K, f.dOut->probs, PROB_CAP,
                                              f.dOut->probOff, f.dOut->status, f.dOut->nFound, f.ws, f.wsBytes, s);
}

bool read_doubles(double* x, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (std::scanf("%lf", x + i) != 1) return false;
    return true;
}

}  // namespace

int main() {
    size_t nFrames;
    double nonassign;
    if (std::scanf("%zu %lf", &nFrames, &nonassign) != 2) return 2;
    if (nonassign != 10.0) { std::fprintf(stderr, "the graphs are captured with nonassign = 10\n"); return 2; }
    cudaStream_t s;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    Inputs *hIn, *dIn;
    Outputs* hOut;
    CK(cudaHostAlloc(reinterpret_cast<void**>(&hIn), sizeof(Inputs), cudaHostAllocDefault));
    CK(cudaHostAlloc(reinterpret_cast<void**>(&hOut), sizeof(Outputs), cudaHostAllocDefault));
    CK(cudaMalloc(reinterpret_cast<void**>(&dIn), sizeof(Inputs)));
    std::memset(hIn, 0, sizeof(Inputs));  // a 0 x 0 frame for the warm-up call
    CK(cudaMemcpy(dIn, hIn, sizeof(Inputs), cudaMemcpyHostToDevice));
    Form forms[2] = {{"kbest", false, nullptr, nullptr, 0, nullptr}, {"perm", true, nullptr, nullptr, 0, nullptr}};
    for (Form& f : forms) {
        f.wsBytes = f.perm ? pda_association_perm_from_moments_workspace_bytes(1, MAX_NL, MAX_NM, PROB_CAP)
                           : pda_association_from_moments_workspace_bytes(1, MAX_NL, MAX_NM, PROB_CAP, K);
        if (f.wsBytes < 0) { std::fprintf(stderr, "workspace: %s\n", pda_last_error()); return 1; }
        CK(cudaMalloc(reinterpret_cast<void**>(&f.dOut), sizeof(Outputs)));
        CK(cudaMalloc(&f.ws, f.wsBytes));
        PK(call(f, dIn, s));  // warm-up: first-use attributes outside the capture
        CK(cudaStreamSynchronize(s));
        cudaGraph_t g;
        CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
        CK(cudaMemcpyAsync(dIn, hIn, sizeof(Inputs), cudaMemcpyHostToDevice, s));
        PK(call(f, dIn, s));
        CK(cudaMemcpyAsync(hOut, f.dOut, sizeof(Outputs), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamEndCapture(s, &g));
        CK(cudaGraphInstantiate(&f.exec, g, 0));
        CK(cudaGraphDestroy(g));
    }
    for (size_t fr = 0; fr < nFrames; ++fr) {
        int nL, nM;
        if (std::scanf("%d %d", &nL, &nM) != 2 || nL < 0 || nM < 0 || nL > MAX_NL || nM > MAX_NM) return 2;
        if (!read_doubles(hIn->landMean, 3 * (size_t)nL) || !read_doubles(hIn->landCov, 9 * (size_t)nL) ||
            !read_doubles(hIn->measMean, 3 * (size_t)nM) || !read_doubles(hIn->measCov, 9 * (size_t)nM))
            return 2;
        hIn->landOff[0] = 0; hIn->landOff[1] = nL;
        hIn->measOff[0] = 0; hIn->measOff[1] = nM;
        for (const Form& f : forms) {
            CK(cudaGraphLaunch(f.exec, s));
            CK(cudaStreamSynchronize(s));
            for (int m = 0; m < nM; ++m) {
                std::printf("%s %zu %d", f.name, fr, m);
                for (int l = 0; l <= nL; ++l) std::printf(" %.17g", hOut->probs[hOut->probOff[0] + (int64_t)m * (nL + 1) + l]);
                std::printf("\n");
            }
            std::printf("status %s %zu %d %lld %d\n", f.name, fr, hOut->status[0], (long long)hOut->probOff[1],
                        f.perm ? -1 : hOut->nFound[0]);
        }
    }
    for (Form& f : forms) {
        cudaGraphExecDestroy(f.exec);
        cudaFree(f.dOut);
        cudaFree(f.ws);
    }
    cudaFree(dIn);
    cudaFreeHost(hIn);
    cudaFreeHost(hOut);
    cudaStreamDestroy(s);
    return 0;
}
