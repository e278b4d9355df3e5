// bbox_driver.cpp -- the stereo box association (asgnBB) from C++, two ways: every frame in one asgnBBRawBatch call
// spread over a list of devices (include/assignment.h), and the per-frame call of a SLAM loop through one CUDA graph:
// the device-pointer form pda_asgn_bb_batch captured once with fixed bounds (one frame, at most 64 left boxes and 128
// boxes in all) together with the upload of the boxes and offsets from a page-locked buffer and the download of the
// assignment and status.  Every frame then only fills the page-locked buffer and launches the graph, whatever its
// shape.  Reads "nFrames nonassign nDevices device..." and then, per frame, "nL nR" and the flattened boxes (left,
// then right; five doubles each) from stdin; prints "batch f a..." per frame and then "graph f status a..." per frame.
// tests/test_gpu_bbox_device.py compares them with the Python face of the library.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "assignment.h"
#include "pda_b200.h"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { std::fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)
#define PK(x) do { int rc = (x); if (rc != PDA_OK) { std::fprintf(stderr, "%s: %d %s\n", #x, rc, pda_last_error()); return 1; } } while (0)

namespace {

constexpr int MAX_NL = 64, MAX_BOXES = 128;

// the upload, one contiguous block: boxes at their capacities, then the two offset pairs
struct Inputs {
    double boxesL[5 * MAX_NL], boxesR[5 * MAX_BOXES];
    int64_t offL[2], offR[2];
};
struct Outputs {
    int32_t assignment[MAX_NL];
    int32_t status[1];
};

bool read_doubles(std::vector<double>& x, size_t n) {
    x.resize(n);
    for (size_t i = 0; i < n; ++i)
        if (std::scanf("%lf", &x[i]) != 1) return false;
    return true;
}

}  // namespace

int main() {
    size_t nFrames;
    double nonassign;
    int nDevices;
    if (std::scanf("%zu %lf %d", &nFrames, &nonassign, &nDevices) != 3 || nDevices < 0) return 2;
    std::vector<int> devices((size_t)nDevices);
    for (int& d : devices)
        if (std::scanf("%d", &d) != 1) return 2;
    std::vector<std::vector<double> > L(nFrames), R(nFrames);
    for (size_t f = 0; f < nFrames; ++f) {
        int nL, nR;
        if (std::scanf("%d %d", &nL, &nR) != 2 || nL < 0 || nR < 0) return 2;
        if (!read_doubles(L[f], 5 * (size_t)nL) || !read_doubles(R[f], 5 * (size_t)nR)) return 2;
    }

    const std::vector<std::vector<int> > batch = asgnBBRawBatch(L, R, nonassign, devices);
    for (size_t f = 0; f < nFrames; ++f) {
        std::printf("batch %zu", f);
        for (int a : batch[f]) std::printf(" %d", a);
        std::printf("\n");
    }

    CK(cudaSetDevice(devices.empty() ? 0 : devices[0]));
    cudaStream_t s;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    Inputs *hIn, *dIn;
    Outputs *hOut, *dOut;
    CK(cudaHostAlloc(reinterpret_cast<void**>(&hIn), sizeof(Inputs), cudaHostAllocDefault));
    CK(cudaHostAlloc(reinterpret_cast<void**>(&hOut), sizeof(Outputs), cudaHostAllocDefault));
    CK(cudaMalloc(reinterpret_cast<void**>(&dIn), sizeof(Inputs)));
    CK(cudaMalloc(reinterpret_cast<void**>(&dOut), sizeof(Outputs)));
    std::memset(hIn, 0, sizeof(Inputs));  // a frame without boxes for the warm-up call
    CK(cudaMemcpy(dIn, hIn, sizeof(Inputs), cudaMemcpyHostToDevice));
    const int64_t wsBytes = pda_asgn_bb_workspace_bytes(1, MAX_NL, MAX_BOXES);
    if (wsBytes < 0) { std::fprintf(stderr, "workspace: %s\n", pda_last_error()); return 1; }
    void* ws;
    CK(cudaMalloc(&ws, wsBytes));
    auto call = [&]() {
        return pda_asgn_bb_batch(dIn->boxesL, dIn->offL, MAX_NL, dIn->boxesR, dIn->offR, MAX_BOXES, 1, MAX_NL, MAX_BOXES, nonassign,
                                 dOut->assignment, dOut->status, ws, wsBytes, s);
    };
    PK(call());  // warm-up: first-use attributes outside the capture
    CK(cudaStreamSynchronize(s));
    cudaGraph_t g;
    cudaGraphExec_t exec;
    CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
    CK(cudaMemcpyAsync(dIn, hIn, sizeof(Inputs), cudaMemcpyHostToDevice, s));
    PK(call());
    CK(cudaMemcpyAsync(hOut, dOut, sizeof(Outputs), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamEndCapture(s, &g));
    CK(cudaGraphInstantiate(&exec, g, 0));
    CK(cudaGraphDestroy(g));
    for (size_t f = 0; f < nFrames; ++f) {
        const size_t nL = L[f].size() / 5, nR = R[f].size() / 5;
        if (nL > MAX_NL || nL + nR > MAX_BOXES) return 2;
        std::memcpy(hIn->boxesL, L[f].data(), L[f].size() * sizeof(double));
        std::memcpy(hIn->boxesR, R[f].data(), R[f].size() * sizeof(double));
        hIn->offL[0] = 0; hIn->offL[1] = (int64_t)nL;
        hIn->offR[0] = 0; hIn->offR[1] = (int64_t)nR;
        CK(cudaGraphLaunch(exec, s));
        CK(cudaStreamSynchronize(s));
        std::printf("graph %zu %d", f, hOut->status[0]);
        for (size_t i = 0; i < nL; ++i) std::printf(" %d", hOut->assignment[i]);
        std::printf("\n");
    }
    cudaGraphExecDestroy(exec);
    cudaFree(ws);
    cudaFree(dOut);
    cudaFree(dIn);
    cudaFreeHost(hIn);
    cudaFreeHost(hOut);
    cudaStreamDestroy(s);
    return 0;
}
