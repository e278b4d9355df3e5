// A C++ caller of the device-pointer forms pda_permanent_prob_batch and pda_conditioned_permanent_batch: device buffers,
// one call of each captured in a CUDA graph, replayed on new inputs copied into the same buffers, then the same inputs
// through direct calls.  Prints "replay ..." and "direct ..." lines with every table entry and status as hex bits; they
// must agree (tests/test_gpu_permanent_prob_device.py).
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "pda_b200.h"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { std::fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)
#define PK(x) do { int rc = (x); if (rc != PDA_OK) { std::fprintf(stderr, "%s: %d %s\n", #x, rc, pda_last_error()); return 1; } } while (0)

static void print(const char* tag, const std::vector<double>& v, const std::vector<int32_t>& st) {
    std::printf("%s", tag);
    for (double x : v) { uint64_t b; std::memcpy(&b, &x, 8); std::printf(" %016llx", (unsigned long long)b); }
    for (int32_t s : st) std::printf(" s%d", s);
    std::printf("\n");
}

int main() {
    // problems: nM = 3, 12 (NW sub-permanents) and 1, each against a few landmarks; costs from a fixed formula
    const int nL[3] = {6, 4, 5}, nM[3] = {3, 12, 1};
    std::vector<int64_t> costOff(3), probOff(3);
    int64_t nc = 0, np = 0;
    for (int p = 0; p < 3; ++p) { costOff[p] = nc; probOff[p] = np; nc += (int64_t)(nL[p] + nM[p]) * nM[p]; np += (int64_t)nM[p] * (nL[p] + 1); }
    auto costs = [&](double shift) {
        std::vector<double> c((size_t)nc);
        for (int64_t i = 0; i < nc; ++i) c[(size_t)i] = 1.0 + 30.0 * std::fabs(std::sin(0.7 * (double)i + shift));
        return c;
    };
    const std::vector<double> cA = costs(0.0), cB = costs(1.3);
    double *dC, *dP;
    int64_t *dCO, *dPO;
    int32_t *dL, *dM, *dS;
    CK(cudaMalloc(&dC, nc * 8)); CK(cudaMalloc(&dP, np * 8)); CK(cudaMalloc(&dCO, 24)); CK(cudaMalloc(&dPO, 24));
    CK(cudaMalloc(&dL, 12)); CK(cudaMalloc(&dM, 12)); CK(cudaMalloc(&dS, 12));
    CK(cudaMemcpy(dCO, costOff.data(), 24, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dPO, probOff.data(), 24, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dL, nL, 12, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dM, nM, 12, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dC, cA.data(), nc * 8, cudaMemcpyHostToDevice));
    const int64_t ws = pda_permanent_prob_workspace_bytes(3, nc, np, 16, 12, 1);
    if (ws < 0) { std::fprintf(stderr, "workspace: %s\n", pda_last_error()); return 1; }
    void* dW;
    CK(cudaMalloc(&dW, ws));
    cudaStream_t s;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    auto call = [&]() { return pda_permanent_prob_batch(dC, dCO, dL, dM, 3, nc, np, 16, 12, 1, dP, dPO, dS, dW, ws, s); };
    PK(call());  // warm-up: first-use attributes outside the capture
    CK(cudaStreamSynchronize(s));
    cudaGraph_t g;
    cudaGraphExec_t ge;
    CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
    PK(call());
    CK(cudaStreamEndCapture(s, &g));
    CK(cudaGraphInstantiate(&ge, g, 0));
    std::vector<double> probs((size_t)np);
    std::vector<int32_t> st(3);
    CK(cudaMemcpyAsync(dC, cB.data(), nc * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(dP, 0, np * 8, s));
    CK(cudaGraphLaunch(ge, s));
    CK(cudaMemcpyAsync(probs.data(), dP, np * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(st.data(), dS, 12, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    print("replay prob", probs, st);
    CK(cudaMemsetAsync(dP, 0, np * 8, s));
    PK(call());
    CK(cudaMemcpyAsync(probs.data(), dP, np * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(st.data(), dS, 12, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    print("direct prob", probs, st);

    // conditioned permanents: two 13 x 13 matrices (NW walk) and a 4 x 6 one, read in place
    const int32_t rows[3] = {13, 13, 4}, cols[3] = {13, 13, 6};
    const int64_t matOff[3] = {0, 169, 338};
    auto mats = [&](double shift) {
        std::vector<double> m(362);
        for (size_t i = 0; i < m.size(); ++i) m[i] = std::fabs(std::cos(0.37 * (double)i + shift));
        return m;
    };
    const std::vector<double> mA = mats(0.0), mB = mats(2.1);
    double *dA, *dO;
    int64_t* dAO;
    int32_t *dR, *dCc, *dS2;
    CK(cudaMalloc(&dA, 362 * 8)); CK(cudaMalloc(&dO, 24)); CK(cudaMalloc(&dAO, 24));
    CK(cudaMalloc(&dR, 12)); CK(cudaMalloc(&dCc, 12)); CK(cudaMalloc(&dS2, 12));
    CK(cudaMemcpy(dA, mA.data(), 362 * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dAO, matOff, 24, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dR, rows, 12, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dCc, cols, 12, cudaMemcpyHostToDevice));
    const int64_t ws2 = pda_conditioned_permanent_workspace_bytes(3, 13, 1);
    if (ws2 < 0) { std::fprintf(stderr, "workspace: %s\n", pda_last_error()); return 1; }
    void* dW2;
    CK(cudaMalloc(&dW2, ws2));
    auto call2 = [&]() { return pda_conditioned_permanent_batch(dA, dAO, dR, dCc, 3, 13, 1, dO, dS2, dW2, ws2, s); };
    PK(call2());
    CK(cudaStreamSynchronize(s));
    cudaGraph_t g2;
    cudaGraphExec_t ge2;
    CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
    PK(call2());
    CK(cudaStreamEndCapture(s, &g2));
    CK(cudaGraphInstantiate(&ge2, g2, 0));
    std::vector<double> out(3);
    CK(cudaMemcpyAsync(dA, mB.data(), 362 * 8, cudaMemcpyHostToDevice, s));
    CK(cudaGraphLaunch(ge2, s));
    CK(cudaMemcpyAsync(out.data(), dO, 24, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(st.data(), dS2, 12, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    print("replay cond", out, st);
    PK(call2());
    CK(cudaMemcpyAsync(out.data(), dO, 24, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(st.data(), dS2, 12, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    print("direct cond", out, st);
    cudaGraphExecDestroy(ge); cudaGraphDestroy(g); cudaGraphExecDestroy(ge2); cudaGraphDestroy(g2);
    cudaFree(dC); cudaFree(dP); cudaFree(dCO); cudaFree(dPO); cudaFree(dL); cudaFree(dM); cudaFree(dS); cudaFree(dW);
    cudaFree(dA); cudaFree(dO); cudaFree(dAO); cudaFree(dR); cudaFree(dCc); cudaFree(dS2); cudaFree(dW2);
    cudaStreamDestroy(s);
    return 0;
}
