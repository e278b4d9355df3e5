// perm_association_driver.cpp -- the usePerm forms of the C++ drop-in layer (include/assignment.h) from a C++ caller:
// getAssignmentProbsFromMoments(.., usePerm = true), getAssignmentProbsFromCosts(.., usePerm = true) and the batch form
// getAssignmentProbsBatch.  Reads "nFrames nonassign" and then, per frame, "nL nM" and the flattened moments (landmark
// means, landmark covariances, detection means, detection covariances; covariances column-major) from stdin, and prints
// every table at full precision; tests/test_gpu_association_perm.py compares them with the Python face of the library.
#include <cstdio>
#include <exception>
#include <vector>

#include "assignment.h"

static void print_table(const char* kind, size_t f, const std::vector<std::vector<double> >& t) {
    for (size_t m = 0; m < t.size(); m++) {
        printf("%s %zu %zu", kind, f, m);
        for (double p : t[m]) printf(" %.17g", p);
        printf("\n");
    }
}

int main() {
    size_t nFrames;
    double nonassign;
    if (scanf("%zu %lf", &nFrames, &nonassign) != 2) return 2;
    const size_t k = 200;  // unused with usePerm, passed as a SLAM run would
    std::vector<std::vector<double> > costs(nFrames);
    std::vector<size_t> nLs(nFrames), nMs(nFrames);
    try {
        for (size_t f = 0; f < nFrames; f++) {
            size_t nL, nM;
            if (scanf("%zu %zu", &nL, &nM) != 2) return 2;
            std::vector<double> lm(3 * nL), lc(9 * nL), mm(3 * nM), mc(9 * nM);
            for (double& x : lm) if (scanf("%lf", &x) != 1) return 2;
            for (double& x : lc) if (scanf("%lf", &x) != 1) return 2;
            for (double& x : mm) if (scanf("%lf", &x) != 1) return 2;
            for (double& x : mc) if (scanf("%lf", &x) != 1) return 2;
            print_table("moments", f, getAssignmentProbsFromMoments(lm, lc, mm, mc, nonassign, k, true));
            costs[f] = computeQuadricCostMatrixRaw(lm, lc, mm, mc, nonassign);
            nLs[f] = nL;
            nMs[f] = nM;
            print_table("costs", f, getAssignmentProbsFromCosts(costs[f], nL, nM, k, true));
        }
        const std::vector<std::vector<std::vector<double> > > batch = getAssignmentProbsBatch(costs, nLs, nMs, k, true);
        for (size_t f = 0; f < nFrames; f++) print_table("batch", f, batch[f]);
    } catch (const std::exception& e) {
        printf("throw %s\n", e.what());
        return 1;
    }
    return 0;
}
