// ladder_driver.cpp -- compMethods' per-frame k sweep (comparison.cpp:194-222) through ONE call of the C++ drop-in layer:
// assignmentProbLadder(cond, condL, nM, {1, 20, 100, 200, k}) on the conditioned matrix of every .dat frame named on
// the command line.  Prints "frame <i>" and then "k<k> <m> p0 p1 ..." lines in the format of compmethods_driver.cpp, so
// tests/test_gpu_assignment_ladder.py can compare them with the reference's own output of that driver.
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <fstream>
#include <limits>
#include <sstream>
#include <string>
#include <vector>

#include "assignment.h"

// the .dat wire format of saveAssignmentProb (assignment.cpp:821-831), read like comparison.cpp:39-54
static bool readDat(const std::string& path, std::vector<std::vector<double> >& rows) {
    std::ifstream f(path.c_str());
    if (!f) return false;
    std::string line;
    rows.clear();
    while (std::getline(f, line)) {
        if (line.empty()) continue;
        rows.push_back(std::vector<double>());
        std::stringstream ss(line);
        std::string val;
        while (std::getline(ss, val, ',')) {
            if (val[0] == 'i') rows.back().push_back(std::numeric_limits<double>::infinity());
            else rows.back().push_back(std::stod(val));
        }
    }
    return !rows.empty();
}

int main(int argc, char** argv) {
    size_t k = 150;
    std::vector<std::string> files;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "--k" && i + 1 < argc) k = size_t(std::atoi(argv[++i]));
        else files.push_back(a);
    }
    const std::vector<size_t> ks = {1, 20, 100, 200, k};
    try {
        for (size_t fi = 0; fi < files.size(); fi++) {
            std::vector<std::vector<double> > costs;
            if (!readDat(files[fi], costs)) { std::printf("frame %zu unreadable\n", fi); continue; }
            const size_t nRows = costs.size(), nM = costs[0].size(), nL = nRows - nM;
            std::vector<double> unrolled(nM * nRows);
            for (size_t r = 0; r < nRows; r++)
                for (size_t c = 0; c < nM; c++) unrolled[c * nRows + r] = costs[r][c];
            std::vector<ptrdiff_t> rowIdx;
            const std::vector<double> cond = conditionCosts(unrolled, nL + nM, nM, rowIdx);
            const size_t condL = cond.size() / nM - nM;
            std::printf("frame %zu\n", fi);
            const std::vector<std::vector<std::vector<double> > > t = assignmentProbLadder(cond, condL, nM, ks);
            for (size_t j = 0; j < ks.size(); j++)
                for (size_t m = 0; m < t[j].size(); m++) {
                    std::printf("k%zu %zu", ks[j], m);
                    for (double p : t[j][m]) std::printf(" %.17g", p);
                    std::printf("\n");
                }
        }
    } catch (const std::exception& e) {
        std::printf("throw %s\n", e.what());
        return 1;
    }
    return 0;
}
