"""Generates the golden files whose reference side cannot be compiled from the repository alone:

  quadric_costs.npz   computeQuadricCostMatrix (assignment.cpp:705-722) -- the reference calls Eigen's ldlt().solve
                      (Eigen is not installed).  The stored costs are a 50-digit TRUTH (mpmath: d^T S^-1 d solved
                      exactly to working precision, rounded once to double), so they pin the restatement in
                      oracle/oracle_quadric.c and the CUDA kernel independently of any double-precision solver; the
                      stored weights are the restatement's (getAssignmentProbs chain, k = 200).
  perm_approx.npz     Huber's approximation (nwPerm.cpp:126-211) -- the reference draws from an unseeded rand(); the
                      stored estimates and success counts come from oracle/oracle_perm_approx.c on the counter-based
                      stream (seed 20260217, matrix index = position), the exact permanents from the oracle's NW walk.
  compmethods_k150.npz  what tests/cpp/compmethods_driver.cpp prints, line for line, when built against the
                      reference's own code and run with --k 150 on the .dat files of tests/helpers.py
                      (compmethods_dat_files) -- the reference's sources are not part of the repository, so the lines
                      are produced by the restatement (conditionCosts, kBest2DCutoff, bruteForceProb, assignmentProb,
                      permanentProb of oracle/*.c), which tests/test_oracle_golden.py holds to the reference's goldens.

    python tests/golden/make_golden_restated.py
"""
from __future__ import annotations

import os
import sys
import tempfile

import mpmath as mp
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import compmethods_dat_files  # noqa: E402
from oracle.loader import load_oracle  # noqa: E402
from probabilisticsemslam_b200 import datfile, synth  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
NONASSIGN, K = 10.0, 200
COMPMETHODS_K = 150


def compmethods_stdout(orc, paths, k):
    """The output of compmethods_driver.cpp for these .dat files (same lines, same %.17g formatting)."""
    out = []

    def g(x):
        return "%.17g" % x

    def probs(tag, p):
        for m, row in enumerate(p):
            out.append(f"{tag} {m}" + "".join(" " + g(v) for v in row))

    for fi, path in enumerate(paths):
        C = datfile.read_dat(path)
        nM = C.shape[1]
        cond, idx = orc.condition_costs(C)
        condL = cond.shape[0] - nM
        out.append(f"frame {fi} nL {C.shape[0] - nM} nM {nM} condL {condL} rowIdx" + "".join(f" {i}" for i in idx))
        if nM > 1:
            n, r4c, c4r, gain = orc.kbest2d_cutoff(k, cond, 42.0)
            out.append(f"kbest found {n}")
            for i in range(n):
                out.append(f"h {i} {g(gain[i])} :" + "".join(f" {x}" for x in r4c[i]) + " |" + "".join(f" {x}" for x in c4r[i]))
        probs("truth", orc.brute_force_prob(cond, condL))
        for kk in (1, 20, 100, 200, k):
            probs(f"k{kk}", orc.assignment_prob(cond, condL, kk))
        if condL + nM < 32:
            st, p = orc.permanent_prob(cond, condL, 1)
            assert st == 0
            probs("permExact", p)
    return "\n".join(out) + "\n"


def truth_costs(lm, lc, mm, mc):
    mp.mp.dps = 50
    nL, nM = lm.shape[0], mm.shape[0]
    C = np.full((nL + nM, nM), np.inf)
    for c in range(nM):
        for r in range(nL):
            d = mp.matrix([mp.mpf(float(lm[r, i])) - mp.mpf(float(mm[c, i])) for i in range(3)])
            S = mp.matrix(3, 3)
            for i in range(3):
                for j in range(3):
                    S[i, j] = mp.mpf(float(lc[r, i, j])) + mp.mpf(float(mc[c, i, j]))
            x = mp.lu_solve(S, d)
            C[r, c] = float(sum(d[i] * x[i] for i in range(3)))
        C[nL + c, c] = NONASSIGN
    return C


def main():
    orc = load_oracle()
    frames = synth.quadric_frames(12, first=2024)
    rec = {"n": np.int64(len(frames)), "nonassign": np.float64(NONASSIGN), "k": np.int64(K)}
    for i, (lm, lc, mm, mc) in enumerate(frames):
        rec[f"lm{i}"], rec[f"lc{i}"], rec[f"mm{i}"], rec[f"mc{i}"] = lm, lc, mm, mc
        rec[f"cost{i}"] = truth_costs(lm, lc, mm, mc)
        rec[f"probs{i}"] = orc.association_from_moments(lm, lc, mm, mc, NONASSIGN, K)
    np.savez_compressed(os.path.join(OUT, "quadric_costs.npz"), **rec)

    mats = [synth.dense_square(1, n, first=500 + n)[0].reshape(n, n, order="F") for n in (3, 6, 9, 12, 15, 18)]
    rng = np.random.default_rng(4)
    mats += [rng.random((3, 7)), rng.random((8, 5))]
    pa = {"n": np.int64(len(mats)), "iterations": np.int64(300), "seed": np.int64(20260217)}
    for i, A in enumerate(mats):
        est, succ = orc.permanent_approx(A, 300, 20260217, i)
        pa[f"A{i}"], pa[f"est{i}"], pa[f"succ{i}"], pa[f"exact{i}"] = A, np.float64(est), np.int64(succ), np.float64(orc.permanent_exact(A)[0])
    np.savez_compressed(os.path.join(OUT, "perm_approx.npz"), **pa)

    with tempfile.TemporaryDirectory() as d:
        text = compmethods_stdout(orc, [p for p, _ in compmethods_dat_files(d)], COMPMETHODS_K)
    np.savez_compressed(os.path.join(OUT, "compmethods_k150.npz"), k=np.int64(COMPMETHODS_K), stdout=np.array(text))
    print("wrote quadric_costs.npz, perm_approx.npz, compmethods_k150.npz")


if __name__ == "__main__":
    main()
