"""Shared helpers for the parity tests."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

KBEST_FILES = [
    "kbest_appendixA", "kbest_config1", "kbest_g1_k200", "kbest_g1_k1000", "kbest_g1int_k200",
    "kbest_g1int_nocut_k300", "kbest_g2cond_k200", "kbest_edges_k50", "kbest_edges_nocut_k50",
    "kbest_maximize_k1", "kbest_maximize_k40", "kbest_maximize_cut_k40",
]


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def kbest_cases(z):
    """Yields (C, nFound, row4col[n, numCol], col4row[n, numRow], gain[n]) of a kbest_*.npz file."""
    for i in range(int(z["n"])):
        yield z[f"C{i}"], int(z[f"n{i}"]), z[f"r{i}"].astype(np.int64), z[f"c{i}"].astype(np.int64), z[f"g{i}"]


def check_approx_rule(g, restated, iterations, what="", shape=None):
    """Holds the CUDA approximate permanent's estimate g to its CPU restatement's (estimate, successes, near ties) with
    the same draws.  K = estimate * iterations / successes; the kernel's successes round(g * iterations / K) must equal
    the restatement's give or take its near ties (draws within 1e-12 of a partial sum they were compared with, where
    the kernel's reassociated sums may decide the other way), and where they are equal, |g / estimate - 1| <= 1e-12."""
    est, succ, ties = restated
    what = f"{what} {shape}: kernel {g!r}, restatement {est!r} ({succ} of {iterations}, {ties} near ties)"
    assert np.isnan(g) == np.isnan(est), what
    if np.isnan(est):
        return
    if shape == (0, 0):
        assert g == est == 1.0, what
    elif succ == 0:
        assert g == 0.0 or ties > 0, what
    else:
        s = round(g * iterations / (est * iterations / succ))
        assert abs(s - succ) <= ties, what
        if s == succ:
            assert abs(g / est - 1.0) <= 1e-12, what


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def assert_kbest_equal(got, want, what=""):
    """got/want = (nFound, row4col, col4row, gain); index lists and gains must match bit for bit."""
    n = want[0]
    assert got[0] == n, f"{what}: nFound {got[0]} != {n}"
    if n == 0:
        return
    np.testing.assert_array_equal(got[1][:n], want[1][:n], err_msg=f"{what}: row4col")
    np.testing.assert_array_equal(got[2][:n], want[2][:n], err_msg=f"{what}: col4row")
    np.testing.assert_array_equal(bits(got[3][:n]), bits(want[3][:n]), err_msg=f"{what}: gain bits")


def compmethods_dat_files(directory):
    """Writes the .dat cost-matrix files that the compMethods-style driver reads in tests/test_gpu_dropin.py: ten gated
    G2 frames (the wire format quantises to 6 decimals, so exact ties appear) and three small dense G1 frames.
    Returns [(path, matrix before quantisation)]."""
    from probabilisticsemslam_b200 import datfile, synth
    files = []
    for run_id, pb in (("o30_p0_k200_perm0_net1", synth.g2_gated(10, first=900)),
                       ("small", synth.g1_dense(3, nL=9, nM=3, first=77))):
        for p in range(len(pb)):
            path = datfile.frame_path(directory, run_id, p + 1)
            datfile.write_dat(path, pb.matrix(p))
            files.append((path, pb.matrix(p)))
    return files


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    d = np.abs(a - b)
    s = np.maximum(np.abs(b), 1e-300)
    return float(np.max(np.where(d == 0, 0.0, d / s))) if a.size else 0.0
