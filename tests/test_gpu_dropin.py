"""Drop-in demonstration: ONE compMethods-style C++ caller (tests/cpp/compmethods_driver.cpp, modelled on
comparison.cpp:146-247) built against include/*.h + libpda_b200_shims.so (tests/cpp/build/compmethods_b200)
must print the same k-best lists and gains and the same probabilities (1e-9) for the same .dat cost-matrix
files as the reference's side: the same caller built against the reference's own code
(oracle/_ref/compmethods_ref) where that has been built, else its output as stored in
tests/golden/compmethods_k150.npz (tests/golden/make_golden_restated.py)."""
import os
import resource
import subprocess

import numpy as np
import pytest

from helpers import compmethods_dat_files, golden
from probabilisticsemslam_b200 import datfile, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "compmethods_ref")
GPU_BIN = os.path.join(ROOT, "tests", "cpp", "build", "compmethods_b200")


def _big_stack():
    resource.setrlimit(resource.RLIMIT_STACK, (resource.RLIM_INFINITY, resource.RLIM_INFINITY))


def _parse(text):
    recs = []
    for line in text.splitlines():
        t = line.split()
        if not t:
            continue
        if t[0] == "h":          # h <i> <gain> : r4c... | c4r...
            recs.append(("h", [float(t[2])], [int(x) for x in t[4:] if x != "|"]))
        elif t[0] in ("frame", "kbest"):
            recs.append((line, [], []))
        else:                     # <tag> <m> p0 p1 ...
            recs.append((t[0] + " " + t[1], [float(x) for x in t[2:]], []))
    return recs


def test_same_caller_two_backends(tmp_path, gpu_api):
    assert os.path.exists(GPU_BIN), "tests/cpp/build/compmethods_b200 missing: run __graft_entry__.build()"
    files = []
    for path, C in compmethods_dat_files(str(tmp_path)):
        np.testing.assert_allclose(datfile.read_dat(path), np.round(C, 6), rtol=0, atol=1e-6)
        files.append(path)
    if os.path.exists(REF_BIN):
        ref = subprocess.run([REF_BIN, "--k", "150"] + files, capture_output=True, text=True, preexec_fn=_big_stack, timeout=600)
        assert ref.returncode == 0, ref.stderr[-500:]
        ref_out = ref.stdout
    else:
        ref_out = str(golden("compmethods_k150")["stdout"])
    gpu = subprocess.run([GPU_BIN, "--k", "150"] + files, capture_output=True, text=True, timeout=600)
    assert gpu.returncode == 0, gpu.stderr[-500:]
    a, b = _parse(ref_out), _parse(gpu.stdout)
    assert len(a) == len(b) and len(a) > 100
    # permExact lines: the reference's NW sum cancels on some of these problems (SURVEY.md F5).  The device path is
    # cancellation-free, so it is held to 1e-9 against the truth (tests/truth.py) always, and to 1e-9 against the
    # reference wherever the reference's own line is that accurate.
    from truth import permanent_prob_truth
    truths = {}
    for fi, path in enumerate(files):
        C = datfile.read_dat(path)
        cond, _ = gpu_api.conditionCosts(C)
        if cond.shape[0] < 32:
            truths[fi] = permanent_prob_truth(cond, cond.shape[0] - cond.shape[1])
    frame = None
    n_perm = 0
    for (ta, fa, ia), (tb, fb, ib) in zip(a, b):
        assert ta == tb
        assert ia == ib, f"{ta}: index lists differ"
        if ta == "h":
            assert fa == fb, "gains must be bit-identical"
        elif ta.startswith("frame"):
            frame = int(ta.split()[1])
        elif ta.startswith("permExact"):
            t = truths[frame][int(ta.split()[1])]
            np.testing.assert_allclose(fb, t, rtol=1e-9, atol=1e-300)
            m = t > 0
            if np.max(np.abs(np.asarray(fa)[m] - t[m]) / t[m]) < 1e-10:
                np.testing.assert_allclose(fb, fa, rtol=1e-9, atol=1e-300)
            n_perm += 1
        else:
            np.testing.assert_allclose(fb, fa, rtol=1e-9, atol=0)
    assert n_perm > 0


def test_moments_and_approximation_through_the_cpp_headers(gpu_api, oracle):
    """computeQuadricCostMatrixRaw, getAssignmentProbsFromMoments and permanentApproximationRaw (include/assignment.h,
    include/nwPerm.h) from a C++ caller: same numbers as the Python face of the library and as the CPU oracle."""
    exe = os.path.join(ROOT, "tests", "cpp", "build", "moments_b200")
    assert os.path.exists(exe), "tests/cpp/build/moments_b200 missing: run __graft_entry__.build()"
    lm, lc, mm, mc = synth.quadric_frames(1, first=31)[0]
    col = lambda c: c.transpose(0, 2, 1).reshape(-1)          # column-major 3x3, Eigen's layout
    text = f"{lm.shape[0]} {mm.shape[0]} 10.0 200\n" + " ".join(repr(float(x)) for x in
                                                                np.concatenate([lm.reshape(-1), col(lc), mm.reshape(-1), col(mc)]))
    run = subprocess.run([exe], input=text, capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stderr[-500:]
    lines = {ln.split()[0] + (" " + ln.split()[1] if ln.startswith("probs") else ""): ln.split() for ln in run.stdout.splitlines()}
    costs = np.array([float(x) for x in lines["costs"][1:]]).reshape((lm.shape[0] + mm.shape[0], mm.shape[0]), order="F")
    want = oracle.quadric_cost_matrix(lm, lc, mm, mc, 10.0)
    np.testing.assert_array_equal(costs.view(np.int64), want.view(np.int64))
    probs = np.array([[float(x) for x in lines[f"probs {m}"][2:]] for m in range(mm.shape[0])])
    np.testing.assert_array_equal(probs, gpu_api.getAssignmentProbs(lm, lc, mm, mc, 10.0, 200))
    np.testing.assert_allclose(probs, oracle.association_from_moments(lm, lc, mm, mc, 10.0, 200), rtol=1e-9, atol=1e-300)
    assert abs(float(lines["approx"][1]) / 720.0 - 1.0) < 0.2     # 300 trials, ~68 % accepted: 4 % standard error


def test_reference_typed_overloads(gpu_api, oracle):
    """The overloads that take the reference's own argument types (const Eigen::MatrixXd&, std::vector<Eigen::Vector3d>,
    const semConsts&) -- compiled against tests/cpp/eigen_stub because Eigen is not installed -- give the numbers of the
    raw forms: permanentExact / Square / Long (nwPerm.h:22-25), conditionedPermanent (assignment.h), the sharded
    permanent, and computeQuadricCostMatrix with runConsts (assignment.h:31-32)."""
    exe = os.path.join(ROOT, "tests", "cpp", "build", "eigen_overloads_b200")
    assert os.path.exists(exe), "tests/cpp/build/eigen_overloads_b200 missing: run __graft_entry__.build()"
    run = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stderr[-500:]
    out = {ln.split()[0]: ln.split()[1:] for ln in run.stdout.splitlines() if ln.strip()}
    A = np.array([[0.25 + 0.5 * ((7 * i + 3 * j) % 5) for j in range(5)] for i in range(5)])
    B = np.array([[1.0 + 0.125 * ((5 * i + 2 * j) % 7) for j in range(5)] for i in range(3)])
    wantA = oracle.permanent_exact_square(A)[0]
    from truth import perm_injective
    wantB = perm_injective(B)
    for tag in ("permanentExact", "permanentExactSquare", "permanentExactLong", "permanentExactSharded"):
        np.testing.assert_allclose(float(out[tag][0]), wantA, rtol=1e-12)
    for tag in ("permanentExactRect", "permanentExactLongRect"):
        np.testing.assert_allclose(float(out[tag][0]), wantB, rtol=1e-12)
    # conditionedPermanent divides by the product of ALL column scales (assignment.cpp:387-402), which is not perm(B) for a
    # matrix wider than tall: the reference's value is the expectation, not the mathematical permanent
    st, wantC = oracle.conditioned_permanent(B, 1)[1], oracle.conditioned_permanent(B, 1)[0]
    assert st == 0
    for tag in ("conditionedPermanent", "conditionedPermanentLong"):
        np.testing.assert_allclose(float(out[tag][0]), wantC, rtol=1e-9)
    assert out["throwsAbove32"] == ["1"] and out["quadricCostsSame"] == ["1"]
    lm = np.array([[2.0 * i + 0.3 * d for d in range(3)] for i in range(4)])
    lc = np.zeros((4, 3, 3))
    for i in range(4):
        lc[i] = np.diag([0.5 + 0.1 * i + 0.05 * d for d in range(3)]); lc[i][0, 1] = lc[i][1, 0] = 0.02
    mm = np.array([[2.0 * i + 0.4 + 0.2 * d for d in range(3)] for i in range(2)])
    mc = np.zeros((2, 3, 3))
    for i in range(2):
        mc[i] = np.diag([0.4 + 0.07 * d for d in range(3)]); mc[i][1, 2] = mc[i][2, 1] = -0.03
    want = gpu_api.computeQuadricCostMatrix(lm, lc, mm, mc, 10.0)
    got = np.array([float(x) for x in out["quadricCosts"]]).reshape(want.shape, order="F")
    np.testing.assert_array_equal(got.view(np.int64), want.view(np.int64))


def test_permanent_exact_long(gpu_api, oracle):
    """permanentExactLong (nwPerm.cpp:386-400): the reference runs the same double kernel and only divides in long
    double, so the double result must agree to 1e-9 (observed: to the last bits) for square and rectangular input."""
    for n in (1, 4, 9, 14):
        A = synth.dense_square(1, n, first=600 + n)[0].reshape(n, n, order="F")
        np.testing.assert_allclose(gpu_api.permanentExactLong(A), oracle.permanent_exact_square(A)[0], rtol=1e-9)
    from truth import perm_injective
    R = synth.dense_square(1, 6, first=77)[0].reshape(6, 6, order="F")[:4, :]
    np.testing.assert_allclose(gpu_api.permanentExactLong(R), perm_injective(R), rtol=1e-9)
    with pytest.raises(RuntimeError):
        gpu_api.permanentExactLong(np.ones((33, 33)))
