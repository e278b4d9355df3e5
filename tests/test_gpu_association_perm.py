"""getAssignmentProbs with usePerm (assignment.cpp:57-74, :64) as one device pipeline: conditionCosts -> likelihoods ->
every sub-permanent by the fused conditioned-permanent kernel -> finish and scatter through rowIdx.

The tables must equal, bit for bit, what the composition of the separate entry points gives (conditionCosts ->
permanentProb(.., 1) -> scatter through rowIdx), which is how getAssignmentProbsFromCosts(usePerm=True) ran before the
pipeline existed; and they must be within 1e-9 of the cancellation-free truth.  The CPU tests at the bottom check the
argument handling, which runs before any device work."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import bits, golden
from perm_route import composed
from probabilisticsemslam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-9
gpu = pytest.mark.gpu


def assert_same(got, want, what):
    (gt, gs), (wt, ws) = got, want
    np.testing.assert_array_equal(gs, ws, err_msg=f"{what}: status")
    for p in range(len(wt)):
        np.testing.assert_array_equal(bits(gt[p]), bits(wt[p]), err_msg=f"{what}: problem {p} (status {ws[p]})")


def truth_table(api, C, nL):
    """permanentProb on the conditioned problem with every sub-permanent evaluated cancellation-free, scattered back."""
    from truth import permanent_prob_truth
    nM = C.shape[1]
    if nL == 0:
        return np.ones((nM, 1))
    cond, rows = api.conditionCosts(C)
    condL = cond.shape[0] - nM
    tc = permanent_prob_truth(cond, condL)
    t = np.zeros((nM, nL + 1))
    t[:, rows[:condL]] = tc[:, :condL]
    t[:, nL] = tc[:, condL]
    return t


def frames_to_costs(api, frames):
    mats = api.quadric_cost_batch(frames, 10.0)
    return synth.pack(mats, [f[0].shape[0] for f in frames])


def ragged_batch():
    """Every edge the pipeline has: nL = 0, nM = 1, condL = 0, the largest fused DP (nM = 11), the routed sizes (nM = 12,
    14), a sub-matrix with more than 32 kept rows (status 1), gated-away dummy rows leaving fewer rows than detections
    (status 3) and a gated-away dummy row with goodRows >= nM (computed, as the reference does), among ordinary gated
    problems."""
    g2 = synth.g2_gated(6, first=600)
    mats, nls = [g2.matrix(p) for p in range(3)], [30] * 3
    mats.append(np.array([[10.0, np.inf], [np.inf, 10.0]])); nls.append(0)                      # nL = 0
    mats.append(np.concatenate([g2.matrix(3)[:30, :1], [[10.0]]])); nls.append(30)               # nM = 1
    c = np.full((8, 3), np.inf); c[:5] = 100.0; c[5 + np.arange(3), np.arange(3)] = 10.0
    mats.append(c); nls.append(5)                                                                # condL = 0
    for nl, nm in ((20, 11), (8, 12), (6, 14)):                                                  # largest DP, routed
        mats.append(synth.g1_dense(1, nL=nl, nM=nm, first=700 + nm).matrix(0)); nls.append(nl)
    mats.append(synth.g1_dense(1, nL=40, nM=3, first=800, scale=10.0).matrix(0)); nls.append(40)  # long side > 32
    c = np.full((5, 3), np.inf); c[:2] = [[0.5, 1.0, 2.0], [1.5, 0.2, 3.0]]; c[2 + np.arange(3), np.arange(3)] = 100.0
    mats.append(c); nls.append(2)                                                                # dummy rows gated away
    mats += [g2.matrix(p) for p in range(3, 6)]; nls += [30] * 3
    c = np.full((5, 2), np.inf); c[:3] = [[0.5, 0.3], [1.0, 2.0], [60.0, 70.0]]; c[3, 0] = 100.0; c[4, 1] = 10.0
    mats.append(c); nls.append(3)                                 # dummy row 0 gated away, goodRows = 3 >= nM: condL = 1
    return synth.pack(mats, nls)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_golden_association_g2(gpu_api):
    z = golden("association_g2")
    n = int(z["n"])
    pb = synth.pack([z[f"C{p}"] for p in range(n)], [30] * n)
    tabs, st = gpu_api.association_perm_probs_batch(pb)
    assert not st.any()
    checked = 0
    for p in range(n):
        truth = truth_table(gpu_api, z[f"C{p}"], 30)
        np.testing.assert_allclose(tabs[p], truth, rtol=RTOL, atol=1e-300)
        if f"perm_{p}" in z:
            m = truth > 0
            if np.max(np.abs(z[f"perm_{p}"][m] - truth[m]) / truth[m]) < 1e-10:   # the reference's own table is accurate
                np.testing.assert_allclose(tabs[p], z[f"perm_{p}"], rtol=RTOL, atol=1e-300)
                checked += 1
    assert checked > 0


@gpu
def test_bit_identical_to_the_composition(gpu_api):
    pb = synth.g2_gated(2000, first=9000)
    assert_same(gpu_api.association_perm_probs_batch(pb), composed(gpu_api, pb), "g2_gated")
    pb = frames_to_costs(gpu_api, synth.quadric_frames(2000, first=3000))
    assert_same(gpu_api.association_perm_probs_batch(pb), composed(gpu_api, pb), "quadric_frames")
    pb = ragged_batch()
    got = gpu_api.association_perm_probs_batch(pb)
    want = composed(gpu_api, pb)
    assert_same(got, want, "ragged")
    assert list(got[1]) == [0] * 9 + [1, 3] + [0] * 4
    np.testing.assert_array_equal(got[0][3], np.ones((2, 1)))
    assert got[0][5][:, :5].sum() == 0 and np.all(got[0][5][:, 5] > 0)          # condL = 0: only non-assignment
    assert got[0][14].any()                                                       # a table, not an error
    for p in (0, 4, 6, 14):                                                       # fused problems against the truth
        np.testing.assert_allclose(got[0][p], truth_table(gpu_api, pb.matrix(p), int(pb.nL[p])), rtol=RTOL, atol=1e-300)


@gpu
def test_moments(gpu_api, oracle):
    frames = synth.quadric_frames(400, first=12_000)
    tabs, st = gpu_api.association_perm_from_moments_batch(frames, 10.0)
    pb = frames_to_costs(gpu_api, frames)
    want_t, want_s = gpu_api.association_perm_probs_batch(pb)
    np.testing.assert_array_equal(st, want_s)
    for f in range(len(frames)):
        np.testing.assert_array_equal(bits(tabs[f]), bits(want_t[f]))
    for f in range(0, len(frames), 20):
        C = oracle.quadric_cost_matrix(*frames[f], 10.0)
        np.testing.assert_allclose(tabs[f], truth_table(gpu_api, C, frames[f][0].shape[0]), rtol=RTOL, atol=1e-300)
    one = gpu_api.getAssignmentProbs(*frames[7], 10.0, 200, usePerm=True)
    np.testing.assert_array_equal(bits(one), bits(tabs[7]))
    np.testing.assert_array_equal(bits(gpu_api.getAssignmentProbsFromCosts(pb.matrix(7), int(pb.nL[7]), 200, usePerm=True)),
                                  bits(tabs[7]))


@gpu
def test_one_hundred_thousand_problems_in_one_call(gpu_api):
    pb = synth.g2_gated(100_000, first=1_000_000)
    tabs, st = gpu_api.association_perm_probs_batch(pb)
    assert not st.any()
    sample = np.sort(np.random.default_rng(5).choice(len(pb), 500, replace=False))
    sub = pb.take(sample)
    want_t, want_s = composed(gpu_api, sub)
    assert not want_s.any()
    for i, p in enumerate(sample):
        np.testing.assert_array_equal(bits(tabs[p]), bits(want_t[i]))


@gpu
def test_device_form_under_a_cuda_graph(gpu_api):
    import torch
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    dev = torch.device("cuda:0")
    pb = synth.g2_gated(500, first=42_000)
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    nr = (nL + nM).astype(np.int64)
    row_off = np.concatenate([[0], np.cumsum(nr)[:-1]]).astype(np.int64)
    sizes = nM.astype(np.int64) * (nL.astype(np.int64) + 1)
    prob_off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    costs, cost_off, d_nL, d_nM, d_row, d_poff = t(pb.costs), t(pb.cost_off), t(nL), t(nM), t(row_off), t(prob_off)
    total_p = int(sizes.sum())
    ws_bytes = lib.pda_association_perm_workspace_bytes(n, pb.costs.size, int(nr.sum()), total_p, int(nr.max()), int(nM.max()))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    probs = torch.zeros(total_p, dtype=torch.float64, device=dev)
    status = torch.full((n,), -7, dtype=torch.int32, device=dev)

    def call():
        return lib.pda_association_perm_probs_batch(
            costs.data_ptr(), cost_off.data_ptr(), d_nL.data_ptr(), d_nM.data_ptr(), d_row.data_ptr(), n, pb.costs.size,
            int(nr.sum()), total_p, int(nr.max()), int(nM.max()), probs.data_ptr(), d_poff.data_ptr(), status.data_ptr(),
            ws.data_ptr(), ws_bytes, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        assert call() == 0                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        rc = call()                         # a host synchronisation inside would invalidate the capture
    assert rc == 0
    for scale in (1.0, 0.7):
        host = synth.ProblemBatch(np.ascontiguousarray(pb.costs * scale), pb.cost_off, pb.nL, pb.nM)
        costs.copy_(t(host.costs))
        graph.replay()
        torch.cuda.synchronize()
        want_t, want_s = gpu_api.association_perm_probs_batch(host)
        got = probs.cpu().numpy()
        np.testing.assert_array_equal(status.cpu().numpy(), want_s)
        np.testing.assert_array_equal(got.view(np.int64), np.concatenate([w.reshape(-1) for w in want_t]).view(np.int64))


@gpu
def test_multi_device_slices(gpu_api):
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    if lib.pda_device_count() < 2:
        pytest.skip("needs two devices")
    pb = synth.g2_gated(3000, first=77_000)
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    sizes = nM.astype(np.int64) * (nL.astype(np.int64) + 1)
    prob_off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    devs = np.arange(lib.pda_device_count(), dtype=np.int32)
    p = lambda a: a.ctypes.data
    probs, st = np.zeros(int(sizes.sum())), np.zeros(n, np.int32)
    _lib.check(lib.pda_association_perm_probs_batch_host_multi(p(pb.costs), p(pb.cost_off), p(nL), p(nM), n, p(probs), p(prob_off),
                                                               p(st), p(devs), len(devs)))
    want_t, want_s = gpu_api.association_perm_probs_batch(pb)
    np.testing.assert_array_equal(st, want_s)
    np.testing.assert_array_equal(probs.view(np.int64), np.concatenate([w.reshape(-1) for w in want_t]).view(np.int64))
    probs = np.zeros(int(sizes.sum()))
    _lib.check(lib.pda_association_probs_batch_host_multi(p(pb.costs), p(pb.cost_off), p(nL), p(nM), n, 200, p(probs), p(prob_off),
                                                          p(devs), len(devs)))
    want = gpu_api.association_probs_batch(pb, 200)
    np.testing.assert_array_equal(probs.view(np.int64), np.concatenate([w.reshape(-1) for w in want]).view(np.int64))


@gpu
def test_cpp_driver(gpu_api):
    exe = os.path.join(ROOT, "tests", "cpp", "build", "perm_association_b200")
    assert os.path.exists(exe), "tests/cpp/build/perm_association_b200 missing: run __graft_entry__.build()"
    frames = synth.quadric_frames(6, first=555)
    col = lambda c: c.transpose(0, 2, 1).reshape(-1)          # column-major 3x3, Eigen's layout
    parts = [f"{len(frames)} 10.0"]
    for lm, lc, mm, mc in frames:
        parts.append(f"{lm.shape[0]} {mm.shape[0]} " + " ".join(repr(float(x)) for x in
                                                               np.concatenate([lm.reshape(-1), col(lc), mm.reshape(-1), col(mc)])))
    run = subprocess.run([exe], input="\n".join(parts) + "\n", capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout[-500:] + run.stderr[-500:]
    got = {}
    for ln in run.stdout.splitlines():
        w = ln.split()
        got.setdefault((w[0], int(w[1])), []).append([float(x) for x in w[3:]])
    tabs, st = gpu_api.association_perm_from_moments_batch(frames, 10.0)
    assert not st.any()
    for kind in ("moments", "costs", "batch"):
        for f in range(len(frames)):
            np.testing.assert_array_equal(bits(np.array(got[(kind, f)])), bits(tabs[f]), err_msg=f"{kind} {f}")


# ---------------------------------------------------------------------------------------------------------------------
# CPU: no device needed
# ---------------------------------------------------------------------------------------------------------------------
def test_cpp_driver_compiles():
    src = os.path.join(ROOT, "tests", "cpp", "perm_association_driver.cpp")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), src],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-800:]


def test_shim_exports_the_batch_form():
    path = os.path.join(ROOT, "probabilisticsemslam_b200", "libpda_b200_shims.so")
    assert os.path.exists(path), "libpda_b200_shims.so missing: run __graft_entry__.build()"
    out = os.popen(f"nm -DC --defined-only {path}").read()
    assert "getAssignmentProbsBatch(" in out
    assert out.count("getAssignmentProbsFromMoments(") >= 2       # the six-argument form and the usePerm overload


def test_host_entries_reject_bad_arguments_before_any_device_work():
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    costs, probs = np.zeros(64), np.zeros(64)
    coff, poff, st = np.zeros(1, np.int64), np.zeros(1, np.int64), np.zeros(1, np.int32)

    def call(nl, nm, cost_off=0, prob_off=0, null=False):
        coff[0], poff[0] = cost_off, prob_off
        a, b = np.array([nl], np.int32), np.array([nm], np.int32)
        return lib.pda_association_perm_probs_batch_host(None if null else p(costs), p(coff), p(a), p(b), 1, p(probs), p(poff), p(st), 0)

    assert call(3, 2, null=True) == -1 and b"NULL" in lib.pda_last_error()
    assert call(-1, 2) == -1 and b"nL=-1" in lib.pda_last_error()
    assert call(3, 0) == -1 and b"nM=0" in lib.pda_last_error()
    assert call(3, 2, cost_off=-4) == -1 and b"negative offset" in lib.pda_last_error()
    assert call(3, 2, prob_off=-1) == -1 and b"negative offset" in lib.pda_last_error()
    assert call(200, 2) == -3                                                     # nL + nM above PDA_MAX_DIM
    assert lib.pda_association_perm_probs_batch_host(p(costs), p(coff), None, None, 0, p(probs), p(poff), p(st), 0) == 0
    devs = np.zeros(2, np.int32)
    a, b = np.array([3], np.int32), np.array([2], np.int32)
    assert lib.pda_association_perm_probs_batch_host_multi(p(costs), p(coff), p(a), p(b), 1, p(probs), p(poff), p(st), None, 0) == -1
    assert lib.pda_association_probs_batch_host_multi(None, p(coff), p(a), p(b), 1, 10, p(probs), p(poff), p(devs), 2) == -1
    lo, mo = np.array([0, 2], np.int64), np.array([3, 1], np.int64)                # detection offsets descending
    z = np.zeros(64)
    assert lib.pda_association_perm_from_moments_batch_host(p(z), p(z), p(lo), p(z), p(z), p(mo), 1, 10.0, p(probs), p(st), 0) == -1
    assert lib.pda_association_perm_from_moments_batch_host(p(z), p(z), p(lo), p(z), p(z), None, 1, 10.0, p(probs), p(st), 0) == -1


def test_device_form_takes_up_to_eleven_detections():
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    d, i64, i32 = np.zeros(64), np.zeros(4, np.int64), np.zeros(4, np.int32)
    assert lib.pda_association_perm_workspace_bytes(1, 14, 14, 3, 14, 12) == -3
    assert lib.pda_association_perm_workspace_bytes(1, 14, 14, 3, 14, 11) > 0
    assert lib.pda_association_perm_probs_batch(p(d), p(i64), p(i32), p(i32), p(i64), 1, 14, 14, 3, 14, 12, p(d), p(i64), p(i32),
                                                p(d), 512, None) == -3
    assert b"maxNumCol 12" in lib.pda_last_error()
    assert lib.pda_association_perm_probs_batch(None, p(i64), p(i32), p(i32), p(i64), 1, 14, 14, 3, 14, 3, p(d), p(i64), p(i32),
                                                p(d), 512, None) == -1
    assert lib.pda_association_perm_probs_batch(p(d), p(i64), p(i32), p(i32), p(i64), 1, 14, 14, 3, 14, 3, p(d), p(i64), p(i32),
                                                p(d), 16, None) == -4                # workspace too small


def test_no_device_means_an_error_not_a_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from probabilisticsemslam_b200 import _lib, api
    lib = _lib.lib()
    pb = synth.g2_gated(2, first=1)
    with pytest.raises(_lib.PdaError) as e:
        api.association_perm_probs_batch(pb)
    assert e.value.code == -2
    with pytest.raises(_lib.PdaError) as e:
        api.association_perm_from_moments_batch(synth.quadric_frames(1), 10.0)
    assert e.value.code == -2
    with pytest.raises(_lib.PdaError):
        api.getAssignmentProbsFromCosts(pb.matrix(0), 30, 200, usePerm=True)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    prob_off = np.array([0, int(nM[0]) * 31], np.int64)
    probs, st, devs = np.zeros(int(nM.sum()) * 31), np.zeros(2, np.int32), np.array([0, 1], np.int32)
    p = lambda a: a.ctypes.data
    assert lib.pda_association_perm_probs_batch_host_multi(p(pb.costs), p(pb.cost_off), p(nL), p(nM), 2, p(probs), p(prob_off), p(st),
                                                           p(devs), 2) == -2
    assert lib.pda_association_probs_batch_host_multi(p(pb.costs), p(pb.cost_off), p(nL), p(nM), 2, 50, p(probs), p(prob_off),
                                                      p(devs), 2) == -2
