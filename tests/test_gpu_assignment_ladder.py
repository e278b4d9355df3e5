"""assignmentProb for several k from one Murty enumeration (pda_assignment_prob_ladder_batch and its layers).

Every slot must be bit-identical (NaN positions included) to a separate assignment_prob_batch call with its k, and
carry that call's nFound, under all three Murty kernels; the C++ drop-in form is held to the reference's own tables;
the device-pointer and page-locked forms to the host form.  The argument checks run without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import compmethods_dat_files, golden, rel_err
from probabilisticsemslam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LADDER_BIN = os.path.join(ROOT, "tests", "cpp", "build", "ladder_b200")


def _assert_matches_single_calls(api, pb, ks):
    tabs, nf = api.assignment_prob_ladder_batch(pb, ks)
    assert nf.shape == (len(pb), len(ks))
    for j, k in enumerate(ks):
        one = api.assignment_prob_batch(pb, int(k))
        np.testing.assert_array_equal(nf[:, j], one.n_found, err_msg=f"nFound of slot {j} (k={k})")
        for p in range(len(pb)):
            want = one.prob_table(pb, p)
            assert np.array_equal(tabs[p][j], want, equal_nan=True), f"problem {p}, slot {j} (k={k})"
            assert np.array_equal(np.isnan(tabs[p][j]), np.isnan(want))
    return tabs, nf


@pytest.mark.gpu
def test_g1(murty_path, gpu_api):
    _assert_matches_single_calls(gpu_api, synth.g1_dense(2000, first=41000), [1, 20, 100, 200])


@pytest.mark.gpu
def test_g1_int_ties(murty_path, gpu_api):
    """Integer costs tie, so the pruning kernel hands problems to the exact ladder kernel."""
    _assert_matches_single_calls(gpu_api, synth.g1_dense(600, first=43000, integer=True), [1, 7, 50, 200])


@pytest.mark.gpu
def test_g2_conditioned_unsorted_with_duplicate(murty_path, gpu_api):
    """compMethods' own order of k, plus a duplicate: many problems stop at the cutoff below some k."""
    pb, _ = gpu_api.condition_costs_batch(synth.g2_gated(2000, first=47000))
    ks = [1, 20, 1000, 100, 200, 150, 200]
    _, nf = _assert_matches_single_calls(gpu_api, pb, ks)
    assert (nf[:, 2] < 1000).mean() > 0.5, "the cutoff should end most G2 enumerations early"
    np.testing.assert_array_equal(nf[:, 4], nf[:, 6])


def _edge_batch():
    rng = np.random.default_rng(7)
    mats, nls = [], []
    for nM, nL in ((1, 5), (3, 4), (1, 0), (4, 2), (2, 30), (5, 9)):
        mats.append(rng.uniform(0.0, 20.0, (nL + nM, nM)))
        nls.append(nL)
    bad = rng.uniform(0.0, 5.0, (6, 3))
    bad[:, 1] = np.inf                      # a detection nobody can take: infeasible
    mats.append(bad); nls.append(3)
    few = rng.uniform(0.0, 5.0, (3, 2))     # 3 x 2: 6 assignments, fewer than most k below
    mats.append(few); nls.append(1)
    return synth.pack(mats, nls)


@pytest.mark.gpu
def test_ragged_edges(murty_path, gpu_api):
    pb = _edge_batch()
    tabs, nf = _assert_matches_single_calls(gpu_api, pb, [1, 3, 7, 50, 1000])
    assert (nf[6] == 0).all() and np.isnan(tabs[6]).all()        # infeasible
    assert nf[7, -1] == 6                                          # k above the number of assignments
    _assert_matches_single_calls(gpu_api, pb, [20])               # nK = 1


@pytest.mark.gpu
def test_against_oracle(gpu_api, oracle):
    pb, _ = gpu_api.condition_costs_batch(synth.g2_gated(200, first=51000))
    ks = [1, 20, 100, 200]
    tabs, _ = gpu_api.assignment_prob_ladder_batch(pb, ks)
    for p in range(len(pb)):
        for j, k in enumerate(ks):
            want = oracle.assignment_prob(pb.matrix(p), int(pb.nL[p]), k)
            assert rel_err(tabs[p][j], want) <= 1e-9, f"problem {p}, k={k}"
    single = gpu_api.assignmentProbLadder(pb.matrix(0), int(pb.nL[0]), ks)
    assert np.array_equal(single, tabs[0], equal_nan=True)


def _parse_tables(text):
    """frame <i> / <tag> <m> p0 p1 ... lines -> {(frame, tag): [rows]}"""
    out, frame = {}, -1
    for line in text.splitlines():
        t = line.split()
        if not t:
            continue
        if t[0] == "frame":
            frame += 1
        elif t[0] in ("k1", "k20", "k100", "k200", "k150"):
            out.setdefault((frame, t[0]), []).append([float(x) for x in t[2:]])
    return out


@pytest.mark.gpu
def test_cpp_driver_against_reference_output(tmp_path, gpu_api):
    assert os.path.exists(LADDER_BIN), "tests/cpp/build/ladder_b200 missing: run __graft_entry__.build()"
    files = [path for path, _ in compmethods_dat_files(str(tmp_path))]
    run = subprocess.run([LADDER_BIN, "--k", "150"] + files, capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-500:] + run.stderr[-500:]
    got, want = _parse_tables(run.stdout), _parse_tables(str(golden("compmethods_k150")["stdout"]))
    assert set(got) == set(want) and len(want) == 5 * len(files)
    for key in want:
        a, b = np.asarray(got[key]), np.asarray(want[key])
        assert a.shape == b.shape, key
        assert rel_err(a, b) <= 1e-9, key


def _device_call(api, pb, ks, ws_bytes=None):
    import torch
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    dev = torch.device("cuda:0")
    nk = len(ks)
    nL = pb.nL.astype(np.int32)
    cells = pb.nM.astype(np.int64) * (nL.astype(np.int64) + 1)
    prob_off = np.zeros(len(pb), np.int64)
    prob_off[1:] = np.cumsum(cells * nk)[:-1]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    costs, cost_off, nr, nc, nl, poff = t(pb.costs), t(pb.cost_off), t(pb.num_row), t(pb.nM.astype(np.int32)), t(nL), t(prob_off)
    probs = torch.full((int(cells.sum()) * nk,), -7.0, dtype=torch.float64, device=dev)
    nf = torch.full((len(pb) * nk,), -7, dtype=torch.int32, device=dev)
    maxr, maxc = int(pb.num_row.max()), int(pb.nM.max())
    full = lib.pda_murty_workspace_bytes(len(pb), int(max(ks)), maxr, maxc)
    assert full > 0
    ws = torch.empty(int(full if ws_bytes is None else ws_bytes(full)), dtype=torch.uint8, device=dev)
    ks32 = np.ascontiguousarray(ks, np.int32)
    stream = torch.cuda.current_stream().cuda_stream
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    _lib.check(lib.pda_assignment_prob_ladder_batch(p(costs), p(cost_off), p(nr), p(nc), p(nl), len(pb), maxr, maxc,
                                                    ks32.ctypes.data, nk, p(probs), p(poff), p(nf), p(ws), ws.numel(),
                                                    ctypes.c_void_p(stream)))
    torch.cuda.synchronize()
    return probs.cpu().numpy(), nf.cpu().numpy().reshape(len(pb), nk)


@pytest.mark.gpu
def test_device_pointer_form(murty_path, gpu_api):
    pb, _ = gpu_api.condition_costs_batch(synth.g2_gated(1500, first=53000))
    ks = [200, 1, 20, 100]
    tabs, nf = gpu_api.assignment_prob_ladder_batch(pb, ks)
    host = np.concatenate([t.reshape(-1) for t in tabs])
    for ws in (None, lambda full: 256 + 4 * (full - 256) // max(len(pb), 1)):   # full, then a workspace for a few warps
        probs, nfd = _device_call(gpu_api, pb, ks, ws)
        np.testing.assert_array_equal(nfd, nf)
        assert np.array_equal(probs, host, equal_nan=True)


@pytest.mark.gpu
def test_page_locked_buffers(gpu_api):
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    pb = synth.g1_dense(3000, first=55000)
    ks = np.asarray([1, 20, 100], np.int32)
    tabs, nf = gpu_api.assignment_prob_ladder_batch(pb, ks)
    nk, nL = len(ks), pb.nL.astype(np.int32)
    num_row, num_col = pb.num_row, pb.nM.astype(np.int32)   # held: ctypes gets bare addresses
    cells = pb.nM.astype(np.int64) * (nL.astype(np.int64) + 1)
    prob_off = np.zeros(len(pb), np.int64)
    prob_off[1:] = np.cumsum(cells * nk)[:-1]
    n_out = int(cells.sum()) * nk
    pin_in, pin_out = lib.pda_host_alloc(pb.costs.nbytes), lib.pda_host_alloc(n_out * 8)
    assert pin_in and pin_out
    try:
        costs = np.ctypeslib.as_array((ctypes.c_double * pb.costs.size).from_address(pin_in))
        costs[:] = pb.costs
        probs = np.ctypeslib.as_array((ctypes.c_double * n_out).from_address(pin_out))
        probs[:] = -7.0
        found = np.zeros((len(pb), nk), np.int32)
        _lib.check(lib.pda_assignment_prob_ladder_batch_host(pin_in, pb.cost_off.ctypes.data, num_row.ctypes.data,
                                                             num_col.ctypes.data, nL.ctypes.data, len(pb),
                                                             ks.ctypes.data, nk, pin_out, prob_off.ctypes.data,
                                                             found.ctypes.data, 0))
        np.testing.assert_array_equal(found, nf)
        assert np.array_equal(probs, np.concatenate([t.reshape(-1) for t in tabs]), equal_nan=True)
    finally:
        lib.pda_host_free(pin_in)
        lib.pda_host_free(pin_out)


# ---- CPU only ------------------------------------------------------------------------------------------
def _host_call(ks, nk):
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    costs = np.zeros(12)
    off, poff = np.zeros(1, np.int64), np.zeros(1, np.int64)
    nr, nc, nl = np.array([4], np.int32), np.array([2], np.int32), np.array([2], np.int32)
    probs, found = np.zeros(6 * 17), np.zeros(17, np.int32)
    ksp = None if ks is None else np.ascontiguousarray(ks, np.int32).ctypes.data
    return lib.pda_assignment_prob_ladder_batch_host(costs.ctypes.data, off.ctypes.data, nr.ctypes.data, nc.ctypes.data,
                                                     nl.ctypes.data, 1, ksp, nk, probs.ctypes.data, poff.ctypes.data,
                                                     found.ctypes.data, 0)


def test_ladder_argument_checks_without_a_device():
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    assert _host_call([5], 0) == -1 and b"nK" in lib.pda_last_error()
    assert _host_call(list(range(1, 18)), 17) == -1 and b"nK" in lib.pda_last_error()
    assert _host_call([5, 0, 3], 3) == -1 and b"k >= 1" in lib.pda_last_error()
    assert _host_call(None, 2) == -1 and b"NULL ks" in lib.pda_last_error()
    ks = np.array([5], np.int32)
    assert lib.pda_assignment_prob_ladder_batch(None, None, None, None, None, 1, 4, 2, ks.ctypes.data, 0, None, None, None,
                                                None, 0, None) == -1


def test_ladder_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from probabilisticsemslam_b200 import _lib
    assert _host_call([1, 20, 5], 3) == -2 and b"no CUDA device" in _lib.lib().pda_last_error()
