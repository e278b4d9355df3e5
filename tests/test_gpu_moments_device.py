"""The device-pointer moments-to-weights calls, pda_association_from_moments_batch (k-best) and
pda_association_perm_from_moments_batch (usePerm): frame shapes read on the device against caller-given bounds, so one
CUDA graph serves frames of any shape within them.

Every computed table, its status, nFound and probOff must equal the _host forms (and the host prefix sums) bit for bit,
for bounds equal to the batch's maxima and for loose ones; rejected frames (status 2) must leave the tables untouched.
The CPU tests at the bottom check the argument handling, which runs before any device work."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import bits
from probabilisticsemslam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NONASSIGN = 10.0
SENTINEL = -7.25
gpu = pytest.mark.gpu


def unpack(lm, lc, lo, mm, mc, mo, f):
    """Frame f of packed moments back as the (land_mean, land_cov, meas_mean, meas_cov) tuple of synth.quadric_frames."""
    cov = lambda c: c.reshape(-1, 3, 3).transpose(0, 2, 1)  # stored column-major
    return (lm[lo[f]:lo[f + 1]], cov(lc[lo[f]:lo[f + 1]]), mm[mo[f]:mo[f + 1]], cov(mc[mo[f]:mo[f + 1]]))


def expected(api, packed, max_nL, max_nM, cap, k):
    """What the device form must produce, from the contract and the _host forms: (probOff, status, {frame: table},
    nFound or None).  k None = the usePerm form."""
    lm, lc, lo, mm, mc, mo = packed
    n = len(lo) - 1
    passing = [0 <= lo[f] <= lo[f + 1] <= len(lm) and 0 <= mo[f] <= mo[f + 1] <= len(mm) and lo[f + 1] - lo[f] <= max_nL
               and mo[f + 1] - mo[f] <= max_nM for f in range(n)]
    spans = np.array([(mo[f + 1] - mo[f]) * (lo[f + 1] - lo[f] + 1) if passing[f] else 0 for f in range(n)], np.int64)
    prob_off = np.concatenate([[0], np.cumsum(spans)]).astype(np.int64)
    run = [f for f in range(n) if passing[f] and not (spans[f] > 0 and prob_off[f + 1] > cap)]
    status = np.full(n, 2, np.int32)
    nf = np.full(n, -1, np.int32) if k is not None else None
    frames = [unpack(*packed, f) for f in run]
    if k is None:
        tabs, st = api.association_perm_from_moments_batch(frames, NONASSIGN) if frames else ([], [])
        status[run] = st
    else:
        tabs = api.association_from_moments_batch(frames, NONASSIGN, k) if frames else []
        status[run] = 0
        solved = [i for i, f in enumerate(frames) if f[2].shape[0] > 0]
        if solved:
            pb = synth.pack(api.quadric_cost_batch([frames[i] for i in solved], NONASSIGN), [frames[i][0].shape[0] for i in solved])
            cond, _ = api.condition_costs_batch(pb)
            nf[[run[i] for i in solved]] = api.assignment_prob_batch(cond, k).n_found
    return prob_off, status, dict(zip(run, tabs)), nf


def run_device(api, packed, max_nL, max_nM, k, cap=None):
    import torch
    lm, lc, lo, mm, mc, mo = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in packed]
    n = lo.shape[0] - 1
    cap = n * max_nM * (max_nL + 1) if cap is None else cap
    probs = torch.full((max(cap, 1),), SENTINEL, dtype=torch.float64, device="cuda")
    if k is None:
        out = api.association_perm_from_moments_batch_device(lm, lc, lo, mm, mc, mo, max_nL, max_nM, NONASSIGN, cap, probs)
    else:
        nf = torch.full((max(n, 1),), -9, dtype=torch.int32, device="cuda")
        out = api.association_from_moments_batch_device(lm, lc, lo, mm, mc, mo, max_nL, max_nM, NONASSIGN, k, cap, probs, n_found=nf)
    torch.cuda.synchronize()
    res = [t.cpu().numpy() for t in out]
    res[2] = res[2][:n]
    if k is not None:
        res[3] = res[3][:n]
    return res


def assert_matches(got, want, cap, what):
    probs, prob_off, status = got[:3]
    w_off, w_status, w_tabs, w_nf = want
    np.testing.assert_array_equal(prob_off, w_off, err_msg=f"{what}: probOff")
    np.testing.assert_array_equal(status, w_status, err_msg=f"{what}: status")
    if w_nf is not None:
        np.testing.assert_array_equal(got[3], w_nf, err_msg=f"{what}: nFound")
    touched = np.zeros(max(cap, 1), bool)
    for f, tab in w_tabs.items():
        span = slice(int(w_off[f]), int(w_off[f + 1]))
        np.testing.assert_array_equal(bits(probs[span]), bits(tab.reshape(-1)), err_msg=f"{what}: frame {f}")
        touched[span] = True
    assert np.all(probs[~touched] == SENTINEL), f"{what}: a table entry outside the computed frames was written"


def maxima(frames):
    return max(f[0].shape[0] for f in frames), max(f[2].shape[0] for f in frames)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [1, 200, None], ids=["k1", "k200", "usePerm"])
def test_bit_identical_to_the_host_forms(gpu_api, k):
    frames = synth.quadric_frames(2000, first=31_000)
    packed = gpu_api._pack_moments(frames)
    for max_nL, max_nM in (maxima(frames), (60, 11)):
        cap = int(sum(f[2].shape[0] * (f[0].shape[0] + 1) for f in frames))
        want = expected(gpu_api, packed, max_nL, max_nM, cap, k)
        assert not (want[1] == 2).any()
        assert_matches(run_device(gpu_api, packed, max_nL, max_nM, k, cap), want, cap, f"bounds {max_nL}/{max_nM}")


def ragged_packed():
    """Frames of every shape the bounds (30 landmarks, 6 detections) allow and several they do not: nL = 0, nM = 0,
    nM = 1, nM = 6, nM = 7..8 and nL = 35 (above the bounds), interleaved with ordinary frames; then offsets that
    descend and offsets that reach past the arrays' capacities."""
    base = synth.quadric_frames(40, first=4_400)
    big = synth.quadric_frames(3, nL=35, first=4_500)
    frames = []
    for i, f in enumerate(base):
        lm, lc, mm, mc = f
        if i % 8 == 1:
            f = (lm[:0], lc[:0], mm, mc)            # nL = 0
        elif i % 8 == 3:
            f = (lm, lc, mm[:0], mc[:0])            # nM = 0
        elif i % 8 == 5:
            f = (lm, lc, mm[:1], mc[:1])            # nM = 1
        frames.append(f)
        if i % 13 == 6:
            frames.append(big[i % 3])               # nL above the bound
    lm, lc, lo, mm, mc, mo = (np.array(a) for a in synth_pack(frames))
    n = len(lo) - 1
    lo[12] = lo[11] - 1                             # frame 11 descends (frame 12 grows)
    mo[20] = len(mm) + 3                            # frame 19 ends past the detection capacity, frame 20 descends
    lo[30] = len(lm) + 1                            # frame 29 past the landmark capacity, frame 30 descends
    mo[n - 4] = -1                                  # a negative offset
    return lm, lc, lo, mm, mc, mo


def synth_pack(frames):
    from probabilisticsemslam_b200 import api
    return api._pack_moments(frames)


@gpu
@pytest.mark.parametrize("k", [200, None], ids=["k200", "usePerm"])
def test_ragged_batch(gpu_api, k):
    packed = ragged_packed()
    lo, mo = packed[2], packed[5]
    n = len(lo) - 1
    nLs, nMs = np.diff(lo), np.diff(mo)
    ok = [(0 <= nLs[f] <= 30 and 0 <= nMs[f] <= 6) for f in range(n)]
    assert {0, 1, 6} <= {int(nMs[f]) for f in range(n) if ok[f]} and any(nLs[f] == 0 and ok[f] for f in range(n))
    assert any(nMs > 6) and any(nLs > 30) and any(nLs < 0) and any(nMs < 0)
    full = expected(gpu_api, packed, 30, 6, 1 << 40, k)[0][-1]
    for cap in (int(full), int(full) // 2):        # the second capacity cuts the batch in the middle
        want = expected(gpu_api, packed, 30, 6, cap, k)
        assert len(want[2]) >= (15 if cap == full else 5)
        if cap < full:
            assert any(want[1][f] == 2 and want[0][f + 1] > want[0][f] for f in range(n))  # kept span, not computed
        got = run_device(gpu_api, packed, 30, 6, k, cap)
        assert_matches(got, want, cap, f"ragged, capacity {cap}")


@gpu
@pytest.mark.parametrize("k", [200, None], ids=["k200", "usePerm"])
@pytest.mark.parametrize("n", [1, 64])
def test_graph_replay_across_shapes(gpu_api, k, n):
    import torch
    from probabilisticsemslam_b200 import _lib
    max_nL, max_nM = 40, 8
    dev = torch.device("cuda:0")
    lm = torch.zeros(n * max_nL * 3, dtype=torch.float64, device=dev)
    lc = torch.zeros(n * max_nL * 9, dtype=torch.float64, device=dev)
    mm = torch.zeros(n * max_nM * 3, dtype=torch.float64, device=dev)
    mc = torch.zeros(n * max_nM * 9, dtype=torch.float64, device=dev)
    lo = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    mo = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    cap = n * max_nM * (max_nL + 1)
    probs = torch.full((cap,), SENTINEL, dtype=torch.float64, device=dev)
    prob_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    nf = torch.empty(n, dtype=torch.int32, device=dev)
    lib = _lib.lib()
    ws_bytes = (lib.pda_association_from_moments_workspace_bytes(n, max_nL, max_nM, cap, k) if k is not None else
                lib.pda_association_perm_from_moments_workspace_bytes(n, max_nL, max_nM, cap))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def call():
        if k is None:
            return gpu_api.association_perm_from_moments_batch_device(lm, lc, lo, mm, mc, mo, max_nL, max_nM, NONASSIGN, cap,
                                                                      probs, prob_off, status, ws)
        return gpu_api.association_from_moments_batch_device(lm, lc, lo, mm, mc, mo, max_nL, max_nM, NONASSIGN, k, cap, probs,
                                                             prob_off, status, nf, ws)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()                                       # warm-up outside the capture (all-zero offsets: 0 x 0 frames)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()                                       # a host synchronisation inside would invalidate the capture
    shapes = [(30, 20), (12, 40), (2, 7), (40, 3), (25, 33), (1, 18)]
    for rep, (a, b) in enumerate(shapes):            # landmark counts of the two halves of the batch
        frames = synth.quadric_frames((n + 1) // 2, nL=a, first=9_000 + 100 * rep)
        if n > 1:
            frames += synth.quadric_frames(n // 2, nL=b, first=9_050 + 100 * rep)
        packed = gpu_api._pack_moments(frames)
        for buf, host in zip((lm, lc, lo, mm, mc, mo), packed):
            flat = torch.from_numpy(np.ascontiguousarray(host).reshape(-1)).to(dev)
            buf[:flat.numel()].copy_(flat)
        probs.fill_(SENTINEL)
        graph.replay()
        torch.cuda.synchronize()
        want = expected(gpu_api, packed, max_nL, max_nM, cap, k)
        got = [probs.cpu().numpy(), prob_off.cpu().numpy(), status.cpu().numpy()] + ([nf.cpu().numpy()] if k is not None else [])
        assert not (want[1] == 2).any()
        assert_matches(got, want, cap, f"replay {rep} (nL {a} / {b})")


@gpu
@pytest.mark.parametrize("k", [200, None], ids=["k200", "usePerm"])
def test_one_hundred_thousand_frames_in_one_call(gpu_api, k):
    frames = synth.quadric_frames(100_000, first=2_000_000)
    packed = gpu_api._pack_moments(frames)
    got = run_device(gpu_api, packed, *maxima(frames), k)
    assert not (got[2] == 2).any()
    sample = np.sort(np.random.default_rng(11).choice(len(frames), 500, replace=False))
    sub = [frames[f] for f in sample]
    spans = np.array([f[2].shape[0] * (f[0].shape[0] + 1) for f in frames], np.int64)
    np.testing.assert_array_equal(got[1], np.concatenate([[0], np.cumsum(spans)]))
    _, w_status, w_tabs, w_nf = expected(gpu_api, gpu_api._pack_moments(sub), *maxima(frames), 1 << 40, k)
    for i, f in enumerate(sample):
        np.testing.assert_array_equal(bits(got[0][got[1][f]:got[1][f + 1]]), bits(w_tabs[i].reshape(-1)), err_msg=f"frame {f}")
        assert got[2][f] == w_status[i]
        if k is not None:
            assert got[3][f] == w_nf[i]


@gpu
def test_smallest_workspace(gpu_api):
    import torch
    from probabilisticsemslam_b200._lib import PdaError
    frames = synth.quadric_frames(50, first=8_100)
    args = gpu_api.moments_to_device(frames)
    for k in (200, None):
        name = "pda_association_from_moments" if k is not None else "pda_association_perm_from_moments"
        extra = (k,) if k is not None else ()
        need = getattr(gpu_api.lib(), name + "_workspace_bytes")(50, 30, 8, 50 * 8 * 31, *extra)
        assert need > 0
        call = (lambda ws: gpu_api.association_from_moments_batch_device(*args, 30, 8, NONASSIGN, k, workspace=ws)) if k else \
               (lambda ws: gpu_api.association_perm_from_moments_batch_device(*args, 30, 8, NONASSIGN, workspace=ws))
        smallest = call(torch.empty(need, dtype=torch.uint8, device="cuda"))
        full = call(None)
        torch.cuda.synchronize()
        for a, b in zip(smallest, full):
            np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy())
        with pytest.raises(PdaError, match="error -4"):
            call(torch.empty(need - 1, dtype=torch.uint8, device="cuda"))


@gpu
def test_cpp_graph_driver(gpu_api):
    exe = os.path.join(ROOT, "tests", "cpp", "build", "moments_graph_b200")
    assert os.path.exists(exe), "tests/cpp/build/moments_graph_b200 missing: run __graft_entry__.build()"
    frames = synth.quadric_frames(4, first=777) + synth.quadric_frames(1, nL=12, first=778) + synth.quadric_frames(1, nL=40, first=779)
    col = lambda c: c.transpose(0, 2, 1).reshape(-1)
    parts = [f"{len(frames)} {NONASSIGN}"]
    for lm, lc, mm, mc in frames:
        parts.append(f"{lm.shape[0]} {mm.shape[0]} " + " ".join(repr(float(x)) for x in
                                                               np.concatenate([lm.reshape(-1), col(lc), mm.reshape(-1), col(mc)])))
    run = subprocess.run([exe], input="\n".join(parts) + "\n", capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout[-500:] + run.stderr[-500:]
    rows, stats = {}, {}
    for ln in run.stdout.splitlines():
        w = ln.split()
        if w[0] == "status":
            stats[(w[1], int(w[2]))] = [int(x) for x in w[3:]]
        else:
            rows.setdefault((w[0], int(w[1])), []).append([float(x) for x in w[3:]])
    kbest = gpu_api.association_from_moments_batch(frames, NONASSIGN, 200)
    perm, st = gpu_api.association_perm_from_moments_batch(frames, NONASSIGN)
    for f, (lm, _, mm, _) in enumerate(frames):
        span = mm.shape[0] * (lm.shape[0] + 1)
        np.testing.assert_array_equal(bits(np.array(rows[("kbest", f)])), bits(kbest[f]), err_msg=f"k-best frame {f}")
        np.testing.assert_array_equal(bits(np.array(rows[("perm", f)])), bits(perm[f]), err_msg=f"usePerm frame {f}")
        assert stats[("kbest", f)][:2] == [0, span] and stats[("kbest", f)][2] > 0
        assert stats[("perm", f)][:2] == [int(st[f]), span]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: no device needed
# ---------------------------------------------------------------------------------------------------------------------
def test_cpp_graph_driver_compiles():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cuda_inc = os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "include")
    assert os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")), f"no CUDA headers at {cuda_inc}"
    src = os.path.join(ROOT, "tests", "cpp", "moments_graph_driver.cpp")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", cuda_inc, src],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-800:]


def _buf():
    buf = ctypes.create_string_buffer(1 << 16)
    return buf, ctypes.cast(buf, ctypes.c_void_p).value


def _kbest_args(p):
    #       lm lc lo cap mm mc mo cap  n  maxNL maxNM nonassign k  probs cap probOff status nFound ws  wsBytes    stream
    return [p, p, p, 40, p, p, p, 8, 1, 30, 8, 10.0, 200, p, 248, p, p, p, p, 1 << 16, None]


def _perm_args(p):
    return [p, p, p, 40, p, p, p, 8, 1, 30, 8, 10.0, p, 248, p, p, p, 1 << 16, None]


def test_argument_errors():
    from probabilisticsemslam_b200._lib import lib
    L = lib()
    keep, p = _buf()
    for fn, args, null_ok in ((L.pda_association_from_moments_batch, _kbest_args(p), {17, 20}),
                              (L.pda_association_perm_from_moments_batch, _perm_args(p), {18})):
        def call(**kw):
            a = list(args)
            for i, v in kw.items():
                a[int(i[1:])] = v
            return fn(*a)
        ptr_slots = [i for i, v in enumerate(args) if v == p]
        for i in ptr_slots:
            if i not in null_ok:
                assert call(**{f"a{i}": None}) == -1, i
                assert b"NULL" in L.pda_last_error()
        assert call(a3=-1) == -1 and call(a7=-1) == -1   # negative capacities
        assert call(a8=-1) == -1                          # nFrames
        assert call(a9=-1) == -1 and call(a10=0) == -1    # maxNL < 0, maxNM < 1
        assert call(a9=121, a10=8) == -3                  # maxNL + maxNM above 128
        assert b"above 128" in L.pda_last_error()
    assert L.pda_association_from_moments_batch(*_kbest_args(p)[:12], 0, *_kbest_args(p)[13:]) == -1  # k < 1
    assert L.pda_association_from_moments_workspace_bytes(-1, 30, 8, 248, 200) == -1
    assert L.pda_association_from_moments_workspace_bytes(1, 30, 8, 248, 0) == -1
    assert L.pda_association_from_moments_workspace_bytes(1, 100, 29, 248, 200) == -3
    # usePerm: at most 11 detections (the fused pipeline); the workspace size needs no device
    assert L.pda_association_perm_from_moments_workspace_bytes(1, 30, 12, 248) == -3
    assert L.pda_association_perm_from_moments_workspace_bytes(1, 30, 11, 248) > 0
    a = _perm_args(p)
    a[10] = 12
    assert L.pda_association_perm_from_moments_batch(*a) == -3
    need = L.pda_association_perm_from_moments_workspace_bytes(1, 30, 8, 248)
    a = _perm_args(p)
    a[17] = need - 1
    assert L.pda_association_perm_from_moments_batch(*a) == -4
    assert b"workspace" in L.pda_last_error()


def test_no_device_is_a_cuda_error():
    from probabilisticsemslam_b200._lib import lib
    L = lib()
    if L.pda_device_count() > 0:
        pytest.skip("a device is visible")
    keep, p = _buf()
    assert L.pda_association_from_moments_batch(*_kbest_args(p)) == -2
    assert L.pda_association_from_moments_workspace_bytes(1, 30, 8, 248, 200) == -2
    assert L.pda_association_perm_from_moments_batch(*_perm_args(p)) == -2
