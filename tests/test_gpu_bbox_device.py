"""The device-pointer stereo box association, pda_asgn_bb_batch: frame shapes read on the device against caller-given
bounds (left boxes, and left + right boxes), so one CUDA graph serves frames of any shape within them; its multi-device
form pda_asgn_bb_batch_host_multi; and the _host form on a slice of a larger batch (offL[0] > 0).

Every computed frame must equal the _host form (and the oracle) entry for entry, for bounds equal to the batch's maxima
and for loose ones; frames that are not computed (status 2) and entries outside every computed frame must keep what the
caller put there.  The CPU tests at the bottom check the argument handling, which runs before any device work."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import golden
from probabilisticsemslam_b200 import synth
from test_gpu_lap_conditioning_bbox import box_frame, box_frames

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NONASSIGN = 0.2
SENTINEL = -9
gpu = pytest.mark.gpu


def pack(lefts, rights):
    """Frames back to back: (flat left boxes, offL, flat right boxes, offR)."""
    off = lambda bs: np.concatenate([[0], np.cumsum([len(b) for b in bs])]).astype(np.int64)
    flat = lambda bs: np.concatenate([np.asarray(b, np.float64).reshape(-1, 5) for b in bs] + [np.zeros((0, 5))])
    return flat(lefts), off(lefts), flat(rights), off(rights)


def maxima(lefts, rights):
    return max(1, max(len(L) for L in lefts)), max(1, max(len(L) + len(R) for L, R in zip(lefts, rights)))


def run_device(api, bl, ol, br, orr, max_nL, max_boxes, nonassign=NONASSIGN, workspace=None):
    """pda_asgn_bb_batch on host arrays moved to the device; assignment starts as SENTINEL.  -> (assignment, status)."""
    import torch
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    asg = torch.full((max(len(bl), 1),), SENTINEL, dtype=torch.int32, device="cuda")
    a, st = api.asgn_bb_batch_device(t(bl), t(ol), t(br), t(orr), max_nL, max_boxes, nonassign, asg, workspace=workspace)
    torch.cuda.synchronize()
    return a.cpu().numpy(), st.cpu().numpy()


def assert_frames(got, ol, want, what):
    for f, w in enumerate(want):
        np.testing.assert_array_equal(got[ol[f]:ol[f + 1]], w, err_msg=f"{what}: frame {f}")


@gpu
@pytest.mark.parametrize("bounds", ["tight", "loose"])
def test_device_form_matches_host_form_and_oracle(gpu_api, oracle, bounds):
    lefts, rights = synth.stereo_boxes(2000, first=50_000)
    bl, ol, br, orr = pack(lefts, rights)
    max_nL, max_boxes = maxima(lefts, rights) if bounds == "tight" else (64, 128)
    got, st = run_device(gpu_api, bl, ol, br, orr, max_nL, max_boxes)
    assert not st.any()
    host = gpu_api.asgn_bb_batch(lefts, rights, NONASSIGN)
    assert_frames(got, ol, host, f"{bounds} bounds vs _host")
    for f in range(0, 2000, 7):
        np.testing.assert_array_equal(host[f], oracle.asgn_bb(lefts[f], rights[f], NONASSIGN)[:len(lefts[f])], err_msg=f"oracle {f}")


@gpu
def test_golden_through_device_form(gpu_api):
    z = golden("asgn_bb")
    n = int(z["n"])
    lefts, rights = [z[f"L{i}"].reshape(-1, 5) for i in range(n)], [z[f"R{i}"].reshape(-1, 5) for i in range(n)]
    bl, ol, br, orr = pack(lefts, rights)
    got, st = run_device(gpu_api, bl, ol, br, orr, *maxima(lefts, rights), float(z["nonassign"]))
    assert not st.any()
    assert_frames(got, ol, [z[f"a{i}"] for i in range(n)], "golden")


@gpu
@pytest.mark.parametrize("nonassign", [0.0, 0.2, 1.5])
def test_wide_frames_in_one_call(murty_path, gpu_api, oracle, nonassign):
    """box_frames(): 5 + 123 and 123 + 5 boxes side by side, so only a bound on nL + nR takes them in one call."""
    frames = box_frames()
    lefts, rights = [L for L, _ in frames], [R for _, R in frames]
    bl, ol, br, orr = pack(lefts, rights)
    got, st = run_device(gpu_api, bl, ol, br, orr, max(len(L) for L in lefts), 128, nonassign)
    assert not st.any()
    assert_frames(got, ol, [oracle.asgn_bb(L, R, nonassign)[:len(L)] for L, R in frames], f"{murty_path} vs oracle")
    assert_frames(got, ol, gpu_api.asgn_bb_batch(lefts, rights, nonassign), f"{murty_path} vs _host")


# frame f: left boxes [OFF_L[f], OFF_L[f+1]), right boxes [OFF_R[f], OFF_R[f+1]); capacities 66 / 30, bounds 12 / 24
OFF_L = [5, 15, 7, 8, 20, 26, 26, 30, 32, 34, 36, 49, 59, 62, 70]
OFF_R = [0, 8, 10, 12, 14, 20, 23, 23, 31, -2, 3, 6, 21, 24, 26]
RAGGED_STATUS = [0,  # [5, 15): computed though it starts past 0
                 2,  # left range descending
                 2,  # [7, 8) starts below offL[1] = 15: frame 0 owns those entries
                 2,  # [8, 20): the same
                 0,
                 0,  # no left box
                 0,  # no right box: every left box -1
                 2,  # right range past capR
                 2,  # right range descending
                 2,  # right range starts below 0
                 2,  # nL = 13 > maxNL
                 2,  # nL + nR = 25 > maxBoxes
                 0,  # computed after all of the above
                 2]  # left range past capL


@gpu
def test_ragged_batch_every_rejection(gpu_api):
    lefts, rights = synth.stereo_boxes(40, first=70_000)
    poolL = np.concatenate(lefts)[:66].copy()
    poolR = np.concatenate(rights)[:30].copy()
    assert len(poolL) == 66 and len(poolR) == 30
    poolR[0:8, 4] = 0.0
    poolL[5:13] = poolR[0:8]                          # frame 0 has pairs to find
    ol, orr = np.array(OFF_L, np.int64), np.array(OFF_R, np.int64)
    got, st = run_device(gpu_api, poolL, ol, poolR, orr, 12, 24)
    np.testing.assert_array_equal(st, RAGGED_STATUS)
    want = np.full(66, SENTINEL, np.int32)
    for f in np.flatnonzero(st == 0):
        L, R = poolL[ol[f]:ol[f + 1]], poolR[orr[f]:orr[f + 1]]
        want[ol[f]:ol[f + 1]] = gpu_api.asgn_bb_batch([L], [R], NONASSIGN)[0]
    assert (want[5:15] >= 0).any() and (want[26:30] == -1).all()
    np.testing.assert_array_equal(got, want)


@gpu
def test_overlap_example_from_the_header(gpu_api):
    """offL = [0, 10, 2, 3, 4]: frame 1 descends, frames 2 and 3 lie inside frame 0; only frame 0 is computed."""
    L, R0 = box_frame(10, 6, 77)
    R = np.concatenate([R0, box_frame(2, 2, 78)[1]])
    ol = np.array([0, 10, 2, 3, 4], np.int64)
    orr = np.array([0, 6, 6, 7, 8], np.int64)
    got, st = run_device(gpu_api, L, ol, R, orr, 10, 20)
    np.testing.assert_array_equal(st, [0, 2, 2, 2])
    np.testing.assert_array_equal(got, gpu_api.asgn_bb_batch([L], [R0], NONASSIGN)[0])


@gpu
@pytest.mark.parametrize("n", [1, 64])
def test_graph_replay_across_shapes(gpu_api, n):
    import torch
    from probabilisticsemslam_b200 import _lib
    max_nL, max_boxes = 24, 40
    dev = torch.device("cuda:0")
    bl = torch.zeros(n * max_nL * 5, dtype=torch.float64, device=dev)
    br = torch.zeros(n * max_boxes * 5, dtype=torch.float64, device=dev)
    ol = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    orr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    asg = torch.full((n * max_nL,), SENTINEL, dtype=torch.int32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    ws_bytes = _lib.lib().pda_asgn_bb_workspace_bytes(n, max_nL, max_boxes)
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def call():
        return gpu_api.asgn_bb_batch_device(bl, ol, br, orr, max_nL, max_boxes, NONASSIGN, asg, status, ws)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()                                       # warm-up outside the capture (all-zero offsets: empty frames)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()                                       # a host synchronisation inside would invalidate the capture
    shapes = [((5, 4), (24, 16)), ((1, 1), (0, 7)), ((12, 0), (17, 3)), ((24, 1), (3, 37)), ((8, 8), (2, 2)), ((0, 0), (20, 20))]
    for rep, (a, b) in enumerate(shapes):            # (nL, nR) of the two halves of the batch
        frames = [box_frame(*(a if f < (n + 1) // 2 else b), 600 + 100 * rep + f) for f in range(n)]
        lefts, rights = [L for L, _ in frames], [R for _, R in frames]
        hl, hol, hr, hor = pack(lefts, rights)
        for buf, host in zip((bl, ol, br, orr), (hl, hol, hr, hor)):
            flat = torch.from_numpy(np.ascontiguousarray(host).reshape(-1)).to(dev)
            buf[:flat.numel()].copy_(flat)
        asg.fill_(SENTINEL)
        graph.replay()
        torch.cuda.synchronize()
        got, st = asg.cpu().numpy(), status.cpu().numpy()
        assert not st.any(), f"replay {rep}"
        assert_frames(got, hol, gpu_api.asgn_bb_batch(lefts, rights, NONASSIGN), f"replay {rep} ({a} / {b})")
        assert (got[hol[-1]:] == SENTINEL).all()


@gpu
def test_one_hundred_thousand_frames_in_one_call(gpu_api):
    lefts, rights = synth.stereo_boxes(100_000, first=3_000_000)
    bl, ol, br, orr = pack(lefts, rights)
    got, st = run_device(gpu_api, bl, ol, br, orr, *maxima(lefts, rights))
    assert not st.any()
    sample = np.sort(np.random.default_rng(12).choice(len(lefts), 2000, replace=False))
    want = gpu_api.asgn_bb_batch([lefts[f] for f in sample], [rights[f] for f in sample], NONASSIGN)
    for i, f in enumerate(sample):
        np.testing.assert_array_equal(got[ol[f]:ol[f + 1]], want[i], err_msg=f"frame {f}")


@gpu
def test_smallest_workspace(gpu_api):
    import torch
    from probabilisticsemslam_b200._lib import PdaError
    lefts, rights = synth.stereo_boxes(300, first=72_000)
    args = pack(lefts, rights)
    need = gpu_api.lib().pda_asgn_bb_workspace_bytes(300, 16, 32)
    assert need > 0
    smallest = run_device(gpu_api, *args, 16, 32, workspace=torch.empty(need, dtype=torch.uint8, device="cuda"))
    full = run_device(gpu_api, *args, 16, 32)
    for a, b in zip(smallest, full):
        np.testing.assert_array_equal(a, b)
    with pytest.raises(PdaError, match="error -4"):
        run_device(gpu_api, *args, 16, 32, workspace=torch.empty(need - 1, dtype=torch.uint8, device="cuda"))


def _devices():
    from probabilisticsemslam_b200 import _lib
    n = _lib.lib().pda_device_count()
    return list(range(n)) if n > 1 else [0, 0, 0]


@gpu
def test_multi_device_form_equals_one_call(gpu_api):
    lefts, rights = synth.stereo_boxes(2000, first=73_000)
    one = gpu_api.asgn_bb_batch(lefts, rights, NONASSIGN)
    for devices in (_devices(), [0, 0, 0]):
        got = gpu_api.asgn_bb_batch(lefts, rights, NONASSIGN, devices=devices)
        for f in range(len(one)):
            np.testing.assert_array_equal(got[f], one[f], err_msg=f"devices {devices}, frame {f}")
    few = gpu_api.asgn_bb_batch(lefts[:2], rights[:2], NONASSIGN, devices=[0] * 5)    # more devices than frames
    for f in range(2):
        np.testing.assert_array_equal(few[f], one[f])


@gpu
def test_host_form_on_a_slice_leaves_the_rest_alone(gpu_api):
    """A _host call whose frames start at offL[0] > 0 -- a shard of a larger batch -- writes only its own range."""
    from probabilisticsemslam_b200._lib import check, lib
    lefts, rights = synth.stereo_boxes(50, first=74_000)
    bl, ol, br, orr = pack(lefts, rights)
    f0 = 20
    asg = np.full(len(bl), SENTINEL, np.int32)
    sub_l, sub_r = np.ascontiguousarray(ol[f0:]), np.ascontiguousarray(orr[f0:])
    assert sub_l[0] > 0 and sub_r[0] > 0
    check(lib().pda_asgn_bb_batch_host(bl.ctypes.data, sub_l.ctypes.data, br.ctypes.data, sub_r.ctypes.data, 50 - f0, NONASSIGN,
                                       asg.ctypes.data, 0))
    assert (asg[:ol[f0]] == SENTINEL).all()
    assert_frames(asg[ol[f0]:], ol[f0:] - ol[f0], gpu_api.asgn_bb_batch(lefts[f0:], rights[f0:], NONASSIGN), "slice")


@gpu
def test_cpp_driver(gpu_api):
    exe = os.path.join(ROOT, "tests", "cpp", "build", "bbox_b200")
    assert os.path.exists(exe), "tests/cpp/build/bbox_b200 missing: run __graft_entry__.build()"
    lefts, rights = synth.stereo_boxes(12, first=75_000)
    for i, (nL, nR) in enumerate([(5, 123), (64, 64), (0, 20), (20, 0), (3, 4), (64, 1)]):
        L, R = box_frame(nL, nR, 900 + i)
        lefts.append(L)
        rights.append(R)
    devices = _devices() + [0]
    parts = [f"{len(lefts)} {NONASSIGN!r} {len(devices)} " + " ".join(map(str, devices))]
    for L, R in zip(lefts, rights):
        parts.append(f"{len(L)} {len(R)} " + " ".join(repr(float(x)) for x in np.concatenate([L.reshape(-1), R.reshape(-1)])))
    run = subprocess.run([exe], input="\n".join(parts) + "\n", capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout[-500:] + run.stderr[-500:]
    batch, graph = {}, {}
    for ln in run.stdout.splitlines():
        w = ln.split()
        if w[0] == "batch":
            batch[int(w[1])] = [int(x) for x in w[2:]]
        else:
            graph[int(w[1])] = (int(w[2]), [int(x) for x in w[3:]])
    want = gpu_api.asgn_bb_batch(lefts, rights, NONASSIGN)
    for f in range(len(lefts)):
        assert batch[f] == want[f].tolist(), f"asgnBBRawBatch frame {f}"
        assert graph[f] == (0, want[f].tolist()), f"graph replay frame {f}"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: no device needed
# ---------------------------------------------------------------------------------------------------------------------
def test_cpp_driver_compiles():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cuda_inc = os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "include")
    assert os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")), f"no CUDA headers at {cuda_inc}"
    src = os.path.join(ROOT, "tests", "cpp", "bbox_driver.cpp")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", cuda_inc, src],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-800:]


def _buf():
    buf = ctypes.create_string_buffer(1 << 16)
    return buf, ctypes.cast(buf, ctypes.c_void_p).value


def _args(p):
    #       bL oL capL bR oR capR n maxNL maxBoxes nonassign asg status ws wsBytes stream
    return [p, p, 8, p, p, 8, 1, 8, 16, 0.2, p, p, p, 1, None]   # a 1-byte workspace: nothing is ever launched


def test_argument_errors():
    from probabilisticsemslam_b200._lib import lib
    L = lib()
    keep, p = _buf()

    def call(**kw):
        a = _args(p)
        for i, v in kw.items():
            a[int(i[1:])] = v
        return L.pda_asgn_bb_batch(*a)

    for i in (0, 1, 3, 4, 10, 11, 12):
        assert call(**{f"a{i}": None}) == -1, i
        assert b"NULL" in L.pda_last_error()
    assert call(a2=-1) == -1 and call(a5=-1) == -1          # negative capacities
    assert call(a6=-1) == -1                                 # nFrames
    assert call(a7=0) == -1 and call(a8=7) == -1             # maxNL < 1, maxBoxes < maxNL
    assert call(a8=129) == -3 and b"above 128" in L.pda_last_error()
    assert call(a0=None, a2=0) in (-2, -4) and call(a3=None, a5=0) in (-2, -4)   # boxes may be NULL at capacity 0
    assert L.pda_asgn_bb_workspace_bytes(-1, 8, 16) == -1
    assert L.pda_asgn_bb_workspace_bytes(1, 0, 16) == -1
    assert L.pda_asgn_bb_workspace_bytes(1, 8, 7) == -1
    assert L.pda_asgn_bb_workspace_bytes(1, 8, 129) == -3


def test_multi_form_argument_errors_without_a_device():
    from probabilisticsemslam_b200._lib import lib
    L = lib()
    if L.pda_device_count() > 0:
        pytest.skip("a device is visible")
    keep, p = _buf()
    dev = (ctypes.c_int32 * 2)(0, 1)
    off = (ctypes.c_int64 * 2)(0, 1)
    assert L.pda_asgn_bb_batch_host_multi(p, off, p, off, 1, 0.2, p, None, 0) == -1
    assert L.pda_asgn_bb_batch_host_multi(p, off, p, off, 1, 0.2, p, dev, 0) == -1
    assert L.pda_asgn_bb_batch_host_multi(p, off, p, off, -1, 0.2, p, dev, 2) == -1
    assert L.pda_asgn_bb_batch_host_multi(p, None, p, off, 1, 0.2, p, dev, 2) == -1
    assert L.pda_asgn_bb_batch_host_multi(p, off, p, off, 1, 0.2, p, dev, 2) == -2
    assert b"no CUDA device" in L.pda_last_error()
    assert L.pda_asgn_bb_workspace_bytes(1, 8, 16) == -2
    assert L.pda_asgn_bb_batch(*_args(p)) == -2
