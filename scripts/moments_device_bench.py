"""getAssignmentProbs from quadric moments: the device-pointer forms (pda_association_from_moments_batch and
pda_association_perm_from_moments_batch, frame shapes read on the device) against the _host forms.

  (a) 100 000 synth.quadric_frames in one call, k-best (k = 200) and usePerm: the device form on resident inputs, timed
      with CUDA events, against the _host form, timed with a host clock around the call (its copies and synchronisation
      included).  The arms alternate in one process, and their tables, statuses and probOff are compared bit for bit.
  (b) One frame, the per-frame call of the SLAM loop: a CUDA graph captured once with fixed bounds (40 landmarks, 8
      detections), which holds the upload of the moments and offsets from page-locked buffers, the call and the download
      of table, probOff and status, replayed per frame, against the _host call.  The six frames of
      scripts/frame_latency.py; host clock, median of 40 after 5 warm-up calls.
Writes profiles/moments_device_b200.json (or the path given as the first argument) with the GPU's name, power limit and
max SM clock, read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from probabilisticsemslam_b200 import _lib, api, synth  # noqa: E402

REPS = 5
K = 200
NONASSIGN = 10.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60).stdout.strip()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def host_call(packed, perm, probs, status):
    p = lambda a: a.ctypes.data
    lm, lc, lo, mm, mc, mo = packed
    n = len(lo) - 1
    if perm:
        rc = _lib.lib().pda_association_perm_from_moments_batch_host(p(lm), p(lc), p(lo), p(mm), p(mc), p(mo), n, NONASSIGN,
                                                                    p(probs), p(status), 0)
    else:
        rc = _lib.lib().pda_association_from_moments_batch_host(p(lm), p(lc), p(lo), p(mm), p(mc), p(mo), n, NONASSIGN, K,
                                                               p(probs), 0)
    _lib.check(rc)


def batch_workload(perm):
    frames = synth.quadric_frames(100_000, first=3_000_000)
    packed = api._pack_moments(frames)
    max_nL = max(f[0].shape[0] for f in frames)
    max_nM = max(f[2].shape[0] for f in frames)
    spans = np.array([f[2].shape[0] * (f[0].shape[0] + 1) for f in frames], np.int64)
    cap = int(spans.sum())
    args = api.moments_to_device(frames)
    probs = torch.zeros(cap, dtype=torch.float64, device="cuda")
    prob_off = torch.empty(len(frames) + 1, dtype=torch.int64, device="cuda")
    status = torch.empty(len(frames), dtype=torch.int32, device="cuda")
    if perm:
        run = lambda ws: api.association_perm_from_moments_batch_device(*args, max_nL, max_nM, NONASSIGN, cap, probs, prob_off,
                                                                        status, ws)
    else:
        n_found = torch.empty(len(frames), dtype=torch.int32, device="cuda")
        run = lambda ws: api.association_from_moments_batch_device(*args, max_nL, max_nM, NONASSIGN, K, cap, probs, prob_off,
                                                                   status, n_found, ws)
    name = "pda_association_perm_from_moments" if perm else "pda_association_from_moments"
    extra = () if perm else (K,)
    ws = torch.empty(int(getattr(_lib.lib(), name + "_workspace_bytes")(len(frames), max_nL, max_nM, cap, *extra)),
                     dtype=torch.uint8, device="cuda")
    h_probs, h_status = np.zeros(cap), np.zeros(len(frames), np.int32)
    run(ws); torch.cuda.synchronize()
    host_call(packed, perm, h_probs, h_status)
    dev_ms, host_ms = [], []
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(REPS):
        start.record()
        run(ws)
        stop.record()
        stop.synchronize()
        dev_ms.append(start.elapsed_time(stop))
        t0 = time.perf_counter()
        host_call(packed, perm, h_probs, h_status)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    same = (np.array_equal(probs.cpu().numpy().view(np.int64), h_probs.view(np.int64)) and
            np.array_equal(prob_off.cpu().numpy(), np.concatenate([[0], np.cumsum(spans)])) and
            (np.array_equal(status.cpu().numpy(), h_status) if perm else not status.cpu().numpy().any()))
    return {"workload": f"quadric_frames_100000_{'useperm' if perm else 'k200'}", "frames": len(frames), "max_nL": max_nL,
            "max_nM": max_nM, "device_ms": dev_ms, "host_ms": host_ms, "device_ms_median": float(np.median(dev_ms)),
            "host_ms_median": float(np.median(host_ms)), "bit_identical": bool(same)}


class FrameGraph:
    """One graph per weighting: page-locked inputs -> device, the call, table / probOff / status -> page-locked outputs."""
    MAX_NL, MAX_NM = 40, 8

    def __init__(self, perm):
        L, M = self.MAX_NL, self.MAX_NM
        pin = lambda n, dt: torch.zeros(n, dtype=dt).pin_memory()
        self.h_in = [pin(3 * L, torch.float64), pin(9 * L, torch.float64), pin(2, torch.int64), pin(3 * M, torch.float64),
                     pin(9 * M, torch.float64), pin(2, torch.int64)]
        self.d_in = [torch.zeros_like(t, device="cuda") for t in self.h_in]
        cap = M * (L + 1)
        self.perm = perm
        d_probs = torch.zeros(cap, dtype=torch.float64, device="cuda")
        d_off = torch.zeros(2, dtype=torch.int64, device="cuda")
        d_status = torch.zeros(1, dtype=torch.int32, device="cuda")
        name = "pda_association_perm_from_moments" if perm else "pda_association_from_moments"
        extra = () if perm else (K,)
        ws = torch.empty(int(getattr(_lib.lib(), name + "_workspace_bytes")(1, L, M, cap, *extra)), dtype=torch.uint8,
                         device="cuda")
        d_nf = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.h_probs, self.h_off, self.h_status = (torch.zeros_like(t, device="cpu").pin_memory() for t in (d_probs, d_off, d_status))
        self.d_out = (d_probs, d_off, d_status, d_nf, ws)  # the graph replays into these: they must outlive it

        def call():
            if perm:
                api.association_perm_from_moments_batch_device(*self.d_in, L, M, NONASSIGN, cap, d_probs, d_off, d_status, ws)
            else:
                api.association_from_moments_batch_device(*self.d_in, L, M, NONASSIGN, K, cap, d_probs, d_off, d_status, d_nf, ws)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            call()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            for d, h in zip(self.d_in, self.h_in):
                d.copy_(h, non_blocking=True)
            call()
            for h, d in zip((self.h_probs, self.h_off, self.h_status), (d_probs, d_off, d_status)):
                h.copy_(d, non_blocking=True)

    def run(self, packed):
        lm, lc, lo, mm, mc, mo = packed
        for h, a in zip(self.h_in, (lm, lc, lo, mm, mc, mo)):
            flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
            h[:flat.numel()].copy_(flat)
        self.graph.replay()
        torch.cuda.synchronize()
        return self.h_probs.numpy()[:int(self.h_off[1])], int(self.h_status[0])


def median_us(f, reps=40, warm=5):
    for _ in range(warm):
        f()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        t.append(time.perf_counter() - t0)
    return 1e6 * float(np.median(t))


def frame_workloads():
    rows = []
    graphs = {False: FrameGraph(False), True: FrameGraph(True)}
    for i, f in enumerate(synth.quadric_frames(8, first=50)[:6]):  # the frames of scripts/frame_latency.py
        packed = api._pack_moments([f])
        nL, nM = f[0].shape[0], f[2].shape[0]
        for perm, g in graphs.items():
            h_probs, h_status = np.zeros(nM * (nL + 1)), np.zeros(1, np.int32)
            host_us, graph_us = [], []
            for _ in range(2):  # alternated
                graph_us.append(median_us(lambda: g.run(packed)))
                host_us.append(median_us(lambda: host_call(packed, perm, h_probs, h_status)))
            got, st = g.run(packed)
            host_call(packed, perm, h_probs, h_status)
            same = np.array_equal(got.view(np.int64), h_probs.view(np.int64)) and st == int(h_status[0])
            row = {"workload": f"frame_{i}_{'useperm' if perm else 'k200'}", "nL": nL, "nM": nM, "graph_replay_us": graph_us,
                   "host_call_us": host_us, "bit_identical": bool(same)}
            print(json.dumps(row), flush=True)
            rows.append(row)
    return rows


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "moments_device_b200.json")
    res = {"card": card(), "reps": REPS, "k": K, "workloads": []}
    for perm in (False, True):
        row = batch_workload(perm)
        print(json.dumps(row), flush=True)
        res["workloads"].append(row)
    res["workloads"] += frame_workloads()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
