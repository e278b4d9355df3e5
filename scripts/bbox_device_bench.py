"""The stereo box association (asgnBB): the device-pointer form pda_asgn_bb_batch (frame shapes read on the device)
and the multi-device form pda_asgn_bb_batch_host_multi against the _host form.

  (a) 100 000 synth.stereo_boxes frames in one call: the device form on resident inputs, timed with CUDA events, against
      the _host form, timed with a host clock around the call (its copies and synchronisation included).  The arms
      alternate in one process, medians of 5, and their assignments are compared entry for entry.
  (b) One frame, the per-frame call of the SLAM loop (dataframe.cpp:306): a CUDA graph captured once with fixed bounds
      (16 left boxes, 32 boxes in all), which holds the upload of boxes and offsets from page-locked buffers, the call
      and the download of assignment and status, replayed per frame, against the _host call.  Six stereo_boxes frames;
      host clock, median of 40 after 5 warm-up calls, the two arms alternated twice.
  (c) The batch of (a) through the multi-device form on every GPU present (host clock, median of 5), against (a)'s
      _host result.
Writes profiles/bbox_device_b200.json (or the path given as the first argument) with the GPU's name, power limit and
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
NONASSIGN = 0.2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.splitlines()}


def pack(lefts, rights):
    off = lambda bs: np.concatenate([[0], np.cumsum([len(b) for b in bs])]).astype(np.int64)
    flat = lambda bs: np.ascontiguousarray(np.concatenate([b.reshape(-1, 5) for b in bs] + [np.zeros((0, 5))]))
    return flat(lefts), off(lefts), flat(rights), off(rights)


def host_call(packed, out, devices=None):
    bl, ol, br, orr = packed
    p = lambda a: a.ctypes.data if a.size else None
    n = len(ol) - 1
    if devices is None:
        rc = _lib.lib().pda_asgn_bb_batch_host(p(bl), p(ol), p(br), p(orr), n, NONASSIGN, p(out), 0)
    else:
        d = np.asarray(devices, np.int32)
        rc = _lib.lib().pda_asgn_bb_batch_host_multi(p(bl), p(ol), p(br), p(orr), n, NONASSIGN, p(out), p(d), len(d))
    _lib.check(rc)


def batch_workloads():
    lefts, rights = synth.stereo_boxes(100_000, first=3_000_000)
    packed = pack(lefts, rights)
    bl, ol, br, orr = packed
    max_nL = max(len(L) for L in lefts)
    max_boxes = max(len(L) + len(R) for L, R in zip(lefts, rights))
    t = lambda a: torch.from_numpy(a).cuda()
    d_bl, d_ol, d_br, d_or = t(bl), t(ol), t(br), t(orr)
    asg = torch.full((len(bl),), -1, dtype=torch.int32, device="cuda")
    status = torch.empty(len(lefts), dtype=torch.int32, device="cuda")
    ws = torch.empty(int(_lib.lib().pda_asgn_bb_workspace_bytes(len(lefts), max_nL, max_boxes)), dtype=torch.uint8, device="cuda")
    run = lambda: api.asgn_bb_batch_device(d_bl, d_ol, d_br, d_or, max_nL, max_boxes, NONASSIGN, asg, status, ws)
    h_out = np.full(len(bl), -7, np.int32)
    run(); torch.cuda.synchronize()
    host_call(packed, h_out)
    dev_ms, host_ms = [], []
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(REPS):
        start.record()
        run()
        stop.record()
        stop.synchronize()
        dev_ms.append(start.elapsed_time(stop))
        t0 = time.perf_counter()
        host_call(packed, h_out)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    same = np.array_equal(asg.cpu().numpy(), h_out) and not status.cpu().numpy().any()
    in_mb = (bl.nbytes + br.nbytes + ol.nbytes + orr.nbytes) / 1e6
    rows = [{"workload": "stereo_boxes_100000", "frames": len(lefts), "left_boxes": int(ol[-1]), "right_boxes": int(orr[-1]),
             "max_nL": max_nL, "max_boxes": max_boxes, "input_MB": in_mb, "device_ms": dev_ms, "host_ms": host_ms,
             "device_ms_median": float(np.median(dev_ms)), "host_ms_median": float(np.median(host_ms)),
             "bit_identical": bool(same)}]
    devices = list(range(torch.cuda.device_count()))
    m_out = np.full(len(bl), -7, np.int32)
    host_call(packed, m_out, devices)
    multi_ms = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        host_call(packed, m_out, devices)
        multi_ms.append((time.perf_counter() - t0) * 1e3)
    rows.append({"workload": "stereo_boxes_100000_multi", "devices": devices, "host_ms": multi_ms,
                 "host_ms_median": float(np.median(multi_ms)), "bit_identical": bool(np.array_equal(m_out, h_out))})
    return rows


class FrameGraph:
    """Page-locked boxes and offsets -> device, pda_asgn_bb_batch, assignment and status -> page-locked outputs."""
    MAX_NL, MAX_BOXES = 16, 32

    def __init__(self):
        pin = lambda n, dt: torch.zeros(n, dtype=dt).pin_memory()
        self.h_in = [pin(5 * self.MAX_NL, torch.float64), pin(2, torch.int64), pin(5 * self.MAX_BOXES, torch.float64),
                     pin(2, torch.int64)]
        self.d_in = [torch.zeros_like(h, device="cuda") for h in self.h_in]
        d_asg = torch.full((self.MAX_NL,), -1, dtype=torch.int32, device="cuda")
        d_status = torch.zeros(1, dtype=torch.int32, device="cuda")
        ws = torch.empty(int(_lib.lib().pda_asgn_bb_workspace_bytes(1, self.MAX_NL, self.MAX_BOXES)), dtype=torch.uint8, device="cuda")
        self.h_asg, self.h_status = (torch.zeros_like(t, device="cpu").pin_memory() for t in (d_asg, d_status))
        self.d_out = (d_asg, d_status, ws)  # the graph replays into these: they must outlive it
        bl, ol, br, orr = self.d_in
        call = lambda: api.asgn_bb_batch_device(bl, ol, br, orr, self.MAX_NL, self.MAX_BOXES, NONASSIGN, d_asg, d_status, ws)
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
            for h, d in zip((self.h_asg, self.h_status), (d_asg, d_status)):
                h.copy_(d, non_blocking=True)

    def run(self, packed):
        for h, a in zip(self.h_in, packed):
            flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
            h[:flat.numel()].copy_(flat)
        self.graph.replay()
        torch.cuda.synchronize()
        return self.h_asg.numpy()[:int(packed[1][1])], int(self.h_status[0])


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
    g = FrameGraph()
    lefts, rights = synth.stereo_boxes(6, first=50)
    for i, (L, R) in enumerate(zip(lefts, rights)):
        packed = pack([L], [R])
        h_out = np.full(max(len(L), 1), -7, np.int32)
        host_us, graph_us = [], []
        for _ in range(2):  # alternated
            graph_us.append(median_us(lambda: g.run(packed)))
            host_us.append(median_us(lambda: host_call(packed, h_out)))
        got, st = g.run(packed)
        host_call(packed, h_out)
        same = np.array_equal(got, h_out[:len(L)]) and st == 0
        row = {"workload": f"frame_{i}", "nL": len(L), "nR": len(R), "graph_replay_us": graph_us, "host_call_us": host_us,
               "bit_identical": bool(same)}
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bbox_device_b200.json")
    res = {"card": card(), "reps": REPS, "nonassign": NONASSIGN, "workloads": []}
    for row in batch_workloads():
        print(json.dumps(row), flush=True)
        res["workloads"].append(row)
    res["workloads"] += frame_workloads()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    assert all(w["bit_identical"] for w in res["workloads"]), "an arm differs"


if __name__ == "__main__":
    main()
