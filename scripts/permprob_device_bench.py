"""permanentProb: the device-pointer form (pda_permanent_prob_batch, inputs resident on the GPU, CUDA events) against the
host form (pda_permanent_prob_batch_host, host clock around the call, which includes its copies and synchronisations).

Workloads, arms alternated in one process on the same seeded inputs:
  * 10 000 conditioned G2 problems, permOpt 1 and permOpt 0: the per-frame permanentProb calls of compMethods, batched;
  * one compMethods-shaped frame (conditioned G2, one problem), permOpt 1: the latency of a single call;
  * 64 problems with 12-14 detections: every sub-permanent goes to the NW walk.
Tables and statuses of the two arms are compared bit for bit in the same run.  Under permOpt 0 they are identical only
within one host chunk (65 536 sub-permanents): the draws are keyed by the item index, which the host form counts per
chunk, so the 10 000-problem batch (six chunks) differs by design.  Writes profiles/permprob_device_b200.json
(or the path given as the first argument) with the GPU's name, power limit and max SM clock."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from probabilisticsemslam_b200 import _lib, api, device, synth  # noqa: E402

REPS = 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60).stdout.strip()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def workloads():
    g2, _ = api.condition_costs_batch(synth.g2_gated(10_000, first=20_000))
    frame = g2.take(np.array([0]))
    nw = synth.pack([synth.g1_dense(1, nL=6, nM=12 + p % 3, first=500 + p).matrix(0) for p in range(64)],
                    [6] * 64)
    return [("g2_10000_permopt1", g2, 1, 1), ("g2_10000_permopt0", g2, 0, 1), ("single_frame_permopt1", frame, 1, 20),
            ("nm12_14_x64_permopt1", nw, 1, 1)]


def time_device(plan, inner):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(inner):
        plan.run()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / inner


def time_host(pb, perm_opt, inner):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(inner):
        out = api.permanent_prob_batch(pb, perm_opt)
    return (time.perf_counter() - t0) * 1e3 / inner, out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "permprob_device_b200.json")
    _lib.lib().pda_set_approx_seed(20260217)
    res = {"card": card(), "reps": REPS, "workloads": []}
    for name, pb, perm_opt, inner in workloads():
        plan = device.PermanentProbPlan(pb, perm_opt)
        plan.run(); torch.cuda.synchronize()                     # warm-up of both arms
        _, want = time_host(pb, perm_opt, 1)
        dev_ms, host_ms = [], []
        for _ in range(REPS):                                     # alternated
            dev_ms.append(time_device(plan, inner))
            host_ms.append(time_host(pb, perm_opt, inner)[0])
        got = plan.result()
        same = bool(np.array_equal(got[1], want[1]) and all(
            np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64)) for a, b in zip(got[0], want[0])))
        items = int((pb.nM.astype(np.int64) * (pb.nL + 1)).sum())
        row = {"workload": name, "problems": len(pb), "sub_permanents": items, "perm_opt": perm_opt,
               "device_ms": dev_ms, "host_ms": host_ms, "device_ms_median": float(np.median(dev_ms)),
               "host_ms_median": float(np.median(host_ms)), "bit_identical": same}
        print(json.dumps(row), flush=True)
        res["workloads"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
