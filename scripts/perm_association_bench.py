"""getAssignmentProbs with usePerm: the fused device pipeline (pda_association_perm_probs_batch[_host]) against the route
it replaces (conditionCosts -> permanentProb(.., 1) -> scatter through rowIdx, three separate calls), on one GPU.

Per workload (100 000 synth.g2_gated problems; 100 000 synth.quadric_frames turned into cost matrices on the device):
  fused_host      pda_association_perm_probs_batch_host on host arrays (copy in, run, copy out)
  composed        condition_costs_batch -> permanent_prob_batch -> numpy scatter (what getAssignmentProbsFromCosts ran)
  device          pda_association_perm_probs_batch on resident device inputs, CUDA events, after a warm-up
The fused and composed arms run alternately in one process; their tables are compared bit for bit on the timed inputs.
Also: the moments host form on the quadric frames, single-frame latency (median of 40 calls after warm-up) on the six
frames of scripts/frame_latency.py, and the CPU oracle (usePerm) on a sample over all host threads.

    python scripts/perm_association_bench.py --out profiles/perm_association_b200.json
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from probabilisticsemslam_b200 import _lib, api, synth  # noqa: E402
from perm_route import composed as _composed  # noqa: E402  the route the tests compare against, too


def composed(pb):
    """conditionCosts -> permanentProb(.., 1) -> scatter, as three separate library calls and numpy."""
    return _composed(api, pb)


def card():
    """Name and power limit of GPU 0, read in the same run as the numbers."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    import torch
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def flat(tabs):
    return np.concatenate([t.reshape(-1) for t in tabs])


def wall(f):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = f()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def device_arm(pb, reps):
    """pda_association_perm_probs_batch on resident inputs, timed with CUDA events."""
    import torch
    lib = _lib.lib()
    dev = torch.device("cuda:0")
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
    _lib.check(int(ws_bytes) if ws_bytes < 0 else 0)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    probs = torch.zeros(total_p, dtype=torch.float64, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()

    def call():
        _lib.check(lib.pda_association_perm_probs_batch(
            costs.data_ptr(), cost_off.data_ptr(), d_nL.data_ptr(), d_nM.data_ptr(), d_row.data_ptr(), n, pb.costs.size,
            int(nr.sum()), total_p, int(nr.max()), int(nM.max()), probs.data_ptr(), d_poff.data_ptr(), status.data_ptr(),
            ws.data_ptr(), ws_bytes, ctypes.c_void_p(stream.cuda_stream)))

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms, probs.cpu().numpy(), status.cpu().numpy(), ws_bytes


def run_workload(name, pb, reps, extra=None):
    n = len(pb)
    rec = {"problems": n, "mean_nM": float(pb.nM.mean()), "mean_nL": float(pb.nL.mean()), "fused_host_s": [], "composed_s": []}
    api.association_perm_probs_batch(pb.slice(0, min(n, 1000)))     # warm-up of every shape the timed window uses
    composed(pb.slice(0, min(n, 1000)))
    same = True
    for _ in range(reps):                                             # alternate new and old in one process
        dt, new = wall(lambda: api.association_perm_probs_batch(pb))
        rec["fused_host_s"].append(dt)
        dt, old = wall(lambda: composed(pb))
        rec["composed_s"].append(dt)
        same = same and np.array_equal(new[1], old[1])
        same = same and all(np.array_equal(a.view(np.int64), b.view(np.int64)) for a, b in zip(new[0], old[0]))
    ms, probs, st, ws_bytes = device_arm(pb, reps * 3)
    rec["device_ms"] = ms
    rec["device_workspace_bytes"] = int(ws_bytes)
    same_dev = bool(np.array_equal(st, new[1]) and np.array_equal(probs.view(np.int64), flat(new[0]).view(np.int64)))
    rec["bit_identical_fused_vs_composed"] = bool(same)
    rec["bit_identical_device_vs_host"] = same_dev
    rec["status_nonzero"] = int(np.count_nonzero(new[1]))
    med = lambda v: float(np.median(v))
    rec["fused_host_frames_per_s"] = n / med(rec["fused_host_s"])
    rec["composed_frames_per_s"] = n / med(rec["composed_s"])
    rec["device_frames_per_s"] = n / (med(ms) / 1e3)
    if extra:
        rec.update(extra())
    print(name, json.dumps({k: v for k, v in rec.items() if not isinstance(v, list)}), flush=True)
    return rec


def median_us(f, reps=40, warm=5):
    for _ in range(warm):
        f()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        t.append(time.perf_counter() - t0)
    return 1e6 * float(np.median(t))


def latency():
    out = []
    for i, f in enumerate(synth.quadric_frames(8, first=50)[:6]):       # the frames of scripts/frame_latency.py
        C = api.computeQuadricCostMatrix(*f, 10.0)
        nL = f[0].shape[0]
        pb = synth.pack([C], [nL])
        rec = {"frame": i, "nL": nL, "nM": int(C.shape[1])}
        rec["fused_from_costs_us"] = median_us(lambda: api.association_perm_probs_batch(pb))
        rec["fused_from_moments_us"] = median_us(lambda: api.association_perm_from_moments_batch([f], 10.0))
        rec["composed_from_costs_us"] = median_us(lambda: composed(pb))
        a, b = api.association_perm_probs_batch(pb), composed(pb)
        rec["bit_identical"] = bool(np.array_equal(a[1], b[1]) and np.array_equal(a[0][0].view(np.int64), b[0][0].view(np.int64)))
        out.append(rec)
        print("latency", json.dumps(rec), flush=True)
    return out


def cpu_arm(pb, n_sample):
    from oracle.loader import load_oracle
    o = load_oracle()
    idx = range(min(n_sample, len(pb)))
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(lambda p: o.association_probs(pb.matrix(p), int(pb.nL[p]), 200, use_perm=True), idx))
    dt = time.perf_counter() - t0
    rec = {"problems": len(res), "threads": threads, "seconds": dt, "frames_per_s": len(res) / dt,
           "status_nonzero": sum(1 for s, _ in res if s)}
    print("cpu", json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--problems", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=2000)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("perm_association_bench: no CUDA device (nothing here is measured on the CPU)")
    res = {"card": card(), "problems": a.problems, "reps": a.reps, "workloads": {}}
    g2 = synth.g2_gated(a.problems, first=2_000_000)
    res["workloads"]["g2_gated"] = run_workload("g2_gated", g2, a.reps)
    frames = synth.quadric_frames(a.problems, first=3_000_000)
    qc = synth.pack(api.quadric_cost_batch(frames, 10.0), [f[0].shape[0] for f in frames])

    def moments():
        api.association_perm_from_moments_batch(frames[:1000], 10.0)
        t = [wall(lambda: api.association_perm_from_moments_batch(frames, 10.0))[0] for _ in range(a.reps)]
        return {"fused_from_moments_host_s": t, "fused_from_moments_frames_per_s": len(frames) / float(np.median(t))}

    res["workloads"]["quadric_frames"] = run_workload("quadric_frames", qc, a.reps, moments)
    res["latency"] = latency()
    res["cpu_oracle_g2_gated"] = cpu_arm(g2, a.cpu_sample)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
