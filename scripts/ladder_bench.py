"""assignmentProb for several k: one ladder call (pda_assignment_prob_ladder_batch) against one assignmentProb call per k.

compMethods (comparison.cpp:194-222) asks for k = 1, 20, 100, 200 and more on every frame; BASELINE config 4 studies
weights as a function of k.  Arms alternate in one process, on the same seeded inputs:
  * 100 000 G1 problems and 100 000 conditioned G2 problems, ks = {1, 20, 100, 200} and {1, 20, 100, 200, 1000}:
    device-resident (device-pointer entries, CUDA events, inputs already on the GPU) and host form (host clock).
  * the six frames of scripts/frame_latency.py, conditioned, through the host call on the CTA path (median of 40).
Outputs of the two arms are compared bit for bit in the same run.  Writes profiles/assignment_ladder_b200.json
(or the path given as the first argument) with the GPU's name, power limit and max SM clock."""
import ctypes
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

L = _lib.lib()
N = 100_000
REPS = 3
KSETS = ([1, 20, 100, 200], [1, 20, 100, 200, 1000])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60).stdout.strip()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


class DeviceBatch:
    """A batch resident on the GPU with buffers for both arms."""

    def __init__(self, pb, ks):
        dev = torch.device("cuda:0")
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.n, self.ks = len(pb), np.ascontiguousarray(ks, np.int32)
        nL = pb.nL.astype(np.int32)
        cells = pb.nM.astype(np.int64) * (nL.astype(np.int64) + 1)
        off1 = np.zeros(self.n, np.int64)
        off1[1:] = np.cumsum(cells)[:-1]
        self.costs, self.cost_off, self.nr = t(pb.costs), t(pb.cost_off), t(pb.num_row)
        self.nc, self.nl = t(pb.nM.astype(np.int32)), t(nL)
        self.off_ladder, self.off_one = t(off1 * len(ks)), t(off1)
        self.maxr, self.maxc = int(pb.num_row.max()), int(pb.nM.max())
        self.p_ladder = torch.zeros(int(cells.sum()) * len(ks), dtype=torch.float64, device=dev)
        self.p_one = [torch.zeros(int(cells.sum()), dtype=torch.float64, device=dev) for _ in ks]
        self.f_ladder = torch.zeros(self.n * len(ks), dtype=torch.int32, device=dev)
        self.f_one = [torch.zeros(self.n, dtype=torch.int32, device=dev) for _ in ks]
        ws = max(L.pda_murty_workspace_bytes(self.n, int(k), self.maxr, self.maxc) for k in ks)
        self.ws = torch.empty(int(ws), dtype=torch.uint8, device=dev)
        self.cells, self.off1 = cells, off1

    def ladder(self, stream):
        p = lambda x: ctypes.c_void_p(x.data_ptr())
        _lib.check(L.pda_assignment_prob_ladder_batch(p(self.costs), p(self.cost_off), p(self.nr), p(self.nc), p(self.nl),
                                                      self.n, self.maxr, self.maxc, self.ks.ctypes.data, len(self.ks),
                                                      p(self.p_ladder), p(self.off_ladder), p(self.f_ladder), p(self.ws),
                                                      self.ws.numel(), ctypes.c_void_p(stream)))

    def separate(self, stream):
        p = lambda x: ctypes.c_void_p(x.data_ptr())
        for j, k in enumerate(self.ks):
            _lib.check(L.pda_murty_batch(p(self.costs), p(self.cost_off), p(self.nr), p(self.nc), self.n, self.maxr, self.maxc,
                                         int(k), api.CUT_RELATIVE, api.GATE, 0, 0, None, None, None, None, None,
                                         p(self.f_one[j]), api.WEIGHTS_GATED, p(self.p_one[j]), p(self.off_one), p(self.nl),
                                         p(self.ws), self.ws.numel(), ctypes.c_void_p(stream)))

    def same_bits(self):
        nk = len(self.ks)
        lad = self.p_ladder.cpu().numpy()
        fl = self.f_ladder.cpu().numpy().reshape(self.n, nk)
        idx = (self.off1 * nk)[:, None] + np.arange(nk)[None, :] * self.cells[:, None]
        ok = True
        for j in range(nk):
            one = self.p_one[j].cpu().numpy()
            mine = np.concatenate([lad[idx[p, j]:idx[p, j] + self.cells[p]] for p in range(self.n)])
            ok &= bool(np.array_equal(mine.view(np.int64), one.view(np.int64)))
            ok &= bool(np.array_equal(fl[:, j], self.f_one[j].cpu().numpy()))
        return ok


def device_times(pb, ks):
    b = DeviceBatch(pb, ks)
    stream = torch.cuda.current_stream().cuda_stream
    b.ladder(stream), b.separate(stream)
    torch.cuda.synchronize()
    t = {"ladder": [], "separate": []}
    for _ in range(REPS):
        for arm in ("ladder", "separate"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            getattr(b, arm)(stream)
            e1.record()
            torch.cuda.synchronize()
            t[arm].append(e0.elapsed_time(e1))
    return {"ladder_ms": t["ladder"], "separate_ms": t["separate"], "identical": b.same_bits()}


def host_times(pb, ks):
    t = {"ladder": [], "separate": []}
    lad = sep = None
    for _ in range(REPS):
        t0 = time.perf_counter()
        lad = api.assignment_prob_ladder_batch(pb, ks)
        t["ladder"].append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        sep = [api.assignment_prob_batch(pb, k) for k in ks]
        t["separate"].append(1e3 * (time.perf_counter() - t0))
    same = all(np.array_equal(lad[1][:, j], sep[j].n_found) for j in range(len(ks)))
    for j in range(len(ks)):
        one = np.concatenate([sep[j].prob_table(pb, p).reshape(-1) for p in range(len(pb))])
        mine = np.concatenate([lad[0][p][j].reshape(-1) for p in range(len(pb))])
        same &= bool(np.array_equal(mine.view(np.int64), one.view(np.int64)))
    return {"ladder_ms": t["ladder"], "separate_ms": t["separate"], "identical": same}


def frames():
    """The six frames of scripts/frame_latency.py, conditioned, one host call each, on the CTA path."""
    prev = api.set_murty_path("cta")
    out = []
    ks = [1, 20, 1000, 100, 200, 150]   # compMethods' per-frame sequence with k = 150
    for i, f in enumerate(synth.quadric_frames(8, first=50)[:6]):
        C = api.quadric_cost_batch([f], 10.0)[0]
        pb, _ = api.condition_costs_batch(synth.pack([C], [C.shape[0] - C.shape[1]]))

        def med(fn, reps=40, warm=5):
            for _ in range(warm):
                fn()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                ts.append(time.perf_counter() - t0)
            return 1e6 * float(np.median(ts))
        lad_us = med(lambda: api.assignment_prob_ladder_batch(pb, ks))
        sep_us = med(lambda: [api.assignment_prob_batch(pb, k) for k in ks])
        tabs, nf = api.assignment_prob_ladder_batch(pb, ks)
        same = all(np.array_equal(tabs[0][j], api.assignment_prob_batch(pb, k).prob_table(pb, 0), equal_nan=True)
                   for j, k in enumerate(ks))
        out.append({"frame": i, "nM": int(pb.nM[0]), "cond_rows": int(pb.num_row[0]), "nFound": nf[0].tolist(),
                    "ladder_us": lad_us, "separate_us": sep_us, "identical": same})
    api.set_murty_path(prev)
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "assignment_ladder_b200.json")
    res = {"gpu": card(), "n_problems": N, "reps": REPS, "batches": []}
    g1 = synth.g1_dense(N, first=0)
    g2, _ = api.condition_costs_batch(synth.g2_gated(N, first=0))
    for name, pb in (("G1", g1), ("G2 conditioned", g2)):
        for ks in KSETS:
            r = {"batch": name, "ks": ks, "device": device_times(pb, ks), "host": host_times(pb, ks)}
            print(json.dumps(r), flush=True)
            res["batches"].append(r)
    res["frames_cta_host"] = frames()
    print(json.dumps(res["frames_cta_host"]), flush=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
