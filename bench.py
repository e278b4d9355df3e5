#!/usr/bin/env python
"""bench.py -- headline benchmark of the probabilistic data-association hot path.

Metric (BASELINE.json): k=200 Murty problems/sec at 1/2/4/8 B200; permanent n=24 latency vs host CPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path -- cost matrix in, k-best lists + gains + nM x (nL+1)
association weights out (SURVEY.md 8d) -- over one batch of 100 000 KITTI-shaped synthetic problems
per GPU (BASELINE.json configs[1]; generator G1 of probabilisticsemslam_b200/synth.py).
Problems are independent, so N GPUs each take their own 100 000 (weak scaling, no data-path
collective; one max-reduction of the elapsed time).

  value   problems/s, batch resident in HBM, CUDA events around K steps, max over ranks
  e2e     the same metric through the reference-facing call -- batched assignmentProb
          (pda_murty_batch_host): HOST cost matrices in, HOST weights out, copies inside the timed region
  roofline  HBM: algorithmic bytes of a pass / measured kernel time, against MEASURED_PEAKS.json
  cpu_baseline  the reference's own CPU code (oracle/_ref, built from the reference's sources) or, failing that,
          the oracle port, on this box's host cores over a bounded sample of the same workload
  extra.permanent_n24  latency of one dense 24x24 permanent, GPU vs the same CPU arm

--impl reference times the reference's CPU implementation only (no GPU code on that path).

--dump-outputs DIR writes what the last timed step returned (rank 0's batch) as DIR/<name>.npy, so that two builds
can be compared output for output on identical seeded inputs: see dump_outputs().
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from probabilisticsemslam_b200 import synth  # noqa: E402

METRIC = "murty_k200_problems_per_sec"
UNIT = "problems/s"
N_PER_GPU = 100_000
K_BEST = 200
WORKLOAD = "configs[1]: 100k KITTI-shaped problems (3-8 detections x 30 landmarks + missed-detection slack), k=200, G1 seed 20260217"


def measured_traffic(n, k):
    """DRAM bytes of one launch of the headline kernel from the committed ncu capture (profiles/traffic.json).  The
    capture was taken over fewer problems than a bench launch (ncu replays the kernel ~40 times); problems are
    independent and alike, so the per-problem figure is scaled to this launch's problem count.  None at another k."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)["murty_kernel<2, true>"]
        return int(t["bytes_per_problem"] * n) if t["k"] == k else None
    except (OSError, KeyError, ValueError):
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except OSError:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val == "Active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_checker():
    """The CPU arm: the reference's own code when oracle/_ref was built, else the oracle port."""
    from oracle.loader import load_oracle, load_reference, reference_available
    if reference_available("fast") or reference_available("native"):
        chk = load_reference("timing")
        return chk, "reference", f"oracle/_ref ({chk.kind}: g++ {chk.flags})"
    return load_oracle(), "port", "oracle/liboracle.so (gcc -O2, IEEE-strict)"


def cpu_problems_per_sec(chk, n_problems: int, threads: int, first: int = 0):
    pb = synth.g1_dense(n_problems, first=first)
    out = chk.batch(pb, K_BEST, threads=threads, want_probs=True, want_lists=True)
    return n_problems / out["seconds"], out["seconds"]


def cpu_permanent_ms(chk, threads: int = 1):
    A = synth.dense_square(1, 24, first=4242)
    sec, _ = chk.permanent_batch(A, 24, threads=1)
    return sec * 1e3


DUMP_PROBLEMS = 1024
DUMP_BYTES = 64 << 20
DUMP_SEED = 20260217


def dump_outputs(plan, pb, out_dir):
    """Writes the k-best pass's results for a fixed, seeded sample of problems (at most DUMP_PROBLEMS, at most DUMP_BYTES
    in all), concatenated in sample order:
      problems  the sampled problem indices                        n_found  nFound per problem
      gain      [problems, k], NaN beyond nFound                   probs    the nM x (nL+1) weight table per problem
      row4col   the k x nM list per problem, col4row  the k x (nL+nM) list per problem; -1 beyond nFound
    Index lists are stored as float32 (exact for these small integers), everything else as float64.  Only the first
    nFound hypotheses of a problem are defined, so the rest is masked to make runs comparable bit for bit."""
    import torch
    k = plan.k
    nc = pb.nM.astype(np.int64)
    nr = pb.num_row.astype(np.int64)
    w = nc * (pb.nL.astype(np.int64) + 1)
    order = np.random.default_rng(DUMP_SEED).permutation(len(pb))[:DUMP_PROBLEMS]
    cost = np.cumsum(16 + 8 * k + 4 * k * (nc[order] + nr[order]) + 8 * w[order])
    idx = np.sort(order[:int(np.searchsorted(cost, DUMP_BYTES, side="right"))])
    nf = plan.n_found.cpu().numpy()[idx].astype(np.int64)

    def gather(t, off, size):
        """The segments [off[p], off[p] + size[p]) of device tensor t for the sampled p, and each element's position
        inside its segment."""
        start, size = off[idx], size[idx]
        within = np.arange(int(size.sum())) - np.repeat(np.cumsum(size) - size, size)
        pos = torch.from_numpy(np.repeat(start, size) + within).to(t.device)
        return t[pos].cpu().numpy(), within, size

    def lists(t, off, width):
        v, within, size = gather(t, off, width * k)
        hyp = within // np.repeat(width[idx], size)
        return np.where(hyp < np.repeat(nf, size), v, -1).astype(np.float32)

    gain = plan.gain.view(plan.n, k)[torch.from_numpy(idx).to(plan.gain.device)].cpu().numpy()
    gain[np.arange(k)[None, :] >= nf[:, None]] = np.nan
    out = {"problems": idx.astype(np.float64), "n_found": nf.astype(np.float64), "gain": gain,
           "row4col": lists(plan.row4col, plan.r4c_off_h, nc), "col4row": lists(plan.col4row, plan.c4r_off_h, nr),
           "probs": gather(plan.probs, plan.prob_off_h, w)[0]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    chk, kind, what = cpu_checker()
    cores = os.cpu_count() or 1
    sample = max(cores * 250, 1000)
    for _ in range(args.warmup):
        cpu_problems_per_sec(chk, max(cores * 20, 100), cores)
    t = []
    for s in range(args.steps):
        _, sec = cpu_problems_per_sec(chk, sample, cores, first=s * sample)
        t.append(sec)
    total = sum(t)
    value = sample * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "k": K_BEST, "sample_per_step": sample, "host_threads": cores, "code": what},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{sample} problems per step x {args.steps} steps of the same generator, {cores} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extra": {"permanent_n24": {"cpu_ms": cpu_permanent_ms(chk), "unit": "ms", "threads": 1}},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--problems", type=int, default=N_PER_GPU, help="problems per GPU (default: the BASELINE configuration)")
    ap.add_argument("--k", type=int, default=K_BEST)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--skip-config3", action="store_true", help="skip extra.config3_k1000_strong (profiling runs)")
    ap.add_argument("--skip-config4", action="store_true", help="skip extra.permanent_batch_sharded (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from probabilisticsemslam_b200 import _lib, device as dev

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        # a bounded collective timeout: a stuck exchange ends the run with an error after five minutes instead of hanging it
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=300))
    lib = _lib.lib()
    n, k = args.problems, args.k

    pb = synth.g1_dense(n, first=rank * n)          # rank r owns problems [r*n, (r+1)*n): no data-path collective
    plan = dev.MurtyPlan(pb, k=k, weights=True, pinned_inputs=True)
    for _ in range(max(args.warmup, 3)):
        plan.run()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----------------------------------------------------------------
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    with ClockSampler(local) as clk:
        ev[0].record()
        for s in range(args.steps):
            plan.run()
            ev[s + 1].record()
        torch.cuda.synchronize()
    barrier()
    step_ms = [ev[s].elapsed_time(ev[s + 1]) for s in range(args.steps)]
    total_ms = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * n * args.steps / (total_ms_max * 1e-3)
    alg_bytes = plan.algorithmic_bytes()
    kernel_ms = statistics.mean(step_ms)
    fallback_problems = int(plan.workspace[8:12].view(torch.int32).item())  # problems the pruning kernel handed to the exact one
    if args.dump_outputs and rank == 0:
        dump_outputs(plan, pb, args.dump_outputs)

    # ---- end to end: host buffers through the C ABI (batched assignmentProb) ----------------------------
    nL32, nM32 = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    nR32 = (nL32 + nM32).astype(np.int32)
    prob_off = plan.prob_off_h
    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_costs, h_off, h_nr, h_nc, h_nl, h_poff = pin(pb.costs), pin(pb.cost_off), pin(nR32), pin(nM32), pin(nL32), pin(prob_off)
    h_probs = torch.empty(plan.n_prob, dtype=torch.float64).pin_memory()
    h_found = torch.empty(n, dtype=torch.int32).pin_memory()
    def e2e_step():
        _lib.check(lib.pda_murty_batch_host(h_costs.data_ptr(), h_off.data_ptr(), h_nr.data_ptr(), h_nc.data_ptr(), n, k,
                                            1, 42.0, 0, 0, None, None, None, None, None, h_found.data_ptr(),
                                            1, h_probs.data_ptr(), h_poff.data_ptr(), h_nl.data_ptr(), local))
    del plan.row4col, plan.col4row   # free the resident k-best lists before the host path stages its own buffers
    plan.row4col = plan.col4row = None
    torch.cuda.empty_cache()
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.steps / float(t.item())
    h2d = int(h_costs.numel() * 8 + h_off.numel() * 8 + h_nr.numel() * 4 + h_nc.numel() * 4 + h_nl.numel() * 4 + h_poff.numel() * 8)
    d2h = int(h_probs.numel() * 8 + h_found.numel() * 4)
    probs_dev = plan.probs.cpu().numpy()
    e2e_matches = bool(np.array_equal(probs_dev, h_probs.numpy()))

    # ---- e2e variants (rank 0 of a single-GPU run): the same host call with PAGEABLE buffers (copied through the
    #      staging arena), and kBest2DCutoff semantics -- every k-best list and gain returned to the host -- on 20 000
    #      problems with page-locked buffers (1.3 GB of lists per pass cross the bus device -> host)
    e2e_variants = None
    if world == 1:
        pg_costs, pg_probs, pg_found = pb.costs.copy(), np.zeros(plan.n_prob), np.zeros(n, np.int32)
        def pageable_step():
            _lib.check(lib.pda_murty_batch_host(pg_costs.ctypes.data, pb.cost_off.ctypes.data, nR32.ctypes.data, nM32.ctypes.data, n, k,
                                                1, 42.0, 0, 0, None, None, None, None, None, pg_found.ctypes.data,
                                                1, pg_probs.ctypes.data, prob_off.ctypes.data, nL32.ctypes.data, local))
        pageable_step()
        t0 = time.perf_counter()
        for _ in range(2):
            pageable_step()
        pageable_pps = 2 * n / (time.perf_counter() - t0)
        nl_ = min(n, 20000)
        r4o, c4o = plan.r4c_off_h[:nl_], plan.c4r_off_h[:nl_]
        n_r4c = int(nM32[:nl_].astype(np.int64).sum()) * k
        n_c4r = int(nR32[:nl_].astype(np.int64).sum()) * k
        hl_r4c = torch.empty(n_r4c, dtype=torch.int64).pin_memory()
        hl_c4r = torch.empty(n_c4r, dtype=torch.int64).pin_memory()
        hl_gain = torch.empty(nl_ * k, dtype=torch.float64).pin_memory()
        def lists_step():
            _lib.check(lib.pda_murty_batch_host(h_costs.data_ptr(), h_off.data_ptr(), h_nr.data_ptr(), h_nc.data_ptr(), nl_, k,
                                                1, 42.0, 0, 0, hl_r4c.data_ptr(), r4o.ctypes.data, hl_c4r.data_ptr(), c4o.ctypes.data,
                                                hl_gain.data_ptr(), h_found.data_ptr(), 1, h_probs.data_ptr(), h_poff.data_ptr(),
                                                h_nl.data_ptr(), local))
        lists_step()
        t0 = time.perf_counter()
        for _ in range(2):
            lists_step()
        lists_pps = 2 * nl_ / (time.perf_counter() - t0)
        e2e_variants = {"pageable_buffers_weights_only": {"value": pageable_pps, "unit": UNIT, "problems": n,
                                                          "note": "numpy arrays: inputs and outputs are copied through the staging arena"},
                        "lists_to_host_kBest2DCutoff": {"value": lists_pps, "unit": UNIT, "problems": nl_,
                                                        "d2h_bytes_per_pass": int((n_r4c + n_c4r + nl_ * k) * 8),
                                                        "note": "row4col + col4row (int64) + gains of every hypothesis returned to page-locked host buffers"}}
        del hl_r4c, hl_c4r, hl_gain

    # ---- permanent n = 24 latency (second half of the metric) ----------------------------------------------
    A24 = synth.dense_square(1, 24, first=4242)
    pplan = dev.PermanentPlan(A24, 24)
    for _ in range(5):
        pplan.run()
    torch.cuda.synchronize()
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        pplan.run()
    e1.record()
    torch.cuda.synchronize()
    perm_ms = e0.elapsed_time(e1) / reps
    # ---- config 5: ONE n = 28 permanent, Gray range split over the ranks, (hi, lo) partials all-gathered ----
    from probabilisticsemslam_b200 import shard
    A28 = synth.dense_square(1, 28, first=2828)[0].reshape(28, 28, order="F")
    b28, e28 = shard.gray_range(28, world, rank)
    rplan = dev.PermanentRangePlan(A28, b28, e28)
    parts = torch.zeros(world * 2, dtype=torch.float64, device="cuda")
    def perm28_step():
        if e28 > b28:
            rplan.run()
        if world > 1:
            dist.all_gather_into_tensor(parts, rplan.partial)
        else:
            parts.copy_(rplan.partial)
    for _ in range(3):
        perm28_step()
    # Optional (PDA_BENCH_GRAPH=1): kernel + exchange as ONE CUDA graph, so the collective is queued behind the kernel on
    # the device with no Python and no launch latency between them.  OFF by default: an 8-rank run with the capture
    # enabled did not come back within its time limit in round 2 and could not be re-examined, so the measured path
    # stays the plain stream launches that every earlier run used.
    perm28_run, perm28_how = perm28_step, "stream launches"
    if world > 1 and os.environ.get("PDA_BENCH_GRAPH") == "1":
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                perm28_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph28 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph28):
                perm28_step()
            perm28_run, perm28_how = graph28.replay, "one CUDA graph (kernel + NCCL all_gather)"
        except Exception as exc:  # capture not possible here: plain launches
            perm28_how = f"stream launches (graph capture failed: {type(exc).__name__})"
    for _ in range(3):
        perm28_run()
    barrier()
    e0.record()
    for _ in range(10):
        perm28_run()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 10], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    perm28_ms = float(t.item())
    perm28_value = shard.combine_partials(parts.cpu().numpy(), 28)

    # ---- config 3 as BASELINE words it: the SAME 100k-problem batch at k = 1000, cut into contiguous slices over the
    #      ranks (strong scaling).  Lists, gains and weights are written on the owning rank; the weight tables and
    #      nFound are gathered on rank 0 inside the timed region (assignmentProb's result; the 33 GB of k-best lists
    #      stay where they were produced).  Time = max over ranks.  Present at every N, so the driver's scaling file
    #      carries a strong-scaling series next to the weak-scaling headline.
    cfg3 = None
    if not args.skip_config3:
        k3, n3 = 1000, args.problems
        lo3, hi3 = n3 * rank // world, n3 * (rank + 1) // world
        torch.cuda.empty_cache()
        pb3 = synth.g1_dense(hi3 - lo3, first=lo3)
        plan3 = dev.MurtyPlan(pb3, k=k3, weights=True)
        sizes3 = [n3 * (r + 1) // world - n3 * r // world for r in range(world)]
        # gather buffers on rank 0: equal-sized slots (the largest slice's table), plain NCCL gather
        slot = torch.tensor([plan3.n_prob], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(slot, op=dist.ReduceOp.MAX)
        slot = int(slot.item())
        send_p = torch.zeros(slot, dtype=torch.float64, device="cuda")
        send_f = torch.zeros(max(sizes3), dtype=torch.int32, device="cuda")
        recv_p = [torch.empty(slot, dtype=torch.float64, device="cuda") for _ in range(world)] if rank == 0 else None
        recv_f = [torch.empty(max(sizes3), dtype=torch.int32, device="cuda") for _ in range(world)] if rank == 0 else None
        def cfg3_step():
            plan3.run()
            if world > 1:
                send_p[:plan3.n_prob].copy_(plan3.probs)
                send_f[:plan3.n].copy_(plan3.n_found)
                dist.gather(send_p, recv_p, dst=0)
                dist.gather(send_f, recv_f, dst=0)
        cfg3_step()
        barrier()
        e0c, e1c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps3 = 2
        e0c.record()
        for _ in range(reps3):
            cfg3_step()
        e1c.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0c.elapsed_time(e1c) / reps3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms3 = float(t.item())
        fb3 = int(plan3.workspace[8:12].view(torch.int32).item())
        cfg3 = {"workload": f"configs[2]: the same {n3} problems at k={k3}, contiguous slices over {world} rank(s) (strong scaling)",
                "ms_per_pass": ms3, "problems_per_s": n3 / (ms3 * 1e-3), "ranks": world,
                "problems_on_rank0": hi3 - lo3, "exact_fallback_problems_rank0": fb3,
                "gather": "weight tables + nFound to rank 0 (NCCL gather) inside the timed region; k-best lists stay on the owning rank" if world > 1 else "none (one rank)"}
        del plan3, send_p, send_f, recv_p, recv_f
        torch.cuda.empty_cache()

    # ---- config 4 over the ranks: batched exact permanents n = 12..20 (dense U(0,1)), contiguous slices of every size
    #      class per rank, results gathered on rank 0; and permanentProb weights of gated problems the same way
    cfg4 = None
    if not args.skip_config4:
        per_n = 2000
        plans4 = []
        for nd_ in range(12, 21):
            lo4, hi4 = per_n * rank // world, per_n * (rank + 1) // world
            plans4.append(dev.PermanentPlan(synth.dense_square(hi4 - lo4, nd_, first=5000 * nd_ + lo4), nd_))
        tot_local = sum(pl.n for pl in plans4)
        send4 = torch.zeros(9 * (per_n // world + 1), dtype=torch.float64, device="cuda")
        recv4 = [torch.empty_like(send4) for _ in range(world)] if rank == 0 else None
        def cfg4_step():
            o = 0
            for pl in plans4:
                pl.run()
                send4[o:o + pl.n].copy_(pl.out); o += pl.n
            if world > 1:
                dist.gather(send4, recv4, dst=0)
        cfg4_step()
        barrier()
        e0c, e1c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0c.record()
        for _ in range(3):
            cfg4_step()
        e1c.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0c.elapsed_time(e1c) / 3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms4 = float(t.item())
        flops4 = sum(per_n * 3.0 * nd_ * 2.0 ** (nd_ - 1) for nd_ in range(12, 21))
        # permanentProb (host call per rank on its slice of gated problems)
        from probabilisticsemslam_b200 import api as _api
        g2 = synth.g2_gated(1200, first=40000)
        cond, _ = _api.condition_costs_batch(g2, device=local)
        keep = [q for q in range(len(cond)) if cond.matrix(q).shape[0] - 1 <= 20]
        lo5, hi5 = len(keep) * rank // world, len(keep) * (rank + 1) // world
        sub = synth.pack([cond.matrix(q) for q in keep[lo5:hi5]], [int(cond.nL[q]) for q in keep[lo5:hi5]])
        _api.permanent_prob_batch(sub, 1, device=local)
        barrier()
        t0 = time.perf_counter()
        tabs, _st = _api.permanent_prob_batch(sub, 1, device=local)
        flat = torch.from_numpy(np.concatenate([x.reshape(-1) for x in tabs])).cuda() if len(tabs) else torch.zeros(0, dtype=torch.float64, device="cuda")
        if world > 1:
            sz = torch.tensor([flat.numel()], dtype=torch.int64, device="cuda")
            dist.all_reduce(sz, op=dist.ReduceOp.MAX)
            pad = torch.zeros(int(sz.item()), dtype=torch.float64, device="cuda"); pad[:flat.numel()] = flat
            dist.gather(pad, [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None, dst=0)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        cfg4 = {"workload": f"configs[3]: {per_n} dense matrices for each n = 12..20, contiguous slices over {world} rank(s); results gathered on rank 0",
                "ms_per_pass": ms4, "matrices": 9 * per_n, "matrices_per_s": 9 * per_n / (ms4 * 1e-3),
                "achieved_tflops": flops4 / (ms4 * 1e-3) / 1e12, "ranks": world, "matrices_on_rank0": tot_local,
                "permanent_prob": {"problems": len(keep), "ms": 1e3 * float(t.item()),
                                   "problems_per_s": len(keep) / float(t.item()),
                                   "call": "pda_permanent_prob_batch_host on each rank's slice of gated problems (<= 21 rows), tables gathered on rank 0"}}
        del plans4
        torch.cuda.empty_cache()

    # ---- configs[0]: ONE 5x30 problem, k = 200, through the host call (the per-frame shape of the SLAM loop): the
    #      batch-of-one goes to the one-CTA-per-problem kernel; H2D, launch and D2H are inside the wall-clock time
    from probabilisticsemslam_b200 import api
    C1 = synth.g1_dense(1, nM=5).matrix(0)
    lat = {}
    if rank == 0:
        for path in ("cta", "warp"):
            api.set_murty_path(path)
            for _ in range(5):
                api.assignmentProb(C1, 30, k)
            ts = []
            for _ in range(30):
                t0 = time.perf_counter(); api.assignmentProb(C1, 30, k); ts.append(time.perf_counter() - t0)
            lat[path] = 1e6 * statistics.median(ts)
        api.set_murty_path("auto")
    # ---- "next" row: moments in, weights out (cost matrices built on the device), 20 000 gated frames ------------
    mom = None
    if rank == 0:
        frames = synth.quadric_frames(2000, first=123)
        packed = api._pack_moments(frames * 10)
        nLs, nMs = np.diff(packed[2]), np.diff(packed[5])
        out = np.zeros(int((nMs * (nLs + 1)).sum()))
        def mom_step():
            _lib.check(lib.pda_association_from_moments_batch_host(*[a.ctypes.data for a in packed[:6]], len(nLs), 10.0, k,
                                                                   out.ctypes.data, local))
        mom_step()
        t0 = time.perf_counter()
        for _ in range(3):
            mom_step()
        mom = {"frames": int(len(nLs)), "frames_per_s": 3 * len(nLs) / (time.perf_counter() - t0),
               "call": "pda_association_from_moments_batch_host: quadric moments in (host), weights out (host); "
                       "cost matrices, conditioning, k-best weights and un-compaction on the device"}

    fp64_peak = None
    if hasattr(lib, "pda_diag_dfma_tflops"):
        import ctypes as C
        lib.pda_diag_dfma_tflops.restype = C.c_double
        fp64_peak = float(lib.pda_diag_dfma_tflops())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD if (n == N_PER_GPU and k == K_BEST) else f"G1 x {n} per GPU, k={k}",
                   "problems_per_gpu": n, "k": k, "outputs": "row4col+col4row (int64) + gains + weights per problem",
                   "l2": "inputs (150 MB) and outputs (7 GB) per pass exceed the 126 MB L2; no flush needed",
                   "parallelism": f"{world} x independent shards, no data-path collective"},
        "clocks": clk.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "call": "pda_murty_batch_host (batched assignmentProb: host cost matrices in, host weights out; "
                        "k-best lists stay device-internal as they are stack temporaries in the reference). The buffers are "
                        "page-locked, so the kernel reads each cost matrix and writes each weight table over PCIe itself "
                        "(the bytes below cross the bus inside the timed region, overlapped with computing); e2e can exceed "
                        "`value` because the device-resident pass additionally writes the 7 GB of k-best lists",
                "matches_device_run": e2e_matches},
        # per timed step: order_by_cost_kernel + murty_kernel<2, true> (pruning) + murty_kernel<2, false> (exact, over the
        # problems the pruning kernel handed back: none on this workload, the launch finds an empty list)
        "gpu_launches": 3 * args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                     "traffic": measured_traffic(n, k), "peak_source": pk_kind, "kernel": "murty_kernel<2, true>", "kernel_ms": kernel_ms,
                     "exact_fallback_problems": fallback_problems,
                     "traffic_source": "profiles/traffic.json: ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch over 20 000 problems, scaled per problem",
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "note": "issue/ALU-pipe bound by construction (SURVEY.md 8d), not HBM bound. traffic (ncu, profiles/) exceeds the "
                             "algorithmic bytes by the node arena: every KEPT Murty child (736 B of duals + pairing) is spilled once and the "
                             "ones that reach the top are read back; children that cannot be among the k best are abandoned before they are stored; "
                             "inputs are read once"},
        "extra": {"permanent_n24": {"gpu_ms": perm_ms, "unit": "ms", "flops": pplan.flops(),
                                    "achieved_tflops": pplan.flops() / (perm_ms * 1e-3) / 1e12,
                                    "fp64_peak_tflops_measured": fp64_peak},
                  "config0_single_5x30_k200": {"host_call_us_cta_kernel": lat.get("cta"), "host_call_us_warp_kernel": lat.get("warp"),
                                               "call": "assignmentProb, batch of one, host buffers (H2D + launch + D2H inside)"},
                  "moments_to_weights": mom,
                  "config3_k1000_strong": cfg3,
                  "permanent_batch_sharded": cfg4,
                  "e2e_variants": e2e_variants,
                  "permanent_n28_sharded": {"ms": perm28_ms, "ranks": world, "value": perm28_value,
                                            "exchange": "all_gather of 16-byte (hi, lo) partials, summed in rank order" if world > 1 else "none",
                                            "launch": perm28_how,
                                            "achieved_tflops": 3.0 * 28 * 2.0 ** 27 / (perm28_ms * 1e-3) / 1e12}},
    }
    if world == 1 and not args.no_cpu:
        chk, kind, what = cpu_checker()
        cores = os.cpu_count() or 1
        sample = max(cores * 250, 1000)
        cpu_pps, sec = cpu_problems_per_sec(chk, sample, cores)
        one_pps, _ = cpu_problems_per_sec(chk, 400, 1)
        line["cpu_baseline"] = {"value": cpu_pps, "unit": UNIT, "cores": cores, "kind": kind,
                                "sample": f"first {sample} problems of the same batch, {cores} threads, {what}; single thread: {one_pps:.0f} problems/s"}
        line["extra"]["permanent_n24"]["cpu_ms"] = cpu_permanent_ms(chk)
        tc = []
        for _ in range(10):
            t0 = time.perf_counter(); chk.assignment_prob(C1, 30, k); tc.append(time.perf_counter() - t0)
        line["extra"]["config0_single_5x30_k200"]["cpu_us"] = 1e6 * statistics.median(tc)
        # algorithmic work of the reference's formulation (SURVEY.md 8d), counted by the oracle on a sample
        try:
            import ctypes as C
            from oracle.loader import load_oracle
            orc = load_oracle()
            sample_pb = synth.g1_dense(200)
            tot = np.zeros(5)
            cnt = [C.c_int64(0) for _ in range(5)]
            for q in range(len(sample_pb)):
                orc.kbest2d_cutoff(k, sample_pb.matrix(q), 42.0)
                orc.lib.orc_last_counters(*[C.byref(c) for c in cnt])
                tot += [c.value for c in cnt]
            per = tot / len(sample_pb)
            line["extra"]["reference_formulation_work"] = {
                "per_problem": {"pops": per[0], "child_solves": per[1], "dijkstra_steps": per[2], "reduced_cost_evaluations": per[3]},
                "delivered_per_second": {"dijkstra_steps": per[2] * value, "reduced_cost_evaluations": per[3] * value},
                "note": "work the reference's algorithm performs for these outputs; the kernel retires ~80 % of the steps in bulk (fast-forward)"}
        except Exception as exc:  # the counters are informational
            line["extra"]["reference_formulation_work"] = {"unavailable": str(exc)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
