"""Times the single-device *_host entries at a batch of one and at about 50 MB of inputs + outputs, and
pda_murty_batch_host at 140 000 and 262 144 problems (pageable and page-locked at k = 200, page-locked with every k-best
list returned at k = 20), for one or more builds of libpda_b200.so, and states whether every build returned the same
bytes.

    python scripts/host_stage_bench.py --libs OLD.so NEW.so [--rounds 3] [--out results.json]

Each build runs in its own process (PDA_B200_LIB), and the builds take turns, round after round, so that drift on a
shared machine falls on all of them.  A time is the median host-clock time of one call, which ends in a device
synchronise; the output digest is a SHA-256 over every output array of the last call (of a k-best list, over the
nFound hypotheses the call defines).
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BIG = 50 << 20


def _prefix(sizes):
    off = np.zeros(len(sizes), np.int64)
    off[1:] = np.cumsum(np.asarray(sizes, np.int64))[:-1]
    return off


def _p(a):
    return None if a is None else a.ctypes.data


def cases(lib, big):
    """name -> (call, outputs, bytes of inputs + outputs) for a batch of one (big = False) or about 50 MB."""
    from probabilisticsemslam_b200 import api, synth
    out = {}

    def add(name, call, outs, ins):
        out[name] = (call, outs, sum(a.nbytes for a in list(ins) + list(outs) if a is not None))

    def g1(per_problem):
        return synth.g1_dense(max(1, BIG // per_problem) if big else 1, first=10)

    pb = g1(2400)
    nr, nc = pb.num_row, pb.nM.astype(np.int32)
    ro, co = _prefix(nr), _prefix(nc)
    R, C, n = int(nr.sum()), int(nc.sum()), len(pb)
    lap_out = [np.zeros(R, np.int64), np.zeros(C, np.int64), np.zeros(C), np.zeros(R), np.zeros(R, np.uint8), np.zeros(n),
               np.zeros(n, np.int32)]
    add("lap", lambda: lib.pda_lap_batch_host(_p(pb.costs), _p(pb.cost_off), _p(nr), _p(nc), None, n, 1, 0, _p(ro), _p(co),
                                              *[_p(a) for a in lap_out], 0), lap_out, [pb.costs, pb.cost_off, nr, nc, ro, co])

    cond_out = [np.zeros_like(pb.costs), np.zeros(R, np.int64), np.zeros(n, np.int32)]
    add("condition_costs", lambda: lib.pda_condition_costs_batch_host(_p(pb.costs), _p(pb.cost_off), _p(nr), _p(nc), n, _p(ro),
                                                                      *[_p(a) for a in cond_out], 0),
        cond_out, [pb.costs, pb.cost_off, nr, nc, ro])

    lens = np.full(max(1, BIG // 8 // 1000) if big else 1, 1000, np.int64)
    voff = _prefix(lens)
    vals0 = 60.0 * np.random.default_rng(1).random(int(lens.sum()))
    vals = vals0.copy()

    def to_probs():
        vals[:] = vals0
        return lib.pda_to_probs_batch_host(_p(vals), _p(voff), _p(lens), len(lens), 0)
    add("to_probs", to_probs, [vals], [voff, lens])

    nq = BIG // 200 if big else 1
    q, covs = np.random.default_rng(2).random(nq * 16), np.zeros(nq * 9)
    add("quadric_covs", lambda: lib.pda_quadric_covs_batch_host(_p(q), nq, _p(covs), 0), [covs], [q])

    packed = api._pack_moments(synth.quadric_frames(BIG // 6000 if big else 1, first=20))
    nL, nM = np.diff(packed[2]), np.diff(packed[5])
    nf = len(nL)
    costs = np.zeros(int(((nL + nM) * nM).sum()))
    probs = np.zeros(int((nM * (nL + 1)).sum()))
    status = np.zeros(nf, np.int32)
    add("quadric_cost", lambda: lib.pda_quadric_cost_batch_host(*[_p(a) for a in packed], nf, 10.0, _p(costs), 0), [costs], packed)
    add("association_from_moments", lambda: lib.pda_association_from_moments_batch_host(*[_p(a) for a in packed], nf, 10.0, 50,
                                                                                        _p(probs), 0), [probs], packed)
    add("association_perm_from_moments", lambda: lib.pda_association_perm_from_moments_batch_host(
        *[_p(a) for a in packed], nf, 10.0, _p(probs), _p(status), 0), [probs, status], packed)

    pa = g1(2400)
    cells = pa.nM.astype(np.int64) * (pa.nL + 1)
    poff = _prefix(cells)
    aprobs, ast = np.zeros(int(cells.sum())), np.zeros(len(pa), np.int32)
    add("association_probs", lambda: lib.pda_association_probs_batch_host(_p(pa.costs), _p(pa.cost_off), _p(pa.nL), _p(pa.nM),
                                                                          len(pa), 50, _p(aprobs), _p(poff), 0),
        [aprobs], [pa.costs, pa.cost_off, pa.nL, pa.nM, poff])
    add("association_perm_probs", lambda: lib.pda_association_perm_probs_batch_host(
        _p(pa.costs), _p(pa.cost_off), _p(pa.nL), _p(pa.nM), len(pa), _p(aprobs), _p(poff), _p(ast), 0),
        [aprobs, ast], [pa.costs, pa.cost_off, pa.nL, pa.nM, poff])
    add("permanent_prob", lambda: lib.pda_permanent_prob_batch_host(
        _p(pa.costs), _p(pa.cost_off), _p(pa.nL), _p(pa.nM), len(pa), 1, _p(aprobs), _p(poff), _p(ast), 0),
        [aprobs], [pa.costs, pa.cost_off, pa.nL, pa.nM, poff])

    def mats(dim, per):
        m = BIG // per if big else 1
        flat = np.random.default_rng(dim).random(m * dim * dim)
        return flat, _prefix(np.full(m, dim * dim)), np.full(m, dim, np.int32), np.full(m, dim, np.int32), np.zeros(m), np.zeros(m, np.int32)
    m12 = mats(12, 1200)
    add("permanent_exact", lambda: lib.pda_permanent_batch_host(*[_p(a) for a in m12[:4]], len(m12[2]), _p(m12[4]), _p(m12[5]), 0),
        m12[4:], m12[:4])
    m8 = mats(8, 540)
    add("permanent_approx", lambda: lib.pda_permanent_approx_batch_host(*[_p(a) for a in m8[:4]], len(m8[2]), 20, 7, _p(m8[4]),
                                                                        _p(m8[5]), 0), m8[4:], m8[:4])
    add("conditioned_permanent", lambda: lib.pda_conditioned_permanent_batch_host(*[_p(a) for a in m8[:4]], len(m8[2]), 1,
                                                                                  _p(m8[4]), _p(m8[5]), 0), m8[4:], m8[:4])

    lefts, rights = synth.stereo_boxes(BIG // 500 if big else 1, first=30)
    ol = np.concatenate([[0], np.cumsum([len(b) for b in lefts])]).astype(np.int64)
    orr = np.concatenate([[0], np.cumsum([len(b) for b in rights])]).astype(np.int64)
    bl, br = np.ascontiguousarray(np.concatenate(lefts)), np.ascontiguousarray(np.concatenate(rights))
    asg = np.zeros(int(ol[-1]), np.int32)
    add("asgn_bb", lambda: lib.pda_asgn_bb_batch_host(_p(bl), _p(ol), _p(br), _p(orr), len(lefts), 0.2, _p(asg), 0), [asg],
        [bl, br, ol, orr])

    pk = synth.g1_dense(BIG // 4000 if big else 1, first=40)
    found, knr, knc = np.zeros(len(pk), np.int32), pk.num_row, pk.nM.astype(np.int32)
    kcells = pk.nM.astype(np.int64) * (pk.nL + 1)
    kprobs, koff = np.zeros(int(kcells.sum())), _prefix(kcells)
    add("murty_k200", lambda: lib.pda_murty_batch_host(_p(pk.costs), _p(pk.cost_off), _p(knr), _p(knc), len(pk), 200,
                                                       api.CUT_RELATIVE, 42.0, 0, 0, None, None, None, None, None, _p(found),
                                                       api.WEIGHTS_GATED, _p(kprobs), _p(koff), _p(pk.nL), 0),
        [found, kprobs], [pk.costs, pk.cost_off, knr, knc, koff])
    if not big:
        A, part = np.random.default_rng(3).random(20 * 20), np.zeros(2)
        add("permanent_range", lambda: lib.pda_permanent_range_host(_p(A), 20, 0, 1 << 19, _p(part), 0), [part], [A])
    return out


def kbest_cases(lib, n, allocs):
    """pda_murty_batch_host on n G1 problems: pageable and page-locked (pda_host_alloc) at k = 200, and page-locked with
    every k-best list returned at k = 20.  Page-locked buffers are appended to `allocs`."""
    from probabilisticsemslam_b200 import api, synth
    pk = synth.g1_dense(n, first=50)
    nr, nc, nl = pk.num_row, pk.nM.astype(np.int32), pk.nL.astype(np.int32)
    cells = nc.astype(np.int64) * (nl + 1)
    poff = _prefix(cells)

    def pinned(a):
        p = lib.pda_host_alloc(max(a.nbytes, 8))
        assert p, "pda_host_alloc failed"
        allocs.append(p)
        v = np.ctypeslib.as_array((ctypes.c_uint8 * a.nbytes).from_address(p)).view(a.dtype)
        v[:] = a
        return v

    def call(costs, found, probs, k, r4c=None, r4o=None, c4r=None, c4o=None, gain=None):
        return lambda: lib.pda_murty_batch_host(_p(costs), _p(pk.cost_off), _p(nr), _p(nc), n, k, api.CUT_RELATIVE, 42.0, 0, 0,
                                                _p(r4c), _p(r4o), _p(c4r), _p(c4o), _p(gain), _p(found), api.WEIGHTS_GATED,
                                                _p(probs), _p(poff), _p(nl), 0)
    ins = [pk.costs, pk.cost_off, nr, nc, nl, poff]
    mb = lambda arrays: sum(a.nbytes for a in arrays)
    found, probs = np.zeros(n, np.int32), np.zeros(int(cells.sum()))
    out = {f"murty_k200_pageable/{n}": (call(pk.costs, found, probs, 200), [found, probs], mb(ins + [found, probs]))}
    pc, pf, pp = pinned(pk.costs), pinned(found), pinned(probs)
    out[f"murty_k200_pinned/{n}"] = (call(pc, pf, pp, 200), [pf, pp], mb(ins + [pf, pp]))
    k = 20
    r4o, c4o = _prefix(nc.astype(np.int64) * k), _prefix(nr.astype(np.int64) * k)
    lf, lp = pinned(found), pinned(probs)
    r4c, c4r, gain = pinned(np.zeros(int(nc.sum()) * k, np.int64)), pinned(np.zeros(int(nr.sum()) * k, np.int64)), pinned(np.zeros(n * k))

    def defined():  # only the first nFound hypotheses of a problem are defined
        f = lf.astype(np.int64)
        lists = [gain[(np.arange(k)[None, :] < f[:, None]).reshape(-1)]]
        lists += [r4c[o:o + x * c] for o, x, c in zip(r4o, f, nc)] + [c4r[o:o + x * r] for o, x, r in zip(c4o, f, nr)]
        return [lf, lp] + lists
    out[f"murty_k20_lists_pinned/{n}"] = (call(pc, lf, lp, k, r4c, r4o, c4r, c4o, gain), defined,
                                          mb(ins + [r4o, c4o, lf, lp, r4c, c4r, gain]))
    return out


def worker(reps_small, reps_big):
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    res = {}

    def run(key, call, outs, nbytes, reps):
        times = []
        for i in range(2 + reps):
            t0 = time.perf_counter()
            _lib.check(call())
            if i >= 2:
                times.append(time.perf_counter() - t0)
        h = hashlib.sha256()
        for a in (outs() if callable(outs) else outs):
            h.update(np.ascontiguousarray(a).tobytes())
        res[key] = dict(ms=float(np.median(times)) * 1e3, mb=nbytes / 2**20, digest=h.hexdigest()[:16])

    for big in (False, True):
        for name, case in cases(lib, big).items():
            run(f"{name}/{'50MB' if big else 'one'}", *case, reps_big if big else reps_small)
    for n in (140_000, 262_144):
        allocs = []
        try:
            for name, case in kbest_cases(lib, n, allocs).items():
                run(name, *case, reps_big)
        finally:
            for p in allocs:
                lib.pda_host_free(p)
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", nargs="+", help="builds of libpda_b200.so to compare (default: the in-tree build)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=50, help="timed calls per case at a batch of one (a fifth of that at 50 MB)")
    ap.add_argument("--out", help="write every round's results here as JSON")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.reps, max(2, a.reps // 5))
    libs = a.libs or [os.path.join(ROOT, "probabilisticsemslam_b200", "libpda_b200.so")]
    runs = {lib: [] for lib in libs}
    for r in range(a.rounds):
        for lib in (libs if r % 2 == 0 else libs[::-1]):
            env = dict(os.environ, PDA_B200_LIB=os.path.abspath(lib))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--reps", str(a.reps)], env=env,
                               capture_output=True, text=True, check=True)
            runs[lib].append(json.loads(p.stdout.strip().splitlines()[-1]))
    import torch
    props = torch.cuda.get_device_properties(0)
    print(f"{props.name}; median host-clock ms per call, median over {a.rounds} rounds")
    keys = list(runs[libs[0]][0])
    print(f"{'case':42s} {'MB':>7s} " + " ".join(f"{os.path.basename(os.path.dirname(os.path.abspath(l)))[:14]:>14s}" for l in libs) + "  outputs")
    same_all = True
    for k in keys:
        ms = [float(np.median([r[k]["ms"] for r in runs[lib]])) for lib in libs]
        digests = {r[k]["digest"] for lib in libs for r in runs[lib]}
        same_all &= len(digests) == 1
        print(f"{k:42s} {runs[libs[0]][0][k]['mb']:7.2f} " + " ".join(f"{x:14.3f}" for x in ms) +
              ("  same" if len(digests) == 1 else "  DIFFER"))
    print("every output identical across builds and rounds" if same_all else "OUTPUTS DIFFER")
    if a.out:
        with open(a.out, "w") as f:
            json.dump(dict(device=props.name, libs=libs, runs=runs), f, indent=1)
    return 0 if same_all else 1


if __name__ == "__main__":
    sys.exit(main())
