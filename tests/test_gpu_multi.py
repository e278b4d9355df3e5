"""Multi-device entry points of the C ABI (SURVEY.md 8e, "single process drives all GPUs") and large host batches.

On a one-GPU box the device list names device 0 several times: the slices then queue on that device's lock, which
exercises the sharding, the offset handling and the result placement exactly as several devices would.  On a multi-GPU
box (gpurun --gpus N) every visible device is used."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from probabilisticsemslam_b200 import _lib, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "build", "multi_gpu_b200")


def _devices():
    n = _lib.lib().pda_device_count()
    return list(range(n)) if n > 1 else [0, 0, 0]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _assignment_prob(pb, k, devices=None, lists=False):
    lib = _lib.lib()
    n = len(pb)
    nr = pb.num_row.astype(np.int32)
    nc = pb.nM.astype(np.int32)
    nl = pb.nL.astype(np.int32)
    sizes = (nc.astype(np.int64) * (nl + 1)).astype(np.int64)
    poff = np.zeros(n, np.int64); poff[1:] = np.cumsum(sizes)[:-1]
    probs = np.zeros(int(sizes.sum()), np.float64)
    found = np.zeros(n, np.int32)
    r4c = c4r = gain = r4o = c4o = None
    if lists:
        r4o = np.zeros(n, np.int64); r4o[1:] = np.cumsum(nc.astype(np.int64) * k)[:-1]
        c4o = np.zeros(n, np.int64); c4o[1:] = np.cumsum(nr.astype(np.int64) * k)[:-1]
        r4c = np.full(int(nc.astype(np.int64).sum()) * k, -7, np.int64)
        c4r = np.full(int(nr.astype(np.int64).sum()) * k, -7, np.int64)
        gain = np.zeros(n * k, np.float64)
    args = [_p(pb.costs), _p(pb.cost_off), _p(nr), _p(nc), n, k, 1, 42.0, 0, 0,
            _p(r4c) if lists else None, _p(r4o) if lists else None, _p(c4r) if lists else None, _p(c4o) if lists else None,
            _p(gain) if lists else None, _p(found), 1, _p(probs), _p(poff), _p(nl)]
    if devices is None:
        _lib.check(lib.pda_murty_batch_host(*args, 0))
    else:
        d = np.asarray(devices, np.int32)
        _lib.check(lib.pda_murty_batch_host_multi(*args, _p(d), len(d)))
    return probs, found, r4c, c4r, gain


def test_murty_batch_multi_matches_single():
    pb = synth.g1_dense(3000, first=12345)
    p1, f1, r1, c1, g1 = _assignment_prob(pb, 60, None, lists=True)
    pN, fN, rN, cN, gN = _assignment_prob(pb, 60, _devices(), lists=True)
    assert np.array_equal(f1, fN) and np.array_equal(r1, rN) and np.array_equal(c1, cN)
    assert np.array_equal(g1.view(np.int64), gN.view(np.int64))
    assert np.array_equal(p1.view(np.int64), pN.view(np.int64))
    # more devices than problems: the surplus stays idle
    small = synth.g1_dense(2, first=5)
    a = _assignment_prob(small, 20, None)[0]
    b = _assignment_prob(small, 20, [0, 0, 0, 0, 0])[0]
    assert np.array_equal(a, b)


def test_permanent_multi(oracle):
    lib = _lib.lib()
    mats = [synth.dense_square(1, n, first=100 + i)[0].reshape(n, n, order="F") for i, n in enumerate([3, 8, 12, 12, 14, 16, 9, 11, 15])]
    flat = np.concatenate([m.reshape(-1, order="F") for m in mats])
    off = np.zeros(len(mats), np.int64); off[1:] = np.cumsum([m.size for m in mats])[:-1]
    rows = np.array([m.shape[0] for m in mats], np.int32)
    out1, outN = np.zeros(len(mats)), np.zeros(len(mats))
    st1, stN = np.zeros(len(mats), np.int32), np.zeros(len(mats), np.int32)
    _lib.check(lib.pda_permanent_batch_host(_p(flat), _p(off), _p(rows), _p(rows), len(mats), _p(out1), _p(st1), 0))
    d = np.asarray(_devices(), np.int32)
    _lib.check(lib.pda_permanent_batch_host_multi(_p(flat), _p(off), _p(rows), _p(rows), len(mats), _p(outN), _p(stN), _p(d), len(d)))
    # the NW walk of a matrix is cut by the launch shape, which depends on the batch around it: last-bit differences only
    np.testing.assert_allclose(outN, out1, rtol=1e-13)
    assert not stN.any()
    for m, v in zip(mats, outN):
        np.testing.assert_allclose(v, oracle.permanent_exact_square(m)[0], rtol=1e-9)
    # ONE matrix, Gray range split over the devices, partials combined in device order
    n = 22
    A = np.ascontiguousarray(synth.dense_square(1, n, first=99)[0])
    got = np.zeros(1)
    _lib.check(lib.pda_permanent_sharded_host(_p(A), n, _p(d), len(d), _p(got)))
    np.testing.assert_allclose(got[0], oracle.permanent_exact_square(A.reshape(n, n, order="F"))[0], rtol=1e-9)
    one = np.zeros(1, np.int32)
    _lib.check(lib.pda_permanent_sharded_host(_p(A), n, _p(one), 1, _p(got)))
    np.testing.assert_allclose(got[0], oracle.permanent_exact_square(A.reshape(n, n, order="F"))[0], rtol=1e-9)


def test_permanent_prob_multi(gpu_api):
    lib = _lib.lib()
    g2 = synth.g2_gated(60, first=700)
    cond, _ = gpu_api.condition_costs_batch(g2)
    keep = [p for p in range(len(cond)) if cond.matrix(p).shape[0] - 1 <= 20]
    sub = synth.pack([cond.matrix(p) for p in keep], [int(cond.nL[p]) for p in keep])
    want, st = gpu_api.permanent_prob_batch(sub, 1)
    n = len(sub)
    nl, nm = sub.nL.astype(np.int32), sub.nM.astype(np.int32)
    sizes = nm.astype(np.int64) * (nl + 1)
    poff = np.zeros(n, np.int64); poff[1:] = np.cumsum(sizes)[:-1]
    probs = np.zeros(int(sizes.sum())); status = np.zeros(n, np.int32)
    d = np.asarray(_devices(), np.int32)
    _lib.check(lib.pda_permanent_prob_batch_host_multi(_p(sub.costs), _p(sub.cost_off), _p(nl), _p(nm), n, 1, _p(probs), _p(poff),
                                                       _p(status), _p(d), len(d)))
    assert not status.any()
    for p in range(n):
        got = probs[poff[p]:poff[p] + sizes[p]].reshape(int(nm[p]), int(nl[p]) + 1)
        assert np.array_equal(got, want[p])


def test_cpp_caller_drives_several_devices():
    """tests/cpp/multi_gpu_driver.cpp through include/assignment.h and include/nwPerm.h: no Python on the data path."""
    assert os.path.exists(EXE), "tests/cpp/build/multi_gpu_b200 missing: run __graft_entry__.build()"
    run = subprocess.run([EXE, "1500", "100", "20", ",".join(str(x) for x in _devices())], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-300:] + run.stderr[-500:]
    rec = json.loads(run.stdout.strip().splitlines()[-1])
    assert rec["bit_identical"] and rec["permanent_prob_bit_identical"]
    assert rec["perm_rel_diff"] < 1e-9


@pytest.mark.parametrize("pinned", [False, True])
def test_large_host_batch(pinned):
    """140 000 problems in ONE pda_murty_batch_host call must give what two half-size calls give, with pageable and with
    page-locked buffers (lists and weights returned), and a batch whose problems all SHARE one cost matrix (equal
    offsets) must give every problem that matrix's table."""
    import torch
    lib = _lib.lib()
    n, k = 140000, 4
    pb = synth.g1_dense(n, nL=3, nM=2, first=9000)
    half = n // 2
    a = _assignment_prob(pb.slice(0, half), k, None, lists=True)
    b = _assignment_prob(pb.slice(half, n), k, None, lists=True)
    want = [np.concatenate([x, y]) for x, y in zip(a, b)]
    if not pinned:
        got = _assignment_prob(pb, k, None, lists=True)
    else:
        nr = pb.num_row.astype(np.int32); nc = pb.nM.astype(np.int32); nl = pb.nL.astype(np.int32)
        sizes = nc.astype(np.int64) * (nl + 1)
        poff = np.zeros(n, np.int64); poff[1:] = np.cumsum(sizes)[:-1]
        r4o = np.zeros(n, np.int64); r4o[1:] = np.cumsum(nc.astype(np.int64) * k)[:-1]
        c4o = np.zeros(n, np.int64); c4o[1:] = np.cumsum(nr.astype(np.int64) * k)[:-1]
        costs = torch.from_numpy(pb.costs.copy()).pin_memory()
        probs = torch.zeros(int(sizes.sum()), dtype=torch.float64).pin_memory()
        r4c = torch.full((int(nc.astype(np.int64).sum()) * k,), -7, dtype=torch.int64).pin_memory()
        c4r = torch.full((int(nr.astype(np.int64).sum()) * k,), -7, dtype=torch.int64).pin_memory()
        gain = torch.zeros(n * k, dtype=torch.float64).pin_memory()
        found = torch.zeros(n, dtype=torch.int32).pin_memory()
        _lib.check(lib.pda_murty_batch_host(costs.data_ptr(), _p(pb.cost_off), _p(nr), _p(nc), n, k, 1, 42.0, 0, 0,
                                            r4c.data_ptr(), _p(r4o), c4r.data_ptr(), _p(c4o), gain.data_ptr(), found.data_ptr(),
                                            1, probs.data_ptr(), _p(poff), _p(nl), 0))
        got = (probs.numpy(), found.numpy(), r4c.numpy(), c4r.numpy(), gain.numpy())
    assert np.array_equal(got[1], want[1])
    nf = want[1]
    # only the first nFound hypotheses of a problem are defined
    sel_g = (np.arange(k)[None, :] < nf[:, None]).reshape(-1)
    assert np.array_equal(got[4][sel_g].view(np.int64), want[4][sel_g].view(np.int64))
    assert np.array_equal(got[2].reshape(n, k, 2)[np.arange(k)[None, :] < nf[:, None]], want[2].reshape(n, k, 2)[np.arange(k)[None, :] < nf[:, None]])
    assert np.array_equal(got[3].reshape(n, k, 5)[np.arange(k)[None, :] < nf[:, None]], want[3].reshape(n, k, 5)[np.arange(k)[None, :] < nf[:, None]])
    assert np.array_equal(got[0].view(np.int64), want[0].view(np.int64))
    if not pinned:
        # every problem reads the SAME matrix: the staged cost range is one matrix long
        one = synth.g1_dense(1, nL=3, nM=2, first=77)
        nr = np.full(n, 5, np.int32); nc = np.full(n, 2, np.int32); nl = np.full(n, 3, np.int32)
        off0 = np.zeros(n, np.int64)
        poff = np.arange(n, dtype=np.int64) * 8
        probs = np.zeros(n * 8); found = np.zeros(n, np.int32)
        _lib.check(lib.pda_murty_batch_host(_p(one.costs), _p(off0), _p(nr), _p(nc), n, k, 1, 42.0, 0, 0, None, None, None, None, None,
                                            _p(found), 1, _p(probs), _p(poff), _p(nl), 0))
        ref = _assignment_prob(one, k, None)[0]
        assert np.array_equal(probs.reshape(n, 8), np.broadcast_to(ref, (n, 8)))
