"""Both transports of the single-device *_host entries (HostIO, pda_host_stage.h): a call whose declared arrays total at
most PDA_PACKED_LIMIT (8 MB) moves them with one pinned copy each way, a larger one copies each array straight from and
to the caller's memory -- except, for the k-best entries, cost matrices and weight tables in page-locked memory this
device can address, which the kernel uses in place.  Every entry runs once on each side of that limit (the k-best ones
with pageable, torch-pinned and pda_host_alloc buffers), and its results -- statuses and counts included -- must be
bit-identical to its device-pointer form run on the same inputs from CUDA tensors (asgnBB, which has no device-pointer
form, against the CPU oracle)."""
from __future__ import annotations

import numpy as np
import pytest

from helpers import bits
from probabilisticsemslam_b200 import synth

LIMIT = 8 << 20   # PDA_PACKED_LIMIT
SIDES = [pytest.param(False, id="packed"), pytest.param(True, id="per-array")]


def _side(arrays, large):
    """Asserts that the staged arrays of a call lie clearly on the chosen side of the limit."""
    nbytes = sum(int(a.nbytes) for a in arrays if a is not None)
    assert (nbytes > 1.2 * LIMIT) if large else (nbytes < LIMIT // 2), nbytes


def _prefix(sizes):
    off = np.zeros(len(sizes), np.int64)
    off[1:] = np.cumsum(np.asarray(sizes, np.int64))[:-1]
    return off


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _lib():
    from probabilisticsemslam_b200 import _lib
    return _lib


def _call(rc):
    _lib().check(rc)


def _same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: {got.shape} != {want.shape}"
    if got.dtype == np.float64:
        got, want = bits(got), bits(want)
    np.testing.assert_array_equal(got, want, err_msg=what)


def _problems(large, first):
    return synth.g1_dense(8000 if large else 40, first=first)


# ---- LAP ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_lap(gpu_api, large):
    import torch
    pb = _problems(large, 100)
    n, nr, nc = len(pb), pb.num_row, pb.nM.astype(np.int32)
    ng = np.maximum(nc - 1, 0).astype(np.int32)
    host = gpu_api.lap_batch(pb, make_safe=True, num_col4gain=ng)
    _side([pb.costs, pb.cost_off, nr, nc, ng, host["row_off"], host["col_off"]] +
          [host[k] for k in ("col4row", "row4col", "u", "v", "forbidden", "gain", "feasible")], large)
    R, C = int(nr.sum()), int(nc.sum())
    out = dict(col4row=torch.zeros(R, dtype=torch.int64, device="cuda"), row4col=torch.zeros(C, dtype=torch.int64, device="cuda"),
               u=torch.zeros(C, dtype=torch.float64, device="cuda"), v=torch.zeros(R, dtype=torch.float64, device="cuda"),
               forbidden=torch.zeros(R, dtype=torch.uint8, device="cuda"), gain=torch.zeros(n, dtype=torch.float64, device="cuda"),
               feasible=torch.zeros(n, dtype=torch.int32, device="cuda"))
    ins = [_t(a) for a in (pb.costs, pb.cost_off, nr, nc, ng, host["row_off"], host["col_off"])]
    o = out
    _call(_lib().lib().pda_lap_batch(*[x.data_ptr() for x in ins[:5]], n, int(nr.max()), int(nc.max()), 1, 0,
                                     ins[5].data_ptr(), ins[6].data_ptr(), o["col4row"].data_ptr(), o["row4col"].data_ptr(),
                                     o["u"].data_ptr(), o["v"].data_ptr(), o["forbidden"].data_ptr(), o["gain"].data_ptr(),
                                     o["feasible"].data_ptr(), None))
    for k, t in out.items():
        _same(host[k], _np(t), k)


# ---- conditionCosts -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_condition_costs(gpu_api, large):
    import torch
    pb = synth.g2_gated(8000 if large else 40, first=200)
    n, nr, nc = len(pb), pb.num_row, pb.nM.astype(np.int32)
    row_off = _prefix(nr)
    out, idx, good = np.zeros_like(pb.costs), np.zeros(int(nr.sum()), np.int64), np.full(n, -7, np.int32)
    _side([pb.costs, pb.cost_off, nr, nc, row_off, out, idx, good], large)
    lib = _lib().lib()
    _call(lib.pda_condition_costs_batch_host(pb.costs.ctypes.data, pb.cost_off.ctypes.data, nr.ctypes.data, nc.ctypes.data, n,
                                             row_off.ctypes.data, out.ctypes.data, idx.ctypes.data, good.ctypes.data, 0))
    ins = [_t(a) for a in (pb.costs, pb.cost_off, nr, nc, row_off)]
    d_out, d_idx = torch.zeros_like(ins[0]), torch.zeros(idx.size, dtype=torch.int64, device="cuda")
    d_good = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    _call(lib.pda_condition_costs_batch(*[x.data_ptr() for x in ins[:4]], n, ins[4].data_ptr(), d_out.data_ptr(),
                                        d_idx.data_ptr(), d_good.data_ptr(), None))
    d_out, d_idx, d_good = _np(d_out), _np(d_idx), _np(d_good)
    _same(good, d_good, "goodRows")
    for p in range(n):  # only what the kernel writes: goodRows rows of each problem
        g, o, r = int(good[p]), int(pb.cost_off[p]), int(row_off[p])
        _same(out[o:o + g * int(nc[p])], d_out[o:o + g * int(nc[p])], f"costs of problem {p}")
        _same(idx[r:r + g], d_idx[r:r + g], f"rowIdx of problem {p}")


# ---- toProbs, in place ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_to_probs_in_place(gpu_api, large):
    rng = np.random.default_rng(7)
    lens = rng.integers(1, 20000 if large else 200, 200).astype(np.int64)
    off = _prefix(lens)
    vals = 60.0 * rng.random(int(lens.sum()))
    vals[rng.choice(vals.size, 50, replace=False)] = np.inf
    _side([vals, off, lens], large)
    host = vals.copy()
    lib = _lib().lib()
    _call(lib.pda_to_probs_batch_host(host.ctypes.data, off.ctypes.data, lens.ctypes.data, len(lens), 0))
    dv, do, dl = _t(vals), _t(off), _t(lens)
    _call(lib.pda_to_probs_batch(dv.data_ptr(), do.data_ptr(), dl.data_ptr(), len(lens), None))
    _same(host, _np(dv), "values")
    assert not np.array_equal(bits(host), bits(vals))


# ---- quadric covariances and cost matrices --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_quadric_covs(gpu_api, large):
    import torch
    n = 100_000 if large else 100
    q = np.random.default_rng(3).random(n * 16)
    covs = np.zeros(n * 9)
    _side([q, covs], large)
    lib = _lib().lib()
    _call(lib.pda_quadric_covs_batch_host(q.ctypes.data, n, covs.ctypes.data, 0))
    dq, dc = _t(q), torch.zeros(n * 9, dtype=torch.float64, device="cuda")
    _call(lib.pda_quadric_covs_batch(dq.data_ptr(), n, dc.data_ptr(), None))
    _same(covs, _np(dc), "covariances")


def _moments(large, first):
    from probabilisticsemslam_b200 import api
    packed = api._pack_moments(synth.quadric_frames(3000 if large else 20, first=first))
    nL, nM = np.diff(packed[2]), np.diff(packed[5])
    return packed, nL, nM


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_quadric_cost(gpu_api, large):
    import torch
    packed, nL, nM = _moments(large, 300)
    n = len(nL)
    cost_off = _prefix((nL + nM) * nM)
    costs = np.zeros(int(((nL + nM) * nM).sum()))
    _side(list(packed) + [cost_off, costs], large)
    lib = _lib().lib()
    _call(lib.pda_quadric_cost_batch_host(*[a.ctypes.data for a in packed], n, 10.0, costs.ctypes.data, 0))
    d = [_t(a) for a in packed]
    dc, doff = torch.zeros(costs.size, dtype=torch.float64, device="cuda"), _t(cost_off)
    _call(lib.pda_quadric_cost_batch(*[x.data_ptr() for x in d], n, 10.0, dc.data_ptr(), doff.data_ptr(), None, None, None))
    _same(costs, _np(dc), "costs")


@pytest.mark.gpu
@pytest.mark.parametrize("perm", [False, True], ids=["k50", "usePerm"])
@pytest.mark.parametrize("large", SIDES)
def test_association_from_moments(gpu_api, large, perm):
    packed, nL, nM = _moments(large, 400)
    n = len(nL)
    cells = nM * (nL + 1)
    probs, status = np.full(int(cells.sum()), 7.5), np.full(n, -7, np.int32)
    _side(list(packed) + [probs, status, _prefix(cells), _prefix(cells), _prefix(nL + nM)], large)
    lib = _lib().lib()
    if perm:
        _call(lib.pda_association_perm_from_moments_batch_host(*[a.ctypes.data for a in packed], n, 10.0, probs.ctypes.data,
                                                               status.ctypes.data, 0))
    else:
        _call(lib.pda_association_from_moments_batch_host(*[a.ctypes.data for a in packed], n, 10.0, 50, probs.ctypes.data, 0))
    d = [_t(a) for a in packed]
    max_nL, max_nM = int(nL.max()), int(nM.max())
    if perm:
        got = gpu_api.association_perm_from_moments_batch_device(*d, max_nL, max_nM, 10.0)
    else:
        got = gpu_api.association_from_moments_batch_device(*d, max_nL, max_nM, 10.0, 50)
    d_probs, d_off, d_status = _np(got[0]), _np(got[1]), _np(got[2])
    _same(d_off[:n], _prefix(cells), "table offsets")
    _same(probs, d_probs[:probs.size], "tables")
    if perm:
        _same(status, d_status[:n], "status")


# ---- the association pipelines from cost matrices -------------------------------------------------------------------------
def _association(large, perm):
    import torch
    pb = synth.g1_dense(4000 if large else 40, first=500)
    n, nL, nM = len(pb), pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    cells = nM.astype(np.int64) * (nL + 1)
    rows = (nL + nM).astype(np.int64)
    prob_off, row_off = _prefix(cells), _prefix(rows)
    probs, status = np.full(int(cells.sum()), 7.5), np.full(n, -7, np.int32)
    _side([pb.costs, pb.cost_off, nL, nM, prob_off, row_off, probs] + ([status] if perm else []), large)
    lib = _lib().lib()
    host_in = [pb.costs.ctypes.data, pb.cost_off.ctypes.data, nL.ctypes.data, nM.ctypes.data]
    d = [_t(a) for a in (pb.costs, pb.cost_off, nL, nM, row_off, prob_off)]
    d_probs = torch.full((probs.size,), 7.5, dtype=torch.float64, device="cuda")
    d_status = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    tot = (pb.costs.size, int(rows.sum()), probs.size)
    max_r, max_c = int(rows.max()), int(nM.max())
    if perm:
        _call(lib.pda_association_perm_probs_batch_host(*host_in, n, probs.ctypes.data, prob_off.ctypes.data,
                                                        status.ctypes.data, 0))
        ws_bytes = int(lib.pda_association_perm_workspace_bytes(n, *tot, max_r, max_c))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _call(lib.pda_association_perm_probs_batch(*[x.data_ptr() for x in d[:5]], n, *tot, max_r, max_c, d_probs.data_ptr(),
                                                   d[5].data_ptr(), d_status.data_ptr(), ws.data_ptr(), ws_bytes, None))
        _same(status, _np(d_status), "status")
    else:
        _call(lib.pda_association_probs_batch_host(*host_in, n, 40, probs.ctypes.data, prob_off.ctypes.data, 0))
        ws_bytes = int(lib.pda_association_workspace_bytes(n, *tot, 40, max_r, max_c))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _call(lib.pda_association_probs_batch(*[x.data_ptr() for x in d[:5]], n, *tot, max_r, max_c, 40, d_probs.data_ptr(),
                                              d[5].data_ptr(), None, ws.data_ptr(), ws_bytes, None))
    _same(probs, _np(d_probs), "tables")


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_association_probs(gpu_api, large):
    _association(large, perm=False)


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_association_perm_probs(gpu_api, large):
    _association(large, perm=True)


# ---- permanents ------------------------------------------------------------------------------------------------------------
def _mats(n, dims, seed):
    """n column-major matrices, (rows, cols) drawn from dims -> (flat, off, rows, cols)."""
    rng = np.random.default_rng(seed)
    shape = [dims[i] for i in rng.integers(0, len(dims), n)]
    rows = np.asarray([s[0] for s in shape], np.int32)
    cols = np.asarray([s[1] for s in shape], np.int32)
    sizes = rows.astype(np.int64) * cols
    return rng.random(int(sizes.sum())), _prefix(sizes), rows, cols


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_permanent_exact(gpu_api, large):
    import torch
    # square and above the subset programme's reach (PERM_DP_MAX = 10), where the host and device forms take the same route
    flat, off, rows, cols = _mats(9000 if large else 30, [(11, 11), (12, 12), (13, 13)], 11)
    n = len(rows)
    out, st = np.zeros(n), np.full(n, -7, np.int32)
    _side([flat, off, rows, cols, out, st], large)
    lib = _lib().lib()
    _call(lib.pda_permanent_batch_host(flat.ctypes.data, off.ctypes.data, rows.ctypes.data, cols.ctypes.data, n,
                                       out.ctypes.data, st.ctypes.data, 0))
    d = [_t(a) for a in (flat, off, rows, cols)]
    d_out, d_st = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.full((n,), -7, dtype=torch.int32, device="cuda")
    ws_bytes = int(lib.pda_permanent_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _call(lib.pda_permanent_batch(*[x.data_ptr() for x in d], n, int(max(rows.max(), cols.max())), d_out.data_ptr(),
                                  d_st.data_ptr(), ws.data_ptr(), ws_bytes, None))
    _same(out, _np(d_out), "permanents")
    _same(st, _np(d_st), "status")


@pytest.mark.gpu
def test_permanent_range(gpu_api):
    import torch
    n = 20
    A = np.random.default_rng(5).random(n * n)
    begin, end = 1 << 12, 1 << 18
    part = np.zeros(2)
    lib = _lib().lib()
    _call(lib.pda_permanent_range_host(A.ctypes.data, n, begin, end, part.ctypes.data, 0))
    ws_bytes = 64 + 16 * 8192
    dA, dp, ws = _t(A), torch.zeros(2, dtype=torch.float64, device="cuda"), torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _call(lib.pda_permanent_range(dA.data_ptr(), n, begin, end, dp.data_ptr(), ws.data_ptr(), ws_bytes, None))
    _same(part, _np(dp), "partial")


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_permanent_approx(gpu_api, large):
    import torch
    flat, off, rows, cols = _mats(25000 if large else 50, [(8, 8), (9, 6), (5, 5)], 12)
    n = len(rows)
    out, st = np.zeros(n), np.full(n, -7, np.int32)
    _side([flat, off, rows, cols, out, st], large)
    lib = _lib().lib()
    _call(lib.pda_permanent_approx_batch_host(flat.ctypes.data, off.ctypes.data, rows.ctypes.data, cols.ctypes.data, n, 20,
                                              1234, out.ctypes.data, st.ctypes.data, 0))
    d = [_t(a) for a in (flat, off, rows, cols)]
    d_out, d_st = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.full((n,), -7, dtype=torch.int32, device="cuda")
    _call(lib.pda_permanent_approx_batch(*[x.data_ptr() for x in d], n, 20, 1234, d_out.data_ptr(), d_st.data_ptr(), None))
    _same(out, _np(d_out), "estimates")
    _same(st, _np(d_st), "status")


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_conditioned_permanent(gpu_api, large):
    flat, off, rows, cols = _mats(25000 if large else 50, [(10, 6), (9, 9), (7, 3), (12, 4)], 13)
    n = len(rows)
    out, st = np.zeros(n), np.full(n, -7, np.int32)
    _side([flat, off, rows, cols, out, st], large)
    _call(_lib().lib().pda_conditioned_permanent_batch_host(flat.ctypes.data, off.ctypes.data, rows.ctypes.data,
                                                            cols.ctypes.data, n, 1, out.ctypes.data, st.ctypes.data, 0))
    d_out, d_st = gpu_api.conditioned_permanent_batch_device(*[_t(a) for a in (flat, off, rows, cols)],
                                                             int(max(rows.max(), cols.max())), 1)
    _same(out, _np(d_out), "permanents")
    _same(st, _np(d_st), "status")


@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_permanent_prob_with_gaps(gpu_api, large):
    """Tables three doubles apart: the gaps come back as zeros.  One host chunk holds at most 65 536 sub-permanents, and
    nM = 1 problems add none, so the large call is mostly such problems and still one chunk, as the device form is."""
    rng = np.random.default_rng(14)
    n = 30000 if large else 60
    nM = np.where(rng.random(n) < 0.99 if large else np.zeros(n, bool), 1, rng.integers(2, 6, n)).astype(np.int32)
    nL = rng.integers(10, 40, n).astype(np.int32)
    items = int((nM * (nL + 1))[nM > 1].sum())
    assert items <= 65536
    mats = [5.0 * rng.random((int(l + m), int(m))) for l, m in zip(nL, nM)]
    pb = synth.pack(mats, nL)
    cells = nM.astype(np.int64) * (nL + 1)
    prob_off = _prefix(cells + 3)
    total = int(prob_off[-1] + cells[-1])
    probs, st = np.full(total, 7.5), np.full(n, -7, np.int32)
    _side([pb.costs, pb.cost_off, nL, nM, prob_off, probs, st], large)
    _call(_lib().lib().pda_permanent_prob_batch_host(pb.costs.ctypes.data, pb.cost_off.ctypes.data, nL.ctypes.data,
                                                     nM.ctypes.data, n, 1, probs.ctypes.data, prob_off.ctypes.data,
                                                     st.ctypes.data, 0))
    import torch
    d_probs = torch.zeros(total, dtype=torch.float64, device="cuda")
    got = gpu_api.permanent_prob_batch_device(*[_t(a) for a in (pb.costs, pb.cost_off, nL, nM, prob_off)], items,
                                              int((nL + nM).max()), int(nM.max()), 1, probs=d_probs)
    _same(probs, _np(got[0]), "tables")
    _same(st, _np(got[1]), "status")
    gaps = np.ones(total, bool)
    for o, c in zip(prob_off, cells):
        gaps[o:o + c] = False
    assert gaps.sum() == 3 * (n - 1) and np.all(probs[gaps] == 0.0)


# ---- k-best enumeration (pda_murty_batch_host, pda_assignment_prob_ladder_batch_host) --------------------------------------
class _HostMemory:
    """Copies of host arrays in one kind of memory: pageable numpy, torch.pin_memory() (page-locked by this device's
    context) or pda_host_alloc (portable).  Beyond the limit the k-best entries use the last two in place."""

    def __init__(self, kind):
        self.kind, self.held, self.allocs = kind, [], []

    def __call__(self, a):
        import ctypes
        import torch
        a = np.ascontiguousarray(a)
        if self.kind == "pageable":
            return a.copy()
        if self.kind == "torch_pinned":
            t = torch.from_numpy(a.copy()).pin_memory()
            self.held.append(t)
            return t.numpy()
        p = _lib().lib().pda_host_alloc(max(a.nbytes, 8))
        assert p
        self.allocs.append(p)
        v = np.ctypeslib.as_array((ctypes.c_uint8 * a.nbytes).from_address(p)).view(a.dtype)
        v[:] = a
        return v

    def free(self):
        for p in self.allocs:
            _lib().lib().pda_host_free(p)


KINDS = ["pageable", "torch_pinned", "host_alloc"]


def _kbest_inputs(large):
    pb = _problems(large, 700)
    nr, nc, nL = pb.num_row, pb.nM.astype(np.int32), pb.nL.astype(np.int32)
    return pb, nr, nc, nL, nc.astype(np.int64) * (nL + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("large", SIDES)
def test_murty_lists_and_weights(gpu_api, large, kind):
    import torch
    from probabilisticsemslam_b200 import api
    k = 5
    pb, nr, nc, nL, cells = _kbest_inputs(large)
    n = len(pb)
    r4o, c4o, poff = _prefix(nc.astype(np.int64) * k), _prefix(nr.astype(np.int64) * k), _prefix(cells)
    lib = _lib().lib()
    mem = _HostMemory(kind)
    try:
        costs, off, hnr, hnc, hnl, hr4o, hc4o, hpoff = [mem(a) for a in (pb.costs, pb.cost_off, nr, nc, nL, r4o, c4o, poff)]
        r4c, c4r = mem(np.full(int(nc.sum()) * k, -7, np.int64)), mem(np.full(int(nr.sum()) * k, -7, np.int64))
        gain, found, probs = mem(np.zeros(n * k)), mem(np.full(n, -7, np.int32)), mem(np.full(int(cells.sum()), 7.5))
        _side([costs, off, hnr, hnc, hnl, hr4o, hc4o, hpoff, r4c, c4r, gain, found, probs], large)
        _call(lib.pda_murty_batch_host(costs.ctypes.data, off.ctypes.data, hnr.ctypes.data, hnc.ctypes.data, n, k,
                                       api.CUT_RELATIVE, 42.0, 0, 0, r4c.ctypes.data, hr4o.ctypes.data, c4r.ctypes.data,
                                       hc4o.ctypes.data, gain.ctypes.data, found.ctypes.data, api.WEIGHTS_GATED,
                                       probs.ctypes.data, hpoff.ctypes.data, hnl.ctypes.data, 0))
        got = [np.array(a) for a in (found, gain, r4c, c4r, probs)]
    finally:
        mem.free()
    d = [_t(a) for a in (pb.costs, pb.cost_off, nr, nc, r4o, c4o, poff, nL)]
    d_r4c = torch.full((got[2].size,), -7, dtype=torch.int64, device="cuda")
    d_c4r = torch.full((got[3].size,), -7, dtype=torch.int64, device="cuda")
    d_gain, d_found = torch.zeros(n * k, dtype=torch.float64, device="cuda"), torch.full((n,), -7, dtype=torch.int32, device="cuda")
    d_probs = torch.full((got[4].size,), 7.5, dtype=torch.float64, device="cuda")
    max_r, max_c = int(nr.max()), int(nc.max())
    ws_bytes = int(lib.pda_murty_workspace_bytes(n, k, max_r, max_c))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _call(lib.pda_murty_batch(*[x.data_ptr() for x in d[:4]], n, max_r, max_c, k, api.CUT_RELATIVE, 42.0, 0, 0,
                              d_r4c.data_ptr(), d[4].data_ptr(), d_c4r.data_ptr(), d[5].data_ptr(), d_gain.data_ptr(),
                              d_found.data_ptr(), api.WEIGHTS_GATED, d_probs.data_ptr(), d[6].data_ptr(), d[7].data_ptr(),
                              ws.data_ptr(), ws_bytes, None))
    want = [_np(t) for t in (d_found, d_gain, d_r4c, d_c4r, d_probs)]
    _same(got[0], want[0], "nFound")
    _same(got[4], want[4], "weight tables")
    assert want[0].min() >= 1
    for p in range(n):  # only the first nFound hypotheses of a problem are defined
        f = int(want[0][p])
        _same(got[1][p * k:p * k + f], want[1][p * k:p * k + f], f"gains of problem {p}")
        a, b = int(r4o[p]), int(r4o[p]) + f * int(nc[p])
        _same(got[2][a:b], want[2][a:b], f"row4col of problem {p}")
        a, b = int(c4o[p]), int(c4o[p]) + f * int(nr[p])
        _same(got[3][a:b], want[3][a:b], f"col4row of problem {p}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("large", SIDES)
def test_assignment_prob_ladder(gpu_api, large, kind):
    import torch
    ks = np.asarray([3, 1, 5], np.int32)
    nk = len(ks)
    pb, nr, nc, nL, cells = _kbest_inputs(large)
    n = len(pb)
    poff = _prefix(cells * nk)
    lib = _lib().lib()
    mem = _HostMemory(kind)
    try:
        costs, off, hnr, hnc, hnl, hpoff = [mem(a) for a in (pb.costs, pb.cost_off, nr, nc, nL, poff)]
        found, probs = mem(np.full(n * nk, -7, np.int32)), mem(np.full(int(cells.sum()) * nk, 7.5))
        _side([costs, off, hnr, hnc, hnl, hpoff, found, probs], large)
        _call(lib.pda_assignment_prob_ladder_batch_host(costs.ctypes.data, off.ctypes.data, hnr.ctypes.data, hnc.ctypes.data,
                                                        hnl.ctypes.data, n, ks.ctypes.data, nk, probs.ctypes.data,
                                                        hpoff.ctypes.data, found.ctypes.data, 0))
        got = [np.array(a) for a in (found, probs)]
    finally:
        mem.free()
    d = [_t(a) for a in (pb.costs, pb.cost_off, nr, nc, nL, poff)]
    d_found = torch.full((n * nk,), -7, dtype=torch.int32, device="cuda")
    d_probs = torch.full((got[1].size,), 7.5, dtype=torch.float64, device="cuda")
    max_r, max_c = int(nr.max()), int(nc.max())
    ws_bytes = int(lib.pda_murty_workspace_bytes(n, int(ks.max()), max_r, max_c))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _call(lib.pda_assignment_prob_ladder_batch(*[x.data_ptr() for x in d[:5]], n, max_r, max_c, ks.ctypes.data, nk,
                                               d_probs.data_ptr(), d[5].data_ptr(), d_found.data_ptr(), ws.data_ptr(),
                                               ws_bytes, None))
    _same(got[0], _np(d_found), "nFound")
    _same(got[1], _np(d_probs), "weight tables")


# ---- asgnBB ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("large", SIDES)
def test_asgn_bb_vs_oracle(gpu_api, oracle, large):
    """Frames with an empty side keep the -1 the assignment array arrives with through the in-and-out round trip."""
    n = 25000 if large else 40
    lefts, rights = synth.stereo_boxes(n, first=600)
    for f in range(0, n, 13):
        if f % 2:
            lefts[f] = np.zeros((0, 5))
        else:
            rights[f] = np.zeros((0, 5))
    _side([np.concatenate(lefts), np.concatenate(rights), np.zeros(n * 5, np.int64),
           np.zeros(sum(len(b) for b in lefts), np.int32)], large)
    got = gpu_api.asgn_bb_batch(lefts, rights, 0.2)
    empty = 0
    for f, (L, R) in enumerate(zip(lefts, rights)):
        _same(got[f], oracle.asgn_bb(L, R, 0.2)[:len(L)], f"frame {f}")
        if len(R) == 0 and len(L):
            assert np.all(got[f] == -1)
            empty += 1
    assert empty > 0
