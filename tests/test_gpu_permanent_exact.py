"""The NW permanent kernel (permanent_kernel.cu) held to exact arithmetic at every size, walk variant and launch shape.

Inputs come from tests/perm_exact.py.  In its "exact" regime every NW term and every partial sum, in any summation
order, is an exact double, so the kernel must return perm_exact bit for bit; in its "wide" regime the products are
exact but the running sums round, the double-double's lo part carries the rounding errors exactly, and the kernel must
return the correctly rounded exact permanent.  Either way one missing, repeated or sign-flipped Gray step, a wrong
column in a register-cached step, a bad chunk boundary or a lost lo changes the result.  The tolerance rule:

* exact and wide regimes: equality (to the correctly rounded value of the exact rational);
* ones-padded rectangles, which leave both regimes: the rigorous bound perm_exact.nw_error_bound;
* dense U(0,1) input (no exact value affordable): identities between kernel results (Laplace expansion, permuted and
  transposed input) within the estimated NW rounding error of each side, perm_exact.nw_error_estimate, and, for
  n <= 20, the cancellation-free truth at 1e-12.
"""
from fractions import Fraction

import numpy as np
import pytest

import perm_exact as pe
from truth import perm_injective

pytestmark = pytest.mark.gpu

PDA_ERR_WORKSPACE = -4
MAX_DIM = 32


@pytest.fixture(scope="module")
def dev(gpu_api):
    import torch
    from probabilisticsemslam_b200._lib import lib
    assert torch.cuda.is_available()
    return torch, lib()


def _flat(mats):
    rows = np.asarray([m.shape[0] for m in mats], np.int32)
    cols = np.asarray([m.shape[1] for m in mats], np.int32)
    sizes = rows.astype(np.int64) * cols
    off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    flat = np.concatenate([np.asarray(m, np.float64).reshape(-1, order="F") for m in mats] + [np.zeros(1)])
    return flat, off, rows, cols


def device_batch(dev, mats, max_dim, ws=None, ws_bytes=None):
    """pda_permanent_batch on device buffers -> (rc, out, status).  Outputs start as NaN / -7 so unwritten ones show."""
    torch, L = dev
    flat, off, rows, cols = _flat(mats)
    d = torch.device("cuda", torch.cuda.current_device())
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(d)  # noqa: E731
    tm, to, tr, tc = t(flat), t(off), t(rows), t(cols)
    n = len(mats)
    out = torch.full((n,), float("nan"), dtype=torch.float64, device=d)
    st = torch.full((n,), -7, dtype=torch.int32, device=d)
    if ws is None:
        ws = torch.empty(int(ws_bytes if ws_bytes is not None else L.pda_permanent_workspace_bytes(n)), dtype=torch.uint8, device=d)
    rc = L.pda_permanent_batch(tm.data_ptr(), to.data_ptr(), tr.data_ptr(), tc.data_ptr(), n, max_dim, out.data_ptr(),
                               st.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, out.cpu().numpy(), st.cpu().numpy()


def device_range(dev, A, begin, end, ws_bytes=64 + 16 * 8192):
    """pda_permanent_range on device buffers -> (rc, hi, lo)."""
    torch, L = dev
    d = torch.device("cuda", torch.cuda.current_device())
    tA = torch.from_numpy(np.ascontiguousarray(np.asarray(A, np.float64).reshape(-1, order="F"))).to(d)
    part = torch.full((2,), float("nan"), dtype=torch.float64, device=d)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=d)
    rc = L.pda_permanent_range(tA.data_ptr(), A.shape[0], begin, end, part.data_ptr(), ws.data_ptr(), ws_bytes,
                               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    h, l = part.cpu().tolist()
    return rc, h, l


def exact_set(rng, n, count=2):
    """Signed and unsigned matrices of both regimes."""
    return [pe.exact_matrix(rng, n, signed=s, regime=r, rmax=3 if r == "exact" else 31)
            for r in ("exact", "wide") for s in (False, True) for _ in range(count)]


def want_of(mats):
    return np.array([pe.to_float(pe.perm_exact(m)) for m in mats])


def assert_exact(got, want, what=""):
    bad = np.flatnonzero(~(got == want))
    assert bad.size == 0, f"{what}: {bad.size} wrong, first at {bad[0]}: got {got[bad[0]]!r}, exact {want[bad[0]]!r}"


# ---- 1. every size through the host form ---------------------------------------------------------------------------
def test_host_form_every_size(gpu_api):
    """n = 1..32: the subset DP (n <= 10) and every NW tile 12..32, as one ragged batch, as one batch per size and as
    single calls (three different launch shapes per matrix)."""
    rng = np.random.default_rng(2024)
    per_n = {n: exact_set(rng, n) for n in range(1, MAX_DIM + 1)}
    want = {n: want_of(m) for n, m in per_n.items()}
    allm = [m for n in per_n for m in per_n[n]]
    got, st = gpu_api.permanent_batch(allm)
    assert not st.any()
    assert_exact(got, np.concatenate([want[n] for n in per_n]), "ragged batch")
    for n, mats in per_n.items():
        got, st = gpu_api.permanent_batch(mats)
        assert not st.any()
        assert_exact(got, want[n], f"batch n={n}")
        for i, m in enumerate(mats[::3]):
            got, st = gpu_api.permanent_batch([m])
            assert st[0] == 0
            assert_exact(got, want[n][::3][i:i + 1], f"single n={n}")


# ---- 2. every tile through the device form --------------------------------------------------------------------------
def test_device_form_every_tile(dev, gpu_api):
    """pda_permanent_batch with maxDim = n takes the NW tile of n for every n = 0..32 (tiles 2..32; chunk sizes that
    select the c01, c0 and general walks), and a ragged batch at maxDim = 32.  The host form, which sends n <= 10 to
    the subset DP, must give the same bits."""
    rng = np.random.default_rng(77)
    ragged, ragged_want = [], []
    for n in range(0, MAX_DIM + 1):
        mats = exact_set(rng, n) if n else [np.zeros((0, 0))]
        want = want_of(mats)
        for batch, w in ((mats, want), (mats[:1], want[:1]), (mats[-1:], want[-1:])):
            rc, got, st = device_batch(dev, batch, n)
            assert rc == 0 and not st.any()
            assert_exact(got, w, f"device n={n}")
        hgot, hst = gpu_api.permanent_batch(mats)
        assert not hst.any()
        assert_exact(hgot, want, f"host n={n}")
        ragged += mats[:2]
        ragged_want += list(want[:2])
    order = rng.permutation(len(ragged))
    rc, got, st = device_batch(dev, [ragged[i] for i in order], MAX_DIM)
    assert rc == 0 and not st.any()
    assert_exact(got, np.array(ragged_want)[order], "ragged device batch")


# ---- 3. shapes and status codes -------------------------------------------------------------------------------------
def _rect(rng, r, c, signed=True):
    """r x c integer matrix whose rows have odd absolute sums <= 3 over the long side."""
    short, long_ = min(r, c), max(r, c)
    A = np.zeros((short, long_))
    for j in range(short):
        for k, v in pe._row(rng, int(rng.choice([1, 3])), int(rng.integers(long_)), long_, signed).items():
            A[j, k] = v
    return A if r <= c else A.T


def test_shapes_and_status(dev, gpu_api):
    rng = np.random.default_rng(5)
    # empty sides: permanentExact of an empty product is 1 (nwPerm.cpp:261-264, and k! / k! for 0 x k)
    empties = [np.zeros((0, 0)), np.zeros((0, 1)), np.zeros((0, 5)), np.zeros((3, 0)), np.zeros((0, 32)), np.zeros((32, 0))]
    got, st = gpu_api.permanent_batch(empties)
    assert not st.any() and np.all(got == 1.0)
    for m in empties:
        rc, got, st = device_batch(dev, [m], max(m.shape))
        assert rc == 0 and st[0] == 0
        assert abs(got[0] - 1.0) <= pe.nw_error_bound(m, 1), m.shape
    got, st = gpu_api.permanent_batch([np.array([[2.5]]), np.array([[-3.0]])])
    assert not st.any() and list(got) == [2.5, -3.0]
    rc, got, st = device_batch(dev, [np.array([[2.5]]), np.array([[-3.0]])], 1)
    assert rc == 0 and not st.any() and list(got) == [2.5, -3.0]

    # rectangular.  Short side <= 10 goes to the subset DP in the host form, whose integer arithmetic is exact here;
    # the ones-padded NW walk (short side >= 11, and everything in the device form) is held to the rigorous bound
    rects = [_rect(rng, 10, 32), _rect(rng, 32, 10), _rect(rng, 12, 20), _rect(rng, 20, 12), _rect(rng, 11, 32),
             _rect(rng, 32, 11, signed=False), _rect(rng, 3, 7)]
    exact = [pe.perm_exact(m) for m in rects]
    got, st = gpu_api.permanent_batch(rects)
    assert not st.any()
    rc, dgot, dst = device_batch(dev, rects, MAX_DIM)
    assert rc == 0 and not dst.any()
    for m, e, g, dg in zip(rects, exact, got, dgot):
        if min(m.shape) <= 10:
            assert g == pe.to_float(e), (m.shape, g, e)
        else:
            assert abs(g - e) <= pe.nw_error_bound(m, e), (m.shape, g, e)
        assert abs(dg - e) <= pe.nw_error_bound(m, e), (m.shape, dg, e)

    # status 1 where the reference throws (dimension > 32), in both forms
    big = [np.ones((33, 33)), np.ones((5, 40)), np.ones((2, 2))]
    got, st = gpu_api.permanent_batch(big)
    assert list(st) == [1, 1, 0] and got[2] == 2.0
    rc, got, st = device_batch(dev, big, 40)
    assert rc == 0 and list(st) == [1, 1, 0] and got[2] == 2.0

    # status 2: a matrix above the call's maxDim is reported, not silently returned as 0
    mats = [pe.exact_matrix(rng, 3), pe.exact_matrix(rng, 7), np.ones((5, 2)), np.zeros((0, 6)), pe.exact_matrix(rng, 5)]
    rc, got, st = device_batch(dev, mats, 5)
    assert rc == 0 and list(st) == [0, 2, 0, 2, 0]
    assert got[0] == pe.perm_exact(mats[0]) and got[2] == 20.0 and got[4] == pe.perm_exact(mats[4])
    assert got[1] == 0.0 and got[3] == 0.0
    rc, got, st = device_batch(dev, [np.zeros((0, 0)), np.ones((1, 1)), np.ones((24, 24))], 0)
    assert rc == 0 and list(st) == [0, 2, 2] and got[0] == 1.0
    mats = [pe.exact_matrix(rng, 30), pe.exact_matrix(rng, 20)]
    rc, got, st = device_batch(dev, mats, 24)
    assert rc == 0 and list(st) == [2, 0] and got[0] == 0.0 and got[1] == pe.perm_exact(mats[1])


# ---- 4. range mode --------------------------------------------------------------------------------------------------
RANGE_NS = (2, 3, 11, 16, 17, 24, 28, 31, 32)


def _ranges(n, rng):
    T = 1 << (n - 1)
    out = {(0, 1), (T - 1, T), (0, T) if n <= 17 else (0, 1 << 16)}
    for start in {1, 3, (T // 3) | 1, 12345 % T | 1}:
        for ln in (1, 2, 3, 5, 31, 33, 1000, 65537):
            if start < T:
                out.add((start, min(T, start + ln)))
    for k in range(max(1, n - 4), n - 1):  # straddle large powers of two
        out.add((max(0, (1 << k) - 1001), min(T, (1 << k) + 999)))
        out.add(((1 << k) - 1, (1 << k) + 1))
    if n == 32:
        out |= {((1 << 31) - 65537, 1 << 31), ((1 << 31) - 3, 1 << 31), ((1 << 31) - 40000 - 1, (1 << 31) - 7)}
    return sorted(out)


@pytest.mark.parametrize("n", RANGE_NS)
def test_range_exact(dev, gpu_api, n):
    """hi + lo of pda_permanent_range (device form, three workspace sizes) and pda_permanent_range_host equal the exact
    partial sum as rationals: single indices, odd / unaligned starts of many lengths, ranges across large powers of two
    and, at n = 32, starts near 2^31."""
    rng = np.random.default_rng(1000 + n)
    for regime in ("exact", "wide"):
        A = pe.exact_matrix(rng, n, signed=True, regime=regime, rmax=3 if regime == "exact" else 31)
        for b, e in _ranges(n, rng):
            want = pe.nw_range_exact(A, b, e)[0]
            h, l = gpu_api.permanent_range(A, b, e)
            assert Fraction(h) + Fraction(l) == want, ("host", regime, b, e)
            for ws in (64 + 16 * 8192, 64 + 16 * 3, 64 + 16):  # the last two cap ctasPerMat at 3 and 1
                rc, h, l = device_range(dev, A, b, e, ws)
                assert rc == 0 and Fraction(h) + Fraction(l) == want, ("device", regime, b, e, ws)
    rc, _, _ = device_range(dev, A, 0, 1 << (n - 1), 64 + 15)
    assert rc == PDA_ERR_WORKSPACE


def test_range_pieces_add_up_n28(dev):
    """Bench config 5: shard.gray_range pieces for world = 1..8 through PermanentRangePlan (its 32 KB workspace)."""
    import torch
    from probabilisticsemslam_b200 import device, shard
    rng = np.random.default_rng(28)
    n = 28
    for regime in ("exact", "wide"):
        A = pe.exact_matrix(rng, n, signed=True, regime=regime, rmax=3 if regime == "exact" else 31)
        exact = pe.perm_exact(A)
        for world in range(1, 9):
            parts = []
            for r in range(world):
                b, e = shard.gray_range(n, world, r)
                if e > b:
                    plan = device.PermanentRangePlan(A, b, e)
                    plan.run()
                    torch.cuda.synchronize()
                    parts.append(plan.partial.cpu().numpy().copy())
                else:
                    parts.append(np.zeros(2))
            total = sum(Fraction(float(h)) + Fraction(float(l)) for h, l in parts)
            assert pe.nw_factor(n) * total == exact, (regime, world)
            assert shard.combine_partials(np.array(parts), n) == pe.to_float(exact), (regime, world)


# ---- 5. launch plumbing ---------------------------------------------------------------------------------------------
def _perm3(M):
    """Exact permanents of (N, 3, 3) small-integer matrices."""
    a = M.astype(np.int64)
    return (a[:, 0, 0] * (a[:, 1, 1] * a[:, 2, 2] + a[:, 1, 2] * a[:, 2, 1])
            + a[:, 0, 1] * (a[:, 1, 0] * a[:, 2, 2] + a[:, 1, 2] * a[:, 2, 0])
            + a[:, 0, 2] * (a[:, 1, 0] * a[:, 2, 1] + a[:, 1, 1] * a[:, 2, 0]))


def test_sliced_device_batch(dev):
    """More than 65535 * 8 3x3 matrices in one call: the batch is cut into launches of 65535 CTAs of eight; every
    result, on both sides of each slice boundary, is the exact permanent of its own matrix."""
    torch, L = dev
    per = 65535 * 8
    N = 2 * per + 77
    rng = np.random.default_rng(3)
    M = rng.integers(-4, 5, size=(N, 3, 3))
    want = _perm3(M).astype(np.float64)
    d = torch.device("cuda", torch.cuda.current_device())
    mats = torch.from_numpy(np.ascontiguousarray(M.transpose(0, 2, 1).reshape(-1).astype(np.float64))).to(d)
    off = torch.arange(N, dtype=torch.int64, device=d) * 9
    dims = torch.full((N,), 3, dtype=torch.int32, device=d)
    out = torch.full((N,), float("nan"), dtype=torch.float64, device=d)
    st = torch.full((N,), -7, dtype=torch.int32, device=d)
    ws = torch.empty(int(L.pda_permanent_workspace_bytes(N)), dtype=torch.uint8, device=d)
    rc = L.pda_permanent_batch(mats.data_ptr(), off.data_ptr(), dims.data_ptr(), dims.data_ptr(), N, 3, out.data_ptr(),
                               st.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0
    got = out.cpu().numpy()
    assert not st.cpu().numpy().any()
    for i in (0, per - 1, per, 2 * per - 1, 2 * per, N - 1):
        assert got[i] == want[i], i
    assert_exact(got, want, "sliced batch")


def test_workspace_reuse_and_limits(dev):
    """Two different multi-CTA batches back to back on one workspace and stream (the fused arrival counters are reset
    by the finishing CTA) give the bits of a fresh workspace; a workspace just big enough for one CTA per matrix is
    still exact, one byte less is PDA_ERR_WORKSPACE; repeated calls are bit-identical."""
    torch, L = dev
    rng = np.random.default_rng(9)
    b1 = [pe.exact_matrix(rng, 24, signed=True, regime="wide", rmax=31) for _ in range(3)]
    b2 = [pe.exact_matrix(rng, 22, signed=s, regime="wide", rmax=31) for s in (False, True, True, False, True)]
    w1, w2 = want_of(b1), want_of(b2)
    d = torch.device("cuda", torch.cuda.current_device())
    ws = torch.empty(int(L.pda_permanent_workspace_bytes(5)), dtype=torch.uint8, device=d)
    for _ in range(2):
        for b, w, nd in ((b1, w1, 24), (b2, w2, 22)):
            rc, got, st = device_batch(dev, b, nd, ws=ws)
            assert rc == 0 and not st.any()
            assert_exact(got, w, f"reused workspace n={nd}")
            rc, fresh, _ = device_batch(dev, b, nd)
            assert np.array_equal(got.view(np.int64), fresh.view(np.int64))
    n_m = len(b1)
    need = (n_m * 4 + 15) // 16 * 16 + 16 * n_m  # arrival counters + one double-double partial per matrix
    rc, got, st = device_batch(dev, b1, 24, ws_bytes=need)
    assert rc == 0 and not st.any()
    assert_exact(got, w1, "one CTA per matrix")
    rc, _, _ = device_batch(dev, b1, 24, ws_bytes=need - 1)
    assert rc == PDA_ERR_WORKSPACE
    rc, got, st = device_batch(dev, b1, 24, ws_bytes=need + 16 * n_m * 5)  # a few CTAs per matrix
    assert rc == 0 and not st.any()
    assert_exact(got, w1, "workspace-limited CTAs per matrix")
    # dense input: the fixed-order reduction makes every call give the same bits
    D = [np.random.default_rng(s).random((24, 24)) for s in range(3)]
    runs = [device_batch(dev, D, 24)[1] for _ in range(3)]
    assert all(np.array_equal(runs[0].view(np.int64), r.view(np.int64)) for r in runs[1:])


# ---- 6. dense real input at the large tiles -------------------------------------------------------------------------
def _rel(a, b):
    return abs(a - b) / abs(b)


def test_dense_laplace_and_invariance(dev):
    """U(0,1), n = 23..32: perm(A) = sum_k a[r,k] perm(minor_k) links tile n to tile n - 1 (non-negative terms, no
    cancellation in the check itself); row / column permutations and the transpose walk in different orders.  The NW
    sum cancels on this input, so each side is allowed its estimated error (perm_exact.nw_error_estimate)."""
    import math
    rng = np.random.default_rng(2323)
    est = np.random.default_rng(1)
    for n in range(23, MAX_DIM + 1):
        A = rng.random((n, n))
        r = int(rng.integers(n))
        P, Q = rng.permutation(n), rng.permutation(n)
        variants = [A, A[P][:, Q], A.T]
        rc, whole, st = device_batch(dev, variants, n)
        assert rc == 0 and not st.any()
        minors = [np.delete(np.delete(A, r, axis=0), k, axis=1) for k in range(n)]
        rc, pm, st = device_batch(dev, minors, n - 1)
        assert rc == 0 and not st.any()
        lap = math.fsum(A[r, k] * pm[k] for k in range(n))
        err = [pe.nw_error_estimate(v, est) for v in variants]
        lap_err = math.fsum(A[r, k] * pe.nw_error_estimate(minors[k], est) for k in range(n))
        assert abs(whole[0] - lap) <= err[0] + lap_err, (n, whole[0], lap, err[0] + lap_err)
        for v in (1, 2):
            assert abs(whole[v] - whole[0]) <= err[v] + err[0], (n, v, whole, err)
        assert _rel(whole[0], lap) <= 1e-9  # and never worse than the rest of the suite's tolerance


def test_dense_against_truth(dev, gpu_api):
    """U(0,1), n <= 20, against the cancellation-free DP of truth.py, through both forms."""
    rng = np.random.default_rng(1212)
    for n in (11, 12, 15, 16, 19, 20):
        mats = [rng.random((n, n)) for _ in range(2)]
        truth = [perm_injective(m) for m in mats]
        got, st = gpu_api.permanent_batch(mats)
        assert not st.any()
        rc, dgot, dst = device_batch(dev, mats, n)
        assert rc == 0 and not dst.any()
        for g, dg, t in zip(got, dgot, truth):
            assert _rel(g, t) <= 1e-12 and _rel(dg, t) <= 1e-12, (n, g, dg, t)
