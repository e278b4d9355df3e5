"""The plain LAP, cost conditioning, likelihood and stereo-box kernels at every shape they accept, not only the KITTI
one (about 30 landmarks and 3-8 detections) that the golden files hold.

lap_kernel<R> (murty_kernel.cu) picks its launch from the batch's largest problem: R = 1 / 2 / 4 row slots per lane
and 4 / 2 / 1 warps per CTA, halved until the CTA's shared memory fits the opt-in limit.  This file restates that
choice, asserts that every case of one shape table lands in the regime it names, and runs the table -- in every
cost kind, minimising and maximising, alone, in one host batch and through the device-pointer form -- bit for bit
against the CPU oracle, which is itself first checked against scipy's independent solver.  condition_costs_kernel is
run across its 32-row ballot chunks and up to 128 columns, to_probs_kernel at lengths around one warp and far beyond,
both at the exact gate boundary; the box association at frames of up to 128 boxes, where the k = 1 Murty kernel
takes more than 32 rows and more than 16 columns.  Out-of-range input must come back as errors or as skipped problems
that leave their neighbours untouched."""
from __future__ import annotations

import math

import numpy as np
import pytest

from helpers import bits
from probabilisticsemslam_b200 import synth

GATE = 42.0               # assignment.cpp:9
MAX_DIM = 128             # PDA_MAX_DIM
B200_SMEM_OPTIN = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB); the GPU tests read the device


def _ru(x, m):
    return (x + m - 1) // m * m


# ---- the LAP launch, restated (launch_lap / launch_lap_r, murty_kernel.cu) --------------------------------------------
def lap_regime(max_rows, max_cols, optin):
    """(R, warps per CTA) of a batch whose largest problem is max_rows x max_cols; None past the shared memory."""
    R = (max_rows + 31) // 32
    if R == 3:
        R = 4
    c_cap = _ru(max_rows * max(max_cols, 1), 2)
    smem_per_warp = _ru(8 * (c_cap + 64 * R) + 192 * R, 16)
    if smem_per_warp > optin:
        return None
    wpc = 4
    while wpc > 1 and wpc * smem_per_warp > optin:
        wpc >>= 1
    return R, wpc


# (rows, cols, the regime the shape lands in alone); 65-96 rows round up to R = 4, 128 x 54 is the last with 4 warps
LAP_SHAPES = [
    (1, 1, (1, 4)), (2, 1, (1, 4)), (31, 31, (1, 4)), (32, 32, (1, 4)),
    (33, 1, (2, 4)), (33, 33, (2, 4)), (64, 64, (2, 4)),
    (65, 30, (4, 4)), (96, 60, (4, 4)), (128, 54, (4, 4)),
    (128, 55, (4, 2)), (90, 90, (4, 2)), (128, 110, (4, 2)),
    (128, 111, (4, 1)), (128, 128, (4, 1)),
    (1, 0, (1, 4)), (40, 0, (2, 4)), (128, 0, (4, 4)),
]
ALL_REGIMES = {(1, 4), (2, 4), (4, 4), (4, 2), (4, 1)}
KINDS = ["uniform", "ties", "decades", "gated", "infeasible"]


def lap_cost(rows, cols, kind, maximize):
    """A rows x cols cost matrix of one kind; gated entries are +inf when minimising and -inf when maximising."""
    rng = np.random.default_rng(1000003 * rows + 1009 * cols + 17 * KINDS.index(kind) + int(maximize))
    U = rng.random((rows, cols))
    gate = -np.inf if maximize else np.inf
    if kind == "uniform":
        return U
    if kind == "ties":
        return np.floor(U * 6.0)
    if kind == "decades":
        return 10.0 ** (12.0 * U - 6.0)
    if kind == "gated":
        return np.where(rng.random((rows, cols)) < 0.5, gate, U)
    C = U.copy()  # infeasible: one column with no admissible row
    if cols:
        C[:, cols // 2] = gate
    return C


def lap_cases(include_empty=True):
    for rows, cols, _ in LAP_SHAPES:
        if cols == 0 and not include_empty:
            continue
        for kind in KINDS:
            yield rows, cols, kind


def _shifted(C, maximize=False):
    """The safe matrix assign2D builds (shortestPathCPP.cpp:534-569): C - min, or max - C when maximising."""
    if C.size == 0:
        return C.copy(), 0.0
    d = C.max() if maximize else C.min()
    if not math.isfinite(d):  # an all-gated matrix: already as safe as it gets
        return (-C if maximize else C).copy(), d
    return ((-C + d) if maximize else (C - d)) + 0.0, d


# ---- CPU: the regime restatement ---------------------------------------------------------------------------------------
def test_every_lap_shape_lands_in_its_regime_at_b200_limit():
    for rows, cols, regime in LAP_SHAPES:
        assert lap_regime(rows, cols, B200_SMEM_OPTIN) == regime, (rows, cols)


def test_lap_table_reaches_every_regime():
    assert {regime for _, _, regime in LAP_SHAPES} >= ALL_REGIMES
    assert any(cols == 0 for _, cols, _ in LAP_SHAPES)
    # the two ends of the 4-warp range of a 128-row batch
    assert lap_regime(128, 54, B200_SMEM_OPTIN) == (4, 4) and lap_regime(128, 55, B200_SMEM_OPTIN) == (4, 2)
    assert lap_regime(128, 110, B200_SMEM_OPTIN) == (4, 2) and lap_regime(128, 111, B200_SMEM_OPTIN) == (4, 1)


# ---- CPU: the oracle against an independent solver ---------------------------------------------------------------------
def _scipy_total(C, maximize):
    """scipy's optimal total, or None where it finds the problem infeasible."""
    from scipy.optimize import linear_sum_assignment
    try:
        r, c = linear_sum_assignment(C, maximize=maximize)
    except ValueError:
        return None
    return math.fsum(C[r, c])


@pytest.mark.parametrize("maximize", [False, True])
def test_oracle_assign2d_matches_scipy(oracle, maximize):
    """Optimal totals to 1e-12, the same infeasible problems, and duals that certify optimality on the safe matrix."""
    checked = infeasible = 0
    for rows, cols, kind in lap_cases(include_empty=False):
        C = lap_cost(rows, cols, kind, maximize)
        what = f"{rows}x{cols} {kind} maximize={maximize}"
        ret, r4c, c4r, u, v, g = oracle.assign2d(C, maximize)
        want = _scipy_total(C, maximize)
        assert (ret == 1) == (want is not None), what
        if want is None:
            infeasible += 1
            continue
        cols_idx = np.arange(cols)
        assert sorted(r4c.tolist()) == sorted(set(r4c.tolist())) and np.all(c4r[r4c] == cols_idx), what
        assert abs(g - want) <= 1e-12 * abs(want) + 1e-300, f"{what}: oracle {g!r}, scipy {want!r}"
        S, _ = _shifted(C, maximize)
        reduced = S - u[None, :] - v[:, None]
        scale = max(1.0, float(np.max(np.abs(S[np.isfinite(S)]))))
        fin = np.isfinite(reduced)
        assert np.all(reduced[fin] >= -1e-9 * scale) and np.all(reduced[~fin] > 0), what
        assert np.all(np.abs(reduced[r4c, cols_idx]) <= 1e-9 * scale), what
        checked += 1
    assert checked + infeasible == 15 * len(KINDS) and checked >= 55 and infeasible >= 15


def test_oracle_shortest_path_matches_scipy(oracle):
    """shortestPathCPP on the safe matrix: the same assignment cost as scipy, gains over the first numCol4Gain columns."""
    for rows, cols, kind in lap_cases(include_empty=False):
        S, _ = _shifted(lap_cost(rows, cols, kind, False))
        want = _scipy_total(S, False)
        for ng in sorted({cols, cols - 1, 0}):
            ret, r4c, c4r, u, v, g, fb = oracle.shortest_path(S, ng)
            what = f"{rows}x{cols} {kind} numCol4Gain={ng}"
            assert (ret == 0) == (want is not None), what
            if want is None:
                continue
            assert abs(math.fsum(S[r4c, np.arange(cols)]) - want) <= 1e-12 * abs(want) + 1e-300, what
            assert bits([g])[0] == bits([float(sum(S[r4c[c], c] for c in range(ng)))])[0], what  # in column order
            assert fb.sum() == 1 and fb[r4c[0]] == 1, what


# ---- stereo boxes (shared by the CPU check of the oracle and the GPU tests) --------------------------------------------
BOX_TOTALS = (33, 64, 65, 100, 128)
NONASSIGN = (0.0, 0.2, 1.5)


def _box(x0, y0, w, h, off):
    return [x0, y0, x0 + w, y0 + h, off]


def box_frame(nL, nR, seed):
    """nL left and nR right boxes in a 1242 x 375 image: left boxes seen from right ones (disparity + jitter), some
    spurious; plus two identical right boxes competing for one left box, a pair that only touches, and right boxes
    whose x offset moves them out of the image."""
    rng = np.random.default_rng(seed)
    disp = 5.0 + 60.0 * rng.random()
    R, L = [], []
    for i in range(nR):
        u = rng.random(5)
        R.append(_box(1100.0 * u[0], 300.0 * u[1], 30.0 + 140.0 * u[2], 20.0 + 55.0 * u[3], disp * (0.95 + 0.1 * u[4])))
    for i in range(nL):
        u = rng.random(6)
        if i < nR and u[5] < 0.85:
            j = 6.0 * (u[:2] - 0.5)
            r = R[i]
            L.append([r[0] + disp + j[0], r[1] + j[1], r[2] + disp + j[0], r[3] + j[1], -r[4]])
        else:
            L.append(_box(1000.0 * u[0], 250.0 * u[1], 30.0 + 100.0 * u[2], 20.0 + 50.0 * u[3], -disp))
    if nR >= 2:
        R[1] = list(R[0])                     # identical right boxes: the tie order decides
    if nL >= 2 and nR >= 1:
        L[1] = list(L[0])                     # ... and two identical left boxes after them
    if nL >= 3 and nR >= 3:                   # touching: l == r in both IoU directions (exact integers)
        R[2] = [100.0, 50.0, 180.0, 90.0, 20.0]
        L[2] = [200.0, 50.0, 260.0, 90.0, -20.0]
    for i in range(3, nR, 7):
        R[i][4] = 1.0e4                       # shifted out of the image: IoU 0 seen from this box
    return np.asarray(L, np.float64).reshape(-1, 5), np.asarray(R, np.float64).reshape(-1, 5)


def box_frames():
    shapes = []
    for total in BOX_TOTALS:
        for nL in sorted({5, 17, total // 2, total - 5}):
            if 1 <= nL < total:
                shapes.append((nL, total - nL))
    shapes += [(0, 20), (20, 0), (0, 0), (3, 4)]
    return [box_frame(nL, nR, 4242 + i) for i, (nL, nR) in enumerate(shapes)]


def test_box_frames_cover_the_wide_shapes():
    frames = box_frames()
    totals = {len(L) + len(R) for L, R in frames if len(L) and len(R)}
    assert set(BOX_TOTALS) <= totals
    assert any(len(L) > 16 and len(R) for L, R in frames)
    assert any(len(L) == 0 for L, _ in frames) and any(len(R) == 0 for _, R in frames)


@pytest.mark.parametrize("nonassign", NONASSIGN)
def test_oracle_asgn_bb_matches_scipy(oracle, nonassign):
    """The pairing asgnBB picks scores what scipy's maximum scores on the same cost matrix (-inf made finite)."""
    from scipy.optimize import linear_sum_assignment
    for f, (L, R) in enumerate(box_frames()):
        got = oracle.asgn_bb(L, R, nonassign)
        if len(L) == 0 or len(R) == 0:
            assert np.all(got == -1)
            continue
        M = oracle.bb_cost_matrix(L, R, nonassign)
        nR = len(R)
        total = math.fsum(M[a, c] if a >= 0 else M[nR + c, c] for c, a in enumerate(got))
        F = np.where(np.isfinite(M), M, -1.0e9)
        r, c = linear_sum_assignment(F, maximize=True)
        want = math.fsum(F[r, c])
        assert abs(total - want) <= 1e-12 * max(1.0, abs(want)), f"frame {f} nonassign {nonassign}"
        if nonassign == 1.5:
            assert np.all(got == -1)  # an IoU never exceeds 1


# ---- GPU: the LAP kernel ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def optin():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _prefix(sizes):
    off = np.zeros(len(sizes), np.int64)
    off[1:] = np.cumsum(np.asarray(sizes, np.int64))[:-1]
    return off


def _split(r, mats):
    """Per problem (feasible, row4col, col4row, u, v, gain, forbidden) out of one batch's flat outputs."""
    out = []
    for p, C in enumerate(mats):
        nr, nc = C.shape
        ro, co = int(r["row_off"][p]), int(r["col_off"][p])
        out.append((int(r["feasible"][p]), r["row4col"][co:co + nc].copy(), r["col4row"][ro:ro + nr].copy(),
                    r["u"][co:co + nc].copy(), r["v"][ro:ro + nr].copy(), float(r["gain"][p]),
                    r["forbidden"][ro:ro + nr].copy()))
    return out


def _lap_host(api, mats, make_safe, maximize, ng=None):
    pb = synth.pack(mats, [C.shape[0] - C.shape[1] for C in mats])
    return _split(api.lap_batch(pb, make_safe=make_safe, maximize=maximize, num_col4gain=ng), mats)


def _lap_device(mats, make_safe, maximize, ng, max_rows, max_cols):
    """pda_lap_batch on torch tensors; outputs start as sentinels (-7, 7.5, 9) so that unwritten entries show."""
    import torch
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    nr = np.asarray([C.shape[0] for C in mats], np.int32)
    nc = np.asarray([C.shape[1] for C in mats], np.int32)
    pb = synth.pack(mats, nr - nc)
    row_off, col_off = _prefix(nr), _prefix(nc)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d = lambda x: None if x is None else x.data_ptr()
    costs = t(pb.costs if pb.costs.size else np.zeros(1))
    off, tnr, tnc, tro, tco = t(pb.cost_off), t(nr), t(nc), t(row_off), t(col_off)
    tng = None if ng is None else t(np.asarray(ng, np.int32))
    R, Cn, n = max(int(nr.sum()), 1), max(int(nc.sum()), 1), len(mats)
    c4r = torch.full((R,), -7, dtype=torch.int64, device="cuda")
    r4c = torch.full((Cn,), -7, dtype=torch.int64, device="cuda")
    u = torch.full((Cn,), 7.5, dtype=torch.float64, device="cuda")
    v = torch.full((R,), 7.5, dtype=torch.float64, device="cuda")
    fb = torch.full((R,), 9, dtype=torch.uint8, device="cuda")
    g = torch.full((n,), 7.5, dtype=torch.float64, device="cuda")
    fe = torch.full((n,), 9, dtype=torch.int32, device="cuda")
    rc = lib.pda_lap_batch(d(costs), d(off), d(tnr), d(tnc), d(tng), n, max_rows, max_cols, int(make_safe), int(maximize),
                           d(tro), d(tco), d(c4r), d(r4c), d(u), d(v), d(fb), d(g), d(fe), None)
    assert rc == 0, lib.pda_last_error()
    torch.cuda.synchronize()
    r = dict(col4row=c4r.cpu().numpy(), row4col=r4c.cpu().numpy(), u=u.cpu().numpy(), v=v.cpu().numpy(),
             forbidden=fb.cpu().numpy(), gain=g.cpu().numpy(), feasible=fe.cpu().numpy(), row_off=row_off, col_off=col_off)
    return _split(r, mats)


def _assert_same(got, want, what, forbidden=True):
    """Bit-identical LAP results: (feasible, row4col, col4row, u, v, gain[, forbidden])."""
    assert got[0] == want[0], f"{what}: feasible {got[0]} != {want[0]}"
    np.testing.assert_array_equal(got[1], want[1], err_msg=f"{what}: row4col")
    np.testing.assert_array_equal(got[2], want[2], err_msg=f"{what}: col4row")
    np.testing.assert_array_equal(bits(got[3]), bits(want[3]), err_msg=f"{what}: u bits")
    np.testing.assert_array_equal(bits(got[4]), bits(want[4]), err_msg=f"{what}: v bits")
    assert bits([got[5]])[0] == bits([want[5]])[0], f"{what}: gain {got[5]!r} != {want[5]!r}"
    if forbidden:
        np.testing.assert_array_equal(got[6], want[6], err_msg=f"{what}: forbidden")


def _empty_result(rows):
    """The n x 0 problem: feasible, gain +0.0, every row unassigned with dual 0, nothing forbidden."""
    return (1, np.zeros(0, np.int64), np.full(rows, -1, np.int64), np.zeros(0), np.zeros(rows), 0.0, np.zeros(rows, np.uint8))


def _sp_problems():
    """shortestPathCPP calls: (safe matrix, numCol4Gain, label)."""
    out = []
    for rows, cols, kind in lap_cases():
        S, _ = _shifted(lap_cost(rows, cols, kind, False))
        for ng in sorted({cols, cols - 1, 0}):
            if ng >= 0:
                out.append((S, ng, f"{rows}x{cols} {kind} numCol4Gain={ng}"))
    return out


def _a2d_problems(maximize):
    return [(lap_cost(rows, cols, kind, maximize), f"{rows}x{cols} {kind} maximize={maximize}")
            for rows, cols, kind in lap_cases()]


@pytest.mark.gpu
def test_lap_regimes_on_this_device(optin):
    for rows, cols, regime in LAP_SHAPES:
        assert lap_regime(rows, cols, optin) == regime, (rows, cols, optin)


@pytest.mark.gpu
@pytest.mark.parametrize("maximize", [False, True])
def test_assign2d_every_regime_vs_oracle(gpu_api, oracle, maximize):
    """assign2D alone, in one host batch and through the device-pointer form: the oracle's bits every time."""
    probs = _a2d_problems(maximize)
    mats = [C for C, _ in probs]
    alone = []
    for C, what in probs:
        ret, r4c, c4r, u, v, g = gpu_api.assign2D(C, maximize)
        got = (ret, r4c, c4r, u, v, g, None)
        if C.shape[1] == 0:
            _assert_same(got, _empty_result(C.shape[0]), what, forbidden=False)
        else:
            _assert_same(got, oracle.assign2d(C, maximize) + (None,), what, forbidden=False)
        alone.append(_lap_host(gpu_api, [C], True, maximize)[0])  # the same call, forbidden included
        _assert_same(alone[-1], got, f"{what} (again)", forbidden=False)
    batch = _lap_host(gpu_api, mats, True, maximize)
    dev = _lap_device(mats, True, maximize, None, MAX_DIM, MAX_DIM)
    for (C, what), a, b, c in zip(probs, alone, batch, dev):
        if C.shape[1] == 0:
            _assert_same(a, _empty_result(C.shape[0]), what)
        _assert_same(b, a, f"{what} (host batch)")
        _assert_same(c, a, f"{what} (device form)")
    assert sum(a[0] == 0 for a in alone) >= 15  # the infeasible kind, at least


@pytest.mark.gpu
def test_shortest_path_every_regime_vs_oracle(gpu_api, oracle):
    """shortestPathCPP on the oracle's safe matrix, numCol4Gain = numCol, numCol - 1 and 0; forbidden included."""
    probs = _sp_problems()
    alone = []
    for S, ng, what in probs:
        ret, r4c, c4r, u, v, g, fb = gpu_api.shortestPathCPP(S, ng)
        got = (1 - ret, r4c, c4r, u, v, g, fb)
        w = oracle.shortest_path(S, ng)
        _assert_same(got, (1 - w[0],) + w[1:], what)
        if S.shape[1] == 0:
            _assert_same(got, _empty_result(S.shape[0]), what)
        alone.append(got)
    mats = [S for S, _, _ in probs]
    ngs = [ng for _, ng, _ in probs]
    batch = _lap_host(gpu_api, mats, False, False, ngs)
    dev = _lap_device(mats, False, False, ngs, MAX_DIM, MAX_DIM)
    for (_, _, what), a, b, c in zip(probs, alone, batch, dev):
        _assert_same(b, a, f"{what} (host batch)")
        _assert_same(c, a, f"{what} (device form)")


@pytest.mark.gpu
def test_lap_small_problem_next_to_the_largest(gpu_api, oracle):
    """A 5 x 3 problem in the R = 4, one-warp-per-CTA launch a 128 x 128 neighbour forces."""
    small, big = lap_cost(5, 3, "uniform", False), lap_cost(128, 128, "ties", False)
    got = _lap_host(gpu_api, [small, big, small], True, False)
    for p, C in ((0, small), (1, big), (2, small)):
        _assert_same(got[p][:6] + (None,), oracle.assign2d(C) + (None,), f"problem {p}", forbidden=False)


@pytest.mark.gpu
def test_lap_empty_problem(gpu_api):
    """n x 0 is feasible with gain +0.0 (not NaN: the extremum of an empty matrix is +-inf), minimising and maximising."""
    for rows in (1, 33, 128):
        for maximize in (False, True):
            got = _lap_host(gpu_api, [np.zeros((rows, 0))], True, maximize)[0]
            _assert_same(got, _empty_result(rows), f"{rows}x0 maximize={maximize}")
            got = _lap_host(gpu_api, [np.zeros((rows, 0))], False, maximize, [0])[0]
            _assert_same(got, _empty_result(rows), f"{rows}x0 shortestPath")


@pytest.mark.gpu
def test_lap_device_form_skips_problems_beyond_the_declared_maxima(gpu_api):
    """Declared 40 x 10: a 50-row problem (inside the R = 2 slots) and a 70-row one (beyond them) get feasible = 0 and
    leave their outputs alone; their neighbours are bit-identical to a run without them."""
    good = [lap_cost(40, 10, "uniform", False), lap_cost(12, 7, "ties", False), lap_cost(33, 10, "gated", False)]
    bad = [lap_cost(50, 5, "uniform", False), lap_cost(70, 5, "uniform", False), lap_cost(20, 11, "uniform", False)]
    mixed = [good[0], bad[0], good[1], bad[1], good[2], bad[2]]
    ref = _lap_device(good, True, False, None, 40, 10)
    got = _lap_device(mixed, True, False, None, 40, 10)
    for i, p in enumerate((0, 2, 4)):
        _assert_same(got[p], ref[i], f"neighbour {p}")
    for p in (1, 3, 5):
        f, r4c, c4r, u, v, g, fb = got[p]
        assert f == 0 and g == 7.5, p
        assert np.all(r4c == -7) and np.all(c4r == -7) and np.all(u == 7.5) and np.all(v == 7.5) and np.all(fb == 9), p


@pytest.mark.gpu
def test_lap_host_form_rejects_malformed_problems(gpu_api):
    from probabilisticsemslam_b200 import _lib
    for mats in ([np.zeros((3, 4))], [np.zeros((5, 2)), np.zeros((0, 0))]):
        with pytest.raises(_lib.PdaError) as e:
            _lap_host(gpu_api, mats, True, False)
        assert e.value.code == -1 and "lap: problem" in str(e.value)


# ---- GPU: conditionCosts ---------------------------------------------------------------------------------------------
COND_ROWS = (1, 31, 32, 33, 63, 64, 65, 100, 128)
COND_COLS = (1, 8, 16, 64, 128)
COND_VARIANTS = ("plain", "edges", "neginf", "allinf")


def cond_cost(rows, cols, variant):
    """200 U (about a fifth of each column within the gate of its minimum), then per variant: rows 31/32 and 63/64
    gated everywhere (the row compaction carries its base across 32-row chunks), rows kept through one column only,
    an entry exactly at colMin + 42 (kept) and one just above (gated); a -inf entry; an all-+inf column."""
    rng = np.random.default_rng(7919 * rows + 31 * cols + COND_VARIANTS.index(variant))
    C = 200.0 * rng.random((rows, cols))
    if variant == "edges":
        big = C.min(axis=0) + 1000.0
        for r in (31, 32, 63, 64):
            if r < rows:
                C[r, :] = big
        m0 = C[:, 0].min() - 1.0
        C[0, 0] = m0  # row 0 holds the minimum of column 0
        edge = m0 + GATE
        for r, x in ((rows // 3, edge), (rows // 2, np.nextafter(edge, np.inf)), (rows - 1, m0 + 1.0)):
            if rows > 4 and r not in (31, 32, 63, 64):
                C[r, :] = big
                C[r, 0] = x  # kept (or not) through column 0 alone
        assert C[:, 0].min() == m0
    elif variant == "neginf":
        C[rows // 2, cols // 2] = -np.inf
    elif variant == "allinf":
        C[:, cols - 1] = np.inf
    return C


def cond_cases():
    for rows in COND_ROWS:
        for cols in COND_COLS:
            if cols <= rows:
                for variant in COND_VARIANTS:
                    yield rows, cols, variant


def _assert_cond_same(got, want, what):
    """Conditioned matrix and rowIdx bit for bit; where the result is NaN (inf - inf, -inf - -inf) only NaN-ness."""
    (gm, gi), (wm, wi) = got, want
    assert gm.shape == wm.shape, f"{what}: {gm.shape} != {wm.shape}"
    np.testing.assert_array_equal(gi, wi, err_msg=f"{what}: rowIdx")
    nan = np.isnan(wm)
    np.testing.assert_array_equal(np.isnan(gm), nan, err_msg=f"{what}: NaN pattern")
    np.testing.assert_array_equal(bits(gm[~nan]), bits(wm[~nan]), err_msg=f"{what}: bits")


@pytest.mark.gpu
def test_condition_costs_every_chunk_and_width_vs_oracle(gpu_api, oracle):
    cases = list(cond_cases())
    mats = [cond_cost(*c) for c in cases]
    want = [oracle.condition_costs(C) for C in mats]
    seen_nan = 0
    for c, C, w in zip(cases, mats, want):
        _assert_cond_same(gpu_api.conditionCosts(C), w, f"{c}")
        seen_nan += bool(np.isnan(w[0]).any())
        if c[2] == "edges" and c[0] > 4:
            kept = set(w[1].tolist())
            assert c[0] // 3 in kept and c[0] // 2 not in kept, c  # colMin + 42 kept, the next double gated
            assert not kept & {31, 32, 63, 64}, c
    assert seen_nan >= 20
    pb, maps = gpu_api.condition_costs_batch(synth.pack(mats, [C.shape[0] - C.shape[1] for C in mats]))
    for p, (c, w) in enumerate(zip(cases, want)):
        _assert_cond_same((pb.matrix(p), maps[p]), w, f"{c} (batch)")


def _condition_device(mats):
    """pda_condition_costs_batch on torch tensors; outputs start as sentinels."""
    import torch
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    pb = synth.pack(mats, [C.shape[0] - C.shape[1] for C in mats])
    nr, nc = pb.num_row, pb.nM.astype(np.int32)
    row_off = _prefix(nr)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    costs, off, tnr, tnc, tro = t(pb.costs), t(pb.cost_off), t(nr), t(nc), t(row_off)
    out = torch.full_like(costs, 7.5)
    idx = torch.full((int(nr.sum()),), -7, dtype=torch.int64, device="cuda")
    good = torch.full((len(mats),), -7, dtype=torch.int32, device="cuda")
    rc = lib.pda_condition_costs_batch(costs.data_ptr(), off.data_ptr(), tnr.data_ptr(), tnc.data_ptr(), len(mats),
                                       tro.data_ptr(), out.data_ptr(), idx.data_ptr(), good.data_ptr(), None)
    assert rc == 0, lib.pda_last_error()
    torch.cuda.synchronize()
    out, idx, good = out.cpu().numpy(), idx.cpu().numpy(), good.cpu().numpy()
    res = []
    for p, C in enumerate(mats):
        o, g, ro = int(pb.cost_off[p]), int(good[p]), int(row_off[p])
        res.append((g, out[o:o + C.size], idx[ro:ro + C.shape[0]]))
    return res


@pytest.mark.gpu
def test_condition_costs_device_form_skips_more_than_max_dim_columns(gpu_api, oracle):
    """A 140 x 130 problem would need more column minima than the kernel keeps: goodRows = 0, nothing written; its
    neighbours are bit-identical to a run without it."""
    good = [cond_cost(64, 16, "edges"), cond_cost(128, 128, "plain"), cond_cost(33, 8, "allinf")]
    big = np.random.default_rng(5).random((140, 130))
    ref = _condition_device(good)
    got = _condition_device([good[0], big, good[1], good[2]])
    assert got[1][0] == 0 and np.all(got[1][1] == 7.5) and np.all(got[1][2] == -7)
    for (g, out, idx), (rg, rout, ridx), C in zip([got[0], got[2], got[3]], ref, good):
        assert g == rg
        np.testing.assert_array_equal(bits(out[:g * C.shape[1]]), bits(rout[:rg * C.shape[1]]))
        np.testing.assert_array_equal(idx[:g], ridx[:rg])
        wm, wi = oracle.condition_costs(C)
        _assert_cond_same((out[:g * C.shape[1]].reshape((g, C.shape[1]), order="F"), idx[:g]), (wm, wi), "device form")


# ---- GPU: the association pipeline's bounds ----------------------------------------------------------------------------
def _association_device(pb, k, max_rows, max_cols, ws_bytes=None):
    """pda_association_probs_batch on torch tensors -> (rc, tables, nFound, workspace after the call); every output
    and the workspace start as sentinels."""
    import torch
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    rows = (nL + nM).astype(np.int64)
    cells = nM.astype(np.int64) * (nL.astype(np.int64) + 1)
    row_off, prob_off = _prefix(rows), _prefix(cells)
    tot_cost, tot_rows, tot_prob = int(pb.costs.size), int(rows.sum()), int(cells.sum())
    if ws_bytes is None:
        ws_bytes = int(lib.pda_association_workspace_bytes(n, tot_cost, tot_rows, tot_prob, k, max_rows, max_cols))
        assert ws_bytes > 0
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    costs, off, tl, tm, tro, tpo = t(pb.costs), t(pb.cost_off), t(nL), t(nM), t(row_off), t(prob_off)
    probs = torch.full((tot_prob,), 7.5, dtype=torch.float64, device="cuda")
    found = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    ws = torch.full((ws_bytes,), 0x5A, dtype=torch.uint8, device="cuda")
    rc = lib.pda_association_probs_batch(costs.data_ptr(), off.data_ptr(), tl.data_ptr(), tm.data_ptr(), tro.data_ptr(), n,
                                         tot_cost, tot_rows, tot_prob, max_rows, max_cols, k, probs.data_ptr(),
                                         tpo.data_ptr(), found.data_ptr(), ws.data_ptr(), ws_bytes, None)
    torch.cuda.synchronize()
    probs, found = probs.cpu().numpy(), found.cpu().numpy()
    tabs = [probs[prob_off[p]:prob_off[p] + cells[p]].reshape(int(nM[p]), int(nL[p]) + 1) for p in range(n)]
    return rc, tabs, found, ws.cpu().numpy()


def _assoc_batch(with_big):
    base = synth.g2_gated(6, first=4100)
    mats = [base.matrix(p) for p in range(len(base))]
    nls = [int(x) for x in base.nL]
    if with_big:
        rng = np.random.default_rng(11)
        max_rows, max_cols = int(max(base.num_row)), int(max(base.nM))
        # more rows than declared, which conditioning would bring under the bound (its last 12 rows are gated away),
        # then more columns than declared
        tall = 30.0 * rng.random((max_rows + 6, 4))
        tall[-12:, :] = 1000.0
        mats[2:2] = [tall, 30.0 * rng.random((max_rows, max_cols + 1))]
        nls[2:2] = [tall.shape[0] - 4, max_rows - max_cols - 1]
    return synth.pack(mats, nls), int(max(base.num_row)), int(max(base.nM))


@pytest.mark.gpu
def test_association_skips_problems_beyond_the_declared_bounds(gpu_api, oracle):
    k = 40
    ref_pb, max_rows, max_cols = _assoc_batch(False)
    pb, _, _ = _assoc_batch(True)
    rc, ref_tabs, ref_found, _ = _association_device(ref_pb, k, max_rows, max_cols)
    assert rc == 0
    rc, tabs, found, _ = _association_device(pb, k, max_rows, max_cols)
    assert rc == 0
    assert found[2] == -1 and found[3] == -1
    keep = [0, 1, 4, 5, 6, 7]
    np.testing.assert_array_equal(found[keep], ref_found)
    for i, p in enumerate(keep):
        np.testing.assert_array_equal(bits(tabs[p]), bits(ref_tabs[i]), err_msg=f"problem {p}")
        st, want = oracle.association_probs(pb.matrix(p), int(pb.nL[p]), k)
        assert st == 0
        np.testing.assert_allclose(tabs[p], want, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_association_rejects_bad_bounds_before_any_launch(gpu_api):
    from probabilisticsemslam_b200 import _lib
    pb, max_rows, max_cols = _assoc_batch(False)
    ws_bytes = int(_lib.lib().pda_association_workspace_bytes(len(pb), pb.costs.size, int(pb.num_row.sum()),
                                                              int((pb.nM * (pb.nL + 1)).sum()), 40, MAX_DIM, max_cols))
    for rows, cols, code in ((MAX_DIM + 1, max_cols, -3), (MAX_DIM + 40, MAX_DIM + 1, -3), (max_rows, 0, -1),
                             (max_rows, max_rows + 1, -1)):
        rc, tabs, found, ws = _association_device(pb, 40, rows, cols, ws_bytes=ws_bytes)
        assert rc == code, (rows, cols, rc)
        assert np.all(ws == 0x5A) and np.all(found == -7), (rows, cols)  # nothing ran
        assert all(np.all(t == 7.5) for t in tabs), (rows, cols)


# ---- GPU: toProbs ----------------------------------------------------------------------------------------------------
PROB_LENGTHS = (1, 31, 32, 33, 1000, 100_000)


def prob_vectors():
    out = []
    for n in PROB_LENGTHS:
        rng = np.random.default_rng(n)
        v = 3.0 + 60.0 * rng.random(n)
        if n >= 8:
            lo = v.min() - 1.5
            v[rng.choice(n, 4, replace=False)] = lo                     # equal minima
            i, j, q = rng.choice(np.flatnonzero(v != lo), 3, replace=False)
            v[i] = lo + GATE                                            # gated: the test is strict
            v[j] = np.nextafter(lo + GATE, -np.inf)                     # the largest double still inside
            v[q] = np.inf
        out.append(v)
    out += [np.array([np.inf, 5.0, np.inf]), np.full(3, np.inf), np.array([-np.inf, 1.0, 2.0]), np.array([7.0])]
    return out


def _probs_want(v):
    lo = v.min()
    keep = lo + GATE > v
    with np.errstate(invalid="ignore", over="ignore"):
        return keep, np.where(keep, np.exp(lo - v), 0.0)


@pytest.mark.gpu
def test_to_probs_every_length_and_the_gate_vs_oracle(gpu_api, oracle):
    from probabilisticsemslam_b200 import _lib
    vecs = prob_vectors()
    lens = np.asarray([v.size for v in vecs], np.int64)
    flat = np.concatenate(vecs)
    off = _prefix(lens)
    _lib.check(_lib.lib().pda_to_probs_batch_host(flat.ctypes.data, off.ctypes.data, lens.ctypes.data, len(vecs), 0))
    for i, v in enumerate(vecs):
        alone = gpu_api.toProbs(v)
        batch = flat[off[i]:off[i] + v.size]
        np.testing.assert_array_equal(bits(batch), bits(alone), err_msg=f"vector {i}: batch vs alone")
        want = oracle.to_probs(v)
        keep, ref = _probs_want(v)
        np.testing.assert_array_equal(alone != 0, want != 0, err_msg=f"vector {i}: gate vs oracle")
        np.testing.assert_array_equal(alone != 0, keep, err_msg=f"vector {i}: gate vs lo + 42 > x")
        np.testing.assert_allclose(alone, want, rtol=1e-14, atol=0, err_msg=f"vector {i} vs oracle")
        np.testing.assert_allclose(alone, ref, rtol=1e-14, atol=0, err_msg=f"vector {i} vs numpy.exp")
        if v.size >= 8:
            lo = v.min()
            assert alone[v == lo + GATE].max() == 0.0 and alone[v == np.nextafter(lo + GATE, -np.inf)].min() > 0.0
            assert np.all(alone[v == lo] == 1.0) and np.all(alone[np.isinf(v)] == 0.0)


# ---- GPU: stereo boxes beyond KITTI ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nonassign", NONASSIGN)
def test_stereo_boxes_wide_frames_vs_oracle(murty_path, gpu_api, oracle, nonassign):
    frames = box_frames()
    got = gpu_api.asgn_bb_batch([L for L, _ in frames], [R for _, R in frames], nonassign)
    matched = 0
    for f, (L, R) in enumerate(frames):
        want = oracle.asgn_bb(L, R, nonassign)
        np.testing.assert_array_equal(got[f], want, err_msg=f"frame {f} ({len(L)} + {len(R)} boxes, {murty_path})")
        np.testing.assert_array_equal(gpu_api.asgnBB(L, R, nonassign), want, err_msg=f"frame {f} alone")
        matched += int((want >= 0).sum())
    assert (matched == 0) == (nonassign == 1.5)


@pytest.mark.gpu
def test_stereo_boxes_beyond_max_dim(gpu_api):
    from probabilisticsemslam_b200 import _lib
    L, R = box_frame(64, 65, 99)
    small = box_frame(5, 6, 98)
    with pytest.raises(_lib.PdaError) as e:
        gpu_api.asgn_bb_batch([small[0], L], [small[1], R], 0.2)
    assert e.value.code == -3
