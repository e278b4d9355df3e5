"""Huber's approximate permanent (permanent_approx_kernel.cu) at every shape it accepts, trial for trial against its CPU
restatement (oracle/oracle_perm_approx.c), and against the exact permanent at sides 21-32, the range permanentFastest
(include/nwPerm.h) sends to it.

Both sides draw the same counter-based stream and do the same arithmetic in the same order, without FMA contraction.
They differ only in the association of the products over rows and of the prefix sum, in log(), and in (|rows-cols|)!,
each by a few ulp.  So a trial can go the other way only where a draw lies within rounding of a partial sum it was
compared with, and the restatement counts such draws (its near ties).  The rule every estimate is held to:

    K = the restatement's estimate * iterations / successes (the bound times the un-scaling);
    the kernel's successes round(g * iterations / K) equal the restatement's, give or take the near ties;
    where the counts are equal, |g / est - 1| <= 1e-12; statuses and NaN-ness are equal.

A kernel that moved one estimate by one trial, or changed the arithmetic of a few matrices, fails it."""
from __future__ import annotations

import math

import numpy as np
import pytest

from helpers import bits, check_approx_rule

gpu = pytest.mark.gpu
SEED = 20260217
N_TRIALS = 300            # apprxIter, assignment.cpp:10
EXACT_TRIALS = 10000      # against the exact permanent; families that accept rarely get more (_FAMILY_TRIALS)
_FAMILY_TRIALS = {"J+tI": 20000, "dense": 40000, "block": 100000}   # acceptance about 18 %, 6 % and 0.5-3 %
MAXD = 32                 # PDA_MAX_PERM_DIM
KINDS = ("u01", "wide", "ones", "rank1", "sparse")


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _matrix(kind, r, c, rng):
    """One (r, c) matrix of the given kind.  "sparse" is the union of three injective maps from the short side into the
    long side, so the ones-padded square matrix has total support and Sinkhorn converges."""
    if kind == "u01":
        return rng.random((r, c))
    if kind == "wide":
        return 10.0 ** rng.uniform(-6, 6, (r, c))
    if kind == "ones":
        return np.ones((r, c))
    if kind == "rank1":
        return np.outer(10.0 ** rng.uniform(-1, 1, r), 10.0 ** rng.uniform(-1, 1, c))
    A = np.zeros((r, c))
    short, long_ = min(r, c), max(r, c)
    for _ in range(3):
        img = rng.permutation(long_)[:short]
        for i in range(short):
            if r <= c:
                A[i, img[i]] = rng.uniform(0.1, 1.0)
            else:
                A[img[i], i] = rng.uniform(0.1, 1.0)
    return A


def _shapes():
    s = [(n, n) for n in range(MAXD + 1)]
    s += [(1, c) for c in range(2, MAXD + 1)] + [(r, 1) for r in range(2, MAXD + 1)]
    s += [(0, 1), (0, 7), (0, 32), (1, 0), (7, 0), (32, 0)]
    s += [(31, 32), (32, 31), (30, 32), (16, 32), (2, 32), (32, 2)]
    return s


def _every_shape():
    rng = np.random.default_rng(20261022)
    return [_matrix(k, r, c, rng) for (r, c) in _shapes() for k in KINDS]


# ---- the two forms of the kernel --------------------------------------------------------------------------------------
def _pack(mats):
    flat = [np.asfortranarray(m, dtype=np.float64).reshape(-1, order="F") for m in mats]
    off = np.zeros(len(mats), np.int64)
    if len(mats) > 1:
        off[1:] = np.cumsum([f.size for f in flat])[:-1]
    buf = np.concatenate(flat + [np.zeros(1)])
    rows = np.asarray([m.shape[0] for m in mats], np.int32)
    cols = np.asarray([m.shape[1] for m in mats], np.int32)
    return buf, off, rows, cols


def _host(mats, iterations=N_TRIALS, seed=SEED):
    from probabilisticsemslam_b200 import api
    return api.permanent_approx_batch(mats, iterations, seed)


def _device_raw(buf, off, rows, cols, iterations=N_TRIALS, seed=SEED):
    """pda_permanent_approx_batch on CUDA tensors -> (estimates, status, return code).  The matrix buffer carries a
    32 x 32 tail, so no shape can read past its allocation."""
    import torch
    from probabilisticsemslam_b200 import _lib
    n = len(rows)
    d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (np.concatenate([buf, np.zeros(MAXD * MAXD)]), off, rows, cols)]
    out = torch.full((max(n, 1),), -7.0, dtype=torch.float64, device="cuda")
    st = torch.full((max(n, 1),), -7, dtype=torch.int32, device="cuda")
    rc = _lib.lib().pda_permanent_approx_batch(*[x.data_ptr() for x in d], n, int(iterations), int(seed), out.data_ptr(),
                                               st.data_ptr(), None)
    torch.cuda.synchronize()
    return out.cpu().numpy()[:n], st.cpu().numpy()[:n], rc


def _device(mats, iterations=N_TRIALS, seed=SEED):
    from probabilisticsemslam_b200 import _lib
    g, st, rc = _device_raw(*_pack(mats), iterations, seed)
    _lib.check(rc)
    return g, st


def _both(mats, iterations=N_TRIALS, seed=SEED):
    """Both forms; their estimates and statuses must be the same bits."""
    g, st = _host(mats, iterations, seed)
    gd, std = _device(mats, iterations, seed)
    np.testing.assert_array_equal(bits(gd), bits(g), err_msg="device-pointer form != _host form")
    np.testing.assert_array_equal(std, st)
    return g, st


# ---- the rule ---------------------------------------------------------------------------------------------------------
_restated = {}


def _restate(oracle, A, iterations, seed, index):
    key = (A.shape, A.tobytes(order="F"), iterations, seed, index)
    if key not in _restated:
        _restated[key] = oracle.permanent_approx(A, iterations, seed, index, near_ties=True)
    return _restated[key]


def _check_rule(oracle, A, g, st, iterations=N_TRIALS, seed=SEED, index=0, what=""):
    """Holds the kernel's estimate g (status st) of A at matrix index `index` to the rule; returns the near ties."""
    restated = _restate(oracle, A, iterations, seed, index)
    assert st == 0, (what, A.shape, index, st)
    check_approx_rule(g, restated, iterations, f"{what} index {index}", tuple(A.shape))
    return restated[2]


def _within_binomial_error(est, exact, successes, trials, sigmas=5.0):
    p = max(successes, 1) / trials
    sd = math.sqrt((1 - p) / (trials * p))
    return abs(est / exact - 1.0) <= sigmas * sd + 0.02   # + the 1e-4 Sinkhorn tolerance's bias allowance


# ---- 1. every shape, both forms -----------------------------------------------------------------------------------------
@gpu
def test_every_shape_both_forms(gpu_api, oracle):
    mats = _every_shape()
    g, st = _both(mats)
    for i, A in enumerate(mats):
        _check_rule(oracle, A, g[i], st[i], index=i, what=KINDS[i % len(KINDS)])
    assert {tuple(A.shape) for A in mats} == set(_shapes())


# ---- 2. against the exact permanent at sides 21-32 ------------------------------------------------------------------------
def _exact_cases():
    """(family, matrix, exact permanent, trials) with closed-form or independently computed permanents."""
    rng = np.random.default_rng(321)
    cases = []
    for n in range(21, MAXD + 1):
        f = math.factorial
        cases.append(("ones", np.ones((n, n)), float(f(n))))
        r = n - 1 - n % 5   # ones r x n: n! / (n - r)! injective maps
        cases.append(("ones-rect", np.ones((r, n)), float(f(n) // f(n - r))))
        cases.append(("ones-rect-t", np.ones((n, r)), float(f(n) // f(n - r))))
        der = [1, 0]
        for k in range(2, n + 1):
            der.append((k - 1) * (der[-1] + der[-2]))
        cases.append(("J-I", np.ones((n, n)) - np.eye(n), float(der[n])))
        t = 0.5
        cases.append(("J+tI", np.ones((n, n)) + t * np.eye(n), sum(math.comb(n, k) * t ** k * f(n - k) for k in range(n + 1))))
        u, v = 10.0 ** rng.uniform(-1, 1, n), 10.0 ** rng.uniform(-1, 1, n)
        cases.append(("rank1", np.outer(u, v), f(n) * float(np.prod(u)) * float(np.prod(v))))
        sizes, left = [], n
        while left:
            b = min(left, int(rng.integers(3, 11)))
            sizes.append(b)
            left -= b
        A, at, blocks = np.zeros((n, n)), 0, []
        for b in sizes:
            A[at:at + b, at:at + b] = rng.uniform(0.1, 1.0, (b, b))
            blocks.append(A[at:at + b, at:at + b].copy())
            at += b
        cases.append(("block", A, blocks))
    for n in range(21, 25):
        cases.append(("dense", rng.random((n, n)), None))
    return cases


def _exact_values(oracle):
    out = []
    for fam, A, exact in _exact_cases():
        if exact is None:
            exact, st = oracle.permanent_exact(A)
            assert st == 0
        elif isinstance(exact, list):
            exact = float(np.prod([oracle.permanent_exact(B)[0] for B in exact]))
        trials = _FAMILY_TRIALS.get(fam, EXACT_TRIALS)
        out.append((fam, A, exact, trials))
    return out


def test_restatement_against_exact_at_long_sides(oracle):
    """The restatement's estimator at sides 21-32, where only the status at 33 used to be checked."""
    for i, (fam, A, exact, trials) in enumerate(_exact_values(oracle)):
        est, succ, _ = _restate(oracle, A, trials, SEED, i)
        assert succ >= 100 and _within_binomial_error(est, exact, succ, trials), (fam, A.shape, est, exact, succ)


@gpu
def test_kernel_against_exact_at_long_sides(gpu_api, oracle):
    cases = _exact_values(oracle)
    for trials in sorted({c[3] for c in cases}):
        idx = [i for i, c in enumerate(cases) if c[3] == trials]
        # matrix index = position in the whole case list, as in the restatement's twin above: pad the batch with 0 x 0
        full = [np.zeros((0, 0))] * len(cases)
        for i in idx:
            full[i] = cases[i][1]
        g, st = _both(full, trials)
        for i in idx:
            fam, A, exact, _ = cases[i]
            est, succ, _ = _restate(oracle, A, trials, SEED, i)
            assert _within_binomial_error(g[i], exact, succ, trials), (fam, A.shape, g[i], exact, succ)
            _check_rule(oracle, A, g[i], st[i], trials, SEED, i, fam)


# ---- 3. degenerate input ------------------------------------------------------------------------------------------------
def _degenerate():
    rng = np.random.default_rng(77)
    zr = rng.random((5, 5)); zr[2, :] = 0
    zc = rng.random((6, 4)); zc[:, 1] = 0
    inf = rng.random((4, 4)); inf[1, 3] = np.inf
    nan = rng.random((3, 7)); nan[2, 2] = np.nan
    sub = rng.random((5, 5)); sub[:, 4] = 1e-310
    big = rng.random((32, 32)); big[31, :] = 0      # every lane live
    return [zr, zc, inf, nan, np.zeros((1, 1)), sub, big]


def _with_neighbours(bad, rng):
    """4 matrices per CTA: each degenerate matrix sits in a CTA with ordinary ones, at slot 1 or 2 of it."""
    mats, where = [], []
    for j, B in enumerate(bad):
        cta = [rng.random((int(rng.integers(2, 12)), int(rng.integers(2, 12)))) for _ in range(4)]
        cta[1 + j % 2] = B
        where.append(4 * j + 1 + j % 2)
        mats += cta
    return mats, where


def test_restatement_gives_nan_on_degenerate_input(oracle):
    for A in _degenerate():
        est, succ = oracle.permanent_approx(A, N_TRIALS, SEED, 0)
        assert np.isnan(est) and succ == 0, A.shape


@gpu
def test_degenerate_input_in_a_shared_cta(gpu_api, oracle):
    rng = np.random.default_rng(5)
    bad = _degenerate()
    mats, where = _with_neighbours(bad, rng)
    g, st = _both(mats)
    plain = list(mats)
    for w in where:
        plain[w] = np.ones((3, 3))
    g0, st0 = _both(plain)
    for i, A in enumerate(mats):
        assert st[i] == 0
        if i in where:
            assert np.isnan(g[i]), (i, A.shape, g[i])
            _check_rule(oracle, A, g[i], st[i], index=i, what="degenerate")
        else:
            assert bits(g[i]) == bits(g0[i]), f"neighbour {i} changed next to a degenerate matrix"


# ---- 4. launch geometry, status and arguments --------------------------------------------------------------------------
def _mixed(n, rng):
    mats = []
    for _ in range(n):
        r, c = int(rng.integers(0, MAXD + 1)), int(rng.integers(0, MAXD + 1))
        if rng.random() < 0.5:
            c = r
        mats.append(_matrix(KINDS[int(rng.integers(len(KINDS)))], r, c, rng))
    return mats


@gpu
def test_batches_around_one_cta(gpu_api, oracle):
    rng = np.random.default_rng(11)
    mats = _mixed(9, rng)
    g9, _ = _both(mats)
    for i, A in enumerate(mats):
        _check_rule(oracle, A, g9[i], 0, index=i, what="batch of 9")
    for b in range(1, 9):
        g, st = _both(mats[:b])
        assert not st.any()
        np.testing.assert_array_equal(bits(g), bits(g9[:b]), err_msg=f"batch of {b}")


@gpu
def test_large_mixed_batch(gpu_api, oracle):
    rng = np.random.default_rng(12)
    mats = _mixed(20000, rng)
    g, st = _both(mats)
    assert not st.any()
    for i in np.sort(rng.choice(len(mats), 500, replace=False)):
        _check_rule(oracle, mats[i], g[i], st[i], index=int(i), what="mixed batch")


@gpu
def test_result_depends_on_index_not_neighbours(gpu_api):
    rng = np.random.default_rng(13)
    a = _mixed(12, rng)
    b = _mixed(12, rng)
    for i in (0, 5, 11):
        b[i] = a[i]
    ga, _ = _both(a)
    gb, _ = _both(b)
    for i in (0, 5, 11):
        assert bits(ga[i]) == bits(gb[i]), i
    moved = [np.ones((1, 1))] + a   # the same matrix at another index draws another stream
    gm, _ = _both(moved)
    assert not np.array_equal(bits(gm[1:]), bits(ga))


@gpu
def test_side_33_is_status_1_beside_ordinary_matrices(gpu_api):
    rng = np.random.default_rng(14)
    mats = _mixed(12, rng)
    plain = list(mats)
    for i, shape in ((1, (33, 33)), (6, (33, 5)), (7, (5, 33)), (11, (40, 1))):
        mats[i] = rng.random(shape)
    g, st = _both(mats)
    g0, st0 = _both(plain)
    assert not st0.any()
    for i in range(12):
        if i in (1, 6, 7, 11):
            assert st[i] == 1 and g[i] == 0.0, i
        else:
            assert st[i] == 0 and bits(g[i]) == bits(g0[i]), i


@gpu
def test_negative_dimension(gpu_api):
    from probabilisticsemslam_b200 import _lib
    rng = np.random.default_rng(15)
    mats = _mixed(8, rng)
    buf, off, rows, cols = _pack(mats)
    g0, st0, rc = _device_raw(buf, off, rows, cols)
    assert rc == 0 and not st0.any()
    bad = {1: (-1, 5), 2: (3, -2), 5: (-4, -4), 6: (-1, 0)}
    for i, (r, c) in bad.items():
        rows[i], cols[i] = r, c
    g, st, rc = _device_raw(buf, off, rows, cols)
    assert rc == 0
    for i in range(8):
        if i in bad:
            assert st[i] == 1 and g[i] == 0.0, (i, bad[i], g[i], st[i])
        else:
            assert st[i] == 0 and bits(g[i]) == bits(g0[i]), i
    out, status = np.zeros(8), np.zeros(8, np.int32)
    rc = _lib.lib().pda_permanent_approx_batch_host(buf.ctypes.data, off.ctypes.data, rows.ctypes.data, cols.ctypes.data, 8,
                                                    N_TRIALS, SEED, out.ctypes.data, status.ctypes.data, 0)
    assert rc == -1   # PDA_ERR_INVALID


@gpu
@pytest.mark.parametrize("iterations", [1, 2, 300, 10000])
def test_iteration_counts(gpu_api, oracle, iterations):
    rng = np.random.default_rng(16)
    mats = _mixed(24, rng)
    g, st = _both(mats, iterations)
    for i, A in enumerate(mats):
        _check_rule(oracle, A, g[i], st[i], iterations, SEED, i, f"{iterations} trials")


@gpu
def test_iterations_below_one_are_an_error(gpu_api):
    from probabilisticsemslam_b200 import _lib
    mats = [np.ones((3, 3))]
    for it in (0, -1):
        with pytest.raises(_lib.PdaError) as e:
            _host(mats, it)
        assert e.value.code == -1
        assert _device_raw(*_pack(mats), it)[2] == -1


# ---- an exact tie: a draw equal to the total picks the last row (pickRowFromProbs uses >=) ------------------------------
_M64, _G = 2 ** 64, 0x9E3779B97F4A7C15


def _unxorshift(z, s):
    x = z
    for _ in range(64 // s + 1):
        x = z ^ (x >> s)
    return x


def _unmix64(z):
    z = _unxorshift(z, 31) * pow(0x94D049BB133111EB, -1, _M64) % _M64
    z = _unxorshift(z, 27) * pow(0xBF58476D1CE4E5B9, -1, _M64) % _M64
    return _unxorshift(z, 30)


def _seed_drawing(u, mat):
    """The seed whose draw of (mat, trial 0, column 0) is exactly u (draw01 inverted: mix64 is a bijection)."""
    k = int(u * 2.0 ** 53)
    assert k / 2.0 ** 53 == u
    key = (_unmix64(k << 11) - _G) % _M64
    return _unmix64(key) ^ (_G * (mat + 1) % _M64)


def _ones2_total():
    """Sum of the pick probabilities of column 0 of the 2 x 2 ones matrix, in the restatement's order.  Sinkhorn and the
    row scaling leave it at exactly ones; at two rows neither the products over rows nor the prefix sum can be
    reassociated, and the one log() is log(2), so the kernel computes the same bits."""
    ee = 2.71828182846
    hl2, hl1 = 2.0 + 0.5 * math.log(2.0) + ee - 1.0, 1.0 + (ee - 1.0) * 1.0
    p = ((1.0 * (hl1 / ee)) * (hl1 / ee)) / ((1.0 * (hl2 / ee)) * (hl2 / ee)) * ee * (1.0 / hl1)
    return p + p


def test_restatement_exact_tie(oracle):
    u, A = _ones2_total(), np.ones((2, 2))
    for mat in (0, 3):
        est, succ, ties = oracle.permanent_approx(A, 1, _seed_drawing(u, mat), mat, near_ties=True)
        assert succ == 1 and ties == 1 and est > 0
        assert oracle.permanent_approx(A, 1, _seed_drawing(np.nextafter(u, 1.0), mat), mat)[1] == 0


@gpu
def test_kernel_exact_tie(gpu_api, oracle):
    u, A = _ones2_total(), np.ones((2, 2))
    for mat in (0, 3):
        seed = _seed_drawing(u, mat)
        for iterations in (1, 300):
            mats = [np.ones((3, 3))] * mat + [A]
            g, st = _both(mats, iterations, seed)
            est, succ = oracle.permanent_approx(A, iterations, seed, mat)
            assert st[mat] == 0 and bits(g[mat]) == bits(est), (mat, iterations, g[mat], est, succ)


# ---- 5. permOpt = 0 through permanentProb and conditionedPermanent at long sides 17-32 ----------------------------------
def _gated_problem(nL, nM, rng):
    """Costs of nL landmarks and nM detections (rows landmarks then one dummy row per detection); cost 100 is gated
    (to_probs gives 0 beyond the gate of 42), every landmark keeps at least one finite cost."""
    C = np.full((nL + nM, nM), 100.0)
    C[:nL] = np.where(rng.random((nL, nM)) < 0.25, 100.0, rng.uniform(0, 8, (nL, nM)))
    C[np.arange(nL), rng.integers(0, nM, nL)] = rng.uniform(0, 8, nL)
    C[nL + np.arange(nM), np.arange(nM)] = 6.0 + rng.uniform(0, 1, nM)
    return C


def _long_sides(oracle, C, nL):
    """The long side of every sub-permanent permanentProb computes: P without column m and without row l (or the dummy
    row of m), zero lines dropped (conditionedPermanent)."""
    nR, nM = C.shape
    P = oracle.to_probs(C.reshape(-1, order="F")).reshape(C.shape, order="F")
    out = set()
    for m in range(nM):
        cols = [c for c in range(nM) if c != m]
        for l in list(range(nL)) + [nL + m]:
            if P[l, m] == 0:
                continue
            S = np.delete(P, l, axis=0)[:, cols]
            out.add(max(int((S != 0).any(axis=1).sum()), int((S != 0).any(axis=0).sum())))
    return out


@gpu
def test_permanent_prob_approx_at_long_sides(gpu_api, oracle):
    from probabilisticsemslam_b200 import _lib
    _lib.lib().pda_set_approx_seed(SEED)
    rng = np.random.default_rng(17)
    seen, ties = set(), 0
    for total in range(18, 34):
        nM = int(rng.integers(2, 5))
        C = _gated_problem(total - nM, nM, rng)
        nL = total - nM
        sides = _long_sides(oracle, C, nL)
        seen |= sides
        got = gpu_api.permanentProb(C, nL, 0)   # batch of one: item indices start at 0, as in the oracle
        oracle.approx_near_ties_reset()
        st, want = oracle.permanent_prob(C, nL, 0)
        t = oracle.approx_near_ties()
        ties += t
        assert st == 0
        if t == 0:
            assert np.max(np.abs(got - want)) <= 1e-12, (C.shape, sides, np.max(np.abs(got - want)))
    assert set(range(17, 33)) <= seen, sorted(seen)


@gpu
def test_conditioned_permanent_approx_at_long_sides(gpu_api, oracle):
    from probabilisticsemslam_b200 import _lib
    _lib.lib().pda_set_approx_seed(SEED)
    rng = np.random.default_rng(18)
    for side in range(17, MAXD + 1):
        short = int(rng.integers(1, side + 1))
        A = rng.random((side + 1, short + 1))
        A[int(rng.integers(0, side + 1)), :] = 0      # a zero row and a zero column are dropped first
        A[:, int(rng.integers(0, short + 1))] = 0
        A = A if rng.random() < 0.5 else A.T
        got = gpu_api.conditionedPermanent(A, 0)
        oracle.set_approx_stream(SEED, 0)
        oracle.approx_near_ties_reset()
        want, st = oracle.conditioned_permanent(A, 0)
        assert st == 0
        if oracle.approx_near_ties() == 0:
            assert abs(got / want - 1.0) <= 1e-12, (A.shape, got, want)
