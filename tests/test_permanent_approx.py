"""Huber's randomised approximate permanent (SURVEY.md 8f rank 4; nwPerm.cpp:36-211, reached through
conditionedPermanent(.., permOpt = 0), assignment.cpp:401).

The reference draws from an unseeded process-wide rand(), so there is no reference sample to match: parity for this
row is statistical by nature.  The CPU restatement (oracle/oracle_perm_approx.c) and the CUDA kernel share one
counter-based stream and the same arithmetic, which makes them comparable trial for trial: the kernel must have the
restatement's success count give or take the restatement's near ties, and then its estimate to 1e-12
(helpers.check_approx_rule).  Both are held to the exact permanent within the estimator's own binomial standard error.
tests/test_gpu_permanent_approx_shapes.py covers every shape the kernel accepts."""
import numpy as np
import pytest

from helpers import check_approx_rule
from probabilisticsemslam_b200 import synth

N_TRIALS = 300   # apprxIter, assignment.cpp:10


def _cases():
    mats = []
    for n in (2, 3, 5, 8, 11, 14, 17, 20):
        for i in range(4):
            mats.append(synth.dense_square(1, n, first=1000 * n + i)[0].reshape(n, n, order="F"))
    rng = np.random.default_rng(9)
    for r, c in ((2, 5), (6, 3), (4, 9), (12, 10)):
        mats.append(rng.random((r, c)))
    for n in (6, 10):   # the shape permanentProb produces: a few likelihood rows over ones (nwPerm.cpp:223-230)
        A = np.ones((n, n)); A[:4, :] = np.exp(-rng.uniform(0, 8, size=(4, n))); mats.append(A)
    return mats


def _within_binomial_error(est, exact, successes, sigmas=5.0):
    p = max(successes, 1) / N_TRIALS
    sd = np.sqrt((1 - p) / (N_TRIALS * p))
    return abs(est / exact - 1.0) <= sigmas * sd + 0.02   # + the 1e-4 Sinkhorn tolerance's bias allowance


def test_oracle_estimator_against_exact(oracle):
    for i, A in enumerate(_cases()):
        exact = oracle.permanent_exact(A)[0]
        est, succ = oracle.permanent_approx(A, N_TRIALS, 20260217, i)
        assert succ > 0 and _within_binomial_error(est, exact, succ), (A.shape, est, exact, succ)
    est, succ = oracle.permanent_approx(np.ones((2, 3)), N_TRIALS, 1, 0)   # 6 injective maps 2 -> 3
    assert abs(est / 6.0 - 1.0) < 0.15


def _golden_cases():
    from helpers import golden
    z = golden("perm_approx")
    return [(z[f"A{i}"], float(z[f"est{i}"]), int(z[f"succ{i}"]), float(z[f"exact{i}"])) for i in range(int(z["n"]))], int(z["seed"])


def test_oracle_reproduces_its_golden_stream(oracle):
    """tests/golden/perm_approx.npz: estimates and success counts of the counter-based stream (regression pin of the
    restatement and of the draw function both sides share)."""
    cases, seed = _golden_cases()
    for i, (A, est, succ, exact) in enumerate(cases):
        got, s = oracle.permanent_approx(A, N_TRIALS, seed, i)
        assert s == succ and abs(got / est - 1.0) < 1e-12
        assert _within_binomial_error(est, exact, succ)


@pytest.mark.gpu
def test_gpu_against_golden_stream(gpu_api, oracle):
    cases, seed = _golden_cases()
    got, st = gpu_api.permanent_approx_batch([c[0] for c in cases], N_TRIALS, seed)
    assert not st.any()
    for i, (g, (A, est, succ, exact)) in enumerate(zip(got, cases)):
        ties = oracle.permanent_approx(A, N_TRIALS, seed, i, near_ties=True)[2]
        check_approx_rule(g, (est, succ, ties), N_TRIALS, "golden", A.shape)
        assert _within_binomial_error(g, exact, succ)


@pytest.mark.gpu
def test_gpu_against_restatement_and_exact(gpu_api, oracle):
    mats = _cases()
    got, st = gpu_api.permanent_approx_batch(mats, N_TRIALS, 20260217)
    assert not st.any()
    for i, A in enumerate(mats):
        restated = oracle.permanent_approx(A, N_TRIALS, 20260217, i, near_ties=True)
        exact = oracle.permanent_exact(A)[0]
        assert _within_binomial_error(got[i], exact, restated[1]), (A.shape, got[i], exact)
        # same draws: the two can only differ where a pick lands within rounding of a partial sum (a near tie)
        check_approx_rule(got[i], restated, N_TRIALS, "case", A.shape)
    again, _ = gpu_api.permanent_approx_batch(mats, N_TRIALS, 20260217)
    np.testing.assert_array_equal(again, got)                                   # reproducible
    other, _ = gpu_api.permanent_approx_batch(mats, N_TRIALS, 12345)
    assert not np.array_equal(other, got)                                        # and seeded
    _, st = gpu_api.permanent_approx_batch([np.ones((33, 33))], N_TRIALS, 1)
    assert st[0] == 1


@pytest.mark.gpu
def test_gpu_permanent_prob_with_approximation(gpu_api, oracle):
    """permanentProb(.., permOpt = 0) on gated problems: against the CPU restatement drawing from the same streams
    (item m*(nL+1)+l of a problem uses stream index m*(nL+1)+l on both sides) to 1e-12 wherever the restatement met no
    near tie, and against permOpt = 1 within what 300 trials per sub-permanent allow -- the restatement itself sits at a
    median max-abs weight error of 0.09 (worst 0.30) on these problems, the order of compMethods' own perm-approx error."""
    g2 = synth.g2_gated(60, first=4242)
    cond, _ = gpu_api.condition_costs_batch(g2)
    keep = [p for p in range(len(cond)) if cond.matrix(p).shape[0] - 1 <= 16]
    sub = synth.pack([cond.matrix(p) for p in keep], [int(cond.nL[p]) for p in keep])
    exact, st1 = gpu_api.permanent_prob_batch(sub, 1)
    approx, st0 = gpu_api.permanent_prob_batch(sub, 0)
    assert not st0.any() and not st1.any()
    vs_exact = []
    for p, (e, a) in enumerate(zip(exact, approx)):
        assert np.all(np.isfinite(a)) and np.all(a >= 0)
        assert np.max(a.sum(axis=1)) <= 1.0 + 1e-9     # normalised by the largest column sum (assignment.cpp:255, 266)
        vs_exact.append(np.max(np.abs(a - e)))
        one = gpu_api.permanentProb(sub.matrix(p), int(sub.nL[p]), 0)      # batch of one: item indices start at 0, as in the oracle
        oracle.approx_near_ties_reset()
        st, want = oracle.permanent_prob(sub.matrix(p), int(sub.nL[p]), 0)
        assert st == 0
        if oracle.approx_near_ties() == 0:
            assert np.max(np.abs(one - want)) <= 1e-12, (p, np.max(np.abs(one - want)))
    assert np.median(vs_exact) < 0.15 and np.max(vs_exact) < 0.6, (np.median(vs_exact), np.max(vs_exact))
    with pytest.raises(RuntimeError):
        gpu_api.permanentProb(sub.matrix(0), int(sub.nL[0]), 7)   # unknown permOpt still throws (assignment.cpp:406)
