"""getAssignmentProbs at every frame shape it accepts, against the exact association marginals (tests/assoc_exact.py).

The table of shapes crosses nM over a warp (32) and two (64), the usePerm path's fused / routed split (11 / 12
detections), nL + nM = PDA_MAX_DIM and the Murty kernel's shared-memory limit: the places where the lane-strided loops of
quadric_cost_kernel, condition_costs_kernel, uncompact_probs_kernel and finish_scatter_kernel, and the host forms' choice
of Murty bounds, change behaviour.  Frames are built with a chosen gate graph (components of a few detections sharing a
few landmarks, everything else out of every gate), so the exact marginals stay cheap at any size and the k-best
enumeration can be made exhaustive.

Per shape: the k-best tables (k = 1, 200 and the frame's hypothesis count) against the truth where exhaustive, against
the CPU oracle always, and bit for bit across the entry points (from costs, from moments, the device-pointer moments form
under tight and loose bounds, alone and inside one mixed batch); the usePerm tables likewise; the cost matrices bit for
bit against the oracle.  Then the degenerate frames: both weight paths must fail the same way."""
from __future__ import annotations

import itertools
import math

import numpy as np
import pytest

from assoc_exact import exact_marginals, gate_graph, perm_status
from perm_route import composed
from test_gpu_murty_geometry import geometry

gpu = pytest.mark.gpu
B200_OPTIN = 227 * 1024
NONASSIGN = 10.0
MAX_DIM = 128
MAX_COUNT = 300  # hypotheses per generated frame: the exhaustive k of a mixed batch stays a few GB of Murty workspace

NLS = (0, 1, 2, 31, 32, 33, 63, 64, 95, 96, 127)
NMS = (1, 2, 3, 8, 11, 12, 16, 31, 32, 33, 64, 65, 96, 112, 113, 127, 128)
SHAPES = [(L, M) for L in NLS for M in NMS if L + M <= MAX_DIM]


def kbest_fits(L, M, k, optin=B200_OPTIN):
    """Whether the Murty kernel takes a frame alone (frames without landmarks never reach it)."""
    return L == 0 or geometry(k, L + M, M, True, optin).error is None


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


# ---- frames with a chosen gate graph ------------------------------------------------------------------------------------
def _groups(rng, nL, nM, max_count):
    """Detection groups, each sharing a set of landmarks (every pair in gate): [(detections, landmarks)], with the
    product of the groups' hypothesis counts at most max_count.  Landmarks and detections are drawn from the whole
    frame, so the kept rows are spread over it."""
    lands, dets = list(rng.permutation(nL)), list(rng.permutation(nM))
    out, count = [], 1
    while lands and dets:
        d, s = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        d, s = min(d, len(dets)), min(s, len(lands))
        c = sum(math.comb(d, j) * math.perm(s, j) for j in range(min(d, s) + 1))
        if count * c > max_count:
            break
        out.append(([int(dets.pop()) for _ in range(d)], [int(lands.pop()) for _ in range(s)]))
        count *= c
    return out


def cost_frame(rng, nL, nM, max_count=MAX_COUNT):
    """(C, intended in-gate [nL, nM]): in-gate costs over 0-40, dummies at 10, everything else at least colMin + 50 or
    +inf, no entry near the 42 boundary."""
    C = np.full((nL + nM, nM), np.inf)
    C[nL + np.arange(nM), np.arange(nM)] = NONASSIGN
    far = rng.uniform(60.0, 160.0, (nL, nM))
    C[:nL] = np.where(rng.random((nL, nM)) < 0.7, far, np.inf)
    adj = np.zeros((nL, nM), bool)
    for ds, ls in _groups(rng, nL, nM, max_count):
        for l in ls:
            for m in ds:
                C[l, m] = rng.uniform(0.0, 40.0)
                adj[l, m] = True
    return C, adj


def _spd(rng, lo, hi):
    q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    return (q * 10.0 ** rng.uniform(lo, hi, 3)) @ q.T


def moments_frame(rng, nL, nM, max_count=MAX_COUNT):
    """(frame moments, intended in-gate [nL, nM]).  Clusters 1e4 apart: the landmarks and detections of one group sit
    within 1 of their cluster centre, every other landmark and detection at a centre of its own.  Landmark covariances
    have eigenvalues over 1e-3..1e3 and detection covariances over 1..1e3, so a pair inside a cluster costs at most 3 and
    a pair in different clusters at least ~5e4."""
    centre = lambda q: 1e4 * np.array([q % 8, (q // 8) % 8, q // 64], np.float64)
    lm, dm = np.zeros((nL, 3)), np.zeros((nM, 3))
    adj = np.zeros((nL, nM), bool)
    q = 0
    used_l, used_m = set(), set()
    for ds, ls in _groups(rng, nL, nM, max_count):
        for l in ls:
            lm[l] = centre(q) + rng.uniform(-0.5, 0.5, 3)
        for m in ds:
            dm[m] = centre(q) + rng.uniform(-0.5, 0.5, 3)
            adj[ls, m] = True
        used_l.update(ls), used_m.update(ds)
        q += 1
    for l in range(nL):
        if l not in used_l:
            lm[l] = centre(q); q += 1
    for m in range(nM):
        if m not in used_m:
            dm[m] = centre(q); q += 1
    lc = np.stack([_spd(rng, -3, 3) for _ in range(nL)]) if nL else np.zeros((0, 3, 3))
    mc = np.stack([_spd(rng, 0, 3) for _ in range(nM)])
    return (lm, lc, dm, mc), adj


def check_gate(C, nL, adj):
    """The cost matrix has the intended gate graph, with every in-gate entry at least 1 inside the 42 boundary and every
    other landmark entry at least 8 outside it."""
    col_min, got = gate_graph(C, nL)
    np.testing.assert_array_equal(got, adj, err_msg="gate graph")
    rel = C[:nL] - col_min[None, :]
    assert np.all(rel[adj] <= 41.0) and np.all(rel[~adj] >= 50.0)


# ---- CPU: the reference itself --------------------------------------------------------------------------------------------
def enumerate_marginals(C, nL):
    """Every hypothesis of the gated problem, one by one."""
    nM = C.shape[1]
    col_min = C.min(axis=0)
    opts = [[l for l in range(nL) if C[l, m] <= col_min[m] + 42.0] + [nL] for m in range(nM)]
    E, Z, n = np.zeros((nM, nL + 1)), 0.0, 0
    for h in itertools.product(*opts):
        ls = [l for l in h if l < nL]
        if len(set(ls)) != len(ls):
            continue
        w = math.exp(-sum((C[l, m] if l < nL else C[nL + m, m]) - col_min[m] for m, l in enumerate(h)))
        for m, l in enumerate(h):
            E[m, l] += w
        Z += w
        n += 1
    return E / Z, n


def tiny(rng, nL, nM, spread=40.0, p_inf=0.3):
    C = np.where(rng.random((nL + nM, nM)) < p_inf, np.inf, rng.uniform(0.0, spread, (nL + nM, nM)))
    C[nL:] = np.inf
    C[nL + np.arange(nM), np.arange(nM)] = rng.uniform(0.0, spread, nM)
    return C


def test_exact_matches_enumeration():
    rng = np.random.default_rng(11)
    for _ in range(150):
        nL, nM = int(rng.integers(0, 6)), int(rng.integers(1, 6))
        C = tiny(rng, nL, nM, spread=rng.choice([5.0, 40.0, 80.0]))
        try:
            E, n = exact_marginals(C, nL)
        except ValueError:
            continue  # a gated-away dummy: outside what E describes
        want, nw = enumerate_marginals(C, nL)
        assert n == nw
        np.testing.assert_allclose(E, want, rtol=0, atol=1e-14)
        np.testing.assert_allclose(E.sum(axis=1), 1.0, rtol=0, atol=1e-14)


def test_exact_matches_permanent_truth():
    from truth import permanent_prob_truth
    rng = np.random.default_rng(12)
    for _ in range(60):
        nL, nM = int(rng.integers(1, 6)), int(rng.integers(1, 5))
        C = tiny(rng, nL, nM)  # every finite entry within 40 of every minimum: both gates keep all of them
        E, _ = exact_marginals(C, nL)
        T = permanent_prob_truth(C, nL)
        if nM == 1:
            T = np.concatenate([T[:, :nL], T[:, nL:].sum(axis=1, keepdims=True)], axis=1)
        np.testing.assert_allclose(E, T / T.sum(axis=1, keepdims=True), rtol=0, atol=1e-13)


def test_exact_matches_brute_force(oracle):
    rng = np.random.default_rng(13)
    for _ in range(60):
        nL = int(rng.integers(1, 10))
        nM = int(rng.integers(1, min(7, 17 - nL)))
        C = tiny(rng, nL, nM)
        E, _ = exact_marginals(C, nL)
        np.testing.assert_allclose(E, oracle.brute_force_prob(C, nL), rtol=0, atol=1e-12)


def test_hypothesis_count_is_exact():
    # one detection, n landmarks: n + 1; n detections sharing n landmarks: sum_j C(n, j)^2 j!
    for n in range(1, 7):
        C = np.full((2 * n, n), np.inf)
        C[:n] = 1.0
        C[n + np.arange(n), np.arange(n)] = 2.0
        assert exact_marginals(C, n)[1] == sum(math.comb(n, j) ** 2 * math.factorial(j) for j in range(n + 1))
    # 40 independent detections with one landmark each: 2^40, past what a float counts exactly
    n = 40
    C = np.full((2 * n, n), np.inf)
    C[np.arange(n), np.arange(n)] = 1.0
    C[n + np.arange(n), np.arange(n)] = 2.0
    assert exact_marginals(C, n)[1] == 2 ** 40


def test_shape_table_reaches_every_regime():
    """The Murty limit here is the B200's (227 KB of opt-in shared memory per block); the GPU tests read the device's."""
    ms = {M for _, M in SHAPES}
    assert {31, 32, 33} <= ms and {64, 65} <= ms               # nM on both sides of one warp and of two
    assert {11, 12} <= ms                                      # the usePerm path's fused / routed split
    assert any(L + M == MAX_DIM for L, M in SHAPES)
    fits = {(L, M): kbest_fits(L, M, MAX_COUNT) for L, M in SHAPES if L > 0}
    assert (1, 113) in fits and fits[(1, 113)]                 # the Murty limit from below: 114 x 113 runs ...
    assert (1, 127) in fits and not fits[(1, 127)]             # ... and from above: 128 x 127 does not
    murty_limited_alone = [M for L, M in SHAPES if L == 0 and geometry(1, M, M, True, B200_OPTIN).error is not None]
    assert murty_limited_alone                                 # nL = 0 frames the Murty kernel could not take


def test_generated_frames_have_their_gate_graph_and_truth(oracle):
    """The cost frames' gate graphs, hypothesis counts and truth, and the oracle's tables against the truth (k-best at the
    exhaustive k, usePerm where it does not throw) at the shapes cheap on the CPU."""
    rng = np.random.default_rng(14)
    for L, M in SHAPES:
        C, adj = cost_frame(rng, L, M)
        check_gate(C, L, adj)
        E, n = exact_marginals(C, L)
        assert n <= MAX_COUNT
        np.testing.assert_allclose(E.sum(axis=1), 1.0, rtol=0, atol=1e-13)
        if L + M > 40:
            continue
        st, got = oracle.association_probs(C, L, n)
        assert st == 0
        np.testing.assert_allclose(got, E, rtol=0, atol=1e-13)
        if M <= 16 and perm_status(C, L) == 0:  # sub-permanents of at most ~2^20 terms on the CPU
            st, got = oracle.association_probs(C, L, 1, use_perm=True)
            assert st == 0
            np.testing.assert_allclose(got, E, rtol=1e-9, atol=1e-300)


# ---- GPU -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def optin():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


@pytest.fixture(scope="module")
def frames(gpu_api):
    """Per shape: a cost frame and a moments frame, the GPU cost matrix of the latter, truth and hypothesis counts."""
    api = gpu_api
    rng = np.random.default_rng(20261022)
    out = {}
    mom = []
    for L, M in SHAPES:
        C, adj = cost_frame(rng, L, M)
        fr, madj = moments_frame(rng, L, M)
        mom.append((fr, madj))
    costs = api.quadric_cost_batch([f for f, _ in mom], NONASSIGN)
    for (L, M), (fr, madj), Cg in zip(SHAPES, mom, costs):
        check_gate(Cg, L, madj)
        C, adj = cost_frame(rng, L, M)
        out[(L, M)] = dict(C=C, E=exact_marginals(C, L), mom=fr, Cg=Cg, Eg=exact_marginals(Cg, L))
    return out


def assert_truth(got, E, what):
    """Exhaustive k-best or usePerm table against E: 1e-13 absolute, 1e-9 relative where E >= 1e-6."""
    d = np.abs(got - E)
    assert d.max() <= 1e-13, f"{what}: max |table - E| = {d.max():.3e}"
    big = E >= 1e-6
    assert np.all(d[big] <= 1e-9 * E[big]), f"{what}: relative {np.max(d[big] / E[big]):.3e}"


def _mixed_groups(shapes, k):
    """Every shape the k-best path takes, in as few batches as its joint bounds allow: one main batch and the frames with
    nM >= 113 and landmarks, which fit alone but not beside 128-row frames."""
    ok = [s for s in shapes if kbest_fits(*s, k)]
    wide = [s for s in ok if s[0] > 0 and s[1] >= 113]
    return [[s for s in ok if s not in wide], wide]


@gpu
def test_kbest_every_shape(gpu_api, oracle, frames, optin):
    api = gpu_api
    import torch
    from probabilisticsemslam_b200 import synth
    worst = 0.0
    K_all = max(max(f["E"][1], f["Eg"][1]) for f in frames.values())
    for k_name in ("1", "200", "K"):
        kk = {"1": 1, "200": 200, "K": K_all}[k_name]
        mixed = {}
        for group in _mixed_groups(SHAPES, kk):
            if not group:
                continue
            tabs = api.association_probs_batch(synth.pack([frames[s]["C"] for s in group], [s[0] for s in group]), kk)
            mt = api.association_from_moments_batch([frames[s]["mom"] for s in group], NONASSIGN, kk)
            for s, t, u in zip(group, tabs, mt):
                mixed[s] = (t.copy(), u.copy())
        for (L, M), f in frames.items():
            if not kbest_fits(L, M, kk, optin):
                continue
            what = f"{L}x{M} k={k_name}"
            (E, n), (Eg, ng) = f["E"], f["Eg"]
            ka = kk if k_name != "K" else max(n, 1)
            t = api.association_probs_batch(synth.pack([f["C"]], [L]), ka)[0]
            np.testing.assert_allclose(t.sum(axis=1), 1.0, rtol=0, atol=1e-12, err_msg=what)
            st, want = oracle.association_probs(f["C"], L, ka)
            assert st == 0
            np.testing.assert_allclose(t, want, rtol=1e-9, atol=0, err_msg=what + " vs oracle")
            if ka >= n:
                assert_truth(t, E, what)
                worst = max(worst, float(np.abs(t - E).max()))
            np.testing.assert_array_equal(bits(t), bits(mixed[(L, M)][0]), err_msg=what + ": alone vs mixed batch")
            # moments: _host from the GPU cost matrix, _host from moments, device form tight and loose, mixed
            kg = kk if k_name != "K" else max(ng, 1)
            tc = api.association_probs_batch(synth.pack([f["Cg"]], [L]), kg)[0]
            tm = api.association_from_moments_batch([f["mom"]], NONASSIGN, kg)[0]
            np.testing.assert_array_equal(bits(tc), bits(tm), err_msg=what + ": from costs vs from moments")
            np.testing.assert_array_equal(bits(tm), bits(mixed[(L, M)][1]), err_msg=what + ": moments alone vs mixed")
            if kg >= ng:
                assert_truth(tm, Eg, what + " (moments)")
                worst = max(worst, float(np.abs(tm - Eg).max()))
            dev = api.moments_to_device([f["mom"]])
            bounds = [(L, M)]
            loose = max((x for x in range(L, MAX_DIM - M + 1) if geometry(kg, x + M, M, True, optin).error is None), default=None)
            if loose is not None and loose != L:
                bounds.append((loose, M))
            for bL, bM in bounds:
                if geometry(kg, bL + bM, bM, True, optin).error is not None:
                    continue
                p, po, st, nf = api.association_from_moments_batch_device(*dev, bL, bM, NONASSIGN, kg)
                torch.cuda.synchronize()
                assert int(st[0]) == 0, what
                td = p[:M * (L + 1)].cpu().numpy().reshape(M, L + 1)
                np.testing.assert_array_equal(bits(td), bits(tm), err_msg=f"{what}: device form at bounds {bL}x{bM}")
    print(f"k-best: worst |table - E| at exhaustive k = {worst:.3e}")


# usePerm frames with 12+ detections whose tables the permanentProb route cannot give to 1e-9: its exact permanent
# (Nijenhuis-Wilf inclusion-exclusion over the ones-padded sub-matrix, as the reference computes it) cancels digits away.
# All are moments frames, measured on a B200 (relative error against E: 1.6e-9 at 1x12 to ~1.0 at 33x16 and 64x12); the
# CPU restatement of the same arithmetic misses by as much.  Every other status-0 frame, fused or routed, meets 1e-9.
CANCELLING = {("moments", L, M) for L, M in ((1, 12), (1, 16), (1, 31), (2, 12), (31, 12), (32, 12), (33, 16), (64, 12),
                                              (96, 12), (96, 16))}


def _perm_tables(api, frames):
    from probabilisticsemslam_b200 import synth
    shapes = list(frames)
    pb = synth.pack([frames[s]["C"] for s in shapes], [s[0] for s in shapes])
    return shapes, api.association_perm_probs_batch(pb), api.association_perm_from_moments_batch(
        [frames[s]["mom"] for s in shapes], NONASSIGN), pb


def same_in_batch(a, b, key, what):
    """The same frame's usePerm table from two calls: bit for bit on the fused pipeline (nM <= 11); to 1e-9 on the
    permanentProb route, which splits its permanent walks by the batch it runs in (the last bits move); status only on
    the CANCELLING frames, where those splits move the cancelled digits too."""
    if key[2] <= 11:
        np.testing.assert_array_equal(bits(a), bits(b), err_msg=what)
    elif key not in CANCELLING:
        np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-300, err_msg=what)


@gpu
def test_perm_every_shape(gpu_api, frames):
    """Status as the helper predicts it, and the same table from every entry point: the _host forms from costs and
    from moments, alone and in one mixed batch, the separate entry points, and the device form (nM <= 11)."""
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    import torch
    shapes, (mt, mst), (gt, gst), pb_all = _perm_tables(api, frames)
    ct, cst = composed(api, pb_all)  # the separate entry points: conditionCosts -> permanentProb -> scatter
    for i, (L, M) in enumerate(shapes):
        f = frames[(L, M)]
        what = f"{L}x{M} usePerm"
        tabs, st = api.association_perm_probs_batch(synth.pack([f["C"]], [L]))
        assert int(st[0]) == perm_status(f["C"], L), what
        assert int(mst[i]) == int(st[0]) == int(cst[i]), what
        same_in_batch(tabs[0], mt[i], ("costs", L, M), what + ": alone vs mixed")
        same_in_batch(tabs[0], ct[i], ("costs", L, M), what + ": vs the separate entry points")
        tc, sc = api.association_perm_probs_batch(synth.pack([f["Cg"]], [L]))
        tm, sm = api.association_perm_from_moments_batch([f["mom"]], NONASSIGN)
        assert int(sc[0]) == int(sm[0]) == int(gst[i]) == perm_status(f["Cg"], L), what + " (moments)"
        np.testing.assert_array_equal(bits(tc[0]), bits(tm[0]), err_msg=what + ": from costs vs from moments")
        same_in_batch(tm[0], gt[i], ("moments", L, M), what + ": moments alone vs mixed")
        if M <= 11:
            dev = api.moments_to_device([f["mom"]])
            for bL, bM in ((L, M), (MAX_DIM - 11, 11)):
                if bL < L:
                    continue
                p, po, st_d = api.association_perm_from_moments_batch_device(*dev, bL, bM, NONASSIGN)
                torch.cuda.synchronize()
                assert int(st_d[0]) == int(sm[0]), what
                td = p[:M * (L + 1)].cpu().numpy().reshape(M, L + 1)
                np.testing.assert_array_equal(bits(td), bits(tm[0]), err_msg=f"{what}: device form at bounds {bL}x{bM}")


PERM_TRUTH_CASES = [pytest.param(fam, L, M, id=f"{fam}-{L}x{M}",
                                 marks=[pytest.mark.xfail(strict=True, reason="cancellation in the permanentProb route")]
                                 if (fam, L, M) in CANCELLING else [])
                    for fam in ("costs", "moments") for L, M in SHAPES]


@gpu
@pytest.mark.parametrize("fam,L,M", PERM_TRUTH_CASES)
def test_perm_tables_equal_exact_marginals(gpu_api, frames, fam, L, M):
    """Wherever usePerm does not throw: its table equals E at the repo's rule (rtol 1e-9, atol 1e-300), its rows sum to 1
    (1e-12 on the fused pipeline, 1e-9 on the route), and where the k-best path can enumerate the frame exhaustively the
    two weight paths agree -- the one check that ties them together -- at the exhaustive k-best table's bound against E."""
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    f = frames[(L, M)]
    C, (E, n) = (f["C"], f["E"]) if fam == "costs" else (f["Cg"], f["Eg"])
    if L == 0 or perm_status(C, L):
        pytest.skip("no table to compare: no landmarks, or status 1")
    tabs, st = api.association_perm_probs_batch(synth.pack([C], [L]))
    assert int(st[0]) == 0
    t = tabs[0]
    rel = float(np.max(np.abs(t - E) / np.maximum(E, 1e-300)))
    print(f"usePerm {fam} {L}x{M}: max relative |table - E| = {rel:.3e}")
    np.testing.assert_allclose(t, E, rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(t.sum(axis=1), 1.0, rtol=0, atol=1e-12 if M <= 11 else 1e-9)
    if kbest_fits(L, M, max(n, 1)):
        kb = api.association_probs_batch(synth.pack([C], [L]), max(n, 1))[0]
        assert_truth(kb, E, f"{fam} {L}x{M} k-best")
        # at the k-best path's own bound: kBest2DCutoff drops hypotheses more than 42 above the best one, which moves
        # entries below ~1e-12 by up to a few 1e-7 relative (1e-19 absolute) while usePerm keeps them
        d = np.abs(kb - t)
        big = E >= 1e-6
        assert d.max() <= 1e-13 and np.all(d[big] <= 1e-9 * E[big]), f"k-best vs usePerm: {d.max():.3e}"


def ldlt_hard_frames(rng):
    """Frames whose S1 + S2 the pivoted LDLT finds hard: equal-magnitude diagonal pivots (the first-maximum rule), a
    singular sum with d inside and outside its range (the pseudo-inverse's DBL_MIN branch), an all-zero sum and an
    indefinite sum."""
    pairs = []
    for _ in range(24):  # ties between diagonal entries, of either sign, with off-diagonal terms
        t = rng.uniform(0.5, 3.0)
        diag = t * rng.choice([-1.0, 1.0], 3)
        diag[rng.integers(0, 3)] = rng.uniform(-0.5 * t, 0.5 * t)
        if rng.random() < 0.5:
            diag[:] = t * rng.choice([-1.0, 1.0], 3)
        A = np.diag(diag)
        for i, j in ((0, 1), (0, 2), (1, 2)):
            A[i, j] = A[j, i] = rng.uniform(-0.4, 0.4) * t
        pairs.append((A, rng.standard_normal(3)))
    for _ in range(8):  # singular: rank 2 and rank 1, d inside and outside the range
        u = rng.standard_normal((3, 2))
        A = u @ u.T
        pairs.append((A, u @ rng.standard_normal(2)))
        pairs.append((A, rng.standard_normal(3)))
        v = rng.standard_normal(3)
        pairs.append((np.outer(v, v), 2.0 * v))
        pairs.append((np.outer(v, v), rng.standard_normal(3)))
    pairs.append((np.zeros((3, 3)), rng.standard_normal(3)))  # all-zero sum
    pairs.append((np.zeros((3, 3)), np.zeros(3)))
    for _ in range(8):  # indefinite
        q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
        pairs.append(((q * np.array([1.0, -2.0, 0.5]) * rng.uniform(0.1, 10.0)) @ q.T, rng.standard_normal(3)))
    frames = []
    for A, d in pairs:
        S1 = rng.uniform(0.0, 1.0) * A
        S2 = A - S1  # the kernel adds S1 + S2 first; the oracle the same
        frames.append((np.zeros((1, 3)) + d, S1[None], np.zeros((1, 3)), S2[None]))
    return frames


@gpu
def test_quadric_costs_every_shape(gpu_api, oracle, frames):
    api = gpu_api
    fr = [f["mom"] for f in frames.values()] + ldlt_hard_frames(np.random.default_rng(15))
    got = api.quadric_cost_batch(fr, NONASSIGN)
    for i, (f, g) in enumerate(zip(fr, got)):
        want = oracle.quadric_cost_matrix(*f, NONASSIGN)
        np.testing.assert_array_equal(bits(g), bits(want), err_msg=f"frame {i} ({len(f[0])} x {len(f[2])})")


# ---- degenerate frames ---------------------------------------------------------------------------------------------------
def few_rows_frame(nonassign):
    """Three detections near landmark 0 only, dummies gated away: conditioning keeps 1 row for 3 detections."""
    C = np.full((5, 3), np.inf)
    C[0] = [1.0, 2.0, 3.0]
    C[1] = [80.0, 90.0, 100.0]
    C[2 + np.arange(3), np.arange(3)] = nonassign
    return C


def few_rows_moments(nonassign):
    lm = np.zeros((1, 3))
    dm = np.array([[0.1, 0, 0], [0, 0.2, 0], [0, 0, 0.3]])
    return (lm, np.eye(3)[None], dm, np.stack([np.eye(3)] * 3)), nonassign


def test_oracle_few_rows_status(oracle):
    for nonassign in (50.0, 100.0):
        for use_perm in (False, True):
            st, tab = oracle.association_probs(few_rows_frame(nonassign), 2, 50, use_perm)
            assert st == 3 and not tab.any()


@gpu
def test_few_rows_fail_the_same_on_both_paths(gpu_api, oracle):
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    for nonassign in (50.0, 100.0):
        C = few_rows_frame(nonassign)
        assert not api.association_probs_batch(synth.pack([C], [2]), 50)[0].any()
        tabs, st = api.association_perm_probs_batch(synth.pack([C], [2]))
        assert int(st[0]) == 3 and not tabs[0].any()
        for use_perm in (False, True):
            with pytest.raises(RuntimeError, match="status 3"):
                api.getAssignmentProbsFromCosts(C, 2, 50, usePerm=use_perm)
        fr, na = few_rows_moments(nonassign)
        assert not api.association_from_moments_batch([fr], na, 50)[0].any()
        for use_perm in (False, True):
            with pytest.raises(RuntimeError, match="status 3"):
                api.getAssignmentProbs(*fr, na, 50, usePerm=use_perm)


@gpu
def test_gated_dummy_with_enough_rows_follows_the_reference(gpu_api, oracle):
    """goodRows >= nM with a dummy gated away: both paths run and give the reference's (different) tables."""
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    C = np.array([[0.5, 0.3], [1, 2], [60, 70], [100, np.inf], [np.inf, 10]], np.float64)
    kb = api.getAssignmentProbsFromCosts(C, 3, 50)
    pm = api.getAssignmentProbsFromCosts(C, 3, 50, usePerm=True)
    for use_perm, got in ((False, kb), (True, pm)):
        st, want = oracle.association_probs(C, 3, 50, use_perm)
        assert st == 0
        np.testing.assert_allclose(got, want, rtol=1e-9, atol=0)
    assert abs(kb[1, 3] - pm[1, 3]) > 0.1  # detection 1 unassigned: ~0.23 from k-best, ~1.2e-4 from usePerm


@gpu
def test_frames_without_landmarks_at_every_nm(gpu_api, frames):
    """nL = 0 gives ones on both paths at any nM, alone and inside a batch with frames the Murty kernel does run."""
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    side = frames[(31, 16)]["C"]
    for M in (1, 32, 33, 64, 112, 113, 127, 128):
        C = np.full((M, M), np.inf)
        C[np.arange(M), np.arange(M)] = NONASSIGN
        for batch in ([C], [side, C]):
            nls = [0] if len(batch) == 1 else [31, 0]
            t = api.association_probs_batch(synth.pack(batch, nls), 200)[-1]
            np.testing.assert_array_equal(t, np.ones((M, 1)))
            p, st = api.association_perm_probs_batch(synth.pack(batch, nls))
            assert int(st[-1]) == 0
            np.testing.assert_array_equal(p[-1], np.ones((M, 1)))
        fr = (np.zeros((0, 3)), np.zeros((0, 3, 3)), 1e4 * np.arange(3 * M, dtype=np.float64).reshape(M, 3), np.stack([np.eye(3)] * M))
        np.testing.assert_array_equal(api.association_from_moments_batch([frames[(31, 16)]["mom"], fr], NONASSIGN, 200)[-1],
                                      np.ones((M, 1)))


@gpu
def test_frames_beyond_the_murty_kernel_are_named(gpu_api, frames, optin):
    api = gpu_api
    from probabilisticsemslam_b200 import synth
    L, M = 1, 127
    assert not kbest_fits(L, M, 50, optin)
    C = frames[(L, M)]["C"]
    with pytest.raises(RuntimeError, match=r"frame 1 \(nL=1, nM=127\)"):
        api.association_probs_batch(synth.pack([frames[(31, 16)]["C"], C], [31, L]), 50)
    with pytest.raises(RuntimeError, match=r"frame 1 \(nL=1, nM=127\)"):
        api.association_from_moments_batch([frames[(31, 16)]["mom"], frames[(L, M)]["mom"]], NONASSIGN, 50)
    # each fits alone, not together: 128 rows beside 113 detections
    a, b = (127, 1), (1, 113)
    assert kbest_fits(*a, 50, optin) and kbest_fits(*b, 50, optin)
    with pytest.raises(RuntimeError, match="do not fit together"):
        api.association_probs_batch(synth.pack([frames[a]["C"], frames[b]["C"]], [a[0], b[0]]), 50)
    # the multi-device form names the frame by its index in the caller's batch, not in its slice: two slices on one device
    from probabilisticsemslam_b200._lib import lib
    pb = synth.pack([frames[(31, 16)]["C"]] * 3 + [C], [31, 31, 31, L])
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    prob_off = np.concatenate([[0], np.cumsum(nM.astype(np.int64) * (nL + 1))[:-1]]).astype(np.int64)
    probs = np.zeros(int((nM.astype(np.int64) * (nL + 1)).sum()))
    devices = np.zeros(2, np.int32)
    rc = lib().pda_association_probs_batch_host_multi(pb.costs.ctypes.data, pb.cost_off.ctypes.data, nL.ctypes.data,
                                                      nM.ctypes.data, len(pb), 50, probs.ctypes.data, prob_off.ctypes.data,
                                                      devices.ctypes.data, 2)
    assert rc == -3
    assert "frame 3 (nL=1, nM=127)" in lib().pda_last_error().decode()


def infeasible_frame():
    """Dummies gated away and detections 0 and 1 in the gate of landmark 0 alone, detection 2 of landmarks 1 and 2:
    conditioning keeps 3 rows for 3 detections (goodRows >= nM), and no assignment of the kept rows is feasible."""
    C = np.full((6, 3), np.inf)
    C[0] = [1.0, 2.0, 80.0]
    C[1] = [90.0, 90.0, 1.0]
    C[2] = [90.0, 90.0, 2.0]
    C[3 + np.arange(3), np.arange(3)] = 100.0
    return C


@gpu
def test_infeasible_conditioned_frame_follows_the_reference(gpu_api, oracle):
    """goodRows >= nM but no feasible assignment: the k-best table has NaN where the reference divides 0 by 0 (so it is
    not the all-zero table of goodRows < nM, and the single-frame entry returns it rather than raising); the usePerm
    table is the reference's too."""
    api = gpu_api
    C = infeasible_frame()
    kb = api.getAssignmentProbsFromCosts(C, 3, 50)
    pm = api.getAssignmentProbsFromCosts(C, 3, 50, usePerm=True)
    for use_perm, got in ((False, kb), (True, pm)):
        st, want = oracle.association_probs(C, 3, 50, use_perm)
        assert st == 0
        np.testing.assert_allclose(got, want, rtol=1e-9, atol=0, equal_nan=True, err_msg=f"usePerm={use_perm}")
    assert np.isnan(kb[:, 3]).all() and not kb[:, :3].any()


def _driver_input(frames, nonassign):
    col = lambda c: np.asarray(c).transpose(0, 2, 1).reshape(-1)  # column-major 3x3, Eigen's layout
    parts = [f"{len(frames)} {nonassign!r}"]
    for lm, lc, mm, mc in frames:
        parts.append(f"{len(lm)} {len(mm)} " + " ".join(repr(float(x)) for x in
                                                      np.concatenate([np.ravel(lm), col(lc), np.ravel(mm), col(mc)])))
    return "\n".join(parts) + "\n"


@gpu
def test_cpp_kbest_entries_raise_on_few_rows(gpu_api, frames):
    """The C++ drop-in layer's k-best getAssignmentProbsFromMoments / getAssignmentProbsFromCosts: the library's tables on
    an ordinary frame, and the usePerm form's exception where conditioning keeps fewer rows than detections."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "build", "perm_association_b200")
    assert os.path.exists(exe), "tests/cpp/build/perm_association_b200 missing: run __graft_entry__.build()"
    fr = frames[(31, 16)]["mom"]
    run = subprocess.run([exe, "kbest"], input=_driver_input([fr], NONASSIGN), capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout[-500:] + run.stderr[-500:]
    want = gpu_api.association_from_moments_batch([fr], NONASSIGN, 200)[0]
    got = {}
    for ln in run.stdout.splitlines():
        w = ln.split()
        got.setdefault(w[0], []).append([float(x) for x in w[3:]])
    for kind in ("moments", "costs", "batch"):
        np.testing.assert_array_equal(bits(np.array(got[kind])), bits(want), err_msg=kind)
    few, na = few_rows_moments(100.0)
    run = subprocess.run([exe, "kbest"], input=_driver_input([few], na), capture_output=True, text=True, timeout=300)
    assert run.returncode == 1 and "throw getAssignmentProbs: conditionCosts kept fewer rows" in run.stdout, run.stdout[-500:]
