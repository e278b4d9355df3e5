"""permanentProb and conditionedPermanent: the device-pointer forms (pda_permanent_prob_batch,
pda_conditioned_permanent_batch) and the host forms, which stage their inputs and run the device form per chunk.

Tables, results and statuses of both forms must equal the bits pinned in tests/golden/permprob_host_bits.npz
(tests/golden/make_golden_permprob.py): the host forms' results from when they ran a separate materialising pipeline
(commit aa4e759).  That covers sub-matrices with a short side of at most 10 through the fused subset programme, larger
ones through the NW walk with its launch shape, negative results through the retry on the device, and permOpt 0 with the
same draws.  The device form must also run on device inputs only: one call captured in a CUDA graph and replayed on new
inputs gives the bits of direct calls.  The CPU tests at the bottom check the argument handling, which runs before any
device work."""
import ctypes
import functools
import hashlib
import os
import subprocess

import numpy as np
import pytest

from helpers import bits, golden
from probabilisticsemslam_b200 import synth

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
gpu = pytest.mark.gpu
HOST_CHUNK = 1 << 16  # sub-permanents per chunk of pda_permanent_prob_batch_host
SEED = 20260217


@pytest.fixture(scope="module")
def papi():
    import torch
    from probabilisticsemslam_b200 import _lib, api
    assert _lib.lib().pda_device_count() > 0, "no CUDA device visible: -m gpu tests must run on the GPU box"
    assert torch.cuda.is_available()
    _lib.lib().pda_set_approx_seed(SEED)
    return api


def run_device(pb, perm_opt, max_row=None, max_col=None, fill=None, ws_extra=0, ws_delta=0):
    """pda_permanent_prob_batch on a fresh upload of pb -> (tables, status), like api.permanent_prob_batch."""
    import torch
    from probabilisticsemslam_b200 import device
    plan = device.PermanentProbPlan(pb, perm_opt, max_num_row=max_row, max_num_col=max_col)
    if fill is not None:
        plan.probs.fill_(fill)
    if ws_extra or ws_delta:
        plan.workspace = torch.empty(plan.workspace.numel() + ws_extra + ws_delta, dtype=torch.uint8, device=plan.probs.device)
    plan.run()
    torch.cuda.synchronize()
    return plan.result()


def run_device_mats(mats, perm_opt, max_dim=None):
    import torch
    from probabilisticsemslam_b200 import device
    plan = device.ConditionedPermanentPlan(mats, perm_opt, max_dim=max_dim)
    plan.run()
    torch.cuda.synchronize()
    return plan.result()


@functools.cache
def _pinned():
    return golden("permprob_host_bits")


def pinned(key, walked):
    """(status, bits) of one pinned host call.  Sub-permanents the NW walk takes follow the launch shape, which follows
    the SM count: such cases run only on a device with the SM count the bits were pinned on."""
    z = _pinned()
    if walked:
        import torch
        sm, want = torch.cuda.get_device_properties(0).multi_processor_count, int(z["sm_count"])
        if sm != want:
            pytest.skip(f"NW-walked bits pinned on {z['device']} with {want} SMs; this device has {sm}")
    return z[key + ".status"], z[key + ".bits"]


def digests(tabs):
    """SHA-256 of each table's bits, as the pinned file stores them."""
    return np.array([np.frombuffer(hashlib.sha256(bits(t).tobytes()).digest(), np.uint8) for t in tabs]).reshape(-1, 32)


def assert_pinned_tables(got, key, what, skip=(), walked=False):
    want_st, want_dg = pinned(key, walked)
    tabs, st = got
    assert len(tabs) == len(want_st), what
    dg = digests(tabs)
    for p in range(len(want_st)):
        if p in skip:
            continue
        assert st[p] == want_st[p], f"{what}: status of problem {p}: {st[p]} != pinned {want_st[p]}"
        assert np.array_equal(dg[p], want_dg[p]), f"{what}: problem {p} (status {st[p]}) differs from the pinned bits"


def assert_pinned_mats(got, key, what, walked=False):
    want_st, want_bits = pinned(key, walked)
    np.testing.assert_array_equal(got[1], want_st, err_msg=f"{what}: status")
    np.testing.assert_array_equal(bits(got[0]), want_bits, err_msg=f"{what}: values")


def assert_tables(got, want, what, skip=()):
    (gt, gs), (wt, ws) = got, want
    for p in range(len(wt)):
        if p in skip:
            continue
        assert gs[p] == ws[p], f"{what}: status of problem {p}: {gs[p]} != {ws[p]}"
        np.testing.assert_array_equal(bits(gt[p]), bits(wt[p]), err_msg=f"{what}: problem {p} (status {ws[p]})")


def assert_mats(got, want, what):
    np.testing.assert_array_equal(got[1], want[1], err_msg=f"{what}: status")
    np.testing.assert_array_equal(bits(got[0]), bits(want[0]), err_msg=f"{what}: values")


def golden_problems():
    z1, za = golden("probs_config1"), golden("probs_appendixA")
    return synth.pack([z1["C"], za["C"]], [int(z1["nL"]), int(za["nL"])])


def golden_mats():
    z = golden("conditioned_permanent")
    return [z[f"A{i}"] for i in range(int(z["n"]))]


def g1_mixed():
    return synth.pack([synth.g1_dense(12, nM=m, first=100 * m).matrix(p) for m in range(2, 9) for p in range(12)],
                      [30] * (7 * 12))


def g2_conditioned(api, n=400):
    cond, _ = api.condition_costs_batch(synth.g2_gated(n, first=900))
    return cond


def nw_problems():
    """nM = 12..16 against a few landmarks: every sub-matrix has a short side of 11..15 and goes to the NW walk."""
    mats, nls = [], []
    for m in range(12, 17):
        pb = synth.g1_dense(2, nL=18 - m, nM=m, first=40 * m)
        mats += [pb.matrix(0), pb.matrix(1)]
        nls += [18 - m] * 2
    return mats, nls


def nw_mats():
    """Square matrices of the NW sizes, as conditioned matrices."""
    return [np.abs(np.sin(np.arange(k * k, dtype=np.float64).reshape(k, k) + k)) for k in (11, 12, 15, 16, 20)]


def ragged(api):
    """nM = 1, nL = 0, the NW sizes, a sub-matrix with more than 32 kept rows (status 1) and, last, two problems above
    maxNumRow = 44 / maxNumCol = 16 (status 2)."""
    g1 = synth.g1_dense(8, nL=30, first=7)
    mats, nls = [g1.matrix(p) for p in range(3)], [30] * 3
    mats.append(g1.matrix(3)[:, :1][np.r_[0:30, 30]]); nls.append(30)              # nM = 1
    mats.append(np.array([[10.0, 50.0], [40.0, 10.0]])); nls.append(0)             # nL = 0
    nw, nwl = nw_problems()
    mats += nw; nls += nwl
    mats.append(synth.g1_dense(1, nL=38, nM=4, first=3, scale=4.0).matrix(0)); nls.append(38)  # kept rows > 32
    mats.append(synth.g1_dense(1, nL=44, nM=3, first=5).matrix(0)); nls.append(44)              # nL + nM > 44
    mats.append(synth.g1_dense(1, nL=2, nM=17, first=6).matrix(0)); nls.append(2)               # nM > 16
    return synth.pack(mats, nls)


def invalid_opt_mats():
    return [np.eye(3) + 0.5, np.ones((2, 4))]


def approx_problems():
    return synth.pack([synth.g1_dense(20, nM=m, first=300 * m).matrix(p) for m in (2, 4, 6) for p in range(20)], [30] * 60)


def approx_mats():
    return [np.abs(np.cos(np.arange(r * c, dtype=np.float64).reshape(r, c))) + 0.05 for r, c in ((4, 4), (6, 5), (8, 8), (12, 12))]


def edge_mats():
    """Shapes at the edges of conditionedPermanent, with a matrix the NW walk takes among them: 0x0, 1xn, nx1, 1x40 and
    36x3 (more than 32 kept rows or columns: status 1) and 130x4 (a side above PDA_MAX_DIM: status 1)."""
    rng = np.random.default_rng(SEED)
    return [rng.uniform(0.1, 1.0, s) for s in ((4, 4), (0, 0), (1, 5), (5, 1), (1, 40), (36, 3), (130, 4), (12, 14))]


def chunked_problems():
    return synth.g1_dense(600, first=50)


# ---- bit identity with the pinned host results -------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("perm_opt", [1, 2])
def test_golden_inputs(papi, perm_opt):
    pb, mats = golden_problems(), golden_mats()
    assert_pinned_tables(run_device(pb, perm_opt), f"golden.{perm_opt}", "probs golden, device")
    assert_pinned_tables(papi.permanent_prob_batch(pb, perm_opt), f"golden.{perm_opt}", "probs golden, host")
    assert_pinned_mats(run_device_mats(mats, perm_opt), f"golden_mats.{perm_opt}", "conditioned golden, device")
    assert_pinned_mats(papi.conditioned_permanent_batch(mats, perm_opt), f"golden_mats.{perm_opt}", "conditioned golden, host")


@gpu
@pytest.mark.parametrize("perm_opt", [1, 2])
def test_g1_and_conditioned_g2(papi, perm_opt):
    for what, pb in (("g1", g1_mixed()), ("g2", g2_conditioned(papi))):
        assert_pinned_tables(run_device(pb, perm_opt), f"{what}.{perm_opt}", f"{what}, device")
        assert_pinned_tables(papi.permanent_prob_batch(pb, perm_opt), f"{what}.{perm_opt}", f"{what}, host")


@gpu
@pytest.mark.parametrize("perm_opt", [1, 2])
def test_ragged_batch_with_nw_items_and_statuses(papi, perm_opt):
    pb = ragged(papi)
    n = len(pb)
    got = run_device(pb, perm_opt, max_row=44, max_col=16, fill=-7.0)
    want = papi.permanent_prob_batch(pb, perm_opt)
    assert_pinned_tables(got, f"ragged.{perm_opt}", "ragged, device", skip=(n - 2, n - 1), walked=True)
    assert_pinned_tables(want, f"ragged.{perm_opt}", "ragged, host", walked=True)
    assert want[1][n - 3] == 1 and got[1][n - 3] == 1
    assert list(got[1][n - 2:]) == [2, 2]
    for p in (n - 2, n - 1):
        assert np.all(got[0][p] == -7.0), "a status-2 table must be left untouched"
    # the same problems one by one as conditioned matrices, NW sizes included
    mats = nw_mats()
    assert_pinned_mats(run_device_mats(mats, perm_opt), f"nw_mats.{perm_opt}", "conditioned NW, device", walked=True)
    assert_pinned_mats(papi.conditioned_permanent_batch(mats, perm_opt), f"nw_mats.{perm_opt}", "conditioned NW, host",
                       walked=True)


@gpu
def test_invalid_perm_opt_matches_host(papi):
    pb = ragged(papi)
    n = len(pb)
    assert_pinned_tables(run_device(pb, 5, max_row=44, max_col=16), "ragged.5", "permOpt 5, device", skip=(n - 2, n - 1))
    assert_pinned_tables(papi.permanent_prob_batch(pb, 5), "ragged.5", "permOpt 5, host")
    mats = invalid_opt_mats()
    assert_pinned_mats(run_device_mats(mats, -1), "invalid_opt_mats.-1", "conditioned permOpt -1, device")
    assert_pinned_mats(papi.conditioned_permanent_batch(mats, -1), "invalid_opt_mats.-1", "conditioned permOpt -1, host")


@gpu
@pytest.mark.parametrize("perm_opt", [0, 1, 2])
def test_host_edge_shapes(papi, perm_opt):
    got = papi.conditioned_permanent_batch(edge_mats(), perm_opt)
    assert_pinned_mats(got, f"edges.{perm_opt}", f"edge shapes, permOpt {perm_opt}", walked=perm_opt != 0)
    assert list(got[1][4:7]) == [1, 1, 1]


# ---- the negative-permanent retry -------------------------------------------------------------------------------
def retry_matrices(seeds):
    """Upper-triangular matrices with tiny diagonals: the permanent is the product of the diagonal, far below the
    rounding error of the NW sum over row sums of order one, so its sign comes out at random."""
    out = []
    for s in seeds:
        rng = np.random.default_rng(s)
        n = 12 + s % 5
        A = np.triu(rng.uniform(0.1, 1.0, (n, n)), 1)
        A[np.arange(n), np.arange(n)] = 10.0 ** -rng.uniform(3, 8, n)
        out.append(A)
    return out


def transposed_conditioned(A):
    """conditionedPermanent's first attempt: positive columns scaled by 1 / sqrt(max * min positive), transposed."""
    keep_c = [j for j in range(A.shape[1]) if A[:, j].max() > 0]
    sc = np.array([1.0 / np.sqrt(A[:, j].max() * A[A[:, j] > 0, j].min()) for j in keep_c])
    B = A[:, keep_c] * sc
    return np.ascontiguousarray(B[B.max(axis=1) > 0].T)


RETRY_SEEDS = list(range(24))


@gpu
def test_retry_of_negative_permanents(papi):
    mats = retry_matrices(RETRY_SEEDS)
    first, _ = papi.permanent_batch([transposed_conditioned(A) for A in mats])
    negative = [i for i in range(len(mats)) if first[i] < 0]
    assert negative, "no seeded input reaches the retry"
    for perm_opt in (1, 2):
        got = run_device_mats(mats, perm_opt)
        assert_pinned_mats(got, f"retry.{perm_opt}", f"retry permOpt {perm_opt}, device", walked=True)
        assert_pinned_mats(papi.conditioned_permanent_batch(mats, perm_opt), f"retry.{perm_opt}",
                           f"retry permOpt {perm_opt}, host", walked=True)
        # the retried values are the untransposed walk's, not the negative first attempt's
        assert all(bits(np.array([got[0][i]]))[0] != bits(np.array([first[i]]))[0] for i in negative)


# ---- permOpt 0 -------------------------------------------------------------------------------------------------
@gpu
def test_approximation_same_draws_as_host(papi):
    from truth import perm_injective
    pb = approx_problems()
    assert_pinned_tables(run_device(pb, 0), "approx.0", "permOpt 0, device")
    assert_pinned_tables(papi.permanent_prob_batch(pb, 0), "approx.0", "permOpt 0, host")
    mats = approx_mats()
    got = run_device_mats(mats, 0)
    assert_pinned_mats(got, "approx_mats.0", "conditioned permOpt 0, device")
    assert_pinned_mats(papi.conditioned_permanent_batch(mats, 0), "approx_mats.0", "conditioned permOpt 0, host")
    for A, est in zip(mats, got[0]):  # 300 trials: the estimator's spread, far inside a factor of two
        exact = perm_injective(A)
        assert abs(est / exact - 1.0) < 0.5, (A.shape, est, exact)


# ---- accuracy ------------------------------------------------------------------------------------------------
@gpu
def test_against_cancellation_free_truth(papi):
    from truth import permanent_prob_truth
    pb = synth.pack([synth.g1_dense(2, nL=20, nM=m, first=70 * m).matrix(p) for m in range(2, 9) for p in range(2)], [20] * 14)
    tabs, st = run_device(pb, 1)  # nL + nM - 1 <= 32 kept rows: nothing throws
    for p in range(len(pb)):
        assert st[p] == 0
        np.testing.assert_allclose(tabs[p], permanent_prob_truth(pb.matrix(p), int(pb.nL[p])), rtol=1e-9, atol=1e-300)


# ---- stream order and graphs -----------------------------------------------------------------------------------
@gpu
def test_graph_capture_and_replay(papi):
    import torch
    from probabilisticsemslam_b200 import device
    a, b = synth.g1_dense(40, first=11), synth.g1_dense(40, first=11)
    b.costs = np.where(np.isfinite(b.costs), b.costs * 0.75 + 1.0, b.costs)  # same shapes, new values
    plan = device.PermanentProbPlan(a, 1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        plan.run()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        plan.run()
    plan.costs.copy_(torch.from_numpy(b.costs).to(plan.costs.device))
    g.replay()
    torch.cuda.synchronize()
    assert_tables(plan.result(), run_device(b, 1), "graph replay")
    # conditioned matrices, with the NW walk and the retry inside the graph
    m1, m2 = retry_matrices(RETRY_SEEDS[:8]), retry_matrices([s + 100 for s in RETRY_SEEDS[:8]])  # same shapes
    cp = device.ConditionedPermanentPlan(m1, 1)
    with torch.cuda.stream(s):
        cp.run()
    torch.cuda.current_stream().wait_stream(s)
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        cp.run()
    flat = np.concatenate([m.reshape(-1, order="F") for m in m2] + [np.zeros(1)])
    cp.mats.copy_(torch.from_numpy(flat).to(cp.mats.device))
    g2.replay()
    torch.cuda.synchronize()
    assert_mats(cp.result(), run_device_mats(m2, 1), "conditioned graph replay")


# ---- scale and workspace ---------------------------------------------------------------------------------------
def host_chunks(pb):
    """The problem slices pda_permanent_prob_batch_host runs as one chunk each."""
    cuts, p0, items = [], 0, 0
    for p in range(len(pb)):
        add = int(pb.nM[p]) * (int(pb.nL[p]) + 1) if pb.nM[p] > 1 else 0
        if p > p0 and items + add > HOST_CHUNK:
            cuts.append((p0, p)); p0, items = p, 0
        items += add
    return cuts + [(p0, len(pb))]


@gpu
def test_beyond_one_host_chunk(papi):
    pb = chunked_problems()
    assert int((pb.nM.astype(np.int64) * (pb.nL + 1)).sum()) > HOST_CHUNK
    tabs, st = run_device(pb, 1)
    assert_pinned_tables((tabs, st), "chunks.1", "600 problems, device")
    assert_pinned_tables(papi.permanent_prob_batch(pb, 1), "chunks.1", "600 problems, host")
    chunks = host_chunks(pb)
    assert len(chunks) > 1
    for lo, hi in chunks:
        wt, ws = papi.permanent_prob_batch(pb.slice(lo, hi), 1)
        assert_tables(([tabs[p] for p in range(lo, hi)], st[lo:hi]), (wt, ws), f"chunk {lo}:{hi}")


@gpu
def test_smallest_workspace(papi):
    from probabilisticsemslam_b200._lib import PdaError
    pb = synth.pack(*nw_problems())
    small = run_device(pb, 1)
    assert_pinned_tables(small, "nw.1", "NW problems, smallest workspace", walked=True)
    assert_pinned_tables(papi.permanent_prob_batch(pb, 1), "nw.1", "NW problems, host", walked=True)
    assert_tables(run_device(pb, 1, ws_extra=1 << 20), small, "full workspace")
    with pytest.raises(PdaError, match="error -4"):
        run_device(pb, 1, ws_delta=-1)


# ---- C++ driver ----------------------------------------------------------------------------------------------------
@gpu
def test_cpp_driver_graph(papi):
    exe = os.path.join(ROOT, "tests", "cpp", "build", "permprob_device_b200")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.split("\n")
    direct = [l for l in lines if l.startswith("direct ")]
    replay = [l for l in lines if l.startswith("replay ")]
    assert direct and [l[7:] for l in direct] == [l[7:] for l in replay]


# ---- CPU: argument handling ----------------------------------------------------------------------------------------
def _lib():
    from probabilisticsemslam_b200._lib import lib
    return lib()


def test_symbols_exported():
    so = ctypes.CDLL(os.path.join(ROOT, "probabilisticsemslam_b200", "libpda_b200.so"))
    for name in ("pda_permanent_prob_workspace_bytes", "pda_permanent_prob_batch",
                 "pda_conditioned_permanent_workspace_bytes", "pda_conditioned_permanent_batch"):
        assert hasattr(so, name), name


def test_argument_errors():
    L = _lib()
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.cast(buf, ctypes.c_void_p).value
    args = [p, p, p, p, 3, 10, 30, 8, 4, 1, p, p, p, p, 1 << 16, None]
    def call(**kw):
        a = list(args)
        for i, v in kw.items():
            a[int(i[1:])] = v
        rc = L.pda_permanent_prob_batch(*a)
        return rc, L.pda_last_error().decode()
    assert call(a0=None) == (-1, "permanent_prob: NULL argument")
    assert call(a13=None)[0] == -1
    assert call(a4=-1) == (-1, "permanent_prob: nProblems < 0")
    assert call(a4=0)[0] == 0
    assert call(a5=-1)[0] == -1
    assert call(a7=200)[0] == -3
    assert call(a8=0)[0] == -1
    rc, msg = call(a14=64)
    assert rc == -4 and "workspace" in msg
    assert L.pda_permanent_prob_workspace_bytes(-1, 0, 0, 8, 4, 1) == -1
    margs = [p, p, p, p, 2, 8, 1, p, p, p, 1 << 16, None]
    def mcall(**kw):
        a = list(margs)
        for i, v in kw.items():
            a[int(i[1:])] = v
        return L.pda_conditioned_permanent_batch(*a), L.pda_last_error().decode()
    assert mcall(a7=None) == (-1, "conditioned_permanent: NULL argument")
    assert mcall(a4=-3)[0] == -1
    assert mcall(a5=-1)[0] == -1
    assert mcall(a5=129)[0] == -3
    rc, msg = mcall(a10=16)
    assert rc == -4 and "workspace" in msg
    assert L.pda_conditioned_permanent_workspace_bytes(-1, 8, 1) == -1


def test_host_argument_errors():
    L = _lib()
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.cast(buf, ctypes.c_void_p).value
    # permOpt outside 0..2, where the reference throws: 0 and status 1, without a device
    out, st = np.full(3, 5.0), np.zeros(3, np.int32)
    assert L.pda_conditioned_permanent_batch_host(p, p, p, p, 3, 7, out.ctypes.data, st.ctypes.data, 0) == 0
    assert list(out) == [0.0] * 3 and list(st) == [1] * 3
    # NULL arguments and negative counts fail before any device call (without a device that would be -2)
    for i in range(6):
        args = [p, p, p, p, 2, 1, p, p, 0]
        args[i if i < 4 else i + 2] = None
        assert L.pda_conditioned_permanent_batch_host(*args) == -1
        assert L.pda_last_error().decode() == "conditioned_permanent: NULL argument"
    assert L.pda_conditioned_permanent_batch_host(p, p, p, p, -1, 1, p, p, 0) == -1
    assert L.pda_last_error().decode() == "conditioned_permanent: nMats < 0"
    for i in (0, 1, 2, 3, 6, 7, 8):
        args = [p, p, p, p, 3, 1, p, p, p, 0]
        args[i] = None
        assert L.pda_permanent_prob_batch_host(*args) == -1
        assert L.pda_last_error().decode() == "permanent_prob: NULL argument"
    assert L.pda_permanent_prob_batch_host(p, p, p, p, -1, 1, p, p, p, 0) == -1
    assert L.pda_last_error().decode() == "permanent_prob: nProblems < 0"


def test_no_device_is_a_cuda_error():
    if _lib().pda_device_count() > 0:
        pytest.skip("a device is visible")
    L = _lib()
    buf = ctypes.create_string_buffer(1 << 20)
    p = ctypes.cast(buf, ctypes.c_void_p).value
    assert L.pda_permanent_prob_batch(p, p, p, p, 3, 10, 30, 8, 4, 1, p, p, p, p, 1 << 20, None) == -2
    assert L.pda_conditioned_permanent_batch(p, p, p, p, 2, 8, 1, p, p, p, 1 << 20, None) == -2
    assert L.pda_permanent_prob_workspace_bytes(3, 10, 30, 8, 4, 1) == -2
