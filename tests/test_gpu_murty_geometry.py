"""The Murty kernels in every launch geometry they choose, against the CPU oracle.

murty_geometry (murty_kernel.cu), the wpc halving of occupancy_one, murty_cta_geometry (murty_cta_kernel.cu) and the
path choice of pda_capi.cu pick, from maxNumRow, maxNumCol, k and whether weights are fused, among distinct regimes:
row slots per lane R = 1 / 2 / 4, a heap top in shared memory or none, 4 / 2 / 1 warps per CTA, the pruning kernel
admitted or not (k <= 2, its open list beyond 2048 slots, its shared memory beyond the opt-in limit), its open list
in shared memory or in the arena, the one-CTA-per-problem kernel (numCol <= 16) or not.  Each regime lays out shared
memory and the arena differently.  This file restates the geometry in Python, pins the restatement to the library
through pda_murty_workspace_bytes, and then runs one table of cases -- each asserted to land in the regime it names --
under all three kernels, bit for bit against the oracle; the same problems under loose declared bounds (what a graph
captured for larger frames runs); the k-ladder form in the same regimes; and the limits, which must come back as
errors."""
from __future__ import annotations

import functools
from dataclasses import dataclass

import numpy as np
import pytest

from helpers import assert_kbest_equal, bits
from probabilisticsemslam_b200 import synth

# ---- the geometry, restated (murty_device.cuh, murty_kernel.cu, murty_cta_kernel.cu, pda_internal.h) ----------------
B200_SMEM_OPTIN = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB); the GPU tests read the device
MAX_DIM = 128             # PDA_MAX_DIM
HEAP_ENTRY = 16           # sizeof(HeapEntry)
MURTY_WPC, MURTY_MINB, FAST_MINB, PQ_SLACK = 4, 6, 5, 8
CTA_MAX_COL, CTA_WARPS, CTA_RECORDS, CTA_MAXTASKS = 16, 16, 64, 48
CTA_TASK, CTA_CTL = 12, 112  # sizeof(Task), sizeof(CtaCtl)
NODE_LIMIT = 1 << 30
WS_LIMIT = 4 << 30           # no call here may ask for more workspace than this


def _ru(x, m):
    return (x + m - 1) // m * m


def _wpc(smem_per_warp, optin):
    wpc = MURTY_WPC
    while wpc > 1 and wpc * smem_per_warp > optin:
        wpc >>= 1
    return wpc


@dataclass
class Geometry:
    error: str | None = None     # None, "invalid", "dim", "nodes" or "smem": what murty_geometry rejects
    R: int = 0
    heap_top_cap: int = 0
    smem_per_warp: int = 0
    wpc: int = 0
    fast_ok: bool = False
    pq_cap: int = 0
    pq_in_smem: bool = False
    fast_smem_per_warp: int = 0
    fast_wpc: int = 0
    arena_stride: int = 0
    cta: bool = False            # the CTA kernel can take it (numCol <= 16 and murty_cta_geometry succeeds)
    cta_arena_stride: int = 0

    @property
    def heap_top(self):
        return self.heap_top_cap > 0


def geometry(k, rows, cols, weights, optin):
    """murty_geometry + occupancy_one's warps per CTA + murty_cta_geometry."""
    if k < 1 or rows < 1 or cols < 1 or cols > rows:
        return Geometry(error="invalid")
    if rows > MAX_DIM:
        return Geometry(error="dim")
    g = Geometry()
    g.R = (rows + 31) // 32
    if g.R == 3:
        g.R = 4
    D = 32 * g.R
    node_stride = _ru(18 * _ru(rows, 8) + 4 * (g.R + 1), 16)
    nodes = 1 + (k - 1) * cols
    if nodes > NODE_LIMIT:
        return Geometry(error="nodes")
    heap_bytes = _ru(nodes, 8) * HEAP_ENTRY
    g.arena_stride = _ru(heap_bytes + nodes * node_stride, 256)
    c_cap = _ru(rows * cols, 2)
    p_cap = c_cap if weights else 0
    base = _ru(8 * (c_cap + p_cap + 2 * D) + 3 * 2 * D, 16)
    budget = (227 * 1024 - MURTY_MINB * 1024) // (MURTY_WPC * MURTY_MINB)
    top = (budget - base) // HEAP_ENTRY if budget > base else 0
    top = min(top, nodes)
    g.heap_top_cap = 0 if top < 3 else top
    g.smem_per_warp = base + g.heap_top_cap * HEAP_ENTRY
    g.pq_cap = _ru(k + 2 * cols + PQ_SLACK + 32, 32)
    g.fast_ok = k > 2 and g.pq_cap <= 64 * 32 and g.pq_cap * 12 <= heap_bytes
    fast_budget = (227 * 1024 - FAST_MINB * 1024) // (MURTY_WPC * FAST_MINB)
    g.pq_in_smem = base + g.pq_cap * 12 + (g.pq_cap >> 5) * 8 <= fast_budget
    g.fast_smem_per_warp = _ru(base + (g.pq_cap >> 5) * 8 + (g.pq_cap * 12 if g.pq_in_smem else 0), 16)
    if g.smem_per_warp > optin:
        return Geometry(error="smem")
    if g.fast_smem_per_warp > optin:
        g.fast_ok = False
    g.wpc = _wpc(g.smem_per_warp, optin)
    g.fast_wpc = _wpc(g.fast_smem_per_warp, optin) if g.fast_ok else g.wpc
    if cols <= CTA_MAX_COL:
        cta_nodes = 1 + k * cols + 16 * cols
        if cta_nodes <= NODE_LIMIT:
            order = k * 16 + ((k + 3) & ~3) * 4 + k * CTA_MAX_COL
            nodes_off = _ru(_ru(cta_nodes, 8) * HEAP_ENTRY + order, 256)
            g.cta_arena_stride = _ru(nodes_off + cta_nodes * node_stride, 256)
            off = _ru(8 * (c_cap + p_cap) + CTA_WARPS * _ru(22 * D, 16) + 8 * CTA_RECORDS * CTA_MAX_COL
                      + 4 * CTA_RECORDS + 2 * CTA_TASK * CTA_MAXTASKS + 32, 16)
            off = _ru(off + CTA_CTL, 16)
            g.cta = (optin - off) // HEAP_ENTRY >= 32
    return g


def workspace_bytes(k, rows, cols, path, optin):
    """pda_murty_workspace_bytes(1, k, rows, cols) under a forced path (weights do not change the arenas)."""
    g = geometry(k, rows, cols, False, optin)
    ws = 256 + g.arena_stride + 2 * 256  # the arena, then the cost order and the fallback list of one problem
    if path == "cta" and g.cta:
        ws = max(ws, 256 + g.cta_arena_stride)
    return ws


@functools.lru_cache(maxsize=None)
def fast_smem_cutoff(rows, cols, weights, optin):
    """The largest k at which the pruning kernel's shared memory still fits (rows x cols, pqCap below its own limit)."""
    k = 3
    while geometry(k + 1, rows, cols, weights, optin).fast_ok:
        k += 1
    return k


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _g1(n, nL, nM, first, integer=False):
    return lambda: synth.g1_dense(n, nL=nL, nM=nM, first=first, integer=integer)


def _square(n, dim, seed):
    """Square and dense (nL = 0, every entry finite): every permutation is feasible."""
    def build():
        rng = np.random.default_rng(seed)
        return synth.pack([rng.uniform(0.0, 20.0, (dim, dim)) for _ in range(n)], [0] * n)
    return build


def _band(n, nM, seed):
    """Detection j may take landmark j or j + 1 and nothing else (its dummy row is +inf): exactly nM + 1 assignments.
    Costs below 0.5, so the relative cut-off of 42 keeps all of them."""
    def build():
        rng = np.random.default_rng(seed)
        mats = []
        for _ in range(n):
            C = np.full((2 * nM + 1, nM), np.inf)
            j = np.arange(nM)
            C[j, j] = rng.uniform(0.0, 0.5, nM)
            C[j + 1, j] = rng.uniform(0.0, 0.5, nM)
            mats.append(C)
        return synth.pack(mats, [nM + 1] * n)
    return build


def _negated(build):
    """For maximize: gated entries become -inf."""
    def neg():
        pb = build()
        return synth.pack([np.where(np.isfinite(m), -m, -np.inf) for m in (pb.matrix(p) for p in range(len(pb)))],
                          list(pb.nL))
    return neg


@dataclass(frozen=True)
class Case:
    name: str
    build: object    # () -> ProblemBatch
    k: object        # int, or "fast_smem_last" / "fast_smem_first": either side of the pruning kernel's smem cut-off
    mode: str        # "gated": CUT_RELATIVE + WEIGHTS_GATED; "nocut": CUT_NONE; "nocut_max": CUT_NONE, maximize
    expect: tuple    # (Geometry field, value) pairs the case must land on
    found: int | None = None  # nFound of every problem when the enumeration runs out before k

    @property
    def weights(self):
        return self.mode == "gated"


CASES = [
    # the CTA kernel at 13-16 detections (16 = a full split record), R = 1 / 2 / 4
    Case("cta_13x31_R1", _g1(3, 18, 13, 60100), 200, "gated", (("cta", True), ("R", 1))),
    Case("cta_14x54_R2", _g1(3, 40, 14, 60200), 200, "gated", (("cta", True), ("R", 2), ("heap_top", False))),
    Case("cta_15x95_R4", _g1(3, 80, 15, 60300), 150, "nocut", (("cta", True), ("R", 4))),
    Case("cta_16x116_R4", _g1(2, 100, 16, 60400), 300, "gated", (("cta", True), ("R", 4), ("heap_top", False))),
    Case("cta_16x32_R1_int", _g1(3, 16, 16, 60500, integer=True), 300, "gated", (("cta", True), ("R", 1))),
    Case("cta_16x16_square", _square(3, 16, 60600), 200, "gated", (("cta", True), ("R", 1))),
    Case("cta_16x33_band", _band(2, 16, 60700), 50, "gated", (("cta", True), ("R", 2)), found=17),
    # heap top in shared memory at R = 4
    Case("heaptop_8x98_R4", _g1(3, 90, 8, 60800), 300, "nocut", (("R", 4), ("heap_top", True), ("wpc", 4))),
    # 17-32 detections
    Case("w24x32_R1", _g1(3, 8, 24, 61000), 300, "gated", (("cta", False), ("R", 1), ("fast_ok", True))),
    Case("w24x64_R2", _g1(3, 40, 24, 61100), 400, "gated", (("cta", False), ("R", 2), ("wpc", 4), ("fast_ok", True))),
    Case("w24x64_int", _g1(3, 40, 24, 61200, integer=True), 200, "nocut", (("cta", False), ("fast_ok", True))),
    # 33-64 detections: two warps per CTA with weights
    Case("w48x88_wpc2", _g1(3, 40, 48, 61300), 200, "gated", (("R", 4), ("wpc", 2), ("fast_ok", True))),
    Case("w64x94_int_wpc2", _g1(2, 30, 64, 61400, integer=True), 100, "gated", (("wpc", 2), ("fast_ok", True))),
    Case("w64x64_square_wpc2", _square(2, 64, 61500), 100, "gated", (("R", 2), ("wpc", 2))),
    Case("w40x40_square_max", _square(2, 40, 61600), 100, "nocut_max", (("R", 2), ("wpc", 4))),
    Case("w40x81_band", _band(2, 40, 61700), 100, "nocut", (("R", 4), ("cta", False)), found=41),
    Case("w60x121_band_wpc1", _band(2, 60, 61800), 100, "gated", (("wpc", 1), ("fast_ok", True)), found=61),
    # 100-112 detections
    Case("w100x120_wpc2", _g1(2, 20, 100, 62000), 60, "nocut", (("wpc", 2), ("heap_top", False), ("fast_ok", True))),
    Case("w100x126_int_wpc1", _g1(2, 26, 100, 62100, integer=True), 60, "gated", (("wpc", 1), ("fast_ok", True))),
    Case("w100x120_k2", _g1(2, 20, 100, 62200), 2, "gated", (("wpc", 1), ("fast_ok", False))),
    Case("w112x128_max", _negated(_g1(2, 16, 112, 62300)), 40, "nocut_max", (("wpc", 1),)),
    Case("w128x128_square_wpc1", _square(1, 128, 62400), 30, "nocut", (("R", 4), ("wpc", 1))),
    # the largest admitted shape: 128 x 112 with weights, one warp per CTA, then k either side of the pruning kernel's
    # shared-memory cut-off
    Case("w112x128_k50", _g1(2, 16, 112, 62500), 50, "gated", (("wpc", 1), ("fast_ok", True), ("fast_wpc", 1))),
    Case("w112x128_fast_last", _g1(1, 16, 112, 62600), "fast_smem_last", "gated", (("wpc", 1), ("fast_ok", True))),
    Case("w112x128_fast_first", _g1(1, 16, 112, 62700, integer=True), "fast_smem_first", "gated",
         (("wpc", 1), ("fast_ok", False))),
    # the pruning kernel's open list: 2048 slots at most (8 detections: k = 1992 fits, 1993 does not)
    Case("pq_8x38_k1992", _g1(2, 30, 8, 62800), 1992, "gated",
         (("fast_ok", True), ("pq_cap", 2048), ("pq_in_smem", False), ("heap_top", True))),
    Case("pq_8x38_k1993", _g1(2, 30, 8, 62900), 1993, "gated", (("fast_ok", False), ("pq_cap", 2080))),
]
CASE_IDS = [c.name for c in CASES]


def _dims(pb):
    return int(pb.num_row.max()), int(pb.nM.max())


def case_k(case, optin):
    if isinstance(case.k, int):
        return case.k
    kmax = fast_smem_cutoff(MAX_DIM, 112, True, optin)
    return kmax if case.k == "fast_smem_last" else kmax + 1


def case_geometry(case, pb, optin):
    rows, cols = _dims(pb)
    return geometry(case_k(case, optin), rows, cols, case.weights, optin)


def _assert_regime(case, pb, optin):
    g = case_geometry(case, pb, optin)
    assert g.error is None, f"{case.name}: the geometry rejects it ({g.error})"
    for field, want in case.expect:
        assert getattr(g, field) == want, f"{case.name}: {field} = {getattr(g, field)}, the case is meant for {want}"
    return g


# ---- CPU: the restatement and the table, at a B200's opt-in limit ----------------------------------------------------
def test_restatement_figures_at_b200_limit():
    optin = B200_SMEM_OPTIN
    big = geometry(50, 128, 112, True, optin)
    assert big.smem_per_warp == 232192 and big.wpc == 1 and big.heap_top_cap == 0
    assert geometry(50, 128, 113, True, optin).error == "smem"
    assert geometry(50, 128, 113, False, optin).error is None
    assert geometry(50, 129, 3, False, optin).error == "dim"
    assert geometry(1 << 24, 65, 65, False, optin).error == "nodes"
    kmax = fast_smem_cutoff(128, 112, True, optin)
    assert 700 < kmax < 800 and geometry(kmax + 1, 128, 112, True, optin).pq_cap <= 2048
    assert geometry(1992, 38, 8, False, optin).fast_ok and not geometry(1993, 38, 8, False, optin).fast_ok
    kitti_graph = geometry(200, 128, 28, True, optin)  # a KITTI frame under bounds maxNL = 100, maxNM = 28
    assert kitti_graph.wpc == 2 and not kitti_graph.heap_top and not kitti_graph.cta


def test_every_case_lands_in_its_regime_at_b200_limit():
    for case in CASES:
        pb = case.build()
        _assert_regime(case, pb, B200_SMEM_OPTIN)


def test_the_table_reaches_every_regime():
    """Across the table: R 1/2/4, heap top on/off, 4/2/1 warps per CTA, the pruning kernel on and off (k <= 2, pqCap,
    shared memory), its list in shared memory and in the arena, CTA on and off, and runs ending before k."""
    seen = set()
    for case in CASES:
        g = case_geometry(case, case.build(), B200_SMEM_OPTIN)
        seen |= {("R", g.R), ("heap_top", g.heap_top), ("wpc", g.wpc), ("fast_ok", g.fast_ok), ("cta", g.cta),
                 ("cols>16", _dims(case.build())[1] > 16), ("exhausted", case.found is not None)}
        if g.fast_ok:
            seen.add(("pq_in_smem", g.pq_in_smem))
    want = {("R", 1), ("R", 2), ("R", 4), ("heap_top", True), ("heap_top", False), ("wpc", 4), ("wpc", 2), ("wpc", 1),
            ("fast_ok", True), ("fast_ok", False), ("pq_in_smem", True), ("pq_in_smem", False), ("cta", True),
            ("cta", False), ("cols>16", True), ("exhausted", True)}
    assert want <= seen, want - seen
    ks = {case.k for case in CASES}
    assert {2, 1992, 1993, "fast_smem_last", "fast_smem_first"} <= ks


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def optin():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


_ORACLE = {}


def _oracle_result(oracle, case, pb, k):
    """Per problem (nFound, row4col, col4row, gain), plus the weight tables of a gated case; computed once per module."""
    key = case.name
    if key not in _ORACLE:
        if case.mode == "gated":
            w = oracle.batch(pb, k, threads=8, want_probs=True, want_lists=True)
            lists = []
            for p in range(len(pb)):
                n, nc, nr = int(w["n_found"][p]), int(pb.nM[p]), int(pb.num_row[p])
                lists.append((n, w["row4col"][w["r4c_off"][p]:w["r4c_off"][p] + n * nc].reshape(n, nc),
                              w["col4row"][w["c4r_off"][p]:w["c4r_off"][p] + n * nr].reshape(n, nr),
                              w["gain"][p * k:p * k + n]))
            _ORACLE[key] = (lists, w["probs"])
        else:
            maxi = case.mode == "nocut_max"
            _ORACLE[key] = ([oracle.kbest2d(k, pb.matrix(p), maxi) for p in range(len(pb))], None)
    return _ORACLE[key]


def _run_case(api, case, pb, k):
    if case.mode == "gated":
        return api.murty_batch(pb, k, cut_mode=api.CUT_RELATIVE, weight_mode=api.WEIGHTS_GATED)
    return api.murty_batch(pb, k, cut_mode=api.CUT_NONE, maximize=case.mode == "nocut_max")


def _workspace_ok(lib, n, k, rows, cols):
    ws = int(lib.pda_murty_workspace_bytes(n, k, rows, cols))
    assert 0 < ws <= WS_LIMIT, f"workspace of {ws} B for {n} problems, k = {k}, {rows} x {cols}"


@pytest.mark.gpu
def test_restatement_matches_workspace_bytes(gpu_api, optin):
    """The restated arenas (warp and CTA kernels) are what the library sizes, over a grid of shapes and k."""
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    prev = gpu_api.set_murty_path("warp")
    bad = []
    try:
        for path in ("warp", "cta"):
            gpu_api.set_murty_path(path)
            for k in (1, 2, 3, 40, 761, 1993):
                for r in (1, 8, 31, 32, 33, 64, 65, 96, 97, 128):
                    for c in sorted({1, r // 2 or 1, min(r, 13), min(r, 16), min(r, 17), min(r, 64), r}):
                        got = int(lib.pda_murty_workspace_bytes(1, k, r, c))
                        want = workspace_bytes(k, r, c, path, optin)
                        if got != want:
                            bad.append((path, k, r, c, got, want))
    finally:
        gpu_api.set_murty_path(prev)
    assert not bad, f"{len(bad)} (path, k, rows, cols, library, restatement) differ, e.g. {bad[:4]}"
    assert lib.pda_murty_workspace_bytes(1, 1 << 24, 65, 65) == -3
    assert lib.pda_murty_workspace_bytes(1, 5, 129, 3) == -3
    assert lib.pda_murty_workspace_bytes(1, 0, 8, 3) == -1


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_case_vs_oracle(case, murty_path, gpu_api, oracle, optin):
    pb = case.build()
    rows, cols = _dims(pb)
    if murty_path == "cta" and cols > CTA_MAX_COL:
        pytest.skip("above 16 detections the cta setting runs the pruning kernel, as the fast setting does")
    _assert_regime(case, pb, optin)
    k = case_k(case, optin)
    from probabilisticsemslam_b200 import _lib
    _workspace_ok(_lib.lib(), len(pb), k, rows, cols)
    want, want_probs = _oracle_result(oracle, case, pb, k)
    got = _run_case(gpu_api, case, pb, k)
    for p in range(len(pb)):
        assert_kbest_equal((int(got.n_found[p]),) + tuple(got.lists(pb, p)), want[p], f"{case.name}[{p}] ({murty_path})")
        if case.found is not None:
            assert int(got.n_found[p]) == case.found < k
    if want_probs is not None:
        np.testing.assert_allclose(got.probs, want_probs, rtol=1e-9, atol=0)


LADDER_CASES = [c for c in CASES if c.mode == "gated"]  # the ladder fuses weights, so these regimes are its own


@pytest.mark.gpu
@pytest.mark.parametrize("case", LADDER_CASES, ids=[c.name for c in LADDER_CASES])
def test_ladder_case_matches_single_calls(case, murty_path, gpu_api, optin):
    """One enumeration to the case's k (its regime: the ladder sizes its geometry from the largest rung) gives, in every
    slot, the bits and nFound of a separate assignment_prob_batch call with that slot's k."""
    pb = case.build()
    if murty_path == "cta" and _dims(pb)[1] > CTA_MAX_COL:
        pytest.skip("above 16 detections the cta setting runs the pruning kernel, as the fast setting does")
    _assert_regime(case, pb, optin)
    k = case_k(case, optin)
    ks = sorted({1, max(1, k // 3), k - 1 if k > 1 else 1, k})
    tabs, nf = gpu_api.assignment_prob_ladder_batch(pb, ks)
    for j, kj in enumerate(ks):
        one = gpu_api.assignment_prob_batch(pb, kj)
        np.testing.assert_array_equal(nf[:, j], one.n_found, err_msg=f"{case.name}: nFound of slot {j} (k = {kj})")
        for p in range(len(pb)):
            assert np.array_equal(bits(tabs[p][j]), bits(one.prob_table(pb, p))), f"{case.name}[{p}], k = {kj}"


# ---- loose declared bounds (device-pointer entry) -----------------------------------------------------------------------
def _loose_batch():
    """KITTI-shaped G1 problems (38 x 8) and two wider ones; tight bounds 38 x 12 keep a heap top and the CTA kernel."""
    mats, nls = [], []
    for src in (synth.g1_dense(3, nL=30, nM=8, first=63000), synth.g1_dense(1, nL=26, nM=12, first=63100),
                synth.g1_dense(1, nL=25, nM=11, first=63200, integer=True)):
        for p in range(len(src)):
            mats.append(src.matrix(p)); nls.append(int(src.nL[p]))
    return synth.pack(mats, nls)


LOOSE_K = 60
# declared (maxNumRow, maxNumCol) -> the regime it puts the same problems in (with weights, k = LOOSE_K)
LOOSE_BOUNDS = [
    ((38, 12), (("R", 2), ("heap_top", True), ("wpc", 4), ("fast_ok", True), ("cta", True))),
    ((38, 16), (("R", 2), ("heap_top", False), ("wpc", 4), ("fast_ok", True), ("cta", True))),
    ((100, 16), (("R", 4), ("heap_top", False), ("wpc", 4), ("cta", True))),
    ((128, 28), (("R", 4), ("wpc", 2), ("fast_ok", True), ("cta", False))),
    ((128, 112), (("wpc", 1), ("fast_ok", True), ("cta", False))),
    ((127, 113), (("wpc", 1), ("fast_ok", False), ("cta", False))),
]


def _plan_result(pb, k, bounds):
    import torch
    from probabilisticsemslam_b200 import device
    plan = device.MurtyPlan(pb, k, weights=True, max_num_row=bounds[0], max_num_col=bounds[1])
    assert plan.workspace_bytes <= WS_LIMIT
    plan.run()
    torch.cuda.synchronize()
    return plan.result()


@pytest.mark.gpu
def test_loose_bounds_same_bits(murty_path, gpu_api, oracle, optin):
    pb = _loose_batch()
    assert _dims(pb) == LOOSE_BOUNDS[0][0]
    want = oracle.batch(pb, LOOSE_K, threads=8, want_probs=True, want_lists=True)
    tight = None
    for bounds, expect in LOOSE_BOUNDS:
        g = geometry(LOOSE_K, bounds[0], bounds[1], True, optin)
        assert g.error is None, bounds
        for field, value in expect:
            assert getattr(g, field) == value, f"bounds {bounds}: {field} = {getattr(g, field)}, meant {value}"
        got = _plan_result(pb, LOOSE_K, bounds)
        np.testing.assert_array_equal(got.n_found, want["n_found"], err_msg=f"bounds {bounds}")
        for p in range(len(pb)):
            n, nc, nr = int(want["n_found"][p]), int(pb.nM[p]), int(pb.num_row[p])
            ref = (n, want["row4col"][want["r4c_off"][p]:want["r4c_off"][p] + n * nc].reshape(n, nc),
                   want["col4row"][want["c4r_off"][p]:want["c4r_off"][p] + n * nr].reshape(n, nr),
                   want["gain"][p * LOOSE_K:p * LOOSE_K + n])
            assert_kbest_equal((int(got.n_found[p]),) + tuple(got.lists(pb, p)), ref, f"bounds {bounds}, problem {p}")
        np.testing.assert_allclose(got.probs, want["probs"], rtol=1e-9, atol=0)
        if tight is None:
            tight = got
        else:
            assert np.array_equal(bits(got.probs), bits(tight.probs)), f"bounds {bounds}: weights differ from tight bounds"


# ---- limits ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_shared_memory_limit_is_an_error(gpu_api, oracle, optin):
    """128 x 113 with weights needs more shared memory per warp than a block may have: -3 and a message, not a launch.
    128 x 112 runs."""
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    assert geometry(5, 128, 113, True, optin).error == "smem" and geometry(5, 128, 112, True, optin).error is None
    pb = synth.g1_dense(1, nL=15, nM=113, first=64000)
    num_row, num_col, nL = pb.num_row, pb.nM.astype(np.int32), pb.nL.astype(np.int32)
    found = np.zeros(1, np.int32)
    probs = np.zeros(113 * 16)
    poff = np.zeros(1, np.int64)
    p = lambda a: a.ctypes.data
    rc = lib.pda_murty_batch_host(p(pb.costs), p(pb.cost_off), p(num_row), p(num_col), 1, 5, 1, 42.0, 0, 0,
                                  None, None, None, None, None, p(found), 1, p(probs), p(poff), p(nL), 0)
    assert rc == -3 and b"shared memory" in lib.pda_last_error()
    ok = synth.g1_dense(1, nL=16, nM=112, first=64100)
    got = gpu_api.murty_batch(ok, 5, weight_mode=gpu_api.WEIGHTS_GATED)
    w = oracle.batch(ok, 5, threads=1)
    np.testing.assert_array_equal(got.n_found, w["n_found"])
    assert np.array_equal(got.row4col, w["row4col"]) and np.array_equal(bits(got.gain.reshape(-1)), bits(w["gain"]))
    np.testing.assert_allclose(got.probs, w["probs"], rtol=1e-9, atol=0)


@pytest.mark.gpu
def test_node_limit_is_an_error(gpu_api):
    """k * numCol beyond 2^30 arena nodes: -3 before anything is staged (NULL lists and gains: nothing to hold 2^30
    entries on the host either)."""
    from probabilisticsemslam_b200 import _lib
    lib = _lib.lib()
    assert geometry(1 << 24, 65, 65, False, B200_SMEM_OPTIN).error == "nodes"
    assert geometry(1 << 24, 64, 64, False, B200_SMEM_OPTIN).error is None  # 2^30 - 63 nodes: the last k that is let in
    C = np.ascontiguousarray(np.random.default_rng(5).uniform(0.0, 1.0, 65 * 65))
    off = np.zeros(1, np.int64)
    nr, nc = np.array([65], np.int32), np.array([65], np.int32)
    found = np.full(1, -7, np.int32)
    p = lambda a: a.ctypes.data
    rc = lib.pda_murty_batch_host(p(C), p(off), p(nr), p(nc), 1, 1 << 24, 0, 0.0, 0, 0,
                                  None, None, None, None, None, p(found), 0, None, None, None, 0)
    assert rc == -3 and b"too large" in lib.pda_last_error()
    assert found[0] == -7
