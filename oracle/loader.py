"""ctypes front-end for the two CPU checkers.  TEST INFRASTRUCTURE ONLY.

    load_oracle()        -> oracle/liboracle.so  (this repo's C restatement, `orc_*`)
    load_reference(kind) -> oracle/_ref/libpda_ref_<kind>.so (the reference's own code, `ref_*`)

Both expose the same methods through `CpuChecker`.  Only tests/, bench.py's CPU legs
and __graft_entry__.smoke() may import this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_i64, _i32, _dbl, _ptr, _int = C.c_int64, C.c_int32, C.c_double, C.c_void_p, C.c_int


def _p(a):
    return None if a is None else a.ctypes.data


class CpuChecker:
    def __init__(self, path: str, prefix: str):
        self.path, self.prefix = path, prefix
        self.lib = C.CDLL(path)
        f = self._fn
        f("kbest2d", _i64, [_i64, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr])
        f("kbest2d_cutoff", _i64, [_i64, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl])
        f("kbest2d_after_cutoff", _i64, [_i64, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _int, _ptr, _dbl])
        f("assign2d", _int, [_i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr])
        f("shortest_path", _int, [_i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr])
        f("condition_costs", _i64, [_ptr, _i64, _i64, _ptr, _ptr])
        f("to_probs", None, [_ptr, _i64])
        f("assignment_prob", _int, [_ptr, _i64, _i64, _i64, _ptr])
        f("brute_force_prob", _int, [_ptr, _i64, _i64, _ptr])
        f("permanent_prob", _int, [_ptr, _i64, _i64, _int, _ptr])
        f("association_probs", _int, [_ptr, _i64, _i64, _i64, _int, _ptr])
        f("permanent_exact", _dbl, [_ptr, _i64, _i64, _ptr])
        f("permanent_exact_square", _dbl, [_ptr, _i64, _ptr])
        f("permanent_exact_long", _dbl, [_ptr, _i64, _i64, _ptr])
        f("conditioned_permanent", _dbl, [_ptr, _i64, _i64, _int, _ptr])
        f("batch", _dbl, [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _dbl, _int, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr])
        f("permanent_batch", _dbl, [_ptr, _i64, _i64, _int, _ptr])
        f("bb_cost_matrix", None, [_ptr, C.c_long, _ptr, C.c_long, _dbl, _ptr])
        f("asgn_bb", None, [_ptr, C.c_long, _ptr, C.c_long, _dbl, _ptr])
        if prefix == "orc":  # restatement only: needs Eigen on the reference side (oracle_quadric.c)
            f("permanent_approx", _dbl, [_ptr, _i64, _i64, _i64, C.c_uint64, _i64, _ptr])
            f("approx_near_ties_reset", None, [])
            f("approx_near_ties", _i64, [])
            f("set_approx_stream", None, [C.c_uint64, _i64])
            f("kbest2d_cutoff_pruned", _i64, [_i64, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr])
            f("quadric_covs", None, [_ptr, _i64, _ptr])
            f("quadric_cost_matrix", None, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _dbl, _ptr])
            f("association_from_moments", _int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _dbl, _i64, _ptr])

    def _fn(self, name, res, args):
        fn = getattr(self.lib, f"{self.prefix}_{name}")
        fn.restype, fn.argtypes = res, args
        setattr(self, "_" + name, fn)

    # ---- k-best -----------------------------------------------------------------
    def _kbest(self, which, k, cmat, maximize, *extra):
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        c4r = np.full((k, nr), -7, np.int64)
        r4c = np.full((k, nc), -7, np.int64)
        g = np.full(k, np.nan)
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        n = getattr(self, which)(k, nr, nc, int(maximize), _p(flat), _p(c4r), _p(r4c), _p(g), *extra)
        return int(n), r4c, c4r, g

    def kbest2d(self, k, cmat, maximize=False):
        return self._kbest("_kbest2d", k, cmat, maximize)

    def kbest2d_cutoff(self, k, cmat, cutoff=42.0, maximize=False):
        return self._kbest("_kbest2d_cutoff", k, cmat, maximize, float(cutoff))

    def kbest2d_cutoff_pruned(self, k, cmat, cutoff=42.0, maximize=False, max_col=None):
        """CPU model of the CUDA pruning kernel's decisions (oracle_murty.c): (n or -2 if the kernel would fall back to the
        exact kernel, row4col, col4row, gains, stats{children, abandoned, dropped_done, kept, tightenings, slots})."""
        stats = np.zeros(6, np.int64)
        mc = int(np.asarray(cmat).shape[1] if max_col is None else max_col)
        n, r4c, c4r, g = self._kbest("_kbest2d_cutoff_pruned", k, cmat, maximize, float(cutoff), mc, _p(stats))
        names = ["children", "abandoned", "dropped_done", "kept", "tightenings", "slots_at_tightening"]
        return n, r4c, c4r, g, dict(zip(names, (int(x) for x in stats)))

    def kbest2d_after_cutoff(self, k, cmat, maximize, first_cmat, first_maximize, first_cutoff):
        first = np.ascontiguousarray(np.asfortranarray(first_cmat, dtype=np.float64).reshape(-1, order="F"))
        return self._kbest("_kbest2d_after_cutoff", k, cmat, maximize, int(first_maximize), _p(first), float(first_cutoff))

    def assign2d(self, cmat, maximize=False):
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        c4r, r4c = np.zeros(nr, np.int64), np.zeros(nc, np.int64)
        u, v, g = np.zeros(nc), np.zeros(nr), np.zeros(1)
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        ret = self._assign2d(nr, nc, int(maximize), _p(flat), _p(c4r), _p(r4c), _p(u), _p(v), _p(g))
        return int(ret), r4c, c4r, u, v, float(g[0])

    def shortest_path(self, cmat, num_col4gain=None):
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        c4r, r4c = np.zeros(nr, np.int64), np.zeros(nc, np.int64)
        u, v, g, fb = np.zeros(nc), np.zeros(nr), np.zeros(1), np.zeros(nr, np.uint8)
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        ret = self._shortest_path(nr, nc, nc if num_col4gain is None else num_col4gain, _p(flat),
                                  _p(c4r), _p(r4c), _p(u), _p(v), _p(g), _p(fb))
        return int(ret), r4c, c4r, u, v, float(g[0]), fb

    # ---- weights ----------------------------------------------------------------
    def condition_costs(self, cmat):
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        out = np.zeros(nr * nc)
        idx = np.zeros(nr, np.int64)
        good = int(self._condition_costs(_p(flat), nr, nc, _p(out), _p(idx)))
        return out[:good * nc].reshape((good, nc), order="F").copy(), idx[:good].copy()

    def to_probs(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64).copy()
        self._to_probs(_p(v), v.size)
        return v

    def _probs(self, fn, cmat, nL, *extra):
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        assert nr == nL + nc
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        out = np.zeros((nc, nL + 1))
        st = fn(_p(flat), nL, nc, *extra, _p(out))
        return int(st), out

    def assignment_prob(self, cmat, nL, k):
        return self._probs(self._assignment_prob, cmat, nL, k)[1]

    def brute_force_prob(self, cmat, nL):
        return self._probs(self._brute_force_prob, cmat, nL)[1]

    def permanent_prob(self, cmat, nL, perm_opt=1):
        return self._probs(self._permanent_prob, cmat, nL, perm_opt)

    def association_probs(self, cmat, nL, k, use_perm=False):
        """getAssignmentProbs from the cost matrix on (assignment.cpp:57-74) -> (status, probs[nM, nL+1])."""
        cmat = np.asfortranarray(cmat, dtype=np.float64)
        nr, nc = cmat.shape
        flat = np.ascontiguousarray(cmat.reshape(-1, order="F"))
        out = np.zeros((nc, nL + 1))
        st = self._association_probs(_p(flat), nL, nc, k, int(use_perm), _p(out))
        return int(st), out

    # ---- permanents -------------------------------------------------------------
    def permanent_exact(self, a):
        a = np.asfortranarray(a, dtype=np.float64)
        st = _int(0)
        flat = np.ascontiguousarray(a.reshape(-1, order="F"))
        r = self._permanent_exact(_p(flat), a.shape[0], a.shape[1], C.byref(st))
        return float(r), st.value

    def permanent_exact_long(self, a):
        a = np.asfortranarray(a, dtype=np.float64)
        st = _int(0)
        flat = np.ascontiguousarray(a.reshape(-1, order="F"))
        r = self._permanent_exact_long(_p(flat), a.shape[0], a.shape[1], C.byref(st))
        return float(r), st.value

    def permanent_exact_square(self, a):
        a = np.asfortranarray(a, dtype=np.float64)
        st = _int(0)
        flat = np.ascontiguousarray(a.reshape(-1, order="F"))
        r = self._permanent_exact_square(_p(flat), a.shape[0], C.byref(st))
        return float(r), st.value

    def conditioned_permanent(self, a, perm_opt=1):
        a = np.asfortranarray(a, dtype=np.float64)
        st = _int(0)
        flat = np.ascontiguousarray(a.reshape(-1, order="F"))
        r = self._conditioned_permanent(_p(flat), a.shape[0], a.shape[1], perm_opt, C.byref(st))
        return float(r), st.value

    # ---- stereo box association (boxes: [n, 5] = xmin, ymin, xmax, ymax, xOffset) -----------------------
    def bb_cost_matrix(self, boxes_l, boxes_r, nonassign):
        bl, br = np.ascontiguousarray(boxes_l, np.float64).reshape(-1, 5), np.ascontiguousarray(boxes_r, np.float64).reshape(-1, 5)
        out = np.zeros((bl.shape[0] + br.shape[0]) * bl.shape[0])
        self._bb_cost_matrix(_p(bl), bl.shape[0], _p(br), br.shape[0], float(nonassign), _p(out))
        return out.reshape((bl.shape[0] + br.shape[0], bl.shape[0]), order="F")

    def asgn_bb(self, boxes_l, boxes_r, nonassign):
        bl, br = np.ascontiguousarray(boxes_l, np.float64).reshape(-1, 5), np.ascontiguousarray(boxes_r, np.float64).reshape(-1, 5)
        out = np.full(max(bl.shape[0], 1), -7, np.int32)
        self._asgn_bb(_p(bl), bl.shape[0], _p(br), br.shape[0], float(nonassign), _p(out))
        return out[:bl.shape[0]]

    # ---- Huber's approximate permanent (restatement only; counter-based draws shared with the CUDA kernel) ----
    def permanent_approx(self, a, iterations=300, seed=20260217, mat_index=0, near_ties=False):
        """-> (estimate, successes), or with near_ties=True (estimate, successes, near ties): the number of draws that lay
        within 1e-12 of a partial sum they were compared with, i.e. how many trials the CUDA kernel may decide the other
        way (oracle_perm_approx.c)."""
        a = np.asfortranarray(a, dtype=np.float64)
        succ = C.c_int64(0)
        self._approx_near_ties_reset()
        est = self._permanent_approx(_p(a), a.shape[0], a.shape[1], int(iterations), int(seed), int(mat_index), C.byref(succ))
        if near_ties:
            return float(est), int(succ.value), int(self._approx_near_ties())
        return float(est), int(succ.value)

    def approx_near_ties_reset(self):
        """Zero this thread's near-tie counter (it also counts the draws of permanent_prob / conditioned_permanent with
        perm_opt 0)."""
        self._approx_near_ties_reset()

    def approx_near_ties(self) -> int:
        return int(self._approx_near_ties())

    def set_approx_stream(self, seed=20260217, index=0):
        """The stream (seed, matrix index) the next conditioned_permanent(.., 0) on this thread draws from."""
        self._set_approx_stream(int(seed), int(index))

    # ---- cost matrices from quadric moments (restatement only) ---------------------------
    def quadric_covs(self, quadrics):
        q = np.ascontiguousarray(quadrics, np.float64).reshape(-1, 16)
        out = np.zeros((q.shape[0], 9))
        self._quadric_covs(_p(q), q.shape[0], _p(out))
        return out.reshape(-1, 3, 3)

    @staticmethod
    def _moments(mean, cov):
        m = np.ascontiguousarray(mean, np.float64).reshape(-1, 3)
        c = np.ascontiguousarray(np.asarray(cov, np.float64).reshape(-1, 3, 3).transpose(0, 2, 1)).reshape(-1, 9)  # column-major 3x3
        return m, c

    def quadric_cost_matrix(self, land_mean, land_cov, meas_mean, meas_cov, nonassign):
        lm, lc = self._moments(land_mean, land_cov)
        mm, mc = self._moments(meas_mean, meas_cov)
        nL, nM = lm.shape[0], mm.shape[0]
        out = np.zeros((nL + nM) * nM)
        self._quadric_cost_matrix(_p(lm), _p(lc), nL, _p(mm), _p(mc), nM, float(nonassign), _p(out))
        return out.reshape((nL + nM, nM), order="F")

    def association_from_moments(self, land_mean, land_cov, meas_mean, meas_cov, nonassign, k):
        lm, lc = self._moments(land_mean, land_cov)
        mm, mc = self._moments(meas_mean, meas_cov)
        nL, nM = lm.shape[0], mm.shape[0]
        out = np.zeros(max(nM * (nL + 1), 1))
        self._association_from_moments(_p(lm), _p(lc), nL, _p(mm), _p(mc), nM, float(nonassign), int(k), _p(out))
        return out[:nM * (nL + 1)].reshape(nM, nL + 1)

    # ---- batches (timing + bulk checks) ----------------------------------------------
    def batch(self, pb, k, *, cutoff=42.0, threads=1, want_probs=True, want_lists=True):
        """Run a synth.ProblemBatch.  Returns dict(seconds, probs, prob_off, row4col, r4c_off,
        col4row, c4r_off, gain, n_found)."""
        n = len(pb)
        nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
        nR = (nL + nM).astype(np.int64)
        prob_sz = nM.astype(np.int64) * (nL.astype(np.int64) + 1)
        prob_off = np.concatenate([[0], np.cumsum(prob_sz)[:-1]]).astype(np.int64) if n else np.zeros(0, np.int64)
        r4c_off = np.concatenate([[0], np.cumsum(nM.astype(np.int64) * k)[:-1]]).astype(np.int64) if n else np.zeros(0, np.int64)
        c4r_off = np.concatenate([[0], np.cumsum(nR * k)[:-1]]).astype(np.int64) if n else np.zeros(0, np.int64)
        probs = np.zeros(int(prob_sz.sum())) if want_probs else None
        r4c = np.full(int(nM.astype(np.int64).sum()) * k, -7, np.int64) if want_lists else None
        c4r = np.full(int(nR.sum()) * k, -7, np.int64) if want_lists else None
        gain = np.full(n * k, np.nan) if want_lists else None
        nf = np.zeros(n, np.int32) if want_lists else None
        sec = self._batch(_p(pb.costs), _p(pb.cost_off), _p(nL), _p(nM), n, k, float(cutoff), int(threads),
                          _p(probs), _p(prob_off), _p(c4r), _p(c4r_off), _p(r4c), _p(r4c_off), _p(gain), _p(nf))
        return dict(seconds=float(sec), probs=probs, prob_off=prob_off, row4col=r4c, r4c_off=r4c_off,
                    col4row=c4r, c4r_off=c4r_off, gain=gain, n_found=nf)

    def permanent_batch(self, mats, dim, threads=1):
        mats = np.ascontiguousarray(mats, dtype=np.float64)
        n = mats.size // (dim * dim)
        out = np.zeros(n)
        sec = self._permanent_batch(_p(mats), dim, n, int(threads), _p(out))
        return float(sec), out


def build_oracle(quiet: bool = True) -> None:
    subprocess.run(["make", "-C", HERE, "oracle"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def build_reference(quiet: bool = True) -> None:
    """(Re)build oracle/_ref from /root/reference when it is mounted; no-op otherwise."""
    subprocess.run(["make", "-C", HERE, "ref"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def load_oracle() -> CpuChecker:
    path = os.path.join(HERE, "liboracle.so")
    if not os.path.exists(path):
        build_oracle()
    return CpuChecker(path, "orc")


def _native_ok() -> bool:
    want = os.path.join(HERE, "_ref", "native_cpu_flags.txt")
    try:
        built = set(open(want).read().split())
        for line in open("/proc/cpuinfo"):
            if line.startswith("flags"):
                return built <= set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return False


def reference_available(kind: str = "strict") -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", f"libpda_ref_{kind}.so"))


def load_reference(kind: str = "strict") -> CpuChecker:
    """kind: 'strict' (IEEE, parity), 'fast' (-Ofast, x86-64-v3), 'native' (the reference's own
    -Ofast -march=native; refused when this host lacks ISA extensions of the build host),
    'timing' (native if loadable here, else fast).

    The -Ofast builds ('fast', 'native', 'timing') are for TIMING on the dense benchmark inputs only: -ffast-math assumes
    there is no infinity, and on gated matrices (most entries +inf after conditionCosts) the reference's own code then does
    not terminate (observed: association_probs on synth.quadric_frames).  Use 'strict' for anything gated."""
    if kind == "timing":
        kind = "native" if (reference_available("native") and _native_ok()) else "fast"
    if kind == "native" and not _native_ok():
        raise OSError("libpda_ref_native.so was built for a CPU with ISA extensions this host lacks")
    path = os.path.join(HERE, "_ref", f"libpda_ref_{kind}.so")
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    chk = CpuChecker(path, "ref")
    chk.kind = kind
    chk.lib.ref_build_flags.restype = C.c_char_p
    chk.flags = chk.lib.ref_build_flags().decode()
    return chk
