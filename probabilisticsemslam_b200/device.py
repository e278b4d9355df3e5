"""Device-resident plans: PyTorch owns the HBM buffers and the stream, libpda_b200.so does the work.

A plan uploads a ragged batch once, keeps inputs, outputs and the kernel workspace resident and
can be re-run any number of times (this is what bench.py times).  torch is plumbing here -- device
memory, streams, torch.distributed -- every kernel is ours, reached through the C ABI with raw
device pointers.
"""
from __future__ import annotations

import numpy as np
import torch

from . import api
from ._lib import alloc_workspace, check, lib
from .synth import ProblemBatch


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream_handle():
    return torch.cuda.current_stream().cuda_stream


class MurtyPlan:
    """k-best enumeration (+ fused assignment weights) of a ProblemBatch on the current CUDA device."""

    def __init__(self, pb: ProblemBatch, k: int, *, weights: bool = False, weight_mode: int | None = None,
                 cut_mode: int = api.CUT_RELATIVE, cutoff: float = api.GATE, maximize: bool = False,
                 cut_maximize: bool = False, want_lists: bool = True, max_arenas: int | None = None,
                 pinned_inputs: bool = False, max_num_row: int | None = None, max_num_col: int | None = None):
        """max_num_row / max_num_col: the bounds the call declares (default: the batch's own maxima).  Looser bounds
        size the kernel geometry as a graph captured for larger frames would; the results do not change."""
        assert torch.cuda.is_available(), "MurtyPlan needs a CUDA device (there is no CPU fallback)"
        self.k, self.n = int(k), len(pb)
        self.cut_mode, self.cutoff, self.maximize, self.cut_maximize = cut_mode, float(cutoff), bool(maximize), bool(cut_maximize)
        self.weight_mode = (api.WEIGHTS_GATED if weights else api.WEIGHTS_NONE) if weight_mode is None else weight_mode
        dev = torch.device("cuda", torch.cuda.current_device())
        self.dev = dev
        num_row, num_col = pb.num_row, pb.nM.astype(np.int32)
        self.max_row = int(num_row.max()) if max_num_row is None else int(max_num_row)
        self.max_col = int(num_col.max()) if max_num_col is None else int(max_num_col)
        self.cost_off_h = pb.cost_off.astype(np.int64)
        self.r4c_off_h = api._prefix(num_col.astype(np.int64) * k)
        self.c4r_off_h = api._prefix(num_row.astype(np.int64) * k)
        self.prob_off_h = api._prefix(num_col.astype(np.int64) * (pb.nL.astype(np.int64) + 1))
        self.n_prob = int((num_col.astype(np.int64) * (pb.nL.astype(np.int64) + 1)).sum())
        # host staging (pinned when asked: the end-to-end path copies from these every step)
        def host(a):
            t = torch.from_numpy(np.ascontiguousarray(a))
            return t.pin_memory() if pinned_inputs else t
        self.h_costs = host(pb.costs)
        self.h_meta = [host(self.cost_off_h), host(num_row), host(num_col), host(pb.nL.astype(np.int32)),
                       host(self.r4c_off_h), host(self.c4r_off_h), host(self.prob_off_h)]
        self.costs = torch.empty(pb.costs.shape[0], dtype=torch.float64, device=dev)
        self.cost_off = torch.empty(self.n, dtype=torch.int64, device=dev)
        self.num_row = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.num_col = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.nL = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.r4c_off = torch.empty(self.n, dtype=torch.int64, device=dev)
        self.c4r_off = torch.empty(self.n, dtype=torch.int64, device=dev)
        self.prob_off = torch.empty(self.n, dtype=torch.int64, device=dev)
        self.upload()
        self.row4col = torch.empty(int(num_col.astype(np.int64).sum()) * k, dtype=torch.int64, device=dev) if want_lists else None
        self.col4row = torch.empty(int(num_row.astype(np.int64).sum()) * k, dtype=torch.int64, device=dev) if want_lists else None
        self.gain = torch.empty(self.n * k, dtype=torch.float64, device=dev)
        self.n_found = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.probs = torch.empty(self.n_prob, dtype=torch.float64, device=dev) if self.weight_mode else None
        ws = int(lib().pda_murty_workspace_bytes(self.n, self.k, self.max_row, self.max_col))
        if ws < 0:
            check(ws)
        if max_arenas is not None:  # testing hook: shrink the workspace to `max_arenas` problems in flight
            per = (ws - 256) // max(1, min(self.n, self._full_warps(ws)))
            ws = 256 + per * max_arenas
        self.workspace = torch.empty(ws, dtype=torch.uint8, device=dev)
        self.workspace_bytes = ws
        # algorithmic bytes of one pass (SURVEY.md 8d): costs in + (row4col, col4row, gain) per hypothesis + weights
        self.bytes_in = int(pb.costs.shape[0]) * 8

    def _full_warps(self, ws):
        one = int(lib().pda_murty_workspace_bytes(1, self.k, self.max_row, self.max_col)) - 256
        return max(1, (ws - 256) // one)

    def upload(self, non_blocking: bool = True):
        """Host -> device copy of the cost matrices and descriptors (part of the end-to-end path)."""
        self.costs.copy_(self.h_costs, non_blocking=non_blocking)
        for d, h in zip([self.cost_off, self.num_row, self.num_col, self.nL, self.r4c_off, self.c4r_off, self.prob_off], self.h_meta):
            d.copy_(h, non_blocking=non_blocking)

    def h2d_bytes(self) -> int:
        return int(self.h_costs.numel() * 8 + sum(t.numel() * t.element_size() for t in self.h_meta))

    def run(self):
        """Enqueue one pass of the hot path on the current stream (no synchronisation)."""
        check(lib().pda_murty_batch(_ptr(self.costs), _ptr(self.cost_off), _ptr(self.num_row), _ptr(self.num_col),
                                    self.n, self.max_row, self.max_col, self.k, self.cut_mode, self.cutoff,
                                    int(self.maximize), int(self.cut_maximize),
                                    _ptr(self.row4col), _ptr(self.r4c_off), _ptr(self.col4row), _ptr(self.c4r_off),
                                    _ptr(self.gain), _ptr(self.n_found),
                                    self.weight_mode, _ptr(self.probs), _ptr(self.prob_off), _ptr(self.nL),
                                    _ptr(self.workspace), self.workspace_bytes, _stream_handle()))

    def algorithmic_bytes(self) -> int:
        """Reference-ABI traffic of the pass just run: 8*numRow*numCol in, nFound*8*(numCol+numRow+1) out,
        8*numCol*(nL+1) weights out (SURVEY.md section 8d)."""
        nf = self.n_found.cpu().numpy().astype(np.int64)
        nr = self.h_meta[1].numpy().astype(np.int64)
        nc = self.h_meta[2].numpy().astype(np.int64)
        nl = self.h_meta[3].numpy().astype(np.int64)
        out = int((nf * 8 * (nc + nr + 1)).sum()) if self.row4col is not None else int((nf * 8).sum())
        w = int((8 * nc * (nl + 1)).sum()) if self.weight_mode else 0
        return int((8 * nr * nc).sum()) + out + w

    def result(self) -> api.KBestResult:
        return api.KBestResult(self.n_found.cpu().numpy(), self.gain.view(self.n, self.k).cpu().numpy(),
                               None if self.row4col is None else self.row4col.cpu().numpy(), self.r4c_off_h,
                               None if self.col4row is None else self.col4row.cpu().numpy(), self.c4r_off_h,
                               None if self.probs is None else self.probs.cpu().numpy(),
                               self.prob_off_h if self.weight_mode else None, self.k)


class PermanentPlan:
    """Batched exact permanents of equally sized dense matrices resident on the device."""

    def __init__(self, mats: np.ndarray, dim: int):
        assert torch.cuda.is_available(), "PermanentPlan needs a CUDA device (there is no CPU fallback)"
        dev = torch.device("cuda", torch.cuda.current_device())
        mats = np.ascontiguousarray(mats, dtype=np.float64).reshape(-1, dim * dim)
        self.n, self.dim = mats.shape[0], dim
        self.mats = torch.from_numpy(mats).to(dev)
        self.off = torch.arange(self.n, dtype=torch.int64, device=dev) * (dim * dim)
        self.rows = torch.full((self.n,), dim, dtype=torch.int32, device=dev)
        self.cols = torch.full((self.n,), dim, dtype=torch.int32, device=dev)
        self.out = torch.empty(self.n, dtype=torch.float64, device=dev)
        self.status = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.ws_bytes = int(lib().pda_permanent_workspace_bytes(self.n))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)

    def run(self):
        check(lib().pda_permanent_batch(_ptr(self.mats), _ptr(self.off), _ptr(self.rows), _ptr(self.cols), self.n,
                                        self.dim, _ptr(self.out), _ptr(self.status), _ptr(self.ws), self.ws_bytes,
                                        _stream_handle()))

    def flops(self) -> float:
        """n DFMA (2 flops) + n DMUL per Gray subset (SURVEY.md 8d): 3 n 2^(n-1) per matrix."""
        return float(self.n) * 3.0 * self.dim * 2.0 ** (self.dim - 1)


class PermanentProbPlan:
    """permanentProb of a ProblemBatch, resident on the current CUDA device: run() enqueues pda_permanent_prob_batch on
    the current stream, result() copies the tables back."""

    def __init__(self, pb: ProblemBatch, perm_opt: int = 1, *, max_num_row: int | None = None, max_num_col: int | None = None):
        assert torch.cuda.is_available(), "PermanentProbPlan needs a CUDA device (there is no CPU fallback)"
        dev = torch.device("cuda", torch.cuda.current_device())
        self.n, self.perm_opt = len(pb), int(perm_opt)
        self.nL_h, self.nM_h = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
        sizes = self.nM_h.astype(np.int64) * (self.nL_h.astype(np.int64) + 1)
        self.prob_off_h = api._prefix(sizes)
        self.total_prob = int(sizes.sum())
        self.max_row = int((self.nL_h + self.nM_h).max()) if max_num_row is None else int(max_num_row)
        self.max_col = int(self.nM_h.max()) if max_num_col is None else int(max_num_col)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.costs = up(pb.costs if pb.costs.size else np.zeros(1))
        self.cost_off, self.nL, self.nM, self.prob_off = up(pb.cost_off.astype(np.int64)), up(self.nL_h), up(self.nM_h), up(self.prob_off_h)
        self.probs = torch.zeros(max(self.total_prob, 1), dtype=torch.float64, device=dev)
        self.status = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.workspace = alloc_workspace(lib().pda_permanent_prob_workspace_bytes(self.n, int(self.costs.numel()), self.total_prob,
                                                                                  self.max_row, self.max_col, self.perm_opt), dev)

    def run(self):
        api.permanent_prob_batch_device(self.costs, self.cost_off, self.nL, self.nM, self.prob_off, self.total_prob,
                                        self.max_row, self.max_col, self.perm_opt, self.probs, self.status, self.workspace)

    def result(self):
        """(list of (nM, nL+1) tables, status), as api.permanent_prob_batch returns them."""
        probs, st = self.probs.cpu().numpy(), self.status.cpu().numpy()
        o, L, M = self.prob_off_h, self.nL_h, self.nM_h
        return [probs[o[p]:o[p] + int(M[p]) * (int(L[p]) + 1)].reshape(int(M[p]), int(L[p]) + 1) for p in range(self.n)], st


class ConditionedPermanentPlan:
    """conditionedPermanent of a list of matrices, resident on the current CUDA device (pda_conditioned_permanent_batch)."""

    def __init__(self, mats: list[np.ndarray], perm_opt: int = 1, *, max_dim: int | None = None):
        assert torch.cuda.is_available(), "ConditionedPermanentPlan needs a CUDA device (there is no CPU fallback)"
        dev = torch.device("cuda", torch.cuda.current_device())
        self.n, self.perm_opt = len(mats), int(perm_opt)
        rows = np.asarray([m.shape[0] for m in mats], np.int32)
        cols = np.asarray([m.shape[1] for m in mats], np.int32)
        flat = np.concatenate([np.asarray(m, np.float64).reshape(-1, order="F") for m in mats] + [np.zeros(1)])
        self.max_dim = int(max(rows.max(), cols.max())) if max_dim is None else int(max_dim)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.mats, self.mat_off = up(flat), up(api._prefix(rows.astype(np.int64) * cols))
        self.rows, self.cols = up(rows), up(cols)
        self.out = torch.zeros(self.n, dtype=torch.float64, device=dev)
        self.status = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.workspace = alloc_workspace(lib().pda_conditioned_permanent_workspace_bytes(self.n, self.max_dim, self.perm_opt), dev)

    def run(self):
        api.conditioned_permanent_batch_device(self.mats, self.mat_off, self.rows, self.cols, self.max_dim, self.perm_opt,
                                               self.out, self.status, self.workspace)

    def result(self):
        return self.out.cpu().numpy(), self.status.cpu().numpy()


class PermanentRangePlan:
    """One large permanent: this rank's share of the Gray-code range, as a double-double partial."""

    def __init__(self, a: np.ndarray, begin: int, end: int):
        dev = torch.device("cuda", torch.cuda.current_device())
        a = np.asarray(a, np.float64)
        self.n = a.shape[0]
        self.begin, self.end = int(begin), int(end)
        self.A = torch.from_numpy(np.ascontiguousarray(a.reshape(-1, order="F"))).to(dev)
        self.partial = torch.zeros(2, dtype=torch.float64, device=dev)
        self.ws_bytes = 64 + 16 * 8 * 256
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)

    def run(self):
        check(lib().pda_permanent_range(_ptr(self.A), self.n, self.begin, self.end, _ptr(self.partial), _ptr(self.ws),
                                        self.ws_bytes, _stream_handle()))

    @staticmethod
    def combine(partials: torch.Tensor, n: int) -> float:
        """Sum (hi, lo) pairs in rank order and apply the NW factor (4(n&1)-2)."""
        hi, lo = 0.0, 0.0
        for h, l in partials.reshape(-1, 2).tolist():
            s = hi + h
            bb = s - hi
            e = (hi - (s - bb)) + (h - bb)
            hi, lo = s, lo + e + l
        return float((4 * (n & 1) - 2) * (hi + lo))
