"""Python face of libpda_b200.so for tests and benchmarks.

The reference's interface for this path is C++ (shortestPathCPP.hpp, assignment.h,
nwPerm.h); the C++ drop-in headers live in include/.  This module mirrors the same
functions name for name on numpy arrays (batch of one -> the *_host C entry points) and
adds the batch forms the GPU is built for.  Everything runs on the CUDA device through
the C ABI; nothing here computes on the CPU and nothing imports the oracle.

Matrices are (numRow, numCol) numpy arrays, rows = landmarks then one dummy row per
detection, exactly the reference's column-major cost matrix viewed in Fortran order.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import alloc_workspace, check, lib
from .synth import ProblemBatch, pack

CUT_NONE, CUT_RELATIVE, CUT_STICKY = 0, 1, 2
WEIGHTS_NONE, WEIGHTS_GATED, WEIGHTS_UNGATED = 0, 1, 2
GATE = 42.0  # assignment.cpp:9


MURTY_PATHS = {"auto": 0, "warp": 1, "cta": 2, "fast": 3}


def set_murty_path(path: str) -> str:
    """Which Murty kernel pda_murty_batch uses: "auto" (by batch size), "warp" (one warp per problem) or "cta" (one
    CTA per problem wherever numCol <= 16).  Results are bit-identical; returns the previous setting."""
    prev = lib().pda_murty_set_path(MURTY_PATHS[path])
    if prev < 0:
        check(prev)
    return {v: k for k, v in MURTY_PATHS.items()}[prev]


def _p(a):
    return None if a is None else a.ctypes.data


def _prefix(sizes: np.ndarray) -> np.ndarray:
    off = np.zeros(len(sizes), dtype=np.int64)
    if len(sizes) > 1:
        off[1:] = np.cumsum(sizes.astype(np.int64))[:-1]
    return off


# ------------------------------------------------------------------------------------------------
# batch forms (host buffers in, host buffers out)
# ------------------------------------------------------------------------------------------------
@dataclass
class KBestResult:
    n_found: np.ndarray   # int32[n]
    gain: np.ndarray      # float64[n, k]
    row4col: np.ndarray   # int64 flat; problem p, hypothesis i at r4c_off[p] + i*numCol[p]
    r4c_off: np.ndarray
    col4row: np.ndarray   # int64 flat; problem p, hypothesis i at c4r_off[p] + i*numRow[p]
    c4r_off: np.ndarray
    probs: np.ndarray | None
    prob_off: np.ndarray | None
    k: int

    def lists(self, pb: ProblemBatch, p: int):
        """(row4col[nFound, numCol], col4row[nFound, numRow], gain[nFound]) of problem p."""
        nf, nc, nr = int(self.n_found[p]), int(pb.nM[p]), int(pb.nL[p] + pb.nM[p])
        r = self.row4col[self.r4c_off[p]:self.r4c_off[p] + nf * nc].reshape(nf, nc)
        c = self.col4row[self.c4r_off[p]:self.c4r_off[p] + nf * nr].reshape(nf, nr)
        return r, c, self.gain[p, :nf]

    def prob_table(self, pb: ProblemBatch, p: int) -> np.ndarray:
        nc, w = int(pb.nM[p]), int(pb.nL[p]) + 1
        return self.probs[self.prob_off[p]:self.prob_off[p] + nc * w].reshape(nc, w)


def murty_batch(pb: ProblemBatch, k: int, *, cut_mode: int = CUT_RELATIVE, cutoff: float = GATE,
                maximize: bool = False, cut_maximize: bool = False, weight_mode: int = WEIGHTS_NONE,
                want_lists: bool = True, device: int = 0) -> KBestResult:
    """k-best enumeration (+ fused weights) for a ragged batch; pda_murty_batch_host."""
    n = len(pb)
    num_row, num_col = pb.num_row, pb.nM.astype(np.int32)
    r4c_off = _prefix(num_col.astype(np.int64) * k)
    c4r_off = _prefix(num_row.astype(np.int64) * k)
    prob_off = _prefix(num_col.astype(np.int64) * (pb.nL.astype(np.int64) + 1))
    r4c = np.full(int(num_col.astype(np.int64).sum()) * k, -7, np.int64) if want_lists else None
    c4r = np.full(int(num_row.astype(np.int64).sum()) * k, -7, np.int64) if want_lists else None
    gain = np.full((n, k), np.nan)
    nf = np.zeros(n, np.int32)
    probs = np.zeros(int((num_col.astype(np.int64) * (pb.nL.astype(np.int64) + 1)).sum())) if weight_mode else None
    nL = pb.nL.astype(np.int32)
    check(lib().pda_murty_batch_host(_p(pb.costs), _p(pb.cost_off), _p(num_row), _p(num_col), n, k, cut_mode,
                                     float(cutoff), int(maximize), int(cut_maximize),
                                     _p(r4c), _p(r4c_off), _p(c4r), _p(c4r_off), _p(gain), _p(nf),
                                     weight_mode, _p(probs), _p(prob_off), _p(nL), device))
    return KBestResult(nf, gain, r4c, r4c_off, c4r, c4r_off, probs, prob_off if weight_mode else None, k)


def assignment_prob_batch(pb: ProblemBatch, k: int, device: int = 0) -> KBestResult:
    """assignmentProb for every problem: weights only (the k-best lists stay on the device)."""
    return murty_batch(pb, k, cut_mode=CUT_RELATIVE, cutoff=GATE, weight_mode=WEIGHTS_GATED,
                       want_lists=False, device=device)


def assignment_prob_ladder_batch(pb: ProblemBatch, ks, device: int = 0):
    """assignmentProb for every problem and every k in ks, from one enumeration to max(ks);
    pda_assignment_prob_ladder_batch_host.  Returns (one (nK, nM, nL+1) array per problem, nFound[n, nK]); slot j is
    bit-identical to assignment_prob_batch(pb, ks[j])."""
    n = len(pb)
    ks = np.ascontiguousarray(ks, dtype=np.int32)
    nk = int(ks.size)
    num_row, num_col, nL = pb.num_row, pb.nM.astype(np.int32), pb.nL.astype(np.int32)
    cells = num_col.astype(np.int64) * (nL.astype(np.int64) + 1)
    prob_off = _prefix(cells * nk)
    probs = np.zeros(max(int(cells.sum()) * nk, 1))
    nf = np.zeros((n, max(nk, 1)), np.int32)
    check(lib().pda_assignment_prob_ladder_batch_host(_p(pb.costs), _p(pb.cost_off), _p(num_row), _p(num_col), _p(nL), n,
                                                      _p(ks), nk, _p(probs), _p(prob_off), _p(nf), device))
    tabs = [probs[prob_off[p]:prob_off[p] + nk * int(cells[p])].reshape(nk, int(num_col[p]), int(nL[p]) + 1)
            for p in range(n)]
    return tabs, nf


def lap_batch(pb: ProblemBatch, *, make_safe: bool = True, maximize: bool = False,
              num_col4gain: np.ndarray | None = None, device: int = 0):
    n = len(pb)
    num_row, num_col = pb.num_row, pb.nM.astype(np.int32)
    row_off, col_off = _prefix(num_row), _prefix(num_col)
    c4r = np.zeros(int(num_row.sum()), np.int64)
    r4c = np.zeros(int(num_col.sum()), np.int64)
    u, v = np.zeros(int(num_col.sum())), np.zeros(int(num_row.sum()))
    fb = np.zeros(int(num_row.sum()), np.uint8)
    gain, feas = np.zeros(n), np.zeros(n, np.int32)
    ng = None if num_col4gain is None else np.ascontiguousarray(num_col4gain, dtype=np.int32)
    check(lib().pda_lap_batch_host(_p(pb.costs), _p(pb.cost_off), _p(num_row), _p(num_col), _p(ng), n,
                                   int(make_safe), int(maximize), _p(row_off), _p(col_off), _p(c4r), _p(r4c),
                                   _p(u), _p(v), _p(fb), _p(gain), _p(feas), device))
    return dict(col4row=c4r, row4col=r4c, u=u, v=v, forbidden=fb, gain=gain, feasible=feas,
                row_off=row_off, col_off=col_off)


def condition_costs_batch(pb: ProblemBatch, device: int = 0):
    """conditionCosts for every problem -> (conditioned ProblemBatch, list of rowIdx arrays)."""
    n = len(pb)
    num_row, num_col = pb.num_row, pb.nM.astype(np.int32)
    row_off = _prefix(num_row)
    out = np.zeros_like(pb.costs)
    idx = np.zeros(int(num_row.sum()), np.int64)
    good = np.zeros(n, np.int32)
    check(lib().pda_condition_costs_batch_host(_p(pb.costs), _p(pb.cost_off), _p(num_row), _p(num_col), n,
                                               _p(row_off), _p(out), _p(idx), _p(good), device))
    mats, nls, maps = [], [], []
    for p in range(n):
        g, nc = int(good[p]), int(num_col[p])
        o = int(pb.cost_off[p])
        mats.append(out[o:o + g * nc].reshape((g, nc), order="F").copy())
        nls.append(g - nc)
        maps.append(idx[row_off[p]:row_off[p] + g].copy())
    return pack(mats, nls), maps


def permanent_batch(mats: list[np.ndarray], device: int = 0):
    """permanentExact of every (rows, cols) matrix -> (values, status)."""
    n = len(mats)
    rows = np.asarray([m.shape[0] for m in mats], np.int32)
    cols = np.asarray([m.shape[1] for m in mats], np.int32)
    off = _prefix(rows.astype(np.int64) * cols)
    flat = np.concatenate([np.asarray(m, np.float64).reshape(-1, order="F") for m in mats]) if n else np.zeros(0)
    flat = np.ascontiguousarray(flat if flat.size else np.zeros(1))
    out, st = np.zeros(n), np.zeros(n, np.int32)
    check(lib().pda_permanent_batch_host(_p(flat), _p(off), _p(rows), _p(cols), n, _p(out), _p(st), device))
    return out, st


def permanent_approx_batch(mats: list[np.ndarray], iterations: int = 300, seed: int = 20260217, device: int = 0):
    """Huber's approximate permanent (nwPerm.cpp:126-211) for a list of (rows, cols) matrices -> (estimates, status)."""
    flat = [np.asfortranarray(m, dtype=np.float64).reshape(-1, order="F") for m in mats]
    sizes = np.asarray([f.size for f in flat], np.int64)
    off = _prefix(sizes)
    buf = np.ascontiguousarray(np.concatenate(flat)) if flat else np.zeros(1)
    rows = np.asarray([m.shape[0] for m in mats], np.int32)
    cols = np.asarray([m.shape[1] for m in mats], np.int32)
    out, st = np.zeros(len(mats)), np.zeros(len(mats), np.int32)
    check(lib().pda_permanent_approx_batch_host(_p(buf), _p(off), _p(rows), _p(cols), len(mats), int(iterations), int(seed),
                                                _p(out), _p(st), device))
    return out, st


def permanentApproximation(A: np.ndarray, iterations: int = 300, seed: int = 20260217, device: int = 0) -> float:
    return float(permanent_approx_batch([A], iterations, seed, device)[0][0])


def conditioned_permanent_batch(mats: list[np.ndarray], perm_opt: int = 1, device: int = 0):
    n = len(mats)
    rows = np.asarray([m.shape[0] for m in mats], np.int32)
    cols = np.asarray([m.shape[1] for m in mats], np.int32)
    off = _prefix(rows.astype(np.int64) * cols)
    flat = np.ascontiguousarray(np.concatenate([np.asarray(m, np.float64).reshape(-1, order="F") for m in mats]))
    out, st = np.zeros(n), np.zeros(n, np.int32)
    check(lib().pda_conditioned_permanent_batch_host(_p(flat), _p(off), _p(rows), _p(cols), n, perm_opt,
                                                     _p(out), _p(st), device))
    return out, st


def permanent_prob_batch(pb: ProblemBatch, perm_opt: int = 1, device: int = 0):
    """permanentProb for every problem -> (list of (nM, nL+1) tables, status)."""
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    prob_off = _prefix(nM.astype(np.int64) * (nL.astype(np.int64) + 1))
    probs = np.zeros(int((nM.astype(np.int64) * (nL.astype(np.int64) + 1)).sum()))
    st = np.zeros(n, np.int32)
    check(lib().pda_permanent_prob_batch_host(_p(pb.costs), _p(pb.cost_off), _p(nL), _p(nM), n, perm_opt,
                                              _p(probs), _p(prob_off), _p(st), device))
    tabs = [probs[prob_off[p]:prob_off[p] + int(nM[p]) * (int(nL[p]) + 1)].reshape(int(nM[p]), int(nL[p]) + 1)
            for p in range(n)]
    return tabs, st


def _device_call_args(tensors, what):
    import torch
    for name, t in tensors.items():
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous()):
            raise ValueError(f"{what}: {name} must be a contiguous CUDA tensor")
    return torch.cuda.current_stream().cuda_stream


def permanent_prob_batch_device(costs, cost_off, nL, nM, prob_off, total_prob_elems: int, max_num_row: int, max_num_col: int,
                                perm_opt: int = 1, probs=None, status=None, workspace=None):
    """pda_permanent_prob_batch on CUDA tensors, enqueued on the current stream (no synchronisation): costs float64,
    cost_off / prob_off int64, nL / nM int32.  The nM x (nL+1) tables go to probs (float64, total_prob_elems; allocated
    when None) at prob_off; status (int32) as in include/pda_b200.h.  Returns (probs, status)."""
    import torch
    dev = costs.device
    probs = torch.zeros(max(int(total_prob_elems), 1), dtype=torch.float64, device=dev) if probs is None else probs
    status = torch.empty(nL.shape[0], dtype=torch.int32, device=dev) if status is None else status
    n = int(nL.shape[0])
    if workspace is None:
        workspace = alloc_workspace(lib().pda_permanent_prob_workspace_bytes(n, int(costs.numel()), int(total_prob_elems),
                                                                             max_num_row, max_num_col, perm_opt), dev)
    stream = _device_call_args(dict(costs=costs, cost_off=cost_off, nL=nL, nM=nM, prob_off=prob_off, probs=probs,
                                    status=status, workspace=workspace), "permanent_prob_batch_device")
    check(lib().pda_permanent_prob_batch(costs.data_ptr(), cost_off.data_ptr(), nL.data_ptr(), nM.data_ptr(), n,
                                         int(costs.numel()), int(total_prob_elems), max_num_row, max_num_col, perm_opt,
                                         probs.data_ptr(), prob_off.data_ptr(), status.data_ptr(), workspace.data_ptr(),
                                         int(workspace.numel()), stream))
    return probs, status


def conditioned_permanent_batch_device(mats, mat_off, rows, cols, max_dim: int, perm_opt: int = 1, out=None, status=None,
                                       workspace=None):
    """pda_conditioned_permanent_batch on CUDA tensors (mats float64 column-major at mat_off int64, rows / cols int32),
    enqueued on the current stream.  Returns (out float64, status int32)."""
    import torch
    dev = mats.device
    n = int(rows.shape[0])
    out = torch.zeros(n, dtype=torch.float64, device=dev) if out is None else out
    status = torch.empty(n, dtype=torch.int32, device=dev) if status is None else status
    if workspace is None:
        workspace = alloc_workspace(lib().pda_conditioned_permanent_workspace_bytes(n, max_dim, perm_opt), dev)
    stream = _device_call_args(dict(mats=mats, mat_off=mat_off, rows=rows, cols=cols, out=out, status=status,
                                    workspace=workspace), "conditioned_permanent_batch_device")
    check(lib().pda_conditioned_permanent_batch(mats.data_ptr(), mat_off.data_ptr(), rows.data_ptr(), cols.data_ptr(), n,
                                                max_dim, perm_opt, out.data_ptr(), status.data_ptr(), workspace.data_ptr(),
                                                int(workspace.numel()), stream))
    return out, status


def association_probs_batch(pb: ProblemBatch, k: int, device: int = 0) -> list[np.ndarray]:
    """getAssignmentProbs from the cost matrices on (assignment.cpp:57-74, usePerm = 0), fused on the device:
    conditionCosts -> assignmentProb -> scatter back through rowIdx.  Returns one (nM, nL+1) table per problem."""
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    prob_off = _prefix(nM.astype(np.int64) * (nL.astype(np.int64) + 1))
    probs = np.zeros(int((nM.astype(np.int64) * (nL.astype(np.int64) + 1)).sum()))
    check(lib().pda_association_probs_batch_host(_p(pb.costs), _p(pb.cost_off), _p(nL), _p(nM), n, k, _p(probs), _p(prob_off), device))
    return [probs[prob_off[p]:prob_off[p] + int(nM[p]) * (int(nL[p]) + 1)].reshape(int(nM[p]), int(nL[p]) + 1) for p in range(n)]


def association_perm_probs_batch(pb: ProblemBatch, device: int = 0):
    """getAssignmentProbs from the cost matrices on with usePerm (assignment.cpp:57-74, :64), fused on the device:
    conditionCosts -> permanentProb(.., 1) -> scatter back through rowIdx.  Returns (one (nM, nL+1) table per problem,
    status): status 1 where the reference throws, 3 where conditioning kept fewer rows than detections."""
    n = len(pb)
    nL, nM = pb.nL.astype(np.int32), pb.nM.astype(np.int32)
    prob_off = _prefix(nM.astype(np.int64) * (nL.astype(np.int64) + 1))
    probs = np.zeros(max(int((nM.astype(np.int64) * (nL.astype(np.int64) + 1)).sum()), 1))
    st = np.zeros(n, np.int32)
    costs = pb.costs if pb.costs.size else np.zeros(1)
    check(lib().pda_association_perm_probs_batch_host(_p(costs), _p(pb.cost_off), _p(nL), _p(nM), n, _p(probs), _p(prob_off), _p(st), device))
    tabs = [probs[prob_off[p]:prob_off[p] + int(nM[p]) * (int(nL[p]) + 1)].reshape(int(nM[p]), int(nL[p]) + 1) for p in range(n)]
    return tabs, st


def _pack_moments(frames):
    """frames: list of (land_mean[nL,3], land_cov[nL,3,3], meas_mean[nM,3], meas_cov[nM,3,3]) -> flat arrays + offsets."""
    lm = [np.asarray(f[0], np.float64).reshape(-1, 3) for f in frames]
    mm = [np.asarray(f[2], np.float64).reshape(-1, 3) for f in frames]
    col = lambda c: np.asarray(c, np.float64).reshape(-1, 3, 3).transpose(0, 2, 1).reshape(-1, 9)  # column-major 3x3
    lc = [col(f[1]) for f in frames]
    mc = [col(f[3]) for f in frames]
    l_off = np.zeros(len(frames) + 1, np.int64); l_off[1:] = np.cumsum([a.shape[0] for a in lm])
    m_off = np.zeros(len(frames) + 1, np.int64); m_off[1:] = np.cumsum([a.shape[0] for a in mm])
    cat = lambda parts, w: np.ascontiguousarray(np.concatenate(parts, axis=0)) if parts else np.zeros((0, w))
    return cat(lm, 3), cat(lc, 9), l_off, cat(mm, 3), cat(mc, 9), m_off


def quadric_cost_batch(frames, nonassign: float, device: int = 0) -> list[np.ndarray]:
    """computeQuadricCostMatrix (assignment.cpp:705-722) for a batch of frames -> list of (nL+nM, nM) matrices."""
    lm, lc, lo, mm, mc, mo = _pack_moments(frames)
    nL, nM = np.diff(lo), np.diff(mo)
    sizes = (nL + nM) * nM
    out = np.zeros(max(int(sizes.sum()), 1))
    check(lib().pda_quadric_cost_batch_host(_p(lm), _p(lc), _p(lo), _p(mm), _p(mc), _p(mo), len(frames), float(nonassign), _p(out), device))
    off = np.concatenate([[0], np.cumsum(sizes)])
    return [out[off[f]:off[f + 1]].reshape((int(nL[f] + nM[f]), int(nM[f])), order="F") for f in range(len(frames))]


def association_from_moments_batch(frames, nonassign: float, k: int, device: int = 0) -> list[np.ndarray]:
    """getAssignmentProbs (assignment.cpp:38-74, usePerm == 0) for a batch of frames, from the quadric moments on, as
    one device pipeline -> list of (nM, nL+1) weight tables."""
    lm, lc, lo, mm, mc, mo = _pack_moments(frames)
    nL, nM = np.diff(lo), np.diff(mo)
    sizes = nM * (nL + 1)
    out = np.zeros(max(int(sizes.sum()), 1))
    check(lib().pda_association_from_moments_batch_host(_p(lm), _p(lc), _p(lo), _p(mm), _p(mc), _p(mo), len(frames), float(nonassign),
                                                        int(k), _p(out), device))
    off = np.concatenate([[0], np.cumsum(sizes)])
    return [out[off[f]:off[f + 1]].reshape(int(nM[f]), int(nL[f]) + 1) for f in range(len(frames))]


def association_perm_from_moments_batch(frames, nonassign: float, device: int = 0):
    """getAssignmentProbs (assignment.cpp:38-74, usePerm == 1) for a batch of frames, from the quadric moments on, as
    one device pipeline -> (list of (nM, nL+1) weight tables, status per frame)."""
    lm, lc, lo, mm, mc, mo = _pack_moments(frames)
    nL, nM = np.diff(lo), np.diff(mo)
    sizes = nM * (nL + 1)
    out = np.zeros(max(int(sizes.sum()), 1))
    st = np.zeros(len(frames), np.int32)
    check(lib().pda_association_perm_from_moments_batch_host(_p(lm), _p(lc), _p(lo), _p(mm), _p(mc), _p(mo), len(frames),
                                                             float(nonassign), _p(out), _p(st), device))
    off = np.concatenate([[0], np.cumsum(sizes)])
    return [out[off[f]:off[f + 1]].reshape(int(nM[f]), int(nL[f]) + 1) for f in range(len(frames))], st


def _moments_device_call(name, land_mean, land_cov, land_off, meas_mean, meas_cov, meas_off, max_nL, max_nM, prob_capacity,
                         probs, prob_off, status, workspace, ws_args, extra_out):
    """Shared body of the two *_from_moments_batch_device calls: outputs and workspace allocated where None, no host read
    of device memory.  A moments array with no rows goes in as a one-element stand-in, since its pointer may not be NULL."""
    import torch
    dev = land_off.device
    n = int(land_off.shape[0]) - 1
    land_cap = min(land_mean.numel() // 3, land_cov.numel() // 9)
    meas_cap = min(meas_mean.numel() // 3, meas_cov.numel() // 9)
    stand_in = lambda t: t if t.numel() else torch.zeros(1, dtype=torch.float64, device=dev)
    land_mean, land_cov, meas_mean, meas_cov = map(stand_in, (land_mean, land_cov, meas_mean, meas_cov))
    if prob_capacity is None:
        prob_capacity = probs.numel() if probs is not None else n * max_nM * (max_nL + 1)
    probs = torch.zeros(max(int(prob_capacity), 1), dtype=torch.float64, device=dev) if probs is None else probs
    prob_off = torch.empty(n + 1, dtype=torch.int64, device=dev) if prob_off is None else prob_off
    status = torch.empty(max(n, 1), dtype=torch.int32, device=dev) if status is None else status
    if workspace is None:
        workspace = alloc_workspace(getattr(lib(), name + "_workspace_bytes")(n, max_nL, max_nM, int(prob_capacity), *ws_args), dev)
    tensors = dict(land_mean=land_mean, land_cov=land_cov, land_off=land_off, meas_mean=meas_mean, meas_cov=meas_cov,
                   meas_off=meas_off, probs=probs, prob_off=prob_off, status=status, workspace=workspace)
    tensors.update({k: v for k, v in extra_out.items() if v is not None})
    stream = _device_call_args(tensors, name)
    return dict(land_cap=land_cap, meas_cap=meas_cap, prob_capacity=int(prob_capacity), probs=probs, prob_off=prob_off,
                status=status, workspace=workspace, stream=stream, means=(land_mean, land_cov, meas_mean, meas_cov))


def association_from_moments_batch_device(land_mean, land_cov, land_off, meas_mean, meas_cov, meas_off, max_nL: int,
                                          max_nM: int, nonassign: float, k: int, prob_capacity: int | None = None,
                                          probs=None, prob_off=None, status=None, n_found=None, workspace=None):
    """pda_association_from_moments_batch on CUDA tensors, enqueued on the current stream (no synchronisation, so it can
    be captured in a CUDA graph): moments float64 (means 3, covariances 9 column-major per row), land_off / meas_off
    int64 with nFrames+1 entries, frame shapes read on the device against the bounds max_nL / max_nM.  probs holds
    prob_capacity doubles (default: probs.numel(), or nFrames * max_nM * (max_nL+1) when probs is None).
    Returns (probs, prob_off, status, n_found); status 2 marks a frame that was not computed (include/pda_b200.h)."""
    import torch
    n = int(land_off.shape[0]) - 1
    n_found = torch.empty(max(n, 1), dtype=torch.int32, device=land_off.device) if n_found is None else n_found
    a = _moments_device_call("pda_association_from_moments", land_mean, land_cov, land_off, meas_mean, meas_cov, meas_off,
                             max_nL, max_nM, prob_capacity, probs, prob_off, status, workspace, (int(k),), dict(n_found=n_found))
    lm, lc, mm, mc = a["means"]
    check(lib().pda_association_from_moments_batch(
        lm.data_ptr(), lc.data_ptr(), land_off.data_ptr(), a["land_cap"], mm.data_ptr(), mc.data_ptr(), meas_off.data_ptr(),
        a["meas_cap"], n, max_nL, max_nM, float(nonassign), int(k), a["probs"].data_ptr(), a["prob_capacity"],
        a["prob_off"].data_ptr(), a["status"].data_ptr(), n_found.data_ptr(), a["workspace"].data_ptr(),
        int(a["workspace"].numel()), a["stream"]))
    return a["probs"], a["prob_off"], a["status"], n_found


def association_perm_from_moments_batch_device(land_mean, land_cov, land_off, meas_mean, meas_cov, meas_off, max_nL: int,
                                               max_nM: int, nonassign: float, prob_capacity: int | None = None, probs=None,
                                               prob_off=None, status=None, workspace=None):
    """pda_association_perm_from_moments_batch (usePerm, max_nM <= 11) on CUDA tensors, as
    association_from_moments_batch_device.  Returns (probs, prob_off, status)."""
    n = int(land_off.shape[0]) - 1
    a = _moments_device_call("pda_association_perm_from_moments", land_mean, land_cov, land_off, meas_mean, meas_cov,
                             meas_off, max_nL, max_nM, prob_capacity, probs, prob_off, status, workspace, (), {})
    lm, lc, mm, mc = a["means"]
    check(lib().pda_association_perm_from_moments_batch(
        lm.data_ptr(), lc.data_ptr(), land_off.data_ptr(), a["land_cap"], mm.data_ptr(), mc.data_ptr(), meas_off.data_ptr(),
        a["meas_cap"], n, max_nL, max_nM, float(nonassign), a["probs"].data_ptr(), a["prob_capacity"],
        a["prob_off"].data_ptr(), a["status"].data_ptr(), a["workspace"].data_ptr(), int(a["workspace"].numel()),
        a["stream"]))
    return a["probs"], a["prob_off"], a["status"]


def moments_to_device(frames, device="cuda"):
    """_pack_moments on CUDA tensors: (land_mean, land_cov, land_off, meas_mean, meas_cov, meas_off), the argument order
    of the *_from_moments_batch_device calls."""
    import torch
    lm, lc, lo, mm, mc, mo = _pack_moments(frames)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
    return t(lm), t(lc), t(lo), t(mm), t(mc), t(mo)


def computeQuadricCostMatrix(land_mean, land_cov, meas_mean, meas_cov, nonassign: float, device: int = 0) -> np.ndarray:
    return quadric_cost_batch([(land_mean, land_cov, meas_mean, meas_cov)], nonassign, device)[0]


def getCovs(quadrics: np.ndarray, device: int = 0) -> np.ndarray:
    """getCovs (assignment.cpp:693-703): n 4x4 dual quadrics -> n 3x3 shape matrices."""
    q = np.ascontiguousarray(quadrics, np.float64).reshape(-1, 16)
    out = np.zeros((q.shape[0], 9))
    check(lib().pda_quadric_covs_batch_host(_p(q), q.shape[0], _p(out), device))
    return out.reshape(-1, 3, 3)


def getAssignmentProbs(land_mean, land_cov, meas_mean, meas_cov, nonassign: float, k: int, device: int = 0,
                       usePerm: bool = False) -> np.ndarray:
    """The reference's SLAM entry point (assignment.cpp:38-74) on the moments getMeans/getCovs return; usePerm selects
    the permanent-based weights (:64) over the k-best ones.  Raises where the reference throws."""
    frame = [(land_mean, land_cov, meas_mean, meas_cov)]
    if not usePerm:
        return association_from_moments_batch(frame, nonassign, k, device)[0]
    tabs, st = association_perm_from_moments_batch(frame, nonassign, device)
    if st[0]:
        raise RuntimeError(f"getAssignmentProbs: the reference throws for this input (status {int(st[0])})")
    return tabs[0]


def asgn_bb_batch(boxes_l: list[np.ndarray], boxes_r: list[np.ndarray], nonassign: float, device: int = 0,
                  devices=None) -> list[np.ndarray]:
    """asgnBB (assignment.cpp:724-775) for a batch of frames; boxes are [count, 5] = xmin, ymin, xmax, ymax, xOffset.
    Returns per frame the right-box index paired with each left box (-1 = none).  devices: a list of CUDA device
    ordinals spreads the frames over them (pda_asgn_bb_batch_host_multi, one contiguous slice each) instead of `device`."""
    n = len(boxes_l)
    cl = np.asarray([len(b) for b in boxes_l], np.int64)
    cr = np.asarray([len(b) for b in boxes_r], np.int64)
    off_l = np.concatenate([[0], np.cumsum(cl)]).astype(np.int64)
    off_r = np.concatenate([[0], np.cumsum(cr)]).astype(np.int64)
    flat_l = np.ascontiguousarray(np.concatenate([np.asarray(b, np.float64).reshape(-1, 5) for b in boxes_l] + [np.zeros((0, 5))]))
    flat_r = np.ascontiguousarray(np.concatenate([np.asarray(b, np.float64).reshape(-1, 5) for b in boxes_r] + [np.zeros((0, 5))]))
    out = np.full(max(int(off_l[-1]), 1), -7, np.int32)
    pl, pr = _p(flat_l) if flat_l.size else None, _p(flat_r) if flat_r.size else None
    if devices is None:
        check(lib().pda_asgn_bb_batch_host(pl, _p(off_l), pr, _p(off_r), n, float(nonassign), _p(out), device))
    else:
        d = np.ascontiguousarray(devices, np.int32)
        check(lib().pda_asgn_bb_batch_host_multi(pl, _p(off_l), pr, _p(off_r), n, float(nonassign), _p(out), _p(d), len(d)))
    return [out[off_l[f]:off_l[f + 1]].copy() for f in range(n)]


def asgn_bb_batch_device(boxes_l, off_l, boxes_r, off_r, max_nL: int, max_boxes: int, nonassign: float, assignment=None,
                         status=None, workspace=None):
    """pda_asgn_bb_batch on CUDA tensors, enqueued on the current stream (no synchronisation, so it can be captured in a
    CUDA graph): boxes float64 (5 per box), off_l / off_r int64 with nFrames+1 entries, frame shapes read on the device
    against the bounds max_nL (left boxes) and max_boxes (left + right boxes).  assignment (int32, one entry per left
    box the boxes_l tensor holds) is allocated filled with -1 when None.  Returns (assignment, status); status 2 marks a
    frame that was not computed (include/pda_b200.h)."""
    import torch
    dev = off_l.device
    n = int(off_l.shape[0]) - 1
    cap_l, cap_r = boxes_l.numel() // 5, boxes_r.numel() // 5
    assignment = torch.full((max(cap_l, 1),), -1, dtype=torch.int32, device=dev) if assignment is None else assignment
    status = torch.empty(max(n, 1), dtype=torch.int32, device=dev) if status is None else status
    if workspace is None:
        workspace = alloc_workspace(lib().pda_asgn_bb_workspace_bytes(n, max_nL, max_boxes), dev)
    stream = _device_call_args(dict(boxes_l=boxes_l, off_l=off_l, boxes_r=boxes_r, off_r=off_r, assignment=assignment,
                                    status=status, workspace=workspace), "asgn_bb_batch_device")
    ptr = lambda t: t.data_ptr() if t.numel() else None
    check(lib().pda_asgn_bb_batch(ptr(boxes_l), off_l.data_ptr(), cap_l, ptr(boxes_r), off_r.data_ptr(), cap_r, n, int(max_nL),
                                  int(max_boxes), float(nonassign), assignment.data_ptr(), status.data_ptr(),
                                  workspace.data_ptr(), int(workspace.numel()), stream))
    return assignment, status


def asgnBB(bbL: np.ndarray, bbR: np.ndarray, nonassign: float, device: int = 0) -> np.ndarray:
    """assignment.h:21 for one frame."""
    return asgn_bb_batch([np.asarray(bbL, np.float64).reshape(-1, 5)], [np.asarray(bbR, np.float64).reshape(-1, 5)], nonassign, device)[0]


def permanent_range(a: np.ndarray, begin: int, end: int, device: int = 0) -> tuple[float, float]:
    """Partial NW sum of one square matrix over Gray indices [begin, end) as (hi, lo)."""
    a = np.asarray(a, np.float64)
    flat = np.ascontiguousarray(a.reshape(-1, order="F"))
    part = np.zeros(2)
    check(lib().pda_permanent_range_host(_p(flat), a.shape[0], begin, end, _p(part), device))
    return float(part[0]), float(part[1])


# ------------------------------------------------------------------------------------------------
# the reference's functions, name for name (batch of one)
# ------------------------------------------------------------------------------------------------
def _one(cmat: np.ndarray, nL: int | None = None) -> ProblemBatch:
    cmat = np.asarray(cmat, np.float64)
    return pack([cmat], [cmat.shape[0] - cmat.shape[1] if nL is None else nL])


def kBest2D(k: int, C: np.ndarray, maximize: bool = False, device: int = 0):
    """shortestPathCPP.hpp:204-212 -> (nFound, row4col[k, numCol], col4row[k, numRow], gain[k])."""
    pb = _one(C)
    r = murty_batch(pb, k, cut_mode=CUT_NONE, maximize=maximize, device=device)
    nr, nc = C.shape
    return int(r.n_found[0]), r.row4col.reshape(k, nc), r.col4row.reshape(k, nr), r.gain[0]


def kBest2DCutoff(k: int, C: np.ndarray, cutoff: float = GATE, maximize: bool = False, device: int = 0):
    """shortestPathCPP.hpp:256-265."""
    pb = _one(C)
    r = murty_batch(pb, k, cut_mode=CUT_RELATIVE, cutoff=cutoff, maximize=maximize, device=device)
    nr, nc = C.shape
    return int(r.n_found[0]), r.row4col.reshape(k, nc), r.col4row.reshape(k, nr), r.gain[0]


def kBest2D_sticky(k: int, C: np.ndarray, maximize: bool, stale_cutoff_gain: float, stale_maximize: bool, device: int = 0):
    """kBest2D on a ScratchSpace that kBest2DCutoff used before (toCut stays set, hpp:84-86)."""
    pb = _one(C)
    r = murty_batch(pb, k, cut_mode=CUT_STICKY, cutoff=stale_cutoff_gain, maximize=maximize,
                    cut_maximize=stale_maximize, device=device)
    nr, nc = C.shape
    return int(r.n_found[0]), r.row4col.reshape(k, nc), r.col4row.reshape(k, nr), r.gain[0]


def assign2D(C: np.ndarray, maximize: bool = False, device: int = 0):
    """shortestPathCPP.hpp:144-149 -> (ret, row4col, col4row, u, v, gain); ret 1 solved / 0 infeasible."""
    r = lap_batch(_one(C), make_safe=True, maximize=maximize, device=device)
    return int(r["feasible"][0]), r["row4col"], r["col4row"], r["u"], r["v"], float(r["gain"][0])


def shortestPathCPP(C: np.ndarray, numCol4Gain: int | None = None, device: int = 0):
    """shortestPathCPP.hpp:178-182 on an already-safe matrix -> (ret, row4col, col4row, u, v, gain, forbidden);
    ret 1 = infeasible (gain -1), 0 = solved."""
    ng = None if numCol4Gain is None else np.asarray([numCol4Gain], np.int32)
    r = lap_batch(_one(C), make_safe=False, num_col4gain=ng, device=device)
    return (0 if r["feasible"][0] else 1), r["row4col"], r["col4row"], r["u"], r["v"], float(r["gain"][0]), r["forbidden"]


def conditionCosts(C: np.ndarray, device: int = 0):
    """assignment.cpp:439-525 -> (conditioned matrix (goodRows, numCol), rowIdx)."""
    pb, maps = condition_costs_batch(_one(C), device)
    return pb.matrix(0), maps[0]


def toProbs(v: np.ndarray, device: int = 0) -> np.ndarray:
    """assignment.cpp:527-542."""
    v = np.ascontiguousarray(v, np.float64).copy()
    if v.size == 0:
        return v
    off, ln = np.zeros(1, np.int64), np.asarray([v.size], np.int64)
    check(lib().pda_to_probs_batch_host(_p(v), _p(off), _p(ln), 1, device))
    return v


def assignmentProb(C: np.ndarray, nL: int, k: int, device: int = 0) -> np.ndarray:
    """assignment.cpp:547-683 -> probs[nM, nL+1]."""
    pb = _one(C, nL)
    return assignment_prob_batch(pb, k, device).prob_table(pb, 0).copy()


def assignmentProbLadder(C: np.ndarray, nL: int, ks, device: int = 0) -> np.ndarray:
    """assignmentProb(C, nL, k) for every k in ks from one enumeration -> probs[nK, nM, nL+1]."""
    tabs, _ = assignment_prob_ladder_batch(_one(C, nL), ks, device)
    return tabs[0].copy()


def brute_force_k(C: np.ndarray) -> int:
    """upperK of bruteForceProb (assignment.cpp:858-868): Minc-type bound on the number of assignments,
    saturated at 20000 (the reference's double->size_t cast is undefined above 2^64)."""
    nr, nc = C.shape
    tau = 6.2831853071
    n, m = float(nr), float(nc)
    bound = tau ** ((m - n) / (2 * n)) * (n / m) ** m * math.exp(m / (12 * n * n) - 1 / (12 * m + 1))
    for r in range(nr):
        card = 1.0 + float(np.count_nonzero(C[r, :] < np.inf))
        bound *= (tau * card) ** (1.0 / (2.0 * card)) * card * math.exp(-1 + 1.0 / (12 * card * card))
        if not bound < 1e300:
            break
    return 20000 if not bound < 20000.0 else int(bound) + 1


def bruteForceProb(C: np.ndarray, nL: int, device: int = 0) -> np.ndarray:
    """assignment.cpp:835-964 -> probs[nM, nL+1]."""
    pb = _one(C, nL)
    k = 1 if C.shape[1] == 1 else brute_force_k(np.asarray(C, np.float64))
    r = murty_batch(pb, k, cut_mode=CUT_NONE, weight_mode=WEIGHTS_UNGATED, want_lists=False, device=device)
    return r.prob_table(pb, 0).copy()


def getAssignmentProbsFromCosts(C: np.ndarray, nL: int, k: int, usePerm: bool = False, device: int = 0) -> np.ndarray:
    """assignment.cpp:57-74: what getAssignmentProbs does once computeQuadricCostMatrix has produced C."""
    C = np.asarray(C, np.float64)
    if not usePerm:
        return association_probs_batch(_one(C, nL), k, device)[0].copy()
    tabs, st = association_perm_probs_batch(_one(C, nL), device)
    if st[0]:
        raise RuntimeError(f"getAssignmentProbsFromCosts: the reference throws for this input (status {int(st[0])})")
    return tabs[0].copy()


def permanentProb(C: np.ndarray, nL: int, permOpt: int = 1, device: int = 0):
    """assignment.cpp:145-290 -> probs[nM, nL+1]; raises where the reference throws."""
    tabs, st = permanent_prob_batch(_one(C, nL), permOpt, device)
    if st[0]:
        raise RuntimeError("permanentProb: the reference throws for this input (dimension > 32 or bad permOpt)")
    return tabs[0]


def conditionedPermanent(A: np.ndarray, permOpt: int = 1, device: int = 0) -> float:
    """assignment.cpp:325-435."""
    out, st = conditioned_permanent_batch([np.asarray(A, np.float64)], permOpt, device)
    if st[0]:
        raise RuntimeError("conditionedPermanent: the reference throws for this input")
    return float(out[0])


def permanentExact(A: np.ndarray, device: int = 0) -> float:
    """nwPerm.cpp:217-231 (rectangular allowed)."""
    out, st = permanent_batch([np.asarray(A, np.float64)], device)
    if st[0]:
        raise RuntimeError("Maximum matrix dimension limited to 32. Error inside permanentExactSquare().")
    return float(out[0])


def permanentExactSquare(A: np.ndarray, device: int = 0) -> float:
    """nwPerm.cpp:251-332."""
    return permanentExact(A, device)


def permanentExactLong(A: np.ndarray, device: int = 0) -> float:
    """nwPerm.cpp:386-400: the same double kernel (the reference divides in long double; below 1 ulp)."""
    return permanentExact(A, device)
