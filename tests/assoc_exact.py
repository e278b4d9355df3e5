"""Exact association marginals, the truth the getAssignmentProbs tables stand for.  Shares no code and no algorithm with
the kernels or the CPU oracle: no LAP, no k-best list, no permanent.

E(C, nL) for an (nL+nM) x nM cost matrix C (rows: landmarks, then one dummy row per detection):
  - detection m goes either to a landmark l with C[l, m] <= colMin_m + 42 (the conditioning gate) or to its own dummy
    row nL+m;
  - no landmark takes two detections;
  - a hypothesis weighs exp(-sum of its costs);
  - E[m, l] is the weight share of the hypotheses that give m to l, E[m, nL] the share that leave m unassigned.

Detections interact only through landmarks they share, so the gate graph is cut into connected components and each is
solved on its own by a forward / backward DP over its landmarks whose state is the set of the component's detections
already taken.  Every term is a sum of products of non-negative numbers (no subtraction anywhere), accumulated in long
double, so each marginal is accurate to a few ulp of float64 relative to itself.
"""
from __future__ import annotations

import numpy as np

GATE = 42.0


def gate_graph(C: np.ndarray, nL: int):
    """(colMin[nM], in-gate boolean [nL, nM]).  Raises ValueError when a dummy row is gated away: the weight paths
    then differ from each other and from E (include/pda_b200.h)."""
    C = np.asarray(C, np.float64)
    nR, nM = C.shape
    assert nR == nL + nM
    col_min = C.min(axis=0)
    dummy = C[nL + np.arange(nM), np.arange(nM)]
    if not np.all(dummy <= col_min + GATE):
        raise ValueError("a dummy row is gated away")
    return col_min, np.isfinite(C[:nL]) & (C[:nL] <= col_min[None, :] + GATE)


def components(adj: np.ndarray):
    """Connected components of the bipartite gate graph: list of (detections, landmarks), detections ascending."""
    nL, nM = adj.shape
    seen_m = np.zeros(nM, bool)
    out = []
    for m0 in range(nM):
        if seen_m[m0]:
            continue
        dets, lands, stack = {m0}, set(), [m0]
        seen_m[m0] = True
        while stack:
            m = stack.pop()
            for l in np.flatnonzero(adj[:, m]):
                if l in lands:
                    continue
                lands.add(int(l))
                for m2 in np.flatnonzero(adj[l]):
                    if not seen_m[m2]:
                        seen_m[m2] = True
                        dets.add(int(m2))
                        stack.append(int(m2))
        out.append((sorted(dets), sorted(lands)))
    return out


def _component_dp(w, dum, one):
    """w[j][i]: weight of landmark j taking detection i (0 where out of gate); dum[i]: weight of i's dummy.  Returns
    (Z, marg[d, n_land + 1]) with marg[:, -1] the unassigned share.  State: bit mask of detections taken."""
    nl, d = len(w), len(dum)
    S = 1 << d
    masks = np.arange(S)
    zero = one - one
    # F[j][A]: landmarks < j took exactly the detections in A
    F = [np.full(S, zero, dtype=object if isinstance(one, int) else np.longdouble)]  # counts: exact Python ints
    F[0][0] = one
    for j in range(nl):
        f = F[j].copy()
        for i in range(d):
            if w[j][i] == zero:
                continue
            has = (masks >> i) & 1 == 1
            f[has] = f[has] + F[j][masks[has] ^ (1 << i)] * w[j][i]
        F.append(f)
    # B[j][R]: ways landmarks >= j and dummies complete the free detections R
    B = [None] * (nl + 1)
    b = np.full(S, one, dtype=F[0].dtype)
    for i in range(d):
        has = (masks >> i) & 1 == 1
        b[has] = b[has] * dum[i]
    B[nl] = b
    for j in range(nl - 1, -1, -1):
        b = B[j + 1].copy()
        for i in range(d):
            if w[j][i] == zero:
                continue
            has = (masks >> i) & 1 == 1
            b[has] = b[has] + B[j + 1][masks[has] ^ (1 << i)] * w[j][i]
        B[j] = b
    full = S - 1
    Z = (F[nl] * B[nl][full ^ masks]).sum()
    marg = np.full((d, nl + 1), zero, dtype=F[0].dtype)
    for i in range(d):
        free_i = (masks >> i) & 1 == 0
        A = masks[free_i]
        for j in range(nl):
            if w[j][i] != zero:
                marg[i, j] = (F[j][A] * B[j + 1][full ^ A ^ (1 << i)]).sum() * w[j][i]
        marg[i, nl] = (F[nl][A] * B[nl][full ^ A]).sum()
    return Z, marg


def exact_marginals(C: np.ndarray, nL: int, max_component: int = 16):
    """(E[nM, nL+1] float64, hypothesis count as a Python int).  max_component bounds the detections of one component
    (the DP holds 2^d states per landmark)."""
    C = np.asarray(C, np.float64)
    nM = C.shape[1]
    col_min, adj = gate_graph(C, nL)
    E = np.zeros((nM, nL + 1))
    count = 1
    for dets, lands in components(adj):
        if len(dets) > max_component:
            raise ValueError(f"a component of {len(dets)} detections")
        # costs relative to each detection's column minimum: the shift multiplies every hypothesis by the same factor
        w = [[np.exp(-np.longdouble(C[l, m] - col_min[m])) if adj[l, m] else np.longdouble(0) for m in dets] for l in lands]
        dum = [np.exp(-np.longdouble(C[nL + m, m] - col_min[m])) for m in dets]
        Z, marg = _component_dp(w, dum, np.longdouble(1))
        for a, m in enumerate(dets):
            for j, l in enumerate(lands):
                E[m, l] = float(marg[a, j] / Z)
            E[m, nL] = float(marg[a, -1] / Z)
        wi = [[1 if adj[l, m] else 0 for m in dets] for l in lands]
        n, _ = _component_dp(wi, [1] * len(dets), 1)
        count *= int(n)
    return E, count


def perm_status(C: np.ndarray, nL: int) -> int:
    """Status of getAssignmentProbs with usePerm on C (its gate graph as above): 1 where permanentProb on the conditioned
    problem meets a sub-matrix that keeps more than 32 rows (the reference throws), else 0."""
    C = np.asarray(C, np.float64)
    nM = C.shape[1]
    if nL == 0 or nM == 1:
        return 0
    col_min, _ = gate_graph(C, nL)
    cond = C - col_min[None, :]
    keep = np.any(cond <= GATE, axis=1)
    P = (cond[keep] < GATE)  # toProbs on the conditioned matrix (its minimum is 0): positive strictly inside 42
    condL = P.shape[0] - nM
    for m in range(nM):
        others = np.delete(np.arange(nM), m)
        live = P[:, others].any(axis=1)
        # sub-matrices of column m: without landmark row l where P[l, m] > 0, and without m's dummy row
        for r in [l for l in range(condL) if P[l, m]] + [condL + m]:
            if int(live.sum()) - int(live[r]) > 32:
                return 1
    return 0
