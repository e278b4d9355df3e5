"""The usePerm body of getAssignmentProbs as separate library calls -- conditionCosts -> permanentProb(cond, condL, nM, 1)
-> scatter of the first condL conditioned rows back through rowIdx (assignment.cpp:57-74) -- which is how
getAssignmentProbsFromCosts(usePerm=True) ran before the fused pipeline existed.  The bit-identity tests
(tests/test_gpu_association_perm.py) and scripts/perm_association_bench.py both compare the fused pipeline with it."""
import numpy as np


def composed(api, pb):
    """-> (tables, status).  The route's only gate is condL = goodRows - nM >= 0 (below that the reference's size_t
    subtraction underflows and the separate calls reject the problem): such problems get an all-zero table and status 3,
    the fused pipeline's convention.  nL == 0 gives {1} per detection (:51-53)."""
    n = len(pb)
    cond, maps = api.condition_costs_batch(pb)
    ok = [p for p in range(n) if pb.nL[p] > 0 and cond.nL[p] >= 0]
    cp, st = api.permanent_prob_batch(cond.take(np.asarray(ok, np.int64)), 1) if ok else ([], [])
    where = {p: i for i, p in enumerate(ok)}
    tabs, status = [], np.zeros(n, np.int32)
    for p in range(n):
        nL, nM = int(pb.nL[p]), int(pb.nM[p])
        t = np.zeros((nM, nL + 1))
        if nL == 0:
            t[:] = 1.0
        elif p not in where:
            status[p] = 3
        else:
            cL = int(cond.nL[p])
            t[:, maps[p][:cL]] = cp[where[p]][:, :cL]
            t[:, nL] = cp[where[p]][:, cL]
            status[p] = st[where[p]]
        tabs.append(t)
    return tabs, status
