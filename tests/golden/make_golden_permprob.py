"""Pins the bits of the permanentProb / conditionedPermanent host entries (pda_permanent_prob_batch_host,
pda_conditioned_permanent_batch_host) on the inputs of tests/test_gpu_permanent_prob_device.py, which checks both the
host and the device-pointer forms against them.

tests/golden/permprob_host_bits.npz was generated once on one NVIDIA B200 with the library of commit aa4e759, the last
in which the host entries ran their own materialising pipeline (build_items_kernel, perm_kernel, finish_probs_kernel):

    PDA_B200_LIB=<that build>/probabilisticsemslam_b200/libpda_b200.so python tests/golden/make_golden_permprob.py [out.npz]

Per call it stores the statuses and, for tables, one SHA-256 digest of each problem's bits (test_gpu_permanent_prob_device
.digests), for conditioned matrices the bits of the results.  Sub-permanents walked by the NW kernel follow its launch
shape, which follows the SM count, so the device name and SM count are stored as well.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

import test_gpu_permanent_prob_device as T  # noqa: E402
from helpers import bits  # noqa: E402


def cases(api):
    """(key, 'tables' | 'mats', inputs, permOpt) of every pinned host call."""
    out = []
    for o in (1, 2):
        out += [(f"golden.{o}", "tables", T.golden_problems(), o), (f"golden_mats.{o}", "mats", T.golden_mats(), o),
                (f"g1.{o}", "tables", T.g1_mixed(), o), (f"g2.{o}", "tables", T.g2_conditioned(api), o),
                (f"ragged.{o}", "tables", T.ragged(api), o), (f"nw_mats.{o}", "mats", T.nw_mats(), o),
                (f"retry.{o}", "mats", T.retry_matrices(T.RETRY_SEEDS), o)]
    out += [(f"edges.{o}", "mats", T.edge_mats(), o) for o in (0, 1, 2)]
    out += [("nw.1", "tables", T.synth.pack(*T.nw_problems()), 1), ("ragged.5", "tables", T.ragged(api), 5),
            ("invalid_opt_mats.-1", "mats", T.invalid_opt_mats(), -1), ("approx.0", "tables", T.approx_problems(), 0),
            ("approx_mats.0", "mats", T.approx_mats(), 0), ("chunks.1", "tables", T.chunked_problems(), 1)]
    return out


def main():
    import torch
    from probabilisticsemslam_b200 import _lib, api
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "permprob_host_bits.npz")
    _lib.lib().pda_set_approx_seed(T.SEED)
    rec = {"device": np.array(torch.cuda.get_device_name(0)),
           "sm_count": np.int64(torch.cuda.get_device_properties(0).multi_processor_count)}
    for key, kind, inputs, perm_opt in cases(api):
        if kind == "tables":
            tabs, st = api.permanent_prob_batch(inputs, perm_opt)
            rec[key + ".bits"] = T.digests(tabs)
        else:
            vals, st = api.conditioned_permanent_batch(inputs, perm_opt)
            rec[key + ".bits"] = bits(vals)
        rec[key + ".status"] = st
        print(key, kind, len(st), "statuses", np.bincount(st).tolist())
    np.savez_compressed(path, **rec)
    print("wrote", path, "on", rec["device"], int(rec["sm_count"]), "SMs")


if __name__ == "__main__":
    main()
