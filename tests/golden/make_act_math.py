"""Generates ``act_math.npz``: points of the action noise's u1 grid where the device's ``logf`` (``rover_policy_math``,
the code ``normal2`` runs) is not the correctly rounded log, with the device's values.

``u1 = (k + 1) * 2^-24`` for every ``k < 2^24`` is evaluated on the device and in float64.  The file keeps up to 128
points where the disagreement reaches ``r = sqrt(-2 logf(u1))`` and up to 32 where it does not, plus the totals.  The
CPU tests (``tests/act_exact.py: RecordedMath``) use them so that a float64 log in place of ``logf`` is visible without
a GPU; ``tests/test_gpu_act_exact.py`` checks the file against the export.  Needs a CUDA device:

    python tests/golden/make_act_math.py [OUT]
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.abspath(os.path.join(HERE, "..", "..")), os.path.abspath(os.path.join(HERE, ".."))]

from isaac_rover_orbit_b200 import _lib  # noqa: E402

F = np.float32


def main(out=os.path.join(HERE, "act_math.npz")):
    dev = torch.device("cuda:0")
    u1 = ((np.arange(1 << 24, dtype=np.int64) + 1).astype(F) * F(2.0 ** -24)).astype(F)
    dev_log = _lib.policy_math(_lib.POLICY_MATH_LOG, torch.from_numpy(u1).to(dev)).cpu().numpy()
    ref_log = np.log(u1.astype(np.float64)).astype(F)
    bad = np.nonzero(dev_log.view(np.uint32) != ref_log.view(np.uint32))[0]
    r_dev = np.sqrt((F(-2) * dev_log[bad]).astype(F))
    r_ref = np.sqrt((F(-2) * ref_log[bad]).astype(F))
    reaches_r = r_dev.view(np.uint32) != r_ref.view(np.uint32)
    pick = lambda idx, k: idx[np.linspace(0, len(idx) - 1, min(k, len(idx))).astype(np.int64)] if len(idx) else idx  # noqa: E731
    keep = np.concatenate([pick(bad[reaches_r], 128), pick(bad[~reaches_r], 32)])
    np.savez(out, log_x=u1[keep], log_y=dev_log[keep], log_mismatches=np.int64(len(bad)),
             log_mismatches_reaching_r=np.int64(reaches_r.sum()), grid=np.int64(1 << 24))
    print(f"{out}: logf differs from the correctly rounded log at {len(bad)} of 2^24 u1 values "
          f"({int(reaches_r.sum())} reach r); kept {len(keep)}")


if __name__ == "__main__":
    main(*sys.argv[1:])
