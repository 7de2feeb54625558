#!/usr/bin/env python
"""Role-level stall breakdown of the fused policy kernel (instrumented build, ocb_policy_debug_profile)."""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diverse_conventions_b200 import _native, layouts  # noqa: E402
from diverse_conventions_b200.overcooked_env import B200Overcooked  # noqa: E402
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet  # noqa: E402

NAMES = ["total", "col_empty", "head_full", "col_full", "a2_full", "w_full", "d1_full", "d2_full", "a2_empty", "d3_full",
         "head_empty", "w_empty", "issue_conv", "issue_fc", "ldg+stage", "cvt+tmem_st"]
NWAIT = 12  # entries [1, NWAIT) are barrier stalls; the rest are sub-intervals of the busy time
ROLES = ["epilogue", "loader", "mma", "producer"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layout", default="simple")
    ap.add_argument("--rows", type=int, default=32768)
    args = ap.parse_args()
    lp = layouts.load_layout(args.layout, 400)
    N = args.rows // 2
    env = B200Overcooked(args.layout, N, 0, horizon=400, seed=1)
    obs = env.rollout_random(37)["obs"][-1].contiguous()
    pol = FusedPolicy(lp, 64, 1)
    pol.set_weights(0, PolicyNet("actor", lp.width, lp.height, 20, 64).init_like_reference(1),
                    PolicyNet("critic", lp.width, lp.height, 20, 64).init_like_reference(2))
    out = pol.forward(obs)
    torch.cuda.synchronize()
    prof = np.zeros((256, 4, 16), dtype=np.int64)
    lib = _native.lib()
    for _ in range(2):
        ctas = _native.check(lib.ocb_policy_debug_profile(pol._h, ctypes.c_void_p(obs.data_ptr()), 2 * N, None,
                                                           ctypes.c_void_p(out["values"].data_ptr()),
                                                           ctypes.c_void_p(out["actions"].data_ptr()),
                                                           prof.ctypes.data_as(ctypes.c_void_p), 256))
    p = prof[:ctas]
    print(json.dumps({"layout": args.layout, "ctas": ctas, "info": pol.info()}))
    print("all CTAs (pair kernel; epilogue = actor group)", "mean cycles over", len(p), "CTAs")
    for r, rn in enumerate(ROLES):
        m = p[:, r, :].mean(axis=0)
        parts = ", ".join("%s %d" % (NAMES[i], m[i]) for i in range(1, len(NAMES)) if m[i] > 0)
        print("  %-9s total %7d  busy %7d | %s" % (rn, m[0], m[0] - m[1:NWAIT].sum(), parts))


if __name__ == "__main__":
    main()
