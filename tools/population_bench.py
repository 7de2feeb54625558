#!/usr/bin/env python
"""Device-timed population self-play: S members, each in self-play on its own slice of worlds, with critic values.

    python tools/population_bench.py --layouts simple,random1 --worlds 8192,32768 --worlds-per-slice 512 --T 400

Arms, run alternately (one rollout of each per repetition, CUDA events around each):
  population : ocb_rollout_population_fused, one persistent launch for all slices (PolicyRollout with a self-play table)
  per_step   : ocb_rollout_policy with the same table (2T+1 launches), replayed through a CUDA graph
  sequential : one single-policy fused launch (ocb_rollout_policy_fused) per slice, back to back on one stream
  ceiling    : one single-policy fused launch over all the worlds (what one member would cost at the whole size)
Every rollout is T env steps of 2 N agents, hidden 64, random-init networks (head gain 2), sampled actions.  Prints one
JSON line per (layout, worlds) with the card name and its power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diverse_conventions_b200 import layouts  # noqa: E402
from diverse_conventions_b200.overcooked_env import B200Overcooked  # noqa: E402
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet  # noqa: E402
from diverse_conventions_b200.rollout import PolicyRollout, pair_tile_policy  # noqa: E402

LAYOUT_NAMES = {"simple": "cramped_room", "random1": "coordination_ring"}


def card():
    name = torch.cuda.get_device_name(torch.cuda.current_device())
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        limit = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        limit = None
    return name, limit


def population(lp, n, seed0=100):
    pol = FusedPolicy(lp, 64, n)
    for i in range(n):
        actor = PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + i, gain=2.0)
        critic = PolicyNet("critic", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + 1000 + i)
        pol.set_weights(i, actor, critic)
    return pol


def run(layout, N, wps, T, reps, horizon):
    S = N // wps
    lp = layouts.load_layout(layout, horizon)
    pol = population(lp, S)
    dev = torch.device("cuda", torch.cuda.current_device())
    table = pair_tile_policy([(s, s) for s in range(S)], wps, dev)
    arms = {}
    env_a = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
    ro_a = PolicyRollout(env_a, pol, T, table, seed=3)
    arms["population"] = [ro_a]
    env_b = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
    arms["per_step"] = [PolicyRollout(env_b, pol, T, table, seed=3, fused=False, use_graph=True)]
    envs_c = [B200Overcooked(layout, wps, 0, horizon=horizon, seed=1, world_offset=s * wps) for s in range(S)]
    arms["sequential"] = [PolicyRollout(e, pol, T, seed=3, fused=True, policy_index=s) for s, e in enumerate(envs_c)]
    env_d = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
    arms["ceiling"] = [PolicyRollout(env_d, pol, T, seed=3, fused=True)]

    def once(ros):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for ro in ros:
            ro.collect()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for ros in arms.values():  # warm-up: module load, graph capture
        once(ros)
    if not ro_a.fused:
        raise RuntimeError("the population launch declined this shape")
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, ros in arms.items():
            ms[k].append(once(ros))
    out = {"layout": LAYOUT_NAMES.get(layout, layout), "worlds": N, "slices": S, "worlds_per_slice": wps, "T": T,
           "horizon": horizon, "reps": reps}
    for k, v in ms.items():
        med = statistics.median(v)
        out[k] = {"ms_median": round(med, 4), "ms_min": round(min(v), 4), "us_per_env_step": round(1000.0 * med / T, 3),
                  "agent_steps_per_s": round(2 * N * T / (med / 1000.0), 1)}
    out["population_over_ceiling"] = round(out["population"]["ms_median"] / out["ceiling"]["ms_median"], 3)
    out["per_step_over_population"] = round(out["per_step"]["ms_median"] / out["population"]["ms_median"], 3)
    out["sequential_over_population"] = round(out["sequential"]["ms_median"] / out["population"]["ms_median"], 3)
    for e in [env_a, env_b, env_d] + envs_c:
        e.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="simple,random1")
    ap.add_argument("--worlds", default="8192,32768")
    ap.add_argument("--worlds-per-slice", type=int, default=512)
    ap.add_argument("--T", type=int, default=400)
    ap.add_argument("--horizon", type=int, default=400)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("population_bench.py measures on the GPU; no CUDA device is visible")
    name, limit = card()
    for layout in args.layouts.split(","):
        for N in (int(w) for w in args.worlds.split(",")):
            res = run(layout, N, args.worlds_per_slice, args.T, args.reps, args.horizon)
            res["device"], res["power_limit_and_max_sm_clock"] = name, limit
            print(json.dumps(res), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
