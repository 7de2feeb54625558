#!/usr/bin/env python
"""Device-timed cross-play TRAINING collection: XD's SP / XP slices and MultiConvention's best-response slices, with values.

    python tools/crossplay_train_bench.py --layouts simple,random1 --T 400 --reps 10

Shapes (1,024 worlds per slice, hidden 64, random-init networks with head gain 2, sampled actions):
  xd : ego 0 in self-play with its SP critic, then ego against each of three earlier conventions in both seatings with
       its XP critics (seat 0 / seat 1 per partner); partners get no critic: 7 slices, 7,168 worlds
  br : ego (actor and critic of set 0) against four fixed partners in both seatings: 8 slices, 8,192 worlds
Arms, alternated within each repetition, each replayed through a CUDA graph (CUDA events around each collection):
  per_step  : PolicyRollout(tile_policy, with_critic=True, fused=False): ocb_rollout_policy, 2T+1 dependent launches with
              both networks of every weight set on every row
  fused     : PolicyRollout(tile_policy, critic_policy=...): ocb_rollout_crossplay_train_fused, the cross-play launch and one
              critic pass over the seat tiles that have a critic
  crossplay : PolicyRollout(tile_policy, with_critic=False, fused=True): ocb_rollout_crossplay_fused alone, so that
              fused - crossplay is the critic pass's share
Before timing, per_step and fused (with critic_policy = tile_policy) are collected once from the same env state and every
buffer must be identical; the fused arm with the shape's own critic table must give the same trajectory.  Launch counts
are kernels per collection, counted with torch.profiler on an eager collection.  Prints one JSON line per (layout, shape)
with the card name, its power limit and maximum SM clock."""
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
from diverse_conventions_b200.rollout import PolicyRollout, crossplay_training_tables  # noqa: E402

LAYOUT_NAMES = {"simple": "cramped_room", "random1": "coordination_ring"}
WPS = 1024


def card():
    name = torch.cuda.get_device_name(torch.cuda.current_device())
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        limit = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        limit = None
    return name, limit


def shape_slices(shape):
    """(slices, weight sets) of a shape; see the module docstring"""
    if shape == "xd":
        partners, xp0, xp1 = [2, 3, 4], [5, 6, 7], [8, 9, 10]
        slices = ([((0, 1), (0, 1))] + [((0, xp0[j]), (p, None)) for j, p in enumerate(partners)] +
                  [((p, None), (0, xp1[j])) for j, p in enumerate(partners)])
        return slices, 11
    partners = [1, 2, 3, 4]
    return [((0, 0), (p, None)) for p in partners] + [((p, None), (0, 0)) for p in partners], 5


def population(lp, n, seed0=100):
    pol = FusedPolicy(lp, 64, n)
    for i in range(n):
        actor = PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + i, gain=2.0)
        critic = PolicyNet("critic", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + 1000 + i)
        pol.set_weights(i, actor, critic)
    return pol


def buffers(b):
    return [None if x is None else x.clone() for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)]


def kernels_per_collection(ro):
    """kernels of one eager collection minus the observe that primes slot 0"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ro._issue(False)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return sum(1 for n in names if not n.lower().startswith(("memcpy", "memset")))


def run(layout, shape, T, reps, horizon):
    slices, n_sets = shape_slices(shape)
    lp = layouts.load_layout(layout, horizon)
    pol = population(lp, n_sets)
    dev = torch.device("cuda", torch.cuda.current_device())
    tile, critic = crossplay_training_tables(slices, WPS, dev)
    N = len(slices) * WPS
    valued_rows = int((critic >= 0).sum()) * 128 * (T + 1)

    # equality at the timed size, eager, from the same env state
    got = {}
    launches = {}
    for arm, kw in (("per_step", dict(fused=False)), ("fused_full", dict(critic_policy=tile)),
                    ("fused", dict(critic_policy=critic)), ("crossplay", dict(with_critic=False, fused=True))):
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
        ro = PolicyRollout(env, pol, T, tile, seed=3, **kw)
        got[arm] = buffers(ro.collect())
        torch.cuda.synchronize()
        if arm != "fused_full":
            launches[arm] = kernels_per_collection(ro)
        env.close()
    for name, x, y in zip(("obs", "actions", "logp", "values", "rewards", "dones"), got["per_step"], got["fused_full"]):
        if not torch.equal(x, y):
            raise RuntimeError("per-step and fused buffers differ (%s) on %s %s" % (name, layout, shape))
    for i in (0, 1, 2, 4, 5):
        if not (torch.equal(got["per_step"][i], got["fused"][i]) and torch.equal(got["per_step"][i], got["crossplay"][i])):
            raise RuntimeError("trajectories differ on %s %s" % (layout, shape))
    del got

    arms = {}
    envs = []
    for arm, kw in (("per_step", dict(fused=False)), ("fused", dict(critic_policy=critic)),
                    ("crossplay", dict(with_critic=False, fused=True))):
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
        envs.append(env)
        arms[arm] = PolicyRollout(env, pol, T, tile, seed=3, use_graph=True, **kw)

    def once(ro):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ro.collect()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for ro in arms.values():  # warm-up: module load, graph capture
        once(ro)
        once(ro)
    if not (arms["fused"].fused and arms["crossplay"].fused):
        raise RuntimeError("a fused arm declined this shape")
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, ro in arms.items():
            ms[k].append(once(ro))
    out = {"layout": LAYOUT_NAMES.get(layout, layout), "shape": shape, "slices": len(slices), "worlds": N, "T": T,
           "horizon": horizon, "reps": reps, "valued_rows": valued_rows, "buffers_identical": True}
    for k, v in ms.items():
        med = statistics.median(v)
        out[k] = {"ms_median": round(med, 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4),
                  "us_per_env_step": round(1000.0 * med / T, 3), "kernels_per_collection": launches[k]}
    crit = out["fused"]["ms_median"] - out["crossplay"]["ms_median"]
    out["critic_pass_ms"] = round(crit, 4)
    out["critic_rows_per_s"] = round(valued_rows / (crit / 1000.0), 1) if crit > 0 else None
    out["per_step_over_fused"] = round(out["per_step"]["ms_median"] / out["fused"]["ms_median"], 3)
    for e in envs:
        e.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="simple,random1")
    ap.add_argument("--shapes", default="xd,br")
    ap.add_argument("--T", type=int, default=400)
    ap.add_argument("--horizon", type=int, default=400)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("crossplay_train_bench.py measures on the GPU; no CUDA device is visible")
    name, limit = card()
    for layout in args.layouts.split(","):
        for shape in args.shapes.split(","):
            res = run(layout, shape, args.T, args.reps, args.horizon)
            res["device"], res["power_limit_and_max_sm_clock"] = name, limit
            print(json.dumps(res), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
