#!/usr/bin/env python
"""Cost of loading a trainer's updated parameters into the policy handle, and of one XD iteration around it.

    python tools/weight_refresh_bench.py --out profiles/r3_weight_refresh_bench_1gpu.jsonl

XD's refresh set with k earlier conventions is 2 + 3k networks: the ego's actor and SP critic (weight set 0) and its 3k
other critics (XP critics per seat and a mixed-play critic per convention; weight sets k + 1 .. 4k, after the k partners'
actors, which do not train).  Every network lives on the device, as a trainer's R_Actor / R_Critic parameters do.
refresh rows (layouts cramped_room / coordination_ring, hidden 64 / 512, k = 3 / 7), two arms alternated per repetition:
  host   : FusedPolicy.set_weights per weight set from the CUDA tensors (copies to the host, host packing, synchronous
           upload): host wall time until the last upload is done
  device : FusedPolicy.set_weights_device(sets): one call; CUDA events around it (device time) and the host time the call
           takes to return (enqueue)
iteration rows (hidden 64, T = 400, 1,024 worlds per slice: XD's SP slice and both seatings against each convention, the
shape of tools/crossplay_train_bench.py), two arms alternated, host wall time until the collection is done:
  host_then_graph : the host refresh, then the graph-replayed PolicyRollout(tile_policy, critic_policy)
  graph_weights   : one replay of the same collection's graph with weights=sets, the refresh inside it
Before timing, the blobs of both refresh arms and the buffers of both iteration arms (one collection each from the same env
state) must be identical.  Each line carries the card name, its power limit and maximum SM clock."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diverse_conventions_b200 import layouts  # noqa: E402
from diverse_conventions_b200.overcooked_env import B200Overcooked  # noqa: E402
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet  # noqa: E402
from diverse_conventions_b200.rollout import PolicyRollout, crossplay_training_tables  # noqa: E402

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


def device_net(kind, lp, hidden, seed):
    src = PolicyNet(kind, lp.width, lp.height, lp.channels, hidden).init_like_reference(seed, gain=2.0 if kind == "actor" else 1.0)
    dev = torch.device("cuda", torch.cuda.current_device())
    params = {k: v.to(dev) for k, v in src.state_dict().items()}
    return PolicyNet(kind, lp.width, lp.height, lp.channels, hidden, device=dev).alias_state_dict(params)


def xd_sets(lp, hidden, k):
    """(refresh sets, partner actors by weight set, number of weight sets)"""
    sets = [(0, device_net("actor", lp, hidden, 1), device_net("critic", lp, hidden, 2))]
    sets += [(k + 1 + j, None, device_net("critic", lp, hidden, 100 + j)) for j in range(3 * k)]
    partners = {1 + j: device_net("actor", lp, hidden, 50 + j) for j in range(k)}
    return sets, partners, 1 + 4 * k


def host_refresh(pol, sets):
    for index, actor, critic in sets:
        pol.set_weights(index, actor, critic)


def stats(v):
    return {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4)}


def perturb(sets, step):
    """stand-in for an optimizer step: every refreshed parameter changes in place"""
    g = torch.Generator(device=torch.device("cuda", torch.cuda.current_device())).manual_seed(step)
    for _, actor, critic in sets:
        for net in (actor, critic):
            if net is not None:
                for t in net.state_dict().values():
                    t.add_(torch.randn(t.shape, generator=g, device=t.device), alpha=1e-3)


def bench_refresh(layout, hidden, k, reps):
    lp = layouts.load_layout(layout, 400)
    sets, partners, n = xd_sets(lp, hidden, k)
    pol_h, pol_d = FusedPolicy(lp, hidden, n), FusedPolicy(lp, hidden, n)
    for pol in (pol_h, pol_d):
        for i, a in partners.items():
            pol.set_weights(i, a)
    host_refresh(pol_h, sets)
    pol_d.set_weights_device(sets)
    torch.cuda.synchronize()
    for i in range(n):
        for net in (0, 1):
            if not torch.equal(pol_h.read_blob(i, net), pol_d.read_blob(i, net)):
                raise RuntimeError("host and device blobs differ: set %d net %d (%s, hidden %d)" % (i, net, layout, hidden))
    host_ms, dev_ms, enq_ms = [], [], []
    for r in range(reps + 2):
        perturb(sets, r)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        host_refresh(pol_h, sets)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t2 = time.perf_counter()
        pol_d.set_weights_device(sets)
        t3 = time.perf_counter()
        e1.record()
        torch.cuda.synchronize()
        if r >= 2:  # two warm-up rounds
            host_ms.append(1e3 * (t1 - t0))
            dev_ms.append(e0.elapsed_time(e1))
            enq_ms.append(1e3 * (t3 - t2))
    weights_bytes = sum(t.numel() * 4 for _, a, c in sets for net in (a, c) if net is not None for t in net.state_dict().values())
    blob_bytes = sum(pol_d.read_blob(i, net).numel() for i, a, c in sets for net, x in ((0, a), (1, c)) if x is not None)
    networks = sum(1 for _, a, c in sets for x in (a, c) if x is not None)
    out = {"kind": "refresh", "layout": layout, "hidden": hidden, "k": k, "networks": networks, "reps": reps,
           "blobs_identical": True, "fp32_weight_bytes": weights_bytes, "packed_bytes": blob_bytes,
           "host_set_weights": stats(host_ms), "device_events": stats(dev_ms), "device_enqueue": stats(enq_ms)}
    out["host_over_device_events"] = round(out["host_set_weights"]["ms_median"] / out["device_events"]["ms_median"], 1)
    pol_h.close(), pol_d.close()
    return out


def buffers(b):
    return [None if x is None else x.clone() for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)]


def bench_iteration(layout, k, T, reps, horizon):
    lp = layouts.load_layout(layout, horizon)
    sets, partners, n = xd_sets(lp, 64, k)
    xp0, xp1 = [k + 1 + j for j in range(k)], [2 * k + 1 + j for j in range(k)]
    slices = ([((0, 0), (0, 0))] + [((0, xp0[j]), (1 + j, None)) for j in range(k)] +
              [((1 + j, None), (0, xp1[j])) for j in range(k)])
    dev = torch.device("cuda", torch.cuda.current_device())
    tile, critic = crossplay_training_tables(slices, WPS, dev)
    N = len(slices) * WPS
    pols, ros, envs = {}, {}, []
    for arm in ("host_then_graph", "graph_weights"):
        pols[arm] = FusedPolicy(lp, 64, n)
        for i, a in partners.items():
            pols[arm].set_weights(i, a)
        host_refresh(pols[arm], sets)
    # equality at the timed size: one collection per arm from the same env state
    got = []
    for arm in pols:
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
        envs.append(env)
        ros[arm] = PolicyRollout(env, pols[arm], T, tile, seed=3, critic_policy=critic, use_graph=True,
                                 weights=sets if arm == "graph_weights" else None)
        if arm == "host_then_graph":
            host_refresh(pols[arm], sets)
        got.append(buffers(ros[arm].collect()))
        torch.cuda.synchronize()
    for name, x, y in zip(("obs", "actions", "logp", "values", "rewards", "dones"), *got):
        if not torch.equal(x, y):
            raise RuntimeError("iteration buffers differ (%s) on %s k=%d" % (name, layout, k))
    del got

    def once(arm):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        if arm == "host_then_graph":
            host_refresh(pols[arm], sets)
        ros[arm].collect()
        e1.record()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0), e0.elapsed_time(e1)

    for arm in ros:  # warm-up
        once(arm)
    wall = {a: [] for a in ros}
    for r in range(reps):
        perturb(sets, 1000 + r)
        for arm in ros:
            wall[arm].append(once(arm)[0])
    out = {"kind": "iteration", "layout": layout, "hidden": 64, "k": k, "networks": 2 + 3 * k, "slices": len(slices),
           "worlds": N, "T": T, "horizon": horizon, "reps": reps, "buffers_identical": True}
    for arm, v in wall.items():
        out[arm] = stats(v)
    out["host_then_graph_over_graph_weights"] = round(out["host_then_graph"]["ms_median"] / out["graph_weights"]["ms_median"], 3)
    for e in envs:
        e.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="cramped_room,coordination_ring")
    ap.add_argument("--hidden", default="64,512")
    ap.add_argument("--k", default="3,7")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--reps512", type=int, default=5)
    ap.add_argument("--T", type=int, default=400)
    ap.add_argument("--horizon", type=int, default=400)
    ap.add_argument("--iter-reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("weight_refresh_bench needs a CUDA device")
    name, limit = card()
    lines = []
    for layout in a.layouts.split(","):
        for hidden in (int(h) for h in a.hidden.split(",")):
            for k in (int(x) for x in a.k.split(",")):
                lines.append(bench_refresh(layout, hidden, k, a.reps if hidden == 64 else a.reps512))
        for k in (int(x) for x in a.k.split(",")):
            lines.append(bench_iteration(layout, k, a.T, a.iter_reps, a.horizon))
    for line in lines:
        line.update({"card": name, "power_limit_and_max_sm_clock": limit})
        print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
