#!/usr/bin/env python
"""Device-timed throughput of the on-device policy rollouts (BASELINE configs 4 and 5), one GPU
or one rank per GPU under torchrun.

    python tools/rollout_bench.py --mode selfplay --layouts simple,random1 --worlds 8192 --T 100
    python tools/rollout_bench.py --mode crossplay --policies 16 --worlds-per-pair 1024

selfplay : MAPPO self-play rollout (actor + critic forward of both seats, sampling, env step,
           PPO buffer write), random-init networks, hidden 64.
mixed    : CoMeDi mixed-play collection: 2L env steps of replicas * (L-1) worlds, main and partner actor per step,
           per-row switch, diagonal / prefix buffer placement, main critic on the recorded rows.  --fused 1: one
           persistent launch + one value launch (ocb_rollout_mixed_fused), 0: 10L+4 per-step launches
           (ocb_rollout_mixed), -1: auto, 2: both arms on identical envs, timed alternately --rounds times.
crossplay: n x n pair matrix on coordination_ring, pairs sharded over the ranks, actors only,
           one 400-step episode per world, matrix gathered with one collective.
Prints one JSON line per configuration (rank 0)."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diverse_conventions_b200 import layouts, sharding  # noqa: E402
from diverse_conventions_b200.overcooked_env import B200Overcooked  # noqa: E402
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet  # noqa: E402
from diverse_conventions_b200.rollout import CrossPlayEvaluator, PolicyRollout  # noqa: E402


def timed(fn, iters, world, dev):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / iters


def power_limit(index):
    """the card's power limit in W (nvidia-smi query), or None where it cannot be read"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="selfplay", choices=["selfplay", "crossplay", "mixed"])
    ap.add_argument("--layouts", default="simple,unident_s,random1,random0,random3")
    ap.add_argument("--worlds", type=int, default=8192)
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--policies", type=int, default=16)
    ap.add_argument("--worlds-per-pair", type=int, default=1024)
    ap.add_argument("--hidden", type=int, default=64, choices=[64, 512])
    ap.add_argument("--L", type=int, default=400, help="mixed: episode_length of the trainer")
    ap.add_argument("--replicas", type=int, default=20, help="mixed: copies of the (L-1)-world scheme per GPU")
    ap.add_argument("--fused", type=int, default=-1, help="1: one persistent launch per rollout, 0: 2T+1 launches, -1: auto"
                    " (mixed: 2 = both arms, alternated)")
    ap.add_argument("--rounds", type=int, default=5, help="mixed --fused 2: alternations of the two arms")
    args = ap.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    if args.mode == "selfplay":
        for layout in args.layouts.split(","):
            lp = layouts.load_layout(layout, 400)
            pol = FusedPolicy(lp, args.hidden, 1, gpu_id=local)
            pol.set_weights(0, PolicyNet("actor", lp.width, lp.height, lp.channels, args.hidden).init_like_reference(1),
                            PolicyNet("critic", lp.width, lp.height, lp.channels, args.hidden).init_like_reference(2))
            env = B200Overcooked(layout, args.worlds, local, horizon=400, seed=1, world_offset=rank * args.worlds)
            ro = PolicyRollout(env, pol, args.T, seed=1, use_graph=bool(args.graph), fused=None if args.fused < 0 else bool(args.fused))
            ro.collect()
            ro.collect()
            ms = timed(ro.collect, args.iters, world, dev)
            rs, ep = sharding.reduce_episode_stats(*env.episode_stats())
            if rank == 0:
                agent_steps = 2 * args.worlds * world * args.T
                print(json.dumps({"mode": "selfplay", "layout": layout, "hidden": args.hidden, "n_gpus": world, "worlds_per_gpu": args.worlds,
                                  "T": args.T, "graph": bool(args.graph), "fused": bool(ro.fused), "ms_per_rollout": round(ms, 4),
                                  "us_per_env_step": round(1e3 * ms / args.T, 3),
                                  "agent_steps_per_s": round(agent_steps / (ms * 1e-3)),
                                  "buffer_mb": round(ro.buf.nbytes() / 2**20, 1),
                                  "episodes": int(ep), "mean_return": (float(rs) / int(ep)) if int(ep) else None}),
                      flush=True)
            env.close()
            pol.close()
    elif args.mode == "mixed":
        from diverse_conventions_b200.mixed import MixedPlayCollector  # noqa: E402
        for layout in args.layouts.split(","):
            lp = layouts.load_layout(layout, 400)
            pol = FusedPolicy(lp, args.hidden, 2, gpu_id=local)
            for i in range(2):
                pol.set_weights(i, PolicyNet("actor", lp.width, lp.height, lp.channels, args.hidden).init_like_reference(1 + 100 * i),
                                PolicyNet("critic", lp.width, lp.height, lp.channels, args.hidden).init_like_reference(2 + 100 * i))
            N = args.replicas * (args.L - 1)
            arms = [False, True] if args.fused == 2 else [None if args.fused < 0 else bool(args.fused)]
            cols, envs = [], []
            for fused in arms:
                env = B200Overcooked(layout, N, local, horizon=400, seed=1, world_offset=rank * N)
                col = MixedPlayCollector(env, pol, args.L, 0, 1, seed=1, mix_seed=7 + rank, use_graph=bool(args.graph),
                                         fused=fused)
                col.collect()
                col.collect()
                envs.append(env)
                cols.append(col)
            times = [[] for _ in cols]
            for _ in range(args.rounds if args.fused == 2 else 1):
                for i, col in enumerate(cols):
                    times[i].append(timed(col.collect, args.iters, world, dev))
            same = None
            if len(cols) == 2:  # both arms ran the same collections from the same state: same buffers, bit for bit
                torch.cuda.synchronize()
                a, b = cols[0].buf, cols[1].buf
                same = all(torch.equal(x, y) for x, y in zip(
                    (a.obs, a.actions, a.action_log_probs, a.value_preds, a.rewards, a.dones),
                    (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)))
            # the fused arm's critic pass on its own: main's critic (weight set 0) over the L * 2 * N recorded rows
            value_ms = None
            if any(col.fused for col in cols):
                rows = cols[-1].buf.obs[:args.L]
                vout = torch.empty((rows.numel() // (lp.width * lp.height * lp.channels),), dtype=torch.float32, device=dev)
                pol.value(rows, out=vout)
                value_ms = timed(lambda: pol.value(rows, out=vout), args.iters, world, dev)
            if rank == 0:
                env_agent_steps = 2 * N * world * 2 * args.L
                for col, t in zip(cols, times):
                    ms = sorted(t)[len(t) // 2]
                    print(json.dumps({"mode": "mixed", "layout": layout, "hidden": args.hidden, "n_gpus": world, "L": args.L,
                                      "replicas_per_gpu": args.replicas, "worlds_per_gpu": N, "world_tiles": (N + 63) // 64,
                                      "graph": bool(args.graph), "fused": bool(col.fused),
                                      "ms_per_collection": round(ms, 4), "ms_rounds": [round(x, 4) for x in t],
                                      "us_per_env_step": round(1e3 * ms / (2 * args.L), 3),
                                      "agent_steps_per_s": round(env_agent_steps / (ms * 1e-3)),
                                      "recorded_agent_steps_per_s": round(env_agent_steps / 2 / (ms * 1e-3)),
                                      # fused: rollout kernel, step-counter add, value pass, slot-L memset and fill
                                      "launches_per_collection": 5 if col.fused else 10 * args.L + 4,
                                      "ms_value_pass": round(value_ms, 4) if col.fused and value_ms is not None else None,
                                      "arms_bit_identical": same, "gpu": torch.cuda.get_device_name(dev),
                                      "power_limit_w": power_limit(local)}), flush=True)
            for env in envs:
                env.close()
            pol.close()
    else:
        layout = "random1"
        lp = layouts.load_layout(layout, 400)
        n = args.policies
        pol = FusedPolicy(lp, args.hidden, n, gpu_id=local)
        for i in range(n):  # seeds 1 + 100 i (seed_skip, train/config.py:315)
            pol.set_weights(i, PolicyNet("actor", lp.width, lp.height, lp.channels, args.hidden).init_like_reference(1 + 100 * i),
                            None)
        pairs = sharding.pair_shard(sharding.all_pairs(n), rank, world)
        ev = CrossPlayEvaluator(layout, pol, pairs, worlds_per_pair=args.worlds_per_pair, horizon=400, gpu_id=local,
                                seed=1, world_offset=rank * len(pairs) * args.worlds_per_pair, chunk_steps=50,
                                use_graph=bool(args.graph), total_worlds=n * n * args.worlds_per_pair)
        ev.run()
        out = {}

        def once():
            out["stats"] = ev.run()

        ms = timed(once, max(args.iters // 2, 1), world, dev)
        mean, eps = sharding.gather_pair_matrix(pairs, out["stats"][0], out["stats"][1], n)
        if rank == 0:
            worlds_total = n * n * args.worlds_per_pair
            print(json.dumps({"mode": "crossplay", "layout": layout, "n_gpus": world, "policies": n,
                              "worlds_per_pair": args.worlds_per_pair, "pairs_per_gpu": len(pairs),
                              "ms_per_matrix": round(ms, 3), "agent_steps_per_s": round(2 * worlds_total * 400 / (ms * 1e-3)),
                              "episodes": int(eps.sum()), "matrix_mean": float(mean.nanmean()),
                              "matrix_diag_mean": float(mean.diagonal().mean()),
                              "matrix_sha256": __import__("hashlib").sha256(mean.cpu().numpy().tobytes()).hexdigest()[:16],
                              "matrix_row0": [round(float(x), 3) for x in mean[0].tolist()]}), flush=True)
        ev.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
