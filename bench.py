#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (baseline/_ref)

Workload of the headline line (BASELINE.json configs[2], the one the metric's target is quoted on):
Overcooked cramped_room, 2 agents, horizon 400, 16,384 worlds per GPU, uniform random actions drawn on the
device, env step + observation encode only.

A bench "step" is one pass of the hot path over one batch: ONE fused launch (ocb_rollout_random) that advances
every world of the job by `--env-steps-per-pass` (default 100) environment steps and writes the
[T, P, N, W, H, C] observation slab (1.3 GB per GPU at the defaults, >> the 126 MB L2, so no flush is needed
between passes).  `value` = agent-steps (P x worlds x env steps) per second over all GPUs.  Every launch is timed
with its own pair of CUDA events on the launching stream; `roofline.launch_ms` is their mean without the first.

`e2e` runs the reference-facing single-step call with HOST (pinned) buffers — H2D of the actions, kernel, D2H of
observations + rewards + dones, every step inside the timed region — through the two-deep pipeline
(ocb_step_host_async / ocb_step_host_wait); the synchronous call (ocb_step_host) and a plain pinned D2H copy of
the same bytes (the PCIe ceiling of this box, all ranks copying at once) are timed beside it.

Further legs on the same line (the "+policy fwd" half of the metric and the gather):
  * `config4`: BASELINE configs[3] as stated — all five classic layouts, 8,192 worlds/GPU, T = 400, MAPPO self-play
    rollout with random-init actor + critic, hidden 64 (one persistent launch) and 512 (per-step launches), each
    with its own HBM / tensor roofline fractions and launch count;
  * `config5`: BASELINE configs[4] — 16 x 16 convention-pair matrix on coordination_ring, 1,024 worlds per pair,
    pairs sharded over the ranks, matrix assembled with one all-gather (sharding.gather_pair_matrix) and hashed.
Prints ONE JSON line on rank 0.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LAYOUT = "simple"  # cramped_room
HORIZON = 400
WORLDS_PER_GPU = 16384
METRIC = "agent-steps/sec (env+obs)"
UNIT = "agent-steps/s"
CLASSIC = ["simple", "unident_s", "random1", "random0", "random3"]  # train/test_vs_bc.py:39-49


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000, help="timed passes (fused launches)")
    ap.add_argument("--warmup", type=int, default=30, help="untimed warm-up passes")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--env-steps-per-pass", type=int, default=100)
    ap.add_argument("--worlds", type=int, default=WORLDS_PER_GPU)
    ap.add_argument("--layout", default=LAYOUT)
    ap.add_argument("--lanes", type=int, default=0, help="lanes per world (kernel tuning), 0 = library default")
    ap.add_argument("--tma", type=int, default=-1, help="1/0 force the TMA bulk-store path, -1 = library default")
    ap.add_argument("--e2e-steps", type=int, default=300, help="single-step host-buffer calls of the e2e measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the '+policy fwd' legs (BASELINE config 4)")
    ap.add_argument("--no-config5", action="store_true", help="skip the cross-play matrix leg (BASELINE config 5)")
    ap.add_argument("--policy-worlds", type=int, default=8192)
    ap.add_argument("--policy-T", type=int, default=400)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--device-warmup-s", type=float, default=2.0, help="untimed device warm-up before the W warm-up passes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the observations, rewards and dones of the last timed pass as float32 DIR/<name>.npy "
                         "(worlds sampled with numpy default_rng(0) to stay under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, n_gpus):
    return {"workload": "overcooked cramped_room (simple.layout), 2 agents, horizon %d, %d worlds/GPU, "
                        "random actions, env step + obs encode" % (HORIZON, args.worlds),
            "layout": args.layout, "worlds_per_gpu": args.worlds, "n_worlds": args.worlds * n_gpus,
            "horizon": HORIZON, "env_steps_per_pass": args.env_steps_per_pass,
            "step_definition": "1 bench step = 1 fused launch = %d env steps of every world" % args.env_steps_per_pass,
            "l2_policy": "outputs larger than L2 (obs slab per launch >> 126 MB); no flush needed",
            "device_warmup_s": args.device_warmup_s,
            "parallelism": "worlds sharded, %d per GPU, no data-path collective" % args.worlds}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------- CPU baselines
def _reference_worker(job):
    """one process = one core: the UNMODIFIED reference CPU path of BASELINE config 1,
    SyncVectorEnv([SimplifiedOvercooked(layout, horizon=400)]) on device cpu (pantheonrl_extension/vectorenv.py:362-396,
    envs/overcooked2_env.py:327-339), `warm` untimed + `passes` timed passes of `steps` n_step calls each"""
    layout, n_worlds, steps, warm, passes, seed = job
    import torch
    torch.set_num_threads(1)
    from oracle import ref_shim
    ns = ref_shim.load()
    env = ns.SyncVectorEnv([lambda: ns.SimplifiedOvercooked(layout, horizon=HORIZON) for _ in range(n_worlds)], device="cpu")
    env.n_reset()
    g = torch.Generator().manual_seed(seed)
    acts = torch.randint(0, 6, (steps, 2, n_worlds, 1), generator=g)
    for _ in range(warm):
        for k in range(steps):
            env.n_step(acts[k])
    times = []
    for _ in range(passes):
        t0 = time.perf_counter()
        for k in range(steps):
            env.n_step(acts[k])
        times.append(time.perf_counter() - t0)
    return times


def reference_throughput(layout, steps, warm, passes, cores, worlds_per_core=1):
    """-> (agent-steps/s over all cores, mean seconds per pass, sample description)"""
    import multiprocessing as mp
    jobs = [(layout, worlds_per_core, steps, warm, passes, 100 + i) for i in range(cores)]
    if cores == 1:
        res = [_reference_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_reference_worker, jobs)
    slowest = max(sum(r) for r in res)
    value = 2 * cores * worlds_per_core * steps * passes / slowest
    sample = "%d processes x SyncVectorEnv([SimplifiedOvercooked]x%d), %d passes of %d n_step calls each (unmodified reference, " \
             "baseline/_ref)" % (cores, worlds_per_core, passes, steps)
    return value, slowest / passes, sample


def _py_port_worker(job):
    """one process: the Python port of the reference env (oracle/overcooked_oracle.py) on `n` worlds for `steps` steps"""
    layout, horizon, n, steps, seed = job
    import numpy as np
    from diverse_conventions_b200 import layouts
    from oracle.overcooked_oracle import OvercookedOracle
    lp = layouts.load_layout(layout, horizon)
    orc = OvercookedOracle(lp, n)
    acts = np.random.default_rng(seed).integers(0, 6, size=(steps, lp.num_players, n))
    t0 = time.perf_counter()
    for k in range(steps):
        orc.step(acts[k])
    return n * steps, time.perf_counter() - t0


def cpu_port_throughput(layout, steps, budget_s, cores):
    import concurrent.futures as cf
    ws, dt = _py_port_worker((layout, HORIZON, 2, 50, 0))  # calibrate: seconds per world-step
    per_ws = dt / ws
    n_per_core = int(max(1, min(256, budget_s / (per_ws * steps))))
    jobs = [(layout, HORIZON, n_per_core, steps, 100 + i) for i in range(cores)]
    with cf.ProcessPoolExecutor(max_workers=cores) as ex:
        res = list(ex.map(_py_port_worker, jobs))
    return 2 * sum(r[0] for r in res) / max(r[1] for r in res), n_per_core * cores, steps


def c_port_throughput(layout, budget_s, threads):
    """agent-steps/s of the C restatement (oracle/ocb_oracle.c), `threads` host threads"""
    import concurrent.futures as cf
    import numpy as np
    from diverse_conventions_b200 import layouts
    from oracle.c_oracle import COracle
    lp = layouts.load_layout(layout, HORIZON)
    n, K = 2048, 50
    acts = np.random.default_rng(0).integers(0, 6, size=(K, 2, n)).astype(np.uint8)

    def work(_):
        orc = COracle(lp, n)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < budget_s:
            orc.rollout(acts)
            reps += 1
        return reps * n * K, time.perf_counter() - t0

    with cf.ThreadPoolExecutor(max_workers=threads) as ex:  # ctypes releases the GIL
        res = list(ex.map(work, range(threads)))
    return 2 * sum(r[0] for r in res) / max(r[1] for r in res)


def cpu_baseline_block(layout, cores, seconds):
    """the reference's CPU path on a bounded sample (plus the ports as secondary figures) for the GPU line"""
    from oracle import ref_shim
    out = {"unit": UNIT, "cores": cores}
    if ref_shim.available():
        steps = 100
        v1, s1, _ = reference_throughput(layout, steps, 1, 4, 1)  # BASELINE.md section 4: N = 1 world, one core
        passes = int(max(2, min(40, seconds / max(s1, 1e-3))))
        v, _, sample = reference_throughput(layout, steps, 1, passes, cores)
        out.update({"value": v, "kind": "reference", "sample": sample, "single_core_value": v1,
                    "single_core_note": "1 process, N = 1 world (BASELINE config 1); 1 of %d cores used" % cores})
    else:
        v, n_worlds, steps_done = cpu_port_throughput(layout, 400, seconds, cores)
        out.update({"value": v, "kind": "port", "sample": "%d worlds x %d steps, python port of the reference env, 1 process per "
                                                           "core (baseline/_ref not installed)" % (n_worlds, steps_done)})
    try:
        out["python_port_value"] = cpu_port_throughput(layout, 400, 3.0, cores)[0]
        out["c_port_value"] = c_port_throughput(layout, 2.0, cores)
        out["port_note"] = "oracle/overcooked_oracle.py (1 process per core) and oracle/ocb_oracle.c (%d threads)" % cores
    except Exception as exc:
        out["port_note"] = "ports failed: %r" % exc
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(1)
    from oracle import c_oracle, ref_shim
    c_oracle.build()
    cores = host_cores()
    t0 = time.perf_counter()
    K, W, spl = max(args.steps, 1), max(args.warmup, 0), args.env_steps_per_pass
    cfg = workload_config(args, args.gpus)
    if ref_shim.available():
        # a pass of the CPU arm = env_steps_per_pass n_step calls on a bounded sample of the workload: one world per
        # process, one process per core (the reference's SyncVectorEnv is a per-world Python loop; more worlds per
        # process scale its time linearly).  K timed passes after W warm-up passes, wall time of the slowest process.
        W = min(W, 100)
        K = min(K, 6000)
        value, pass_s, sample = reference_throughput(args.layout, spl, W, K, cores)
        v1, _, _ = reference_throughput(args.layout, spl, 1, 3, 1)
        kind = "reference"
        extra = {"single_core_value": v1, "single_core_note": "1 process, N = 1 world: BASELINE config 1 as BASELINE.md section 4 "
                                                                "states it; 1 of %d cores used" % cores}
    else:
        _py_port_worker((args.layout, HORIZON, 2, 20, 1))
        value, n_worlds, steps_done = cpu_port_throughput(args.layout, spl * min(K, 4), 20.0, cores)
        pass_s = 2 * n_worlds * spl / value
        sample = "%d worlds x %d steps over %d processes (python port; baseline/_ref not installed)" % (n_worlds, steps_done, cores)
        kind, extra = "port", {}
    try:
        extra["python_port_value"] = cpu_port_throughput(args.layout, 200, 3.0, cores)[0]
        extra["c_port_value"] = c_port_throughput(args.layout, 2.0, cores)
        extra["port_note"] = "oracle/overcooked_oracle.py (1 process per core) and oracle/ocb_oracle.c (%d threads)" % cores
    except Exception as exc:
        extra["port_note"] = "ports failed: %r" % exc
    cb = {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
    cb.update(extra)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * pass_s,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg, "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "steps_requested": args.steps, "warmup_requested": args.warmup,
            "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason samples of one GPU while the bench runs.  NVML in a thread (20 ms period; the pipe of
    `nvidia-smi -lms` is block-buffered on some boxes and delivered nothing inside a short run), `nvidia-smi` as the
    fallback when NVML cannot be loaded.  `index` is torch's device index: the NVML handle is looked up by UUID, so
    CUDA_VISIBLE_DEVICES does not confuse the two numberings."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None):
        self.rows, self.proc, self.nvml, self.source = [], None, None, None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid is not None:
                for cand in ("GPU-" + str(uuid), str(uuid)):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if not isinstance(cand, bytes) else cand)
                        break
                    except Exception:
                        try:
                            h = pynvml.nvmlDeviceGetHandleByUUID(cand)
                            break
                        except Exception:
                            h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml, self.handle = pynvml, h
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.source = "nvml"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.handle
        bits = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                try:
                    util = int(nv.nvmlDeviceGetUtilizationRates(h).gpu)
                except Exception:
                    util = -1
                self.rows.append((time.perf_counter(), (sm, self.sm_max, [n for n, b in bits if mask & b], util)))
            except Exception:
                pass
            self._stop.wait(0.02)

    def _pump(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            try:
                row = (float(f[0]), float(f[1]), [nm for nm, v in zip(names, f[3:7]) if v.lower().startswith("active")], -1)
            except Exception:
                continue
            self.rows.append((time.perf_counter(), row))

    def stop(self, t_begin, t_end):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"], "samples": 0}
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        self._stop.set()
        rows = [r for t, r in self.rows if t_begin - 0.05 <= t <= t_end + 0.15] or [r for _, r in self.rows]
        busy = [r for r in rows if r[3] != 0] or rows  # NVML utilisation 0 = a sample between two legs (host-side setup)
        sm = [r[0] for r in busy]
        reasons = set()
        for r in rows:
            reasons.update(r[2])
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(r[1] for r in rows) if rows else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source}


def measured_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 2250.0, "source": "fallback (B200_PROFILING.md)"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        peaks = {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                 "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                 "source": "MEASURED_PEAKS.json (hbm_gbs copy r+w; bf16 cuBLAS burst / sustained)"}
    except Exception:
        pass
    return peaks


def ncu_traffic_bytes(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_name` from the newest committed
    `ncu --set full` summary under profiles/ (None if there is none for this kernel)"""
    import glob
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_full_*summary.json"))):
        try:
            with open(path) as f:
                rows = json.load(f)
            vals = []
            if isinstance(rows, dict):  # tools/ncu_summary.py: {"launches": [{"kernel": ..., "metric [unit]": value}]}
                for r in rows.get("launches", []):
                    if kernel_name.replace(" ", "") not in r.get("kernel", "").replace(" ", ""):
                        continue
                    tot = 0.0
                    for k, v in r.items():
                        if k.startswith("dram__bytes_read.sum [") or k.startswith("dram__bytes_write.sum ["):
                            tot += float(v) * unit[k[k.index("[") + 1:-1]]
                    vals.append(tot)
                rows = []
            for r in rows:
                if kernel_name.replace(" ", "") not in r.get("Kernel Name", "").replace(" ", ""):
                    continue
                tot = 0.0
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    num, u = r[key].split()
                    tot += float(num) * unit[u]
                vals.append(tot)
            if vals:
                best = statistics.mean(vals)
        except Exception:
            continue
    return best


def bind_to_gpu_local_cores(gpu_index):
    """Pin this rank to the host cores NVML reports as local to its GPU (first-touch placement of the pinned e2e buffers
    and the copy-issuing thread on the GPU's NUMA node).  -> (cores used or None, reason)"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        allowed = os.sched_getaffinity(0)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(allowed | {os.cpu_count() or 1}) + 64) // 64)
        local = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus = local & allowed
        if not cpus:
            return None, "NVML reports no GPU-local core inside this process's cpuset (%d cores allowed)" % len(allowed)
        if cpus == allowed:
            return None, "every allowed core (%d) is already GPU-local: nothing to bind" % len(allowed)
        os.sched_setaffinity(0, cpus)
        return len(cpus), "bound to %d GPU-local cores" % len(cpus)
    except Exception as exc:
        return None, "NVML affinity unavailable: %r" % (exc,)


# ----------------------------------------------------------------------------- policy legs
def policy_flops_per_agent_step(lp, hidden):
    """useful FLOPs of one actor + one critic forward on one observation (2 FLOPs per MAC; the 5 static terrain channels
    are folded into a bias, so 15 of the 20 input channels reach the conv)"""
    npos = (lp.width - 2) * (lp.height - 2)
    co = hidden // 2
    per_net = 2 * (npos * 9 * 15 * co + npos * co * hidden + hidden * hidden)
    return 2 * per_net + 2 * hidden * 7


def config4_leg(args, local, rank, world, dev, barrier, peaks):
    """BASELINE configs[3]: five layouts x hidden {64, 512}, 8,192 worlds/GPU, T = 400, random-init policy forward."""
    import torch
    import torch.distributed as dist
    from diverse_conventions_b200 import layouts
    from diverse_conventions_b200.overcooked_env import B200Overcooked
    from diverse_conventions_b200.policy import FusedPolicy, PolicyNet
    from diverse_conventions_b200.rollout import PolicyRollout
    N, T = args.policy_worlds, args.policy_T
    rows = []
    for hidden in (64, 512):
        for layout in CLASSIC:
            lp = layouts.load_layout(layout, HORIZON)
            pol = FusedPolicy(lp, hidden, 1, gpu_id=local)
            pol.set_weights(0, PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(1),
                            PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(2))
            env = B200Overcooked(layout, N, local, horizon=HORIZON, seed=1, world_offset=rank * N)
            ro = PolicyRollout(env, pol, T, seed=1, use_graph=(hidden == 64))
            warm, iters = (2, 3) if hidden == 64 else (1, 1)
            for _ in range(warm):
                ro.collect()
                ro.buf.compute_returns()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                ro.collect()
                ro.buf.compute_returns()  # GAE + advantage normalisation over the buffer just written
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            ms_rollout = float(ms.item()) / iters
            agent_steps = lp.num_players * N * T
            tflops = policy_flops_per_agent_step(lp, hidden) * lp.num_players * N * (T + 1) / (ms_rollout * 1e-3) / 1e12
            gbs = ro.buf.nbytes() / (ms_rollout * 1e-3) / 1e9
            # launches per rollout: fused = observe + persistent kernel + counter; per-step = observe + T x (policy + env)
            # + bootstrap policy; hidden 512 runs 3 kernels per policy forward; + 2 for GAE / normalisation
            if ro.fused:
                launches = 3 + 2
            else:
                per_fwd = 3 if hidden == 512 else 1
                launches = 1 + T * (per_fwd + 1) + per_fwd + 2
            rows.append({"layout": layout, "hidden": hidden, "worlds_per_gpu": N, "T": T, "fused_single_launch": bool(ro.fused),
                         "cuda_graph": hidden == 64, "ms_per_rollout": ms_rollout, "us_per_env_step": 1e3 * ms_rollout / T,
                         "agent_steps_per_s": agent_steps * world / (ms_rollout * 1e-3), "launches_per_rollout": launches,
                         "roofline": {"hbm": {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                              "bytes": ro.buf.nbytes(), "what": "rollout-buffer bytes written per rollout"},
                                      "tensor": {"achieved": tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                                                 "frac": tflops / peaks["bf16_tflops"],
                                                 "what": "useful fp32-equivalent FLOPs of the actor + critic forwards (the kernels "
                                                         "issue 2-3x that as bf16 hi/lo products)"}}})
            env.close()
            pol.close()
            del ro
            torch.cuda.empty_cache()
    return {"metric": "agent-steps/sec (env+obs+policy fwd+buffer write+GAE)", "unit": UNIT,
            "what": "MAPPO self-play rollout (train/MAPPO/main_player.py:91-112,211-261): actor + critic forward of both seats, "
                    "on-device sampling, env step, seat-major PPO buffer write, then returns / GAE; device-timed, max over ranks",
            "value_cramped_room_h64": next(r["agent_steps_per_s"] for r in rows if r["layout"] == "simple" and r["hidden"] == 64),
            "rows": rows}


def config5_leg(local, rank, world, dev, barrier):
    """BASELINE configs[4]: 16 x 16 pair matrix on coordination_ring, 1,024 worlds per pair, sharded over the ranks."""
    import torch
    import torch.distributed as dist
    from diverse_conventions_b200 import layouts, sharding
    from diverse_conventions_b200.policy import FusedPolicy, PolicyNet
    from diverse_conventions_b200.rollout import CrossPlayEvaluator
    n, wpp, layout = 16, 1024, "random1"
    lp = layouts.load_layout(layout, HORIZON)
    pol = FusedPolicy(lp, 64, n, gpu_id=local)
    for i in range(n):  # seeds 1 + 100 i (seed_skip, train/config.py:315)
        pol.set_weights(i, PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(1 + 100 * i), None)
    pairs = sharding.pair_shard(sharding.all_pairs(n), rank, world)
    ev = CrossPlayEvaluator(layout, pol, pairs, worlds_per_pair=wpp, horizon=HORIZON, gpu_id=local, seed=1,
                            world_offset=rank * len(pairs) * wpp, chunk_steps=50, use_graph=True,
                            total_worlds=n * n * wpp)
    for _ in range(2):  # warm-up (the first run captures the graphs)
        stats = ev.run()
        sharding.gather_pair_matrix(pairs, stats[0], stats[1], n)
    barrier()
    iters = 2
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        stats = ev.run()
        mean, eps = sharding.gather_pair_matrix(pairs, stats[0], stats[1], n)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    out = {"workload": "16 x 16 random-init convention pairs on coordination_ring, %d worlds per pair, one %d-step episode per "
                       "world, pairs sharded over %d rank(s), matrix through sharding.gather_pair_matrix (%s)" % (
                           wpp, HORIZON, world, "NCCL all-gather" if world > 1 else "single rank"),
           "ms_per_matrix": float(ms.item()), "pairs_per_gpu": len(pairs),
           "agent_steps_per_s": 2 * n * n * wpp * HORIZON / (float(ms.item()) * 1e-3),
           "episodes": int(eps.sum()), "matrix_mean": float(mean.nanmean()),
           "matrix_sha256": hashlib.sha256(mean.cpu().numpy().tobytes()).hexdigest()[:16],
           "sha_note": "sampling is keyed by the global (seat, world): the matrix, hence the hash, must not depend on --gpus"}
    ev.close()
    pol.close()
    torch.cuda.empty_cache()
    return out


def dump_outputs(out, directory, limit=60 * 10**6):
    """Write what the last ocb_rollout_random pass handed its caller as float32 .npy files: obs [T, P, n, W, H, C],
    rewards [T, P, n], dones [T, n] for n worlds drawn without replacement by numpy default_rng(0) (all worlds when
    they fit in `limit` bytes), in increasing world order."""
    import numpy as np
    import torch
    arrays = {"obs": (out["obs"], 2), "rewards": (out["rewards"], 2), "dones": (out["dones"], 1)}
    N = out["dones"].shape[1]
    per_world = sum(4 * t.numel() // N for t, _ in arrays.values())
    n = min(N, limit // per_world)
    if n < 1:
        raise SystemExit("bench.py: one world's outputs (%d bytes) exceed the %d-byte dump limit" % (per_world, limit))
    idx = np.sort(np.random.default_rng(0).choice(N, size=n, replace=False))
    idx_t = torch.from_numpy(idx).to(out["dones"].device)
    os.makedirs(directory, exist_ok=True)
    for name, (t, axis) in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.index_select(axis, idx_t).float().cpu().numpy())


# ----------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from diverse_conventions_b200 import layouts
    from diverse_conventions_b200.overcooked_env import B200Overcooked

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    numa_cores, numa_note = bind_to_gpu_local_cores(local) if world > 1 else (None, "single rank: not bound")
    peaks = measured_peaks()

    N, K, W, spl = args.worlds, args.steps, args.warmup, args.env_steps_per_pass
    lp = layouts.load_layout(args.layout, HORIZON)
    P = lp.num_players

    def make_env():
        e = B200Overcooked(args.layout, N, local, horizon=HORIZON, seed=0, world_offset=rank * N)
        if args.lanes or args.tma >= 0:
            e.set_tuning(args.lanes, bool(max(args.tma, 0)))
        return e

    env = make_env()
    out = env.alloc_rollout(spl, obs=True, actions=False)
    bytes_ws = layouts.io_bytes_per_world_step(lp)

    def run_passes(n_passes, events=None, on=None):
        for _ in range(n_passes):
            if events is not None:  # every launch gets its own event pair on the launching stream
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            (on or env).rollout_random(spl, out)
            if events is not None:
                e1.record()
                events.append((e0, e1))
        return n_passes

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None)) if rank == 0 else None
    t_sampler = time.perf_counter()
    # A freshly leased GPU runs its first seconds of work measurably slower (the same binary measured 30 us in the first
    # process of a box and 24.7 us ten seconds later, profiles/README.md): bring the device to its steady state with
    # untimed launches of the same kernel before the W warm-up passes.  They run on a twin of the env, so that the
    # timed env always starts from the same state and step count and its outputs do not depend on the host's speed.
    twin = make_env()
    t_dev = time.perf_counter()
    while time.perf_counter() - t_dev < args.device_warmup_s:
        run_passes(50, on=twin)
        torch.cuda.synchronize()
    twin.close()
    run_passes(max(W, 3))
    barrier()
    t_begin = time.perf_counter()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    events = []
    start.record()
    launches = run_passes(K, events)
    stop.record()
    barrier()
    t_end = time.perf_counter()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    ms = torch.tensor([start.elapsed_time(stop)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = P * N * world * K * spl / (ms_total * 1e-3)

    # average launch duration of the dominant kernel over the timed region (all launches but the first) -> roofline
    per_launch = [e0.elapsed_time(e1) for e0, e1 in events]
    launch_ms = statistics.mean(per_launch[1:] if len(per_launch) > 1 else per_launch)
    achieved = bytes_ws * N * spl / (launch_ms * 1e-3) / 1e9
    tuning = env.get_tuning()
    # (kernel name without the closing bracket: the K-step instance carries a third template argument since round 2)
    kernel_name = "oc_rollout_split_kernel" if tuning["lanes_per_world"] == 16 else \
        "oc_rollout_kernel<%d, %d" % (P, tuning["lanes_per_world"])  # 16 = the role-split kernel (ocb_set_tuning)
    traffic = ncu_traffic_bytes(kernel_name) if (N, spl, args.layout) == (WORLDS_PER_GPU, 100, LAYOUT) else None
    # The GPUs of the pool differ: the same binary streams 0.206-0.226 ms per launch from box to box.  A plain device copy
    # on THIS GPU (1 GiB read + 1 GiB written per iteration, CUDA events) says how much of that is the box.
    box_copy = None
    try:
        src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
        dst = torch.empty_like(src)
        for _ in range(3):
            dst.copy_(src)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(10):
            dst.copy_(src)
        c1.record()
        torch.cuda.synchronize()
        box_copy = 2 * 10 * float(1 << 30) / (c0.elapsed_time(c1) * 1e-3) / 1e9
        del src, dst
        torch.cuda.empty_cache()
    except Exception:
        box_copy = None

    # ---- end-to-end: the reference-facing single-step call with host buffers
    E = max(args.e2e_steps, 10)
    h2d = 4 * P * N
    d2h = P * N * lp.size * lp.channels + 4 * P * N + 4 * N
    slots = [dict(a=torch.randint(0, 6, (P, N), dtype=torch.int32).pin_memory(),
                  o=torch.empty((P, N, lp.width, lp.height, lp.channels), dtype=torch.int8).pin_memory(),
                  r=torch.empty((P, N), dtype=torch.int32).pin_memory(), d=torch.empty((N,), dtype=torch.int32).pin_memory())
             for _ in range(2)]

    def e2e_pipelined(n):
        for t in range(n):
            b = slots[t & 1]
            if t >= 2:
                env.step_host_wait()      # slot t & 1 delivered: its buffers may be reused
            env.step_host_async(b["a"], b["o"], b["r"], b["d"])
        while env.step_host_wait() > 0:
            pass

    def e2e_sync(n, with_obs=True):
        b = slots[0]
        for _ in range(n):
            env.step_host(b["a"], b["o"] if with_obs else None, b["r"], b["d"])

    def timed_host(fn, *a):
        barrier()
        t0 = time.perf_counter()
        fn(*a)
        torch.cuda.synchronize()
        s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(s, op=dist.ReduceOp.MAX)
        return float(s.item())

    e2e_pipelined(6)
    e2e_sync(4)
    s_pipe = timed_host(e2e_pipelined, E)
    s_sync = timed_host(e2e_sync, E)
    s_noobs = timed_host(e2e_sync, E, False)
    e2e_value = P * N * world * E / s_pipe

    # the PCIe ceiling of the same transfer: plain pinned device-to-host copies of d2h bytes, all ranks at once
    d_blob = torch.empty((d2h,), dtype=torch.uint8, device=dev)
    h_blob = torch.empty((d2h,), dtype=torch.uint8).pin_memory()

    def plain_d2h(n):
        for _ in range(n):
            h_blob.copy_(d_blob, non_blocking=True)

    plain_d2h(5)
    s_copy = timed_host(plain_d2h, E)
    copy_gbs_per_gpu = d2h * E / s_copy / 1e9
    e2e_gbs_per_gpu = (d2h + h2d) * E / s_pipe / 1e9

    config4 = None if args.no_config4 else config4_leg(args, local, rank, world, dev, barrier, peaks)
    config5 = None if args.no_config5 else config5_leg(local, rank, world, dev, barrier)
    clocks = None
    if sampler:
        # the headline region lasts milliseconds at the driver's --steps 20, shorter than nvidia-smi's sampling period:
        # the clocks are sampled from the first warm-up pass to the end of the device legs (all of it GPU-bound work)
        clocks = sampler.stop(t_sampler, time.perf_counter())
        clocks["window"] = "warm-up .. headline region .. e2e .. config4 / config5 legs (%.1f s); headline region %.1f ms" % (
            time.perf_counter() - t_sampler, 1e3 * (t_end - t_begin))

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": workload_config(args, world),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                             "kernel": kernel_name.replace(", ", ",") + (">" if "<" in kernel_name else ""), "tuning": tuning,
                             "bytes_per_world_step": bytes_ws, "world_steps_per_launch": N * spl,
                             "launch_ms": launch_ms, "launches_timed": max(len(per_launch) - 1, 1),
                             "launch_ms_first": per_launch[0], "peak_source": peaks["source"],
                             "box_copy_gbs": box_copy, "frac_of_box_copy": (achieved / box_copy) if box_copy else None,
                             "box_copy_note": "torch device-to-device copy of 1 GiB on this GPU (read + written bytes / time): "
                                              "the box's own streaming rate beside the pool-wide peak",
                             "write_only_note": "the kernel reads nothing, so it can (and on fast boxes does) exceed the copy-derived "
                                                "peak: tools/probes/store_probe.cu (profiles/r2g_store_probe.jsonl) measured "
                                                "7.2-7.3 TB/s for 128 SMs writing on a fast box of the pool, 6.6 on a slow one, and "
                                                "at most 62.7 GB/s (32 B/clk) per SM"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "call": "ocb_step_host_async + ocb_step_host_wait (two steps in flight: D2H of step t under the H2D + "
                                "kernel of step t + 1); 1 launch / step, obs + reward + done to pinned host memory every step",
                        "calls": E, "value_sync_call": P * N * world * E / s_sync,
                        "sync_call": "ocb_step_host (H2D -> kernel -> D2H -> wait, nothing overlapped)",
                        "value_without_obs_d2h": P * N * world * E / s_noobs,
                        "pcie_d2h_gbs_per_gpu": copy_gbs_per_gpu, "pcie_d2h_gbs_all_gpus": copy_gbs_per_gpu * world,
                        "pcie_note": "plain pinned cudaMemcpyAsync D2H of the same %d bytes per step, every rank copying at the same "
                                     "time (max over ranks): the ceiling of any host-buffer API on this box" % d2h,
                        "e2e_gbs_per_gpu": e2e_gbs_per_gpu, "pcie_frac": (d2h * E / s_pipe / 1e9) / copy_gbs_per_gpu,
                        "gpu_local_cores_rank0": numa_cores, "numa_note_rank0": numa_note},
                "config4": config4, "config5": config5,
                "gpu_launches": launches, "clocks": clocks,
                "env_steps": K * spl, "us_per_env_step": 1e3 * ms_total / (K * spl)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                from oracle import c_oracle
                c_oracle.build()
                line["cpu_baseline"] = cpu_baseline_block(args.layout, host_cores(), args.cpu_seconds)
            except Exception as exc:  # the baseline must never take the GPU line down
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "failed: %r" % exc}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
