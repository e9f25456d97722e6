"""Flow statistics (rlfc_config.stats_every) on one GPU: what accumulating them costs the RL step.

Workload: 256 default-grid environments from init.bdim, the config-2 actions of bench.py, init_time = -1, RL steps of 16
solver steps on device pointers (rlfc_env_step_device).  Three handles, alive together: stats_every = 0 (no statistics),
1 (a sample after every solver step) and 16 (one per RL step).  env-steps/s comes from CUDA events around --steps RL steps
after --warmup warm-up steps; the handles are alternated over --rounds rounds to show the spread.  Then, in a separate
profiled pass of the stats_every = 1 handle (every launch samples), the per-kernel CUDA-event times of the eager path
(rlfc_env_set_profiling) give k_flow_stats per launch and its effective bandwidth (the profile's algorithmic bytes: 3 floats
read and 7 doubles read and written per cell, 124 B), alternated with cudaMemcpyAsync device to device moving the same
bytes (62 B per cell read and 62 B written, one block far larger than the L2, so both run from HBM).  Records the card's
name and power limit in the same run.  Prints one JSON object; --out also writes it.  Needs a GPU.
    python tools/bench_flow_stats.py --out profiles/flow_stats_b200.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_adaptive import card_info  # noqa: E402

EVERY = (0, 1, 16)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--copies", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    from bench import make_actions
    R.load_library()
    cudart = C.CDLL("libcudart.so.12")       # the runtime librlfc.so is linked against
    cudart.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    B, K, W = args.envs, args.steps, args.warmup
    acts = torch.from_numpy(make_actions(W + K, B, 0, e0=0)).cuda()
    card = card_info()
    runs = {}
    for k in EVERY:
        stream = torch.cuda.Stream()
        env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, stats_every=k)
        runs[k] = dict(env=env, stream=stream, obs=torch.empty((B, 2), dtype=torch.float32, device="cuda"),
                       rew=torch.empty(B, dtype=torch.float32, device="cuda"),
                       done=torch.empty(B, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()

    def rl_step(r, k):
        r["env"].step_device(acts[k].data_ptr(), r["obs"].data_ptr(), r["rew"].data_ptr(), r["done"].data_ptr())

    res = {k: [] for k in EVERY}
    for rnd in range(args.rounds):
        for every in EVERY:
            r = runs[every]
            env = r["env"]
            env.reset(None, reset_accumulators=True)
            if every:
                env.stats_reset()
            with torch.cuda.stream(r["stream"]):
                for k in range(W):
                    rl_step(r, k)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(r["stream"])
                for k in range(W, W + K):
                    rl_step(r, k)
                e1.record(r["stream"])
                e1.synchronize()
            sec = e0.elapsed_time(e1) / 1e3
            assert env.running() == 0 and not env.flags().any()
            if every:
                count, _ = env.stats_sums(0)
                assert count == (W + K) * 16 // every, count
            res[every].append({"env_steps_per_s": B * K / sec, "ms_per_rl_step": sec * 1e3 / K})

    # profiled pass (the event pairs slow the host): k_flow_stats per launch on the handle that samples every step
    r = runs[1]
    env = r["env"]
    env.set_profiling(True)
    with torch.cuda.stream(r["stream"]):
        for k in range(2):
            rl_step(r, k)
    torch.cuda.synchronize()
    p = env.get_profile()
    env.set_profiling(False)
    total = sum(x["ms"] for x in p)
    solver_steps = next(x["launches"] for x in p if x["name"] == "k_force")
    ks = next(x for x in p if x["name"] == "k_flow_stats")
    us = ks["ms"] * 1e3 / ks["launches"]
    kbytes = ks["bytes_per_launch"]
    n, m = env.n, env.m
    for x in runs.values():
        x["env"].close()
    torch.cuda.synchronize()

    # cudaMemcpyAsync D2D of the same traffic, timed by events over --copies copies
    half = int(kbytes // 2)
    src = torch.ones(half, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    stream = torch.cuda.Stream()

    def memcpy_ms():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.copies):
            rc = cudart.cudaMemcpyAsync(C.c_void_p(dst.data_ptr()), C.c_void_p(src.data_ptr()), half, 3, C.c_void_p(stream.cuda_stream))
            assert rc == 0, rc
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / args.copies

    memcpy_ms()
    copies = [memcpy_ms() for _ in range(args.rounds)]
    copy_gbs = 2 * half / (float(np.median(copies)) * 1e-3) / 1e9

    summary = {}
    base = float(np.median([x["env_steps_per_s"] for x in res[0]]))
    for every in EVERY:
        med = float(np.median([x["env_steps_per_s"] for x in res[every]]))
        summary[f"stats_every_{every}"] = {"median_env_steps_per_s": med, "over_no_stats": med / base}
    kern_gbs = kbytes / (us * 1e-6) / 1e9
    summary["k_flow_stats"] = {"us_per_launch": us, "launches": ks["launches"], "algorithmic_bytes_per_launch": kbytes,
                               "gb_per_s": kern_gbs, "memcpy_d2d_gb_per_s": copy_gbs, "over_memcpy": kern_gbs / copy_gbs,
                               "share_of_kernel_time": ks["ms"] / total,
                               "kernel_ms_per_solver_step": total / solver_steps}
    out = {"workload": f"{B} default-grid envs ({n}x{m} incl. ghosts) from init.bdim, config-2 actions, init_time -1, "
                       f"step_device RL steps of 16 solver steps; {K} timed after {W} warm-up, {args.rounds} alternated "
                       f"rounds; profile over 2 RL steps of the stats_every = 1 handle; memcpy of {2 * half} bytes of traffic "
                       f"({half} read + {half} written) per copy",
           "card": card, "rl_steps": {str(k): v for k, v in res.items()}, "memcpy_ms": copies, "summary": summary}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
