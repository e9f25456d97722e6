"""Adaptive vs fixed time stepping on one GPU: 256 default-grid environments from init.bdim, the config-2 actions of
bench.py, RL steps of 16 solver steps on device pointers.  For each mode, in one run:

  * env-steps/s and solver-steps/s (CUDA events around K steps after W warm-up steps);
  * simulated time advanced per wall-clock second: sum over environments of the advance of AFCCylinder.t (dt/resolution
    per solver step), over the timed window;
  * per-kernel times from rlfc_env_set_profiling in a separate, eager run, with the Poisson rebuild kernels' achieved
    bytes/s (bytes each launch must write, from the hierarchy's shapes, plus the del fields the level-0 kernel reads);
  * the card name and its power limit.

Prints one JSON object; --out also writes it to a file.  Needs a GPU (there is no CPU fallback).
    python tools/bench_adaptive.py --envs 256 --steps 20 --warmup 5 --out profiles/adaptive_dt_b200.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

K_TAB_FRONT, K_STAGE_LAG, K_PF = 10, 10, 5      # smooth_rows.cuh (rows_table_entries)


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as exc:   # (the numbers are reported without it, marked as such)
        info["power_limit_w"] = f"unavailable: {exc}"
    return info


def rebuild_bytes(env):
    """Bytes one launch of each rebuild kernel writes for the whole batch (pitched arrays incl. ghosts, row tables), and
    the del fields the level-0 kernel reads."""
    per_level = []
    for l in range(env.num_levels):
        n, m = env.get_coeffs(0, "inv", l).shape
        P = (m + 7) // 8 * 8
        ni, mj = n - 2, m - 2
        C = (mj + 31) // 32
        K, nl = (3 * C + 1 + 3) // 4, (mj + C - 1) // C
        entries = K_TAB_FRONT + ni + nl + K_STAGE_LAG + K_PF + 12
        per_level.append(4 * 4 * n * P + entries * K * 32 * 16)
    n, m = env.get_coeffs(0, "inv", 0).shape
    P = (m + 7) // 8 * 8
    B = env.n_envs
    return {"k_poisson_rebuild0": B * (per_level[0] + 2 * 4 * n * P),
            "k_poisson_rebuild_coarse": B * sum(per_level[1:])}


def run_mode(R, torch, adaptive, B, K, W, acts, profile_steps):
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, adaptive_dt=int(adaptive))
    acts_dev = torch.from_numpy(acts).cuda()
    obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
    rew = torch.empty(B, dtype=torch.float32, device="cuda")
    done = torch.empty(B, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    k = 0
    with torch.cuda.stream(stream):
        for _ in range(W):
            env.step_device(acts_dev[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr()); k += 1
        t0 = env.t.astype(np.float64)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            env.step_device(acts_dev[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr()); k += 1
        e1.record(stream)
        e1.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    t1 = env.t.astype(np.float64)
    assert env.running() == 0 and not env.flags().any() and np.isfinite(obs.cpu().numpy()).all()
    dts = env.dt()
    res = {"env_steps_per_s": B * K / sec, "solver_steps_per_s": B * K * 16 / sec,
           "sim_time_per_wall_s": float((t1 - t0).sum()) / sec, "timed_s": sec,
           "dt_min": float(dts.min()), "dt_median": float(np.median(dts)), "dt_max": float(dts.max())}
    # per-kernel times: eager launches, each bracketed by events (slower than the graph path; a separate run)
    env.set_profiling(True)
    for _ in range(profile_steps):
        env.step(acts[k]); k += 1
    prof = env.get_profile()
    env.set_profiling(False)
    by = rebuild_bytes(env) if adaptive else {}
    table = []
    for p in sorted(prof, key=lambda r: -r["ms"]):
        row = {"kernel": p["name"], "ms_per_launch": p["ms"] / max(p["launches"], 1), "launches": p["launches"]}
        if p["name"] in by:
            row["bytes_per_launch"] = by[p["name"]]
            row["achieved_TB_per_s"] = by[p["name"]] / (row["ms_per_launch"] / 1e3) / 1e12
        table.append(row)
    res["kernels"] = table
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    from bench import make_actions
    acts = make_actions(args.warmup + args.steps + args.profile_steps, args.envs, 0, e0=0)
    out = {"workload": f"{args.envs} default-grid envs from init.bdim, bench.py config-2 actions, init_time=-1, "
                       f"{args.steps} timed RL steps (x16 solver steps) after {args.warmup} warm-up steps",
           "card": card_info()}
    for mode in ("fixed", "adaptive"):
        out[mode] = run_mode(R, torch, mode == "adaptive", args.envs, args.steps, args.warmup, acts, args.profile_steps)
    out["adaptive_over_fixed"] = {k: out["adaptive"][k] / out["fixed"][k]
                                  for k in ("env_steps_per_s", "sim_time_per_wall_s")}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
