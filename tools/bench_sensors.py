"""Flow sensors (rlfc_config.sensors) on one GPU: what sampling them after every solver step costs the RL step.

Workload: 256 default-grid environments from init.bdim, the config-2 actions of bench.py, init_time = -1, RL steps of 16
solver steps on device pointers (rlfc_env_step_device, then rlfc_env_get_sensors_device into a device buffer, the
observation path of a GPU-resident policy).  Four handles, alive together: K = 0 (no sensors), 32 (the SaveScalar points
as p), 151 and 1024 (a wake grid of p, u.x and u.y points).  env-steps/s comes from CUDA events around --steps RL steps
after --warmup warm-up steps; the handles are alternated over --rounds rounds to show the spread.  Then, in a separate
profiled pass, the per-kernel CUDA-event times of the eager path (rlfc_env_set_profiling) give k_sensors per launch and its
share of the kernel time of a solver step.  Records the card's name and power limit in the same run.  Prints one JSON
object; --out also writes it.  Needs a GPU.
    python tools/bench_sensors.py --out profiles/sensors_b200.json
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_adaptive import card_info  # noqa: E402

COUNTS = (0, 32, 151, 1024)


def sensor_sets(res=24, xl=16, yl=8):
    """K -> sensor list: the 32 SaveScalar points (SaveScalar.pde:61-72) as p, and the first K points of a 32 x 32 wake grid
    behind the cylinders, the fields p, u.x, u.y in turn."""
    f = np.float32
    r, cx, cy = f(res), f(xl) * f(res) / f(4), f(yl) * f(res) / f(2)
    ring = []
    for i in range(32):
        a = f(i) / f(32) * f(3.1415927) * f(2)
        ring.append(("p", float(f(np.cos(np.float64(a))) * r / f(2) + cx), float(f(np.sin(np.float64(a))) * r / f(2) + cy)))
    xs = np.linspace(float(cx) + res, xl * res - 4, 32)
    ys = np.linspace(8, yl * res - 8, 32)
    grid = [(("p", "ux", "uy")[k % 3], float(x), float(y)) for k, (x, y) in enumerate((x, y) for x in xs for y in ys)]
    return {0: None, 32: ring, 151: grid[:151], 1024: grid[:1024]}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    from bench import make_actions
    B, K, W = args.envs, args.steps, args.warmup
    acts = torch.from_numpy(make_actions(W + K, B, 0, e0=0)).cuda()
    sets = sensor_sets()
    runs = {}
    for n in COUNTS:
        stream = torch.cuda.Stream()
        env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, sensors=sets[n])
        assert env.n_sensors == n
        runs[n] = dict(env=env, stream=stream, obs=torch.empty((B, 2), dtype=torch.float32, device="cuda"),
                       rew=torch.empty(B, dtype=torch.float32, device="cuda"),
                       done=torch.empty(B, dtype=torch.int32, device="cuda"),
                       sens=torch.empty((B, max(n, 1)), dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()

    def rl_step(r, k):
        r["env"].step_device(acts[k].data_ptr(), r["obs"].data_ptr(), r["rew"].data_ptr(), r["done"].data_ptr())
        if r["env"].n_sensors:
            r["env"].sensors_device(r["sens"].data_ptr())

    res = {n: [] for n in COUNTS}
    for rnd in range(args.rounds):
        for n in COUNTS:
            r = runs[n]
            r["env"].reset(None, reset_accumulators=True)
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
            assert r["env"].running() == 0 and not r["env"].flags().any()
            if n:
                assert torch.isfinite(r["sens"]).all()
            res[n].append({"env_steps_per_s": B * K / sec, "ms_per_rl_step": sec * 1e3 / K})

    # eager per-kernel profile (separate pass: the event pairs slow the host)
    prof = {}
    for n in COUNTS:
        r = runs[n]
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
        ks = [x for x in p if x["name"] == "k_sensors"]
        prof[n] = {"kernel_ms_per_solver_step": total / solver_steps, "solver_steps": solver_steps}
        if ks:
            prof[n].update(k_sensors_us_per_launch=ks[0]["ms"] * 1e3 / ks[0]["launches"], k_sensors_launches=ks[0]["launches"],
                           k_sensors_share_of_kernel_time=ks[0]["ms"] / total)
        env.close()

    summary = {}
    base = float(np.median([x["env_steps_per_s"] for x in res[0]]))
    for n in COUNTS:
        v = [x["env_steps_per_s"] for x in res[n]]
        summary[f"K={n}"] = {"env_steps_per_s": v, "median": float(np.median(v)), "over_K0": float(np.median(v)) / base}
        summary[f"K={n}"].update(prof[n])
    out = {"workload": f"{B} default-grid envs from init.bdim, bench.py config-2 actions, init_time=-1, {K} timed RL steps "
                       f"(x16 solver steps, each followed by sensors_device) after {W} warm-up steps, handles K = "
                       f"{', '.join(map(str, COUNTS))} alternated over {args.rounds} rounds; profile: 2 RL steps on the eager "
                       f"path with per-kernel CUDA events",
           "card": card_info(), "runs": {str(n): v for n, v in res.items()}, "summary": summary}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
