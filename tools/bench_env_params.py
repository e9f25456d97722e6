"""Per-environment constructor arguments (rlfc_config.env_params) on one GPU: 256 default-grid environments from
init.bdim, the config-2 actions of bench.py, init_time = -1, RL steps of 16 solver steps on device pointers.  Cases, each
with fixed and with adaptive dt:

  * shared        -- no env_params (one geometry, the handle-wide kernels in fixed dt);
  * default       -- env_params, every set the scalar config's;
  * random        -- env_params drawn with re in [100, 1000], dR in [0.1, 0.25], gR in [0.1, 0.5], theta in [pi/6, pi/2],
                     t_step in {0.005, 0.0075} (seed 0).

env-steps/s comes from CUDA events around K RL steps after W warm-up steps; the cases run `--rounds` times, alternated,
to show the spread.  Also the latency of rlfc_env_reset_params (host clock around the call, which synchronises) for 1 and
for all environments, and the card's name and power limit.  Prints one JSON object; --out also writes it.  Needs a GPU.
    python tools/bench_env_params.py --envs 256 --steps 20 --warmup 5 --out profiles/env_params_b200.json
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_adaptive import card_info  # noqa: E402


def random_params(n, seed):
    rng = np.random.default_rng(seed)
    out = np.zeros(n, dtype=[("re", np.int32), ("dR", np.float32), ("gR", np.float32), ("theta", np.float32),
                             ("t_step", np.float32)])
    out["re"] = rng.integers(100, 1001, n)
    out["dR"] = rng.uniform(0.1, 0.25, n)
    out["gR"] = rng.uniform(0.1, 0.5, n)
    out["theta"] = rng.uniform(np.pi / 6, np.pi / 2, n)
    out["t_step"] = rng.choice([0.005, 0.0075], n)
    return out


def run_case(R, torch, params, adaptive, B, K, W, acts):
    stream = torch.cuda.Stream()
    t_create = time.perf_counter()
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, adaptive_dt=int(adaptive), env_params=params)
    t_create = time.perf_counter() - t_create
    acts_dev = torch.from_numpy(acts).cuda()
    obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
    rew = torch.empty(B, dtype=torch.float32, device="cuda")
    done = torch.empty(B, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    k = 0
    with torch.cuda.stream(stream):
        for _ in range(W):
            env.step_device(acts_dev[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr()); k += 1
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            env.step_device(acts_dev[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr()); k += 1
        e1.record(stream)
        e1.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    assert env.running() == 0 and not env.flags().any() and np.isfinite(obs.cpu().numpy()).all()
    res = {"env_steps_per_s": B * K / sec, "ms_per_solver_step": sec * 1e3 / (K * 16), "create_s": t_create}
    return env, res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    from bench import make_actions
    B = args.envs
    acts = make_actions(args.warmup + args.steps, B, 0, e0=0)
    cases = {"shared": None, "default": [{}] * B, "random": random_params(B, 0)}
    out = {"workload": f"{B} default-grid envs from init.bdim, bench.py config-2 actions, init_time=-1, "
                       f"{args.steps} timed RL steps (x16 solver steps) after {args.warmup} warm-up steps, "
                       f"{args.rounds} alternated rounds",
           "card": card_info(), "cases": {}}
    for r in range(args.rounds):
        for dt_mode in ("fixed", "adaptive"):
            for name, params in cases.items():
                env, res = run_case(R, torch, params, dt_mode == "adaptive", B, args.steps, args.warmup, acts)
                if name == "random" and dt_mode == "fixed" and r == 0:
                    # rlfc_env_reset_params: geometry built on the host, uploaded, hierarchy rebuilt on the device
                    lat = {}
                    for n in (1, B):
                        ids = np.arange(n, dtype=np.int32)
                        newp = random_params(n, 100 + n)
                        times = []
                        for _ in range(3):
                            t0 = time.perf_counter()
                            env.reset(ids, params=newp)
                            times.append(time.perf_counter() - t0)
                        lat[f"{n}_envs_ms"] = [t * 1e3 for t in times]
                    out["reset_params_latency"] = lat
                env.close()
                out["cases"].setdefault(f"{name}/{dt_mode}", []).append(res)
    summary = {}
    for key, runs in out["cases"].items():
        v = [x["env_steps_per_s"] for x in runs]
        summary[key] = {"env_steps_per_s": v, "median": float(np.median(v))}
    for dt_mode in ("fixed", "adaptive"):
        base = summary[f"shared/{dt_mode}"]["median"]
        for name in ("default", "random"):
            summary[f"{name}/{dt_mode}"]["over_shared"] = summary[f"{name}/{dt_mode}"]["median"] / base
    out["summary"] = summary
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
