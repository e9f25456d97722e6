"""Parameter library (rlfc_config.param_sets) on one GPU: 256 default-grid environments from init.bdim and a library of
--sets parameter sets drawn as tools/bench_env_params.py draws them (re in [100, 1000], dR in [0.1, 0.25], gR in [0.1, 0.5],
theta in [pi/6, pi/2], t_step in {0.005, 0.0075}, seed 0).

  * rlfc_env_reset_sets_device for 1, 16 and 256 environments (environments 0 .. n-1, sets drawn at random): time from
    CUDA events over --calls calls, in fixed and in adaptive dt.  Against rlfc_env_reset_params of the same environments
    with the same sets (host clock around the call, which synchronises before it returns).
  * A device-only loop of --steps RL steps (step_device, 16 solver steps each, init_time = -1, episode_time = --episode):
      - draws:    reset_sets_device(arange(B), where(done, randint(L), -1)) after every step, so that every episode end
                  draws a new set;
      - skip:     the same call with every pair -1 and episodes that never end (the cost of the call itself);
      - no_call:  step_device alone, episodes that never end.
    env-steps/s from CUDA events; the three loops alternate over --rounds rounds to show the spread.

Records the card's name and power limit in the same run.  Prints one JSON object; --out also writes it.  Needs a GPU.
    python tools/bench_param_sets.py --out profiles/param_sets_b200.json
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
from bench_env_params import random_params  # noqa: E402


def time_reset_latency(R, torch, lib, B, adaptive, K):
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, adaptive_dt=int(adaptive), param_sets=lib)
    rng = np.random.default_rng(1)
    out = {}
    for n in (1, 16, B):
        ids = torch.arange(n, dtype=torch.int32, device="cuda")
        draws = torch.from_numpy(rng.integers(0, len(lib), size=(K + 2, n)).astype(np.int32)).cuda()
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            for k in range(2):                    # warm-up
                env.reset_sets_device(ids.data_ptr(), draws[k].data_ptr(), n)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(K):
                env.reset_sets_device(ids.data_ptr(), draws[2 + k].data_ptr(), n)
            e1.record(stream)
            e1.synchronize()
        dev_ms = e0.elapsed_time(e1) / K
        # rlfc_env_reset_params of the same environments with the same sets
        h_ids = np.arange(n, dtype=np.int32)
        host_ms = []
        for k in range(3):
            sets = draws[2 + k].cpu().numpy()
            t0 = time.perf_counter()
            env.reset(h_ids, params=lib[sets])
            host_ms.append((time.perf_counter() - t0) * 1e3)
        out[str(n)] = {"reset_sets_device_ms": dev_ms, "reset_params_ms": host_ms,
                       "speedup": float(np.median(host_ms)) / dev_ms}
    assert not env.flags().any()
    env.close()
    return out


def run_loop(R, torch, lib, B, K, W, mode, episode, acts):
    stream = torch.cuda.Stream()
    ep = episode if mode == "draws" else 1e9
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, episode_time=ep, param_sets=lib)
    ids = torch.arange(B, dtype=torch.int32, device="cuda")
    obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
    rew = torch.empty(B, dtype=torch.float32, device="cuda")
    done = torch.zeros(B, dtype=torch.int32, device="cuda")
    minus1 = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    resets = torch.zeros((), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()

    def one(k):
        env.step_device(acts[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr())
        if mode == "draws":
            draw = torch.randint(0, len(lib), (B,), dtype=torch.int32, device="cuda", generator=gen)
            sets = torch.where(done != 0, draw, minus1)
            resets.add_((done != 0).sum())
            env.reset_sets_device(ids.data_ptr(), sets.data_ptr(), B, reset_accumulators=True)
        elif mode == "skip":
            env.reset_sets_device(ids.data_ptr(), minus1.data_ptr(), B, reset_accumulators=True)

    with torch.cuda.stream(stream):
        for k in range(W):
            one(k)
        resets.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(W, W + K):
            one(k)
        e1.record(stream)
        e1.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    assert env.running() == 0 and not env.flags().any() and np.isfinite(obs.cpu().numpy()).all()
    res = {"env_steps_per_s": B * K / sec, "episode_ends": int(resets.item())}
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--sets", type=int, default=16)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--episode", type=float, default=1.0, help="episode_time of the draws loop")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    from bench import make_actions
    B, L = args.envs, args.sets
    lib = random_params(L, 0)
    out = {"workload": f"{B} default-grid envs from init.bdim, a library of {L} random sets; reset latency over "
                       f"{args.calls} calls; loops of {args.steps} timed RL steps (x16 solver steps) after {args.warmup} "
                       f"warm-up steps, bench.py config-2 actions, init_time=-1, episode_time={args.episode} for the draws loop, "
                       f"{args.rounds} alternated rounds",
           "card": card_info()}
    out["reset_latency"] = {dt: time_reset_latency(R, torch, lib, B, dt == "adaptive", args.calls) for dt in ("fixed", "adaptive")}
    acts = torch.from_numpy(make_actions(args.warmup + args.steps, B, 0, e0=0)).cuda()
    loops = {m: [] for m in ("draws", "skip", "no_call")}
    for _ in range(args.rounds):
        for m in loops:
            loops[m].append(run_loop(R, torch, lib, B, args.steps, args.warmup, m, args.episode, acts))
    out["loops"] = loops
    med = {m: float(np.median([x["env_steps_per_s"] for x in v])) for m, v in loops.items()}
    out["summary"] = {"loop_env_steps_per_s_median": med,
                      "skip_over_no_call": med["skip"] / med["no_call"], "draws_over_no_call": med["draws"] / med["no_call"]}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
