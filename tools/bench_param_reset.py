"""Device parameter resets (rlfc_env_reset_params_device) on one GPU: default-grid environments from init.bdim and parameter
sets drawn as tools/bench_env_params.py draws them (re in [100, 1000], dR in [0.1, 0.25], gR in [0.1, 0.5], theta in
[pi/6, pi/2], t_step in {0.005, 0.0075}).

  * reset_params_device for 1, 16 and --envs environments (environments 0 .. n-1, sets drawn at random from a library of
    --sets sets): time from CUDA events over --calls calls.  Against rlfc_env_reset_sets_device of the same environments
    and library sets (CUDA events) and rlfc_env_reset_params (host clock around the call, which synchronises before it
    returns).  Fixed dt.
  * A device-only loop of --steps RL steps (step_device, 16 solver steps each, init_time = -1):
      - draws:    reset_params_device(where(done, arange(B), -1), fresh continuous sets drawn with torch on the device)
                  after every step, episode_time = --episode, so every episode end takes a new set;
      - skip:     the same call with every id -1 and episodes that never end (the cost of the call itself);
      - no_call:  step_device alone, episodes that never end.
    env-steps/s from CUDA events; the three loops alternate over --rounds rounds to show the spread.

Records the card's name and power limit in the same run.  Prints one JSON object; --out also writes it.  Needs a GPU.
    python tools/bench_param_reset.py --out profiles/param_reset_b200.json
"""
from __future__ import annotations

import argparse
import json
import math
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_adaptive import card_info  # noqa: E402
from bench_env_params import random_params  # noqa: E402


def pack_np(torch, lib):
    """The library as an (L, 5) int32 device tensor of packed rlfc_env_params."""
    re = torch.tensor(lib["re"].astype(np.int32))
    cols = [torch.from_numpy(np.ascontiguousarray(lib[k], np.float32)).view(torch.int32) for k in ("dR", "gR", "theta", "t_step")]
    return torch.stack([re] + cols, 1).contiguous().cuda()


def draw_sets(torch, n, gen):
    """n continuous random sets on the device, packed: torch.stack([re.int(), dR.view(torch.int32), ...], 1)."""
    u = lambda lo, hi: lo + (hi - lo) * torch.rand(n, device="cuda", generator=gen)   # noqa: E731
    re = torch.randint(100, 1001, (n,), device="cuda", generator=gen, dtype=torch.int32)
    dR, gR, theta = u(0.1, 0.25), u(0.1, 0.5), u(math.pi / 6, math.pi / 2)
    t_step = torch.where(torch.rand(n, device="cuda", generator=gen) < 0.5, 0.005, 0.0075).float()
    return torch.stack([re, dR.view(torch.int32), gR.view(torch.int32), theta.view(torch.int32), t_step.view(torch.int32)], 1)


def time_reset_latency(R, torch, lib, B, K):
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, param_sets=lib)
    d_lib = pack_np(torch, lib)
    rng = np.random.default_rng(1)
    out = {}
    for n in (1, 16, B):
        ids = torch.arange(n, dtype=torch.int32, device="cuda")
        draws = torch.from_numpy(rng.integers(0, len(lib), size=(K + 2, n)).astype(np.int32)).cuda()
        packed = [d_lib[draws[k].long()].contiguous() for k in range(K + 2)]
        torch.cuda.synchronize()
        res = {}
        for name in ("reset_params_device", "reset_sets_device"):
            with torch.cuda.stream(stream):
                call = (lambda k: env.reset_params_device(ids.data_ptr(), packed[k].data_ptr(), n)) \
                    if name == "reset_params_device" else (lambda k: env.reset_sets_device(ids.data_ptr(), draws[k].data_ptr(), n))
                for k in range(2):                    # warm-up
                    call(k)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for k in range(K):
                    call(2 + k)
                e1.record(stream)
                e1.synchronize()
            res[name + "_ms"] = e0.elapsed_time(e1) / K
        h_ids = np.arange(n, dtype=np.int32)
        host_ms = []
        for k in range(3):
            sets = draws[2 + k].cpu().numpy()
            t0 = time.perf_counter()
            env.reset(h_ids, params=lib[sets])
            host_ms.append((time.perf_counter() - t0) * 1e3)
        res["reset_params_ms"] = host_ms
        res["host_over_device"] = float(np.median(host_ms)) / res["reset_params_device_ms"]
        res["device_over_library"] = res["reset_params_device_ms"] / res["reset_sets_device_ms"]
        out[str(n)] = res
    assert not env.flags().any()
    env.close()
    return out


def run_loop(R, torch, B, K, W, mode, episode, acts):
    stream = torch.cuda.Stream()
    ep = episode if mode == "draws" else 1e9
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream, init_time=-1.0, episode_time=ep, env_params=[{}] * B)
    ids = torch.arange(B, dtype=torch.int32, device="cuda")
    obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
    rew = torch.empty(B, dtype=torch.float32, device="cuda")
    done = torch.zeros(B, dtype=torch.int32, device="cuda")
    minus1 = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    fixed = draw_sets(torch, B, gen)
    resets = torch.zeros((), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()

    def one(k):
        env.step_device(acts[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr())
        if mode == "draws":
            sets = draw_sets(torch, B, gen)
            who = torch.where(done != 0, ids, minus1)
            resets.add_((done != 0).sum())
            env.reset_params_device(who.data_ptr(), sets.data_ptr(), B, reset_accumulators=True)
        elif mode == "skip":
            env.reset_params_device(minus1.data_ptr(), fixed.data_ptr(), B, reset_accumulators=True)

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
    out = {"workload": f"{B} default-grid envs from init.bdim; reset latency over {args.calls} calls with sets drawn from a "
                       f"library of {L} random sets, fixed dt; loops of {args.steps} timed RL steps (x16 solver steps) after "
                       f"{args.warmup} warm-up steps, bench.py config-2 actions, init_time=-1, episode_time={args.episode} for "
                       f"the draws loop, {args.rounds} alternated rounds",
           "card": card_info()}
    out["reset_latency"] = time_reset_latency(R, torch, lib, B, args.calls)
    acts = torch.from_numpy(make_actions(args.warmup + args.steps, B, 0, e0=0)).cuda()
    loops = {m: [] for m in ("draws", "skip", "no_call")}
    for _ in range(args.rounds):
        for m in loops:
            loops[m].append(run_loop(R, torch, B, args.steps, args.warmup, m, args.episode, acts))
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
