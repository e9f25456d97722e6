#!/usr/bin/env python
"""bench.py -- throughput of the B200 Lilypad environment step (BASELINE.json metric and configs).

  python bench.py [--config 2|3|4|5] [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu B] [--envs-total T]
                  [--impl b200|reference]

  --config 2 (default)  BASELINE configs[1]: default AFCCylinder grid (384x192), 256 envs PER GPU from init.bdim, synthetic
                        per-env actions; a step = one RL step of every env = 16 solver steps + the draw() accumulation.
                        N > 1 (torchrun): every rank owns its own 256 envs (scaling "weak"), one observation all-gather
                        per env-step, no data-path collective.  metric env-steps/s.
  --config 4            BASELINE configs[3]: --envs-total (4096) envs split contiguously over the N ranks (scaling
                        "strong"), otherwise as config 2.
  --config 3            BASELINE configs[2]: ONE 2048x1024 domain (resolution 128, t_step = 0.18/128, uniform start, SURVEY
                        8d), a step = one solver step (AFCCylinder.update2); metric solver-steps/s; roofline against the
                        240 B/cell model.  N > 1 runs N independent replicas (the path does not shard on one domain
                        without the slab decomposition of config 5).
  --config 5            BASELINE configs[4]: ONE 8192x4096 domain (--resolution 512) slab-decomposed over --gpus devices of
                        one box (rlfc_config.n_devices: shared address range + NVLink peer access, one host process);
                        metric solver-steps/s, scaling "strong"; reports barriers (exchanges) per step and NVLink bytes.

`value`  : device-resident throughput (inputs already in HBM, *_device entry points, CUDA events on the handle's stream).
`e2e`    : the same metric through the host-pointer C-ABI call (pinned host buffers, H2D actions + D2H results inside the
           timed region).
`roofline`: dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured HBM peak; `kernels` has every
           kernel (k_advdif also against the fp32 instruction-issue roofline: it is issue-bound under --fmad=false).
`cpu_baseline`: the oracle (literal C port of the reference step) on all host cores, bounded sample.
`--impl reference`: the CPU arm alone (the reference Java cannot run here: no JVM; the literal C port of oracle/ stands
           in, one single-threaded process per host core); its `config` says exactly what a "step" of that arm is.
`--dump-outputs DIR`: after the timed steps, what the timed (device-resident) path computed in its last timed step is
           written as DIR/<name>.npy in float32: configs 2 / 4 obs, reward, done of every env (what rlfc_env_step_device
           hands its caller), configs 3 / 5 the fields ux, uy, p of the domain.  The inputs depend on the arguments only,
           so two builds run with the same arguments can be compared array for array.  At most 64 MB in all: an array
           over its share is replaced by a fixed sample of its elements (sorted unique flat indices drawn with seed 0).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env-steps/sec (batched BDIM cylinders)"
UNIT = "env-steps/s"


METRIC3 = "solver-steps/sec (single 2048x1024 BDIM domain)"
UNIT3 = "solver-steps/s"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float32 within DUMP_LIMIT_BYTES (see --dump-outputs)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    share = DUMP_LIMIT_BYTES // (4 * len(arrays))
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.size > share:
            a = a.ravel()[np.unique(np.random.default_rng(0).integers(0, a.size, share))]
        np.save(out / f"{name}.npy", a)


def workload_config(envs_per_gpu, n_gpus, config=2, n_total=None):
    n_total = n_total if n_total is not None else envs_per_gpu * n_gpus
    split = (f"{envs_per_gpu} batched envs per GPU" if config == 2 else
             f"{n_total} batched envs split contiguously over {n_gpus} GPU(s) ({envs_per_gpu} on rank 0)")
    return {
        "workload": f"BASELINE config {config}: AFCCylinder default grid 384x192 (386x194 arrays), Re=500, "
                    f"{split}, from init.bdim, 16 solver steps per env-step, "
                    "synthetic per-env actions a=clip(0.8 sin(2 pi k/25 + 2 pi e/256)+0.1 N(0,1)) (env 0: config-1 sequence)",
        "baseline_config": config, "envs_per_gpu": envs_per_gpu, "n_envs_total": n_total, "substeps": 16,
        "mode": "exact (bit-identical to the oracle)", "l2": "per-GPU state >> 126 MB L2 (inputs larger than L2)",
        "parallelism": f"env-sharded x{n_gpus}, no data-path collective (observations all-gathered once per env-step)",
    }


def workload_config3(n_gpus):
    return {
        "workload": "BASELINE config 3: single 2048x1024 cylinder-wake domain (resolution 128, 16x8 lengths, Re=500, "
                    "t_step=0.18/128 so dt=0.18 grid units), uniform start u=(1,0) p=0, actions 0 then (0.5,-0.5); "
                    "one step = one solver step (AFCCylinder.update2: 2 advection-diffusion passes + 2 MG pressure solves)",
        "baseline_config": 3, "grid": "2048x1024", "n_envs_total": n_gpus, "substeps": 1,
        "mode": "exact (bit-identical to the oracle)",
        "l2": "L2 flushed between timed steps: no (working set ~0.5 GB per step >> 126 MB L2: inputs larger than L2)",
        "parallelism": "one domain on one GPU" if n_gpus == 1 else f"{n_gpus} independent replicas (one domain per GPU; a single domain "
                       "only shards with the slab decomposition of config 5, which is not built)",
    }


def make_actions(n_steps, B, rank, e0=None):
    """BASELINE config 2 synthetic actions (SURVEY 8d) for the envs [e0, e0 + B) of the global batch."""
    rng = np.random.default_rng(1234 + rank)
    k = np.arange(n_steps)[:, None]
    e = (np.arange(B) + (rank * B if e0 is None else e0))[None, :]
    a1 = 0.8 * np.sin(2 * np.pi * k / 25 + 2 * np.pi * e / 256) + 0.1 * rng.standard_normal((n_steps, B))
    a2 = -0.8 * np.sin(2 * np.pi * k / 25 + 2 * np.pi * e / 256 + 1.0) + 0.1 * rng.standard_normal((n_steps, B))
    a = np.clip(np.stack([a1, a2], axis=-1), -1, 1).astype(np.float32)
    if (rank == 0 if e0 is None else e0 == 0):
        kk = np.arange(n_steps)
        a[:, 0, 0] = (0.8 * np.sin(2 * np.pi * kk / 25.0)).astype(np.float32)
        a[:, 0, 1] = (-0.8 * np.sin(2 * np.pi * kk / 25.0 + 1.0)).astype(np.float32)
    return a


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle on all host cores (persistent single-threaded worker per core)
# ------------------------------------------------------------------------------------------------
def _cpu_worker(conn, core, state_path, wide):
    try:
        os.sched_setaffinity(0, {core})
    except Exception:
        pass
    from oracle import oracle_py as O
    if wide:                                 # BASELINE config 3: one 2048x1024 domain per process, uniform start
        env = O.OracleEnv(literal=True, resolution=128, xLengths=16, yLengths=8, tStep=float(np.float32(0.18) / np.float32(128)))
        env.set_xi(0.5, -0.5)
    else:
        st = O.read_bdimb(state_path)
        env = O.OracleEnv(literal=True)      # reference behaviour: coefficients rebuilt every step
        env.set_state(st["ux"], st["uy"], st["p"])
    k = 0
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg is None:
            break
        for _ in range(msg):
            if wide:
                env.update2()                # a "step" of config 3 is one solver step
            else:
                a = (0.8 * np.sin(2 * np.pi * k / 25.0), -0.8 * np.sin(2 * np.pi * k / 25.0 + 1.0))
                env.env_step(a)
            k += 1
        conn.send(k)


class CpuArm:
    def __init__(self, cores=None, wide=False):
        from oracle import oracle_py as O
        O.build()
        import rlfluidcontrol_b200 as R
        self.cores = cores or len(os.sched_getaffinity(0))
        ctx = mp.get_context("spawn")
        self.workers = []
        core_ids = sorted(os.sched_getaffinity(0))[: self.cores]
        for c in core_ids:
            parent, child = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(child, c, str(R.default_init_state()), wide), daemon=True)
            p.start()
            self.workers.append((p, parent))
        for _, conn in self.workers:
            assert conn.recv() == "ready"

    def step(self, env_steps_each):
        """Every core advances its own environment by `env_steps_each` RL steps; returns wall seconds."""
        t0 = time.perf_counter()
        for _, conn in self.workers:
            conn.send(env_steps_each)
        for _, conn in self.workers:
            conn.recv()
        return time.perf_counter() - t0

    def close(self):
        for p, conn in self.workers:
            try:
                conn.send(None)
            except Exception:
                pass
        for p, _ in self.workers:
            p.join(timeout=5)


def cpu_baseline(sample_env_steps=4, reps=2):
    arm = CpuArm()
    arm.step(1)   # warm-up
    secs = [arm.step(sample_env_steps) for _ in range(reps)]
    arm.close()
    best = min(secs)
    return {
        "value": arm.cores * sample_env_steps / best, "unit": UNIT, "cores": arm.cores, "kind": "port",
        "sample": f"{arm.cores} single-threaded oracle processes (one per host core, literal C port of the Lilypad step, "
                  f"gcc -O2 -ffp-contract=off, coefficients rebuilt every step as the reference does), each advancing one "
                  f"AFCCylinder env from init.bdim by {sample_env_steps} env-steps (config-1 actions); best of {reps}",
    }


def cpu_baseline_wide(sample_steps=2):
    """Config 3 on the host: every core advances its OWN 2048x1024 domain (the reference is single-threaded per domain), so
    the aggregate is cores x the single-domain rate; both are reported."""
    arm = CpuArm(wide=True)
    arm.step(1)   # warm-up (first step builds the geometry)
    sec = arm.step(sample_steps)
    arm.close()
    return {
        "value": arm.cores * sample_steps / sec, "unit": UNIT3, "cores": arm.cores, "kind": "port",
        "single_domain_value": sample_steps / sec,
        "sample": f"{arm.cores} single-threaded oracle processes (one per host core), each advancing its own 2048x1024 domain "
                  f"(uniform start, actions (0.5,-0.5), coefficients rebuilt every step as the reference does) by {sample_steps} solver "
                  "steps; value = aggregate over the cores, single_domain_value = one domain on one core (what one Lilypad "
                  "instance achieves: it has no intra-domain parallelism)",
    }


def run_reference(args):
    """The CPU arm.  What one "step" of THIS arm is, is stated in its config (it is a bounded sample of the workload, sized
    for the host, not the GPU arm's batch)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wide = args.config == 3
    if args.config == 5:
        print(json.dumps({"impl": "reference", "unavailable": "config 5 (8192x4096 over 8 GPUs) is not built; the CPU port would need ~20 s per solver step"}))
        return
    arm = CpuArm(wide=wide)
    per_step = 1 if wide else args.ref_env_steps
    for _ in range(args.warmup):
        arm.step(per_step)
    secs = [arm.step(per_step) for _ in range(args.steps)]
    arm.close()
    total = sum(secs)
    value = arm.cores * per_step * args.steps / total
    unit = UNIT3 if wide else UNIT
    if wide:
        cfg = workload_config3(args.gpus)
        what = (f"one step of this arm = {arm.cores} single-threaded processes (one per host core), each advancing its own 2048x1024 "
                "domain by 1 solver step")
    else:
        cfg = workload_config(args.envs_per_gpu, args.gpus, args.config, args.envs_total if args.config == 4 else None)
        what = (f"one step of this arm = {arm.cores} single-threaded processes (one per host core) x {per_step} env-steps each = "
                f"{arm.cores * per_step} env-steps of the default-grid AFCCylinder from init.bdim (config-1 actions) -- a bounded sample "
                "of the workload, NOT the GPU arm's batch; compare `value` (env-steps/s), not ms_per_step")
    cfg["reference_arm"] = {"what_ran": what, "cores": arm.cores, "units_per_step": arm.cores * per_step,
                            "implementation": "literal C port of the reference step (oracle/lilypad_oracle.c, gcc -O2 -ffp-contract=off, "
                                              "coefficients rebuilt every step as the reference does); the Java itself cannot run: no JVM in the image"}
    line = {
        "impl": "reference", "metric": METRIC3 if wide else METRIC, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.config == 4 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": unit, "cores": arm.cores, "kind": "port", "sample": what},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampling
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_summary(config=2):
    """The committed `ncu --set full` summary of the same workload (newest round available), or {}."""
    names = ["r02_ncu_summary_cfg3.json"] if config == 3 else ["r02_ncu_summary.json", "r01_ncu_summary.json"]
    for nm in names:
        p = ROOT / "profiles" / nm
        if p.exists():
            try:
                return json.loads(p.read_text())
            except Exception:
                pass
    return {}


def ncu_lookup(tab, kernel, key):
    for name, rec in tab.items():
        base = name.split("<")[0]
        if base == kernel or base.replace("_rows", "").replace("_blk", "").replace("_march", "") == kernel:
            if key in rec:
                return float(rec[key])
    return None


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_table(prof, steps, peak, clk_mhz, ncu):
    """Per-kernel view of the live CUDA-event pass: algorithmic GB/s vs the HBM peak, and for the issue-bound stencil
    (k_advdif, --fmad=false) the warp-instruction rate vs the issue roofline 148 SMs x 4 schedulers x clock."""
    kern = sorted(prof, key=lambda r: -r["ms"])
    tot_ms = sum(r["ms"] for r in kern) or 1.0
    table = []
    for r in kern:
        avg_ms = r["ms"] / max(r["launches"], 1)
        gbs = r["bytes_per_launch"] / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        row = {"kernel": r["name"], "share": round(r["ms"] / tot_ms, 4), "avg_ms": round(avg_ms, 4),
               "launches_per_step": r["launches"] / max(steps, 1),
               "algorithmic_GBps": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 4)}
        if r["name"] == "k_advdif" and clk_mhz:
            inst = ncu_lookup(ncu, "k_advdif", "inst")          # warp instructions per launch (ncu smsp__inst_executed.sum)
            if inst and avg_ms > 0:
                issue_peak = 148 * 4 * clk_mhz * 1e6
                row["fp32_issue"] = {"warp_inst_per_launch": inst, "achieved_Ginst_s": round(inst / (avg_ms * 1e-3) / 1e9, 1),
                                     "peak_Ginst_s": round(issue_peak / 1e9, 1), "frac": round(inst / (avg_ms * 1e-3) / issue_peak, 4),
                                     "note": "instruction count from the committed ncu capture of the same workload; peak = 148 SMs x 4 "
                                             "schedulers x SM clock (one warp instruction per scheduler per cycle)"}
        table.append(row)
    return kern, tot_ms, table


# ------------------------------------------------------------------------------------------------
def dist_setup(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from rlfluidcontrol_b200 import build as product_build
    if rank == 0:
        product_build.build()
    barrier()
    return rank, world, local, barrier


def run_b200(args):
    """Configs 2 and 4: batched default-grid environments, sharded over the ranks (rlfluidcontrol_b200/sharding.py)."""
    import torch
    import torch.distributed as dist

    rank, world, local, barrier = dist_setup(args)
    import rlfluidcontrol_b200 as R
    from rlfluidcontrol_b200 import sharding

    K, W = args.steps, args.warmup
    if args.config == 4:
        if args.envs_total % world:
            raise SystemExit(f"--envs-total {args.envs_total} must divide by the {world} ranks")
        e_lo, e_hi = sharding.shard_range(args.envs_total, rank, world)
        B, total_envs, scaling = e_hi - e_lo, args.envs_total, "strong"
    else:
        B, total_envs, scaling = args.envs_per_gpu, args.envs_per_gpu * world, "weak"
        e_lo = rank * B
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(B, device=local, stream=stream.cuda_stream, init_time=-1.0)
    n_total = 2 * (W + K) + args.profile_steps
    acts_np = make_actions(n_total, B, rank, e0=e_lo)
    acts_dev = torch.from_numpy(acts_np).cuda()
    acts_host = torch.from_numpy(acts_np).pin_memory()
    obs_dev = torch.empty((B, 2), dtype=torch.float32, device="cuda")
    rew_dev = torch.empty(B, dtype=torch.float32, device="cuda")
    done_dev = torch.empty(B, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()

    obs_all = torch.empty((B * world, 2), dtype=torch.float32, device="cuda") if world > 1 else None

    def dev_step(k):
        env.step_device(acts_dev[k].data_ptr(), obs_dev.data_ptr(), rew_dev.data_ptr(), done_dev.data_ptr())
        if world > 1:   # the one exchange of the env-sharded path: every rank sees the whole batch's observations
            sharding.gather_observations_equal(obs_dev, obs_all)

    step_idx = 0
    with torch.cuda.stream(stream):
        # ---- device-resident arm ----
        for _ in range(W):
            dev_step(step_idx); step_idx += 1
        barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        l0 = env.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            dev_step(step_idx); step_idx += 1
        e1.record(stream)
        barrier()
        ms = sharding.max_over_ranks(e0.elapsed_time(e1), world, device="cuda")
        launches = env.launch_count - l0
        clk = clocks.stop() if rank == 0 else None
        obs_check = obs_dev.cpu().numpy()
        assert np.isfinite(obs_check).all(), "non-finite observation"
        assert env.running() == 0 and not env.flags().any()
        if args.dump_outputs:   # the last timed step's results of the whole batch, in global env order
            outputs = {nm: sharding.gather_observations(t, world).cpu().numpy()
                       for nm, t in (("obs", obs_dev), ("reward", rew_dev), ("done", done_dev.float()))}

        # ---- end-to-end arm: host buffers through rlfc_env_step ----
        for _ in range(W):
            env.step(acts_host[step_idx].numpy()); step_idx += 1
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            obs, rew, done = env.step(acts_host[step_idx].numpy()); step_idx += 1
        torch.cuda.synchronize()
        e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, world, device="cuda")
        barrier()

        # ---- per-kernel CUDA-event pass (same workload, live) ----
        prof = []
        if rank == 0 and args.profile_steps > 0:
            env.set_profiling(True)
            for _ in range(args.profile_steps):   # rank 0 alone: no collective in here (the other ranks do not take part)
                env.step_device(acts_dev[step_idx].data_ptr(), obs_dev.data_ptr(), rew_dev.data_ptr(), done_dev.data_ptr())
                step_idx += 1
            torch.cuda.synchronize()
            prof = env.get_profile()
            env.set_profiling(False)
    mg = env.mg_iters()
    env.close()
    barrier()

    if rank == 0:
        value = total_envs * K / (ms / 1e3)
        e2e = total_envs * K / e2e_s
        peak, peak_src = measured_peak()
        ncu = ncu_summary(2)
        kern, tot_ms, table = kernel_table(prof, args.profile_steps, peak, clk.get("sm_mhz") if clk else None, ncu)
        roof = None
        if kern:
            top = kern[0]
            avg_ms = top["ms"] / max(top["launches"], 1)
            ach = top["bytes_per_launch"] / (avg_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": top["name"], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_lookup(ncu, top["name"], "dram_traffic_B_per_launch") if B == 256 else None,
                    "peak_source": peak_src, "share_of_step": top["ms"] / tot_ms,
                    "algorithmic_bytes_per_launch": top["bytes_per_launch"], "avg_launch_ms": avg_ms}
            fp = next((r.get("fp32_issue") for r in table if r["kernel"] == top["name"] and "fp32_issue" in r), None)
            if fp:   # (k_advdif is bound by fp32 instruction issue under --fmad=false, SURVEY H5: the second roofline it is held to)
                roof["fp32_issue"] = fp
        # whole-step view against the SURVEY 8d model: 4 B * N_int * (28 + 13 (kP + kC)) per env per solver step
        nint = 384 * 192
        k_sum = float(mg.sum(axis=1).mean())
        model_bytes_step = 4.0 * nint * (28 + 13 * k_sum) * 16 * B
        whole = {"model_bytes_per_env_step_batch": model_bytes_step, "achieved_GBps": model_bytes_step / (ms / K * 1e-3) / 1e9}
        whole["frac_of_hbm_peak"] = whole["achieved_GBps"] / peak
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, world, args.config, total_envs), "clocks": clk,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(B * 2 * 4), "d2h_bytes_per_step": int(B * (2 + 1 + 1) * 4)},
            "gpu_launches": int(launches), "roofline": roof, "whole_step_roofline": whole, "kernels": table,
            "mg_iters_per_solve": k_sum / 2,
        }
        if world > 1:
            line["nccl_ranks"] = dist.get_world_size()
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_sample_env_steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_wide(args):
    """Config 3: one 2048x1024 domain per GPU, one solver step per bench step."""
    import torch
    import torch.distributed as dist

    rank, world, local, barrier = dist_setup(args)
    import rlfluidcontrol_b200 as R
    from rlfluidcontrol_b200 import sharding

    K, W = args.steps, max(args.warmup, 3)
    res = args.resolution
    t_step = float(np.float32(0.18) / np.float32(res))
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(1, init_state=None, device=local, stream=stream.cuda_stream, resolution=res, x_lengths=16, y_lengths=8,
                             t_step=t_step)
    cells = (env.n - 2) * (env.m - 2)
    act_dev = torch.tensor([[0.5, -0.5]], dtype=torch.float32, device="cuda")
    act_host = np.array([[0.5, -0.5]], np.float32)
    with torch.cuda.stream(stream):
        # SURVEY 8d: actions 0 for the impulsive start (the first solves take several MG iterations), then (0.5, -0.5)
        for _ in range(args.settle_steps):
            env.update2_device()
        env.update2_device(act_dev.data_ptr())
        for _ in range(W):
            env.update2_device()
        barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        l0 = env.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            env.update2_device()
        e1.record(stream)
        barrier()
        ms = sharding.max_over_ranks(e0.elapsed_time(e1), world, device="cuda")
        launches = env.launch_count - l0
        clk = clocks.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:   # (the other ranks run identical replicas)
            outputs = dict(zip(("ux", "uy", "p"), env.get_fields(0)))
        # ---- end-to-end: host action in, force + probes out, every step ----
        for _ in range(W):
            env.update2(act_host, want_probes=True)
        barrier()
        t0 = time.perf_counter()
        its = []
        for _ in range(K):
            f, pr = env.update2(act_host, want_probes=True)
        torch.cuda.synchronize()
        e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, world, device="cuda")
        assert np.isfinite(f).all() and not env.flags().any()
        barrier()
        prof = []
        if rank == 0 and args.profile_steps > 0:
            env.set_profiling(True)
            for _ in range(args.profile_steps):
                env.update2()
                its.append(env.mg_iters()[0].tolist())
            prof = env.get_profile()
            env.set_profiling(False)
    env.close()
    barrier()
    if rank == 0:
        value = world * K / (ms / 1e3)
        e2e = world * K / e2e_s
        peak, peak_src = measured_peak()
        kern, tot_ms, table = kernel_table(prof, args.profile_steps, peak, clk.get("sm_mhz") if clk else None, ncu_summary(3))
        k_sum = float(np.sum(its, axis=1).mean()) if its else 2.0
        # SURVEY 8d, coarse levels off chip: 4 B * N_int * (28 + 16 (kP + kC)) per solver step = 240 B/cell at one iteration per solve
        model_bytes = 4.0 * cells * (28 + 16 * k_sum)
        ach = model_bytes / (ms / K * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "whole solver step (every kernel of the step is a latency chain or a small grid; no single "
                                          "kernel dominates: see `kernels`)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": model_bytes, "avg_launch_ms": ms / K,
                "model": "4 B x N_int x (28 + 16 (kP + kC)) = 240 B/cell at one MG iteration per solve (SURVEY 8d)"}
        if kern:
            top = kern[0]
            roof["dominant_kernel"] = {"kernel": top["name"], "share_of_step": top["ms"] / tot_ms,
                                       "avg_launch_ms": top["ms"] / max(top["launches"], 1)}
        line = {
            "metric": METRIC3, "value": value, "unit": UNIT3, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config3(world), "clocks": clk,
            "e2e": {"value": e2e, "unit": UNIT3, "h2d_bytes_per_step": 8, "d2h_bytes_per_step": int((2 + 32) * 4)},
            "gpu_launches": int(launches), "roofline": roof, "kernels": table, "mg_iters_per_solve": k_sum / 2,
        }
        if res != 128:
            line["config"]["workload"] += f" [scaled run: resolution {res}, grid {env.n - 2}x{env.m - 2}]"
        if world == 1 and not args.no_cpu_baseline and res == 128:
            line["cpu_baseline"] = cpu_baseline_wide(args.cpu_sample_wide_steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


METRIC5 = "solver-steps/sec (single BDIM domain, slab-decomposed over the GPUs of one box)"


NVLINK_NOTE = None


def nvlink_counters(n):
    """Cumulative NVLink data bytes (tx + rx) of devices 0..n-1 from NVML, or None (NVLINK_NOTE says why)."""
    global NVLINK_NOTE
    try:
        import pynvml
        pynvml.nvmlInit()
        tot = 0
        for d in range(n):
            h = pynvml.nvmlDeviceGetHandleByIndex(d)
            vals = pynvml.nvmlDeviceGetFieldValues(h, [(pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF),
                                                       (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)])
            for v in vals:
                if v.nvmlReturn != 0:
                    NVLINK_NOTE = f"NVML field {v.fieldId} on device {d}: nvmlReturn {v.nvmlReturn}"
                    return None
                tot += int(v.value.ullVal) * 1024          # KiB
        return tot
    except Exception as ex:
        NVLINK_NOTE = f"{type(ex).__name__}: {ex}"
        return None


def slab_traffic_model(n, m, nd, k_sum):
    """Bytes that cross device boundaries per solver step in slab mode -- a MODEL (the pool's NVML has no NVLink byte
    counters), stated with its assumptions:
    * stencil halos of the row-slab-distributed plain arrays, per internal boundary and solver step: advection-diffusion reads
      2 rows of ux, uy on either side in both half steps (16 rows), the first MG iteration reads p two rows deep and ux one
      row (5 rows per solve), the projection reads p one row (1 row per solve), the coarse grid-wide levels add about a third
      of level 0's MG halo (geometric sum); one row = 4 (m) bytes;
    * layout conversions between the row-distributed plain arrays and the STRIP-distributed skewed arrays of the chained
      smoother, per MG iteration and level-0 cell: the up pass writes r (4 B) and the tagged sweep-0 value (8 B), the increment
      reads the tagged result (8 B), the coefficient entry (16 B) and r (4 B): 40 B, x 4/3 for the coarser chained levels; a
      fraction (nd - 1)/nd of it is remote."""
    try:
        if nd <= 1:
            return {"halo_bytes_per_step_model": 0, "layout_conversion_bytes_per_step_model": 0}
        row = 4.0 * m
        solves = 2.0
        halo_rows = 16.0 + solves * (5.0 * (k_sum / 2.0) * (4.0 / 3.0) + 1.0)
        halo = (nd - 1) * halo_rows * row
        conv = 40.0 * (4.0 / 3.0) * (n - 2) * (m - 2) * k_sum * (nd - 1) / nd
        return {"halo_bytes_per_step_model": int(halo), "layout_conversion_bytes_per_step_model": int(conv)}
    except Exception:
        return {}


def run_slab(args):
    """Config 5: ONE domain (default 8192x4096, resolution 512) advanced by --gpus devices through the library's slab mode
    (rlfc_config.n_devices): the devices are driven by ONE host process -- rank 0 -- which owns all of them (shared address
    range + peer access); under torchrun the other ranks only take part in the rendezvous."""
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("gloo", init_method="env://")
    nd = args.gpus
    if rank == 0:
        import rlfluidcontrol_b200 as R

        K, W = args.steps, max(args.warmup, 3)
        res = args.resolution
        # SURVEY 8d prescribes t_step = 0.18/resolution (dt = 0.18 grid units).  At resolution 512 (nu = D/Re = 1.024) that violates
        # the reference's own bound BDIM.checkCFL = 1/(max|u| + 3 nu) (BDIM.pde:217-219) once |u| > 2.5, and the impulsive start
        # diverges near solver step 41 -- in the CPU oracle exactly as on the device (profiles/r02_config5_stability.md).  From
        # resolution 512 on the bench therefore runs dt = 0.09 grid units: same work per step, stable.
        dt_grid = 0.18 if res < 512 else 0.09
        t_step = float(np.float32(dt_grid) / np.float32(res))
        env = R.AFCCylinderBatch(1, init_state=None, device=0, resolution=res, x_lengths=16, y_lengths=8, t_step=t_step, n_devices=nd)
        cells = (env.n - 2) * (env.m - 2)
        act_host = np.array([[0.5, -0.5]], np.float32)
        torch.cuda.set_device(0)
        ext = torch.cuda.ExternalStream(env.stream, device=0)
        act_dev = torch.tensor([[0.5, -0.5]], dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        for _ in range(args.settle_steps):
            env.update2_device()
        env.update2_device(act_dev.data_ptr())
        for _ in range(W):
            env.update2_device()
        _ = env.t                                            # (synchronises)
        clocks = ClockSampler(0)
        clocks.start()
        l0, (_, b0, shared) = env.launch_count, env.slab_info()
        nv0 = nvlink_counters(nd)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        for _ in range(K):
            env.update2_device()                             # (the last kernel of a step runs behind a barrier of all devices)
        e1.record(ext)
        _ = env.t
        ms = e0.elapsed_time(e1)
        nv1 = nvlink_counters(nd)
        launches, barriers = env.launch_count - l0, env.slab_info()[1] - b0
        clk = clocks.stop()
        if args.dump_outputs:
            outputs = dict(zip(("ux", "uy", "p"), env.get_fields(0)))
        for _ in range(W):
            env.update2(act_host, want_probes=True)
        t0 = time.perf_counter()
        for _ in range(K):
            f, pr = env.update2(act_host, want_probes=True)
        e2e_s = time.perf_counter() - t0
        assert np.isfinite(f).all() and not env.flags().any()
        prof, its = [], []
        if args.profile_steps > 0:
            env.set_profiling(True)
            for _ in range(args.profile_steps):
                env.update2()
                its.append(env.mg_iters()[0].tolist())
            prof = env.get_profile()
            env.set_profiling(False)
        env_n, env_m = env.n, env.m
        env.close()
        peak, peak_src = measured_peak()
        kern, tot_ms, table = kernel_table(prof, args.profile_steps, peak, clk.get("sm_mhz") if clk else None, {})
        k_sum = float(np.sum(its, axis=1).mean()) if its else 2.0
        model_bytes = 4.0 * cells * (28 + 16 * k_sum)
        ach = model_bytes / (ms / K * 1e-3) / 1e9
        line = {
            "metric": METRIC5, "value": K / (ms / 1e3), "unit": UNIT3, "n_gpus": nd, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"BASELINE config 5: ONE {env.n - 2}x{env.m - 2} cylinder-wake domain (resolution {res}, 16x8 lengths, "
                                   f"Re=500, dt = {dt_grid} grid units, uniform start, actions 0 then (0.5,-0.5)) slab-decomposed over {nd} "
                                   "GPU(s) of one box; one step = one solver step (AFCCylinder.update2)",
                       "baseline_config": 5, "grid": f"{env.n - 2}x{env.m - 2}", "mode": "exact (bit-identical to the single-device run)",
                       "l2": "working set >> 126 MB L2 per device (inputs larger than L2)",
                       "parallelism": f"slab x{nd}: rows / strips distributed over one shared address range (VMM + NVLink peer access), "
                                      "one host process drives all devices"},
            "clocks": clk,
            "e2e": {"value": K / e2e_s, "unit": UNIT3, "h2d_bytes_per_step": 8, "d2h_bytes_per_step": int((2 + 32) * 4)},
            "gpu_launches": int(launches),
            "slab": {"devices": nd, "barriers_per_step": barriers / K, "shared_address_range_bytes": shared,
                     **slab_traffic_model(env_n, env_m, nd, k_sum),
                     "nvlink_bytes_per_step_measured": (None if nv0 is None or nv1 is None else (nv1 - nv0) / K),
                     "nvlink_counter_note": NVLINK_NOTE},
            "roofline": {"bound": "hbm", "kernel": "whole solver step", "achieved": ach, "peak": peak * nd, "unit": "GB/s",
                         "frac": ach / (peak * nd), "traffic": None, "peak_source": peak_src + f" x {nd} devices",
                         "algorithmic_bytes_per_launch": model_bytes, "avg_launch_ms": ms / K,
                         "model": "4 B x N_int x (28 + 16 (kP + kC)) = 240 B/cell at one MG iteration per solve (SURVEY 8d)"},
            "kernels": table, "mg_iters_per_solve": k_sum / 2,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json configs[] entry (1-based)")
    ap.add_argument("--envs-per-gpu", type=int, default=256, help="config 2: environments per GPU (weak scaling)")
    ap.add_argument("--envs-total", type=int, default=4096, help="config 4: environments in total, split over the ranks")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--profile-steps", type=int, default=1)
    ap.add_argument("--cpu-sample-env-steps", type=int, default=4)
    ap.add_argument("--cpu-sample-wide-steps", type=int, default=2)
    ap.add_argument("--ref-env-steps", type=int, default=2, help="env-steps per core per step in --impl reference")
    ap.add_argument("--resolution", type=int, default=None,
                    help="configs 3 / 5: cells per diameter (default 128 = the 2048x1024 domain / 512 = the 8192x4096 domain)")
    ap.add_argument("--settle-steps", type=int, default=12, help="config 3: untimed solver steps after the impulsive start")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed path's outputs of its last timed step as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl b200)")
    if args.resolution is None:
        args.resolution = 512 if args.config == 5 else 128
    if args.steps is None:
        args.steps = 200 if (args.config == 3 and args.impl == "b200") else (20 if args.config == 5 else 8)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 5:
        run_slab(args)
    elif args.config == 3:
        run_wide(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
