"""State records (rlfc_env_export / rlfc_env_import and their _device variants) on one GPU: 256 default-grid
environments from init.bdim.

  * export_device and import_device of all 256 environments (record k <-> environment k): time from CUDA events over
    --calls calls, and the effective bandwidth (the record bytes written by an export; read twice and written to the
    fields by an import, counted once per direction as the snapshot table counts them: record bytes read + written).
    Alternated in the same run with cudaMemcpyAsync device-to-device of the same number of bytes (one block, larger than
    the L2, so it comes from HBM like the record copies).
  * export / import of 1 and of 256 environments through host memory (host clock around each call; both synchronise
    before they return).

The cases run --rounds times, alternated, to show the spread.  Records the card's name and power limit in the same run.
Prints one JSON object; --out also writes it.  Needs a GPU.
    python tools/bench_records.py --out profiles/records_b200.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_adaptive import card_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    import rlfluidcontrol_b200 as R
    R.load_library()
    cudart = C.CDLL("libcudart.so.12")       # the runtime librlfc.so is linked against
    cudart.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    B, K = args.envs, args.calls
    stream = torch.cuda.Stream()
    env = R.AFCCylinderBatch(B, stream=stream.cuda_stream)
    size = env.record_bytes
    moved = B * size
    recs = torch.empty(moved, dtype=torch.uint8, device="cuda")
    src = torch.empty(moved, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(1)
    ids = torch.arange(B, dtype=torch.int32, device="cuda")
    env.reset(None, reset_accumulators=True)
    env.update2()                             # a state that is not the init state everywhere
    torch.cuda.synchronize()

    def memcpy():
        rc = cudart.cudaMemcpyAsync(C.c_void_p(dst.data_ptr()), C.c_void_p(src.data_ptr()), moved, 3, C.c_void_p(stream.cuda_stream))
        assert rc == 0, rc

    cases = {
        "export_device": lambda: env.export_states_device(ids.data_ptr(), B, recs.data_ptr()),
        "import_device": lambda: env.import_states_device(ids.data_ptr(), B, recs.data_ptr(), size),
        "memcpy_d2d": memcpy,
    }

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / K

    for fn in cases.values():                 # warm-up (the first call allocates the scratch)
        fn(); fn()
    torch.cuda.synchronize()
    res = {k: [] for k in cases}
    for _ in range(args.rounds):
        for name, fn in cases.items():
            ms = timed(fn)
            res[name].append({"ms_per_call": ms, "gb_per_s": 2 * moved / (ms * 1e-3) / 1e9})
    assert not env.flags().any()

    host = {}
    for n in (1, B):
        sel = np.arange(n, dtype=np.int32)
        blob = env.export_states(sel)
        ex, im = [], []
        for _ in range(args.rounds * 3):
            t0 = time.perf_counter()
            blob = env.export_states(sel)
            ex.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            env.import_states(sel, blob)
            im.append((time.perf_counter() - t0) * 1e3)
        host[f"export_{n}"], host[f"import_{n}"] = ex, im
    env.close()

    summary = {k: {"median_ms": float(np.median([x["ms_per_call"] for x in v])),
                   "median_gb_per_s": float(np.median([x["gb_per_s"] for x in v]))} for k, v in res.items()}
    for k in ("export_device", "import_device"):
        summary[k]["over_memcpy"] = summary[k]["median_gb_per_s"] / summary["memcpy_d2d"]["median_gb_per_s"]
    for k, v in host.items():
        summary[k] = {"median_ms": float(np.median(v))}
    out = {"workload": f"{B} default-grid envs ({env.n}x{env.m} incl. ghosts) from init.bdim after one step; record "
                       f"{size} bytes; {K} calls per timing, {args.rounds} alternated rounds; {moved} record bytes per call "
                       f"of all {B} pairs",
           "card": card_info(), "device": res, "host_ms": host, "summary": summary}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
