"""State records (include/rlfc.h "State records") read without the library: pure numpy, no device.

`parse_record(buf)` returns the header fields of one record and numpy views of its payload; `checksum(buf)` is the
record checksum that `rlfc_record_checksum` computes.
"""
from __future__ import annotations

import numpy as np

MAGIC = b"RLFCSTAT"
VERSION = 1
HEADER_BYTES = 80
SCALAR_WORDS = 48

HEADER = np.dtype([
    ("magic", "S8"), ("checksum", "<u8"), ("version", "<u4"), ("adaptive_dt", "<u4"), ("length", "<u8"),
    ("resolution", "<i4"), ("x_lengths", "<i4"), ("y_lengths", "<i4"), ("n", "<i4"), ("m", "<i4"),
    ("re", "<i4"), ("dR", "<f4"), ("gR", "<f4"), ("theta", "<f4"), ("t_step", "<f4"),
    ("n_probes", "<u4"), ("n_sensors", "<u4"),
])
assert HEADER.itemsize == HEADER_BYTES
SCALARS = np.dtype([
    ("xi", "<f4", 2), ("t", "<f4"), ("flow_t", "<f4"), ("dt", "<f4"), ("force", "<f4", 2), ("probes", "<f4", 32),
    ("callLearn", "<i4"), ("Cd", "<f4"), ("Cl", "<f4"), ("obs", "<f4", 2), ("frozen", "<i4"), ("non_finite", "<i4"),
    ("iters", "<i4", 2),
])
assert SCALARS.itemsize == 4 * SCALAR_WORDS
SENSOR = np.dtype([("field", "<i4"), ("x", "<f4"), ("y", "<f4")])


def record_bytes(n, m, n_sensors):
    """Bytes of one record of an n x m grid (ghosts included) with n_sensors sensors."""
    return HEADER_BYTES + 4 * SCALAR_WORDS + 16 * n_sensors + 12 * n * m


def _mix(x):
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xFF51AFD7ED558CCD)
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xC4CEB9FE1A85EC53)
    return x ^ (x >> np.uint64(33))


def checksum(buf):
    """Sum mod 2^64 over the words w_i, i >= 4, of mix(i << 32 | w_i) (rlfc.h)."""
    w = np.frombuffer(memoryview(buf), dtype="<u4", count=len(memoryview(buf)) // 4).astype(np.uint64)
    i = np.arange(w.size, dtype=np.uint64)
    with np.errstate(over="ignore"):
        return int(_mix((i << np.uint64(32)) | w)[4:].sum(dtype=np.uint64))


def parse_record(buf):
    """One record: a dict of the header fields (plus "tuple", the five parameters) and read-only views of the payload:
    "scalars" (a structured scalar of SCALARS), "sensor_table" (K entries of SENSOR), "sensors" (K floats) and "ux",
    "uy", "p" ((n, m) float32, reference layout).  Raises ValueError for a buffer that is not a record of its own header."""
    mv = memoryview(buf).cast("B")
    if len(mv) < HEADER_BYTES:
        raise ValueError("shorter than a record header")
    h = np.frombuffer(mv, HEADER, count=1)[0]
    if bytes(h["magic"]) != MAGIC:
        raise ValueError("bad magic")
    out = {name: h[name].item() for name in HEADER.names}
    n, m, K = out["n"], out["m"], out["n_sensors"]
    if out["length"] != record_bytes(n, m, K) or len(mv) < out["length"]:
        raise ValueError(f"length {out['length']} does not match the header or the buffer ({len(mv)} bytes)")
    out["tuple"] = (out["re"], out["dR"], out["gR"], out["theta"], out["t_step"])
    o = HEADER_BYTES
    out["scalars"] = np.frombuffer(mv, SCALARS, count=1, offset=o)[0]
    o += SCALARS.itemsize
    out["sensor_table"] = np.frombuffer(mv, SENSOR, count=K, offset=o)
    o += SENSOR.itemsize * K
    out["sensors"] = np.frombuffer(mv, "<f4", count=K, offset=o)
    o += 4 * K
    for name in ("ux", "uy", "p"):
        out[name] = np.frombuffer(mv, "<f4", count=n * m, offset=o).reshape(n, m)
        o += 4 * n * m
    return out


def split_records(buf, count):
    """The `count` consecutive records of one export, as memoryviews."""
    mv = memoryview(buf).cast("B")
    if count <= 0 or len(mv) % count:
        raise ValueError(f"{len(mv)} bytes do not hold {count} equal records")
    size = len(mv) // count
    return [mv[k * size:(k + 1) * size] for k in range(count)]
