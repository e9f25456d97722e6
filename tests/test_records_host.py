"""CPU tests of state records (include/rlfc.h "State records"): the size and checksum functions of the library, the
pure-numpy reader, and the argument checks that run before any device call."""
import ctypes as C

import numpy as np
import pytest

from rlfluidcontrol_b200 import records


def _config(rlfc, **kw):
    from rlfluidcontrol_b200.env import Config
    c = Config()
    rlfc.load_library().rlfc_default_config(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def _lib_bytes(rlfc, **kw):
    n = C.c_size_t()
    rc = rlfc.load_library().rlfc_record_bytes(C.byref(_config(rlfc, **kw)), C.byref(n))
    return rc, n.value


@pytest.mark.parametrize("grid,K", [((24, 16, 8), 0), ((24, 16, 8), 3), ((64, 16, 8), 0), ((8, 4, 2), 7), ((16, 3, 1), 1)])
def test_record_bytes_follows_the_layout(rlfc, grid, K):
    res, xl, yl = grid
    rc, got = _lib_bytes(rlfc, resolution=res, x_lengths=xl, y_lengths=yl, n_sensors=K)
    n, m = xl * res + 2, yl * res + 2
    # header 80, scalar record 192, sensor table 12 K, sensor values 4 K, three n x m float fields
    assert rc == 0 and got == 80 + 192 + 12 * K + 4 * K + 3 * 4 * n * m == records.record_bytes(n, m, K)
    assert got % 16 == 0


def test_record_bytes_rejects_bad_arguments(rlfc):
    L = rlfc.load_library()
    n = C.c_size_t()
    assert L.rlfc_record_bytes(None, C.byref(n)) == -1
    assert L.rlfc_record_bytes(C.byref(_config(rlfc)), None) == -1
    assert _lib_bytes(rlfc, resolution=0)[0] == -1
    assert _lib_bytes(rlfc, y_lengths=-1)[0] == -1
    assert _lib_bytes(rlfc, n_sensors=-2)[0] == -1
    assert "n_sensors" in L.rlfc_last_error().decode()


def synthetic(n=4, m=6, K=2, seed=0):
    """A record of an n x m grid with K sensors, random payload, consistent header and checksum."""
    rng = np.random.default_rng(seed)
    size = records.record_bytes(n, m, K)
    buf = bytearray(rng.integers(0, 256, size, dtype=np.uint8).tobytes())
    h = np.zeros(1, records.HEADER)
    h["magic"], h["version"], h["adaptive_dt"], h["length"] = records.MAGIC, 1, 1, size
    h["resolution"], h["x_lengths"], h["y_lengths"], h["n"], h["m"] = 1, n - 2, m - 2, n, m
    h["re"], h["dR"], h["gR"], h["theta"], h["t_step"] = 300, 0.125, 0.2, 1.0471976, 0.0075
    h["n_probes"], h["n_sensors"] = 32, K
    buf[:records.HEADER_BYTES] = h.tobytes()
    buf[8:16] = np.uint64(records.checksum(buf)).tobytes()
    return buf


def _lib_checksum(rlfc, buf):
    b = (C.c_char * len(buf)).from_buffer(buf)
    return rlfc.load_library().rlfc_record_checksum(b, len(buf))


def _naive_checksum(buf):
    """The rlfc.h definition word by word, in Python integers."""
    w = np.frombuffer(bytes(buf), "<u4")
    M = (1 << 64) - 1
    s = 0
    for i in range(4, w.size):
        x = (i << 32) | int(w[i])
        x ^= x >> 33
        x = (x * 0xFF51AFD7ED558CCD) & M
        x ^= x >> 33
        x = (x * 0xC4CEB9FE1A85EC53) & M
        x ^= x >> 33
        s = (s + x) & M
    return s


def test_checksum_matches_the_definition(rlfc):
    for seed in range(3):
        buf = synthetic(seed=seed)
        want = _naive_checksum(buf)
        assert records.checksum(buf) == want
        assert _lib_checksum(rlfc, buf) == want
        assert int(np.frombuffer(bytes(buf[8:16]), "<u8")[0]) == want


def test_every_single_bit_flip_changes_the_checksum(rlfc):
    buf = synthetic(n=2, m=2, K=1)
    base = _lib_checksum(rlfc, buf)
    for byte in range(len(buf)):
        for bit in range(8):
            buf[byte] ^= 1 << bit
            got = _lib_checksum(rlfc, buf)
            buf[byte] ^= 1 << bit
            if byte >= 16:
                assert got != base, (byte, bit)
            else:                      # magic and the checksum field itself are not covered
                assert got == base, (byte, bit)


def test_parse_record_synthetic():
    n, m, K = 4, 6, 2
    buf = synthetic(n, m, K)
    w = np.frombuffer(bytes(buf), "<u4")
    r = records.parse_record(buf)
    assert (r["n"], r["m"], r["n_sensors"], r["length"], r["version"], r["adaptive_dt"]) == (n, m, K, len(buf), 1, 1)
    assert r["tuple"] == (300, np.float32(0.125), np.float32(0.2), np.float32(1.0471976), np.float32(0.0075))
    assert r["scalars"]["dt"] == np.frombuffer(bytes(buf[96:100]), "<f4")[0]     # scalar word 4 at 80 + 16
    assert r["scalars"]["iters"].tolist() == w[20 + 46:20 + 48].astype(np.int32).tolist()
    s0 = 272 + 16 * K
    assert r["sensor_table"]["field"].tolist() == w[68:68 + 3 * K:3].astype(np.int32).tolist()
    assert r["sensors"].tobytes() == bytes(buf[272 + 12 * K:s0])
    assert r["ux"].shape == (n, m) and r["ux"].tobytes() == bytes(buf[s0:s0 + 4 * n * m])
    assert r["p"].tobytes() == bytes(buf[s0 + 8 * n * m:])
    two = bytes(buf) + bytes(synthetic(n, m, K, seed=1))
    parts = records.split_records(two, 2)
    assert records.parse_record(parts[1])["ux"].tobytes() == records.parse_record(synthetic(n, m, K, seed=1))["ux"].tobytes()
    bad = bytearray(buf)
    bad[0] ^= 1
    with pytest.raises(ValueError, match="magic"):
        records.parse_record(bad)
    with pytest.raises(ValueError, match="length"):
        records.parse_record(buf[:-4])


def test_null_arguments_rejected_before_any_device_call(rlfc):
    L = rlfc.load_library()
    ids = (C.c_int * 1)(0)
    buf = (C.c_char * 16)()
    assert L.rlfc_env_export(None, ids, 1, buf) == -1
    assert L.rlfc_env_import(None, ids, 1, buf, 0) == -1
    assert L.rlfc_env_export_device(None, None, 0, None) == -1
    assert L.rlfc_env_import_device(None, None, 0, None, 0, 0) == -1
    assert "null handle" in L.rlfc_last_error().decode()
