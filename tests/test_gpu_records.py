"""State records (rlfc_env_export / rlfc_env_import and their _device variants): an environment imported from a record
continues bit-identically to the one that exported it, in another handle, process or device, through every entry point
and read-out.  Records that fail a check change nothing.  Bar: every float compared with ==, as in test_gpu_snapshots."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from rlfluidcontrol_b200 import records
from test_gpu_parity import assert_same
from test_gpu_slab import device_count
from test_gpu_snapshots import RL, X, DeviceRL, assert_readouts, hetero_actions, readouts, rl_actions, rl_sequence

pytestmark = pytest.mark.gpu

F = np.float32
SENS = [("p", 100.0, 96.0), ("ux", 150.5, 90.25), ("uy", 200.0, 100.0)]
CONT = dict(init_time=0.05)          # the RL-step calls of the continuation reach their first observation quickly


def full(env, a):
    return np.tile(np.asarray(a, F).reshape(1, 2), (env.n_envs, 1))


def continuation(torch, env, e, tmp_path=None, tag=""):
    """Environment e through 3 substep, 2 substep_device, 2 step and 2 step_device calls: every read-out after each."""
    out = []

    def take(extra):
        r = readouts(env, e)
        r["extra"] = [np.asarray(x).copy() for x in extra]
        if env.n_sensors:
            r["sensors"] = env.sensors()[e].copy()
        out.append(r)

    for k in range(3):
        f, pr = env.update2(full(env, [0.6, -0.4]) if k == 0 else None, want_probes=True)
        take((f[e], pr[e]))
    d_a = torch.from_numpy(full(env, [-0.3, 0.5])).cuda()
    torch.cuda.synchronize()
    for _ in range(2):
        env.update2_device(d_a.data_ptr())
        torch.cuda.synchronize()
        take(())
    for k in range(2):
        o, r, d = env.step(full(env, rl_actions(k, 1)[0]))
        take((o[e], r[e], d[e]))
    dev = DeviceRL(torch, env)
    for k in range(2):
        o, r, d, _ = dev.round(full(env, rl_actions(k + 2, 1)[0]))
        take((o[e], r[e], d[e]))
    if tmp_path is not None:
        out.append(readouts(env, e, tmp_path, tag))
    return out


def assert_continuation(got, want, what):
    assert len(got) == len(want)
    for c, (g, w) in enumerate(zip(got, want)):
        assert_readouts(g, w, f"{what}, call {c}")
        for i, (a, b) in enumerate(zip(g.get("extra", []), w.get("extra", []))):
            assert a.tobytes() == b.tobytes(), f"{what}, call {c}: read-out {i} {a!r} vs {b!r}"
        if "sensors" in w:
            assert g["sensors"].tobytes() == w["sensors"].tobytes(), f"{what}, call {c}: sensors"


def warm(env, steps=4, seed=3):
    for k in range(steps):
        env.update2(hetero_actions(env.n_envs, seed) if k == 0 else None)


def dev_ints(torch, v):
    return torch.tensor(v, dtype=torch.int32, device="cuda")


def to_device(torch, data):
    return torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()


MIXED = [dict(), X, X, dict(re=100), X, dict(theta=F(1.2))]
WIDE_T = float(F(0.18) / F(64))        # the impulsive start at resolution 64 stays stable (test_gpu_slab)
LIB = [dict(), X, dict(re=100)]

# case: (source kw, destination kw, source env, destination env, environment variable, device path)
ROUND_TRIP = {
    "default": (dict(n_envs=4), dict(n_envs=4), 2, 1, None, False),
    "groups": (dict(n_envs=6), dict(n_envs=3), 4, 0, ("RLFC_GROUPS", "3"), True),
    "no_graph": (dict(n_envs=3), dict(n_envs=2), 0, 1, ("RLFC_NO_GRAPH", "1"), True),
    "snapshots_sensors": (dict(n_envs=3, n_snapshots=2, sensors=SENS), dict(n_envs=2, n_snapshots=1, sensors=SENS), 1, 1,
                          None, True),
    "adaptive": (dict(n_envs=3, adaptive_dt=1), dict(n_envs=4, adaptive_dt=1), 1, 3, None, True),
    "env_params": (dict(n_envs=6, env_params=MIXED), dict(n_envs=3, env_params=[dict(), X, dict()]), 4, 1, None, False),
    "param_sets": (dict(n_envs=3, param_sets=LIB), dict(n_envs=2, param_sets=LIB), 0, 1, None, True),
    "wide_grid": (dict(n_envs=2, resolution=64, init_state=None, t_step=WIDE_T), dict(n_envs=2, resolution=64, init_state=None,
                                                                                      t_step=WIDE_T), 0, 1, None, True),
}


@pytest.mark.parametrize("case", list(ROUND_TRIP))
def test_round_trip(rlfc, monkeypatch, tmp_path, case):
    torch = pytest.importorskip("torch")
    skw, dkw, s, d, envvar, device = ROUND_TRIP[case]
    if envvar:
        monkeypatch.setenv(*envvar)
    skw, dkw = dict(skw, **CONT), dict(dkw, **CONT)
    with rlfc.AFCCylinderBatch(skw.pop("n_envs"), **skw) as src, rlfc.AFCCylinderBatch(dkw.pop("n_envs"), **dkw) as dst:
        if case == "param_sets":               # both on library set 1 (set 2 for the others) after a device reset
            for env in (src, dst):
                ids = dev_ints(torch, list(range(env.n_envs)))
                target = s if env is src else d
                sets = dev_ints(torch, [1 if e == target else 2 for e in range(env.n_envs)])
                torch.cuda.synchronize()
                env.reset_sets_device(ids.data_ptr(), sets.data_ptr(), env.n_envs)
        warm(src)
        warm(dst, 2, seed=8)
        if device:
            buf = torch.empty(src.record_bytes, dtype=torch.uint8, device="cuda")
            ids = dev_ints(torch, [s])
            torch.cuda.synchronize()
            src.export_states_device(ids.data_ptr(), 1, buf.data_ptr())
            torch.cuda.synchronize()
            rec = buf.cpu().numpy().tobytes()
            assert rec == src.export_states([s])
            dbuf, dids = to_device(torch, rec), dev_ints(torch, [d])
            torch.cuda.synchronize()
            dst.import_states_device(dids.data_ptr(), 1, dbuf.data_ptr(), len(rec))
            torch.cuda.synchronize()
        else:
            rec = src.export_states([s])
            dst.import_states([d], rec)
        assert dst.flags()[d] == 0
        assert_readouts(readouts(dst, d), readouts(src, s), f"{case}: right after the import")
        if case == "adaptive":
            for l in range(src.num_levels):
                for nm in ("lower.x", "lower.y", "inv", "diag") + (("c.x", "c.y") if l == 0 else ()):
                    assert_same(dst.get_coeffs(d, nm, l), src.get_coeffs(s, nm, l), f"{nm} level {l}")
        if case == "env_params":               # a record goes only to an equal tuple
            with pytest.raises(rlfc.RlfcError, match=r"record 0 \(env id 0\): parameter tuple"):
                dst.import_states([0], rec)
        want = continuation(torch, src, s, tmp_path, "src")
        got = continuation(torch, dst, d, tmp_path, "dst")
        assert_continuation(got, want, case)


@pytest.mark.parametrize("state", ["uncontrolled_start", "mid_window", "boundary", "after_done"])
def test_rl_step_states(rlfc, state):
    """Records taken at the four kinds of RL-step state, imported into a new handle, continue exactly (obs, reward, done,
    running(), t); keep_accumulators = 0 / 1 does what it does for restore."""
    torch = pytest.importorskip("torch")
    B = 3
    with rlfc.AFCCylinderBatch(B, n_snapshots=1, **RL) as env, rlfc.AFCCylinderBatch(B, **RL) as other:
        dev = DeviceRL(torch, env)
        k = 0
        for _ in range({"uncontrolled_start": 1, "mid_window": 2, "boundary": 3, "after_done": 3}[state]):
            dev.round(rl_actions(k, B))
            k += 1
        if state == "after_done":
            while not env.step(rl_actions(k, B))[2].all():
                k += 1
            k += 1
        rec = env.export_states([0])
        env.snapshot([0], [0])
        other.import_states([0, 1, 2], rec * 3)
        want = rl_sequence(env, dev, k)
        got = rl_sequence(other, DeviceRL(torch, other), k)
        for c, (g, w) in enumerate(zip(got, want)):
            for nm, a, b in zip(("obs", "reward", "done", "running", "t"), g, w):
                assert np.array_equal(np.asarray(a), np.asarray(b)), f"{state}: {nm} call {c}"
        for keep in (0, 1):                       # env 1 restored, env 2 imported: the same state afterwards
            env.restore([1], [0], keep_accumulators=keep)
            env.import_states([2], rec, keep_accumulators=keep)
            for c in range(3):
                o, r, d = env.step(rl_actions(k + c, B))
                assert o[1].tobytes() == o[2].tobytes() and r[1] == r[2] and d[1] == d[2], (state, keep, c)
            assert_readouts(readouts(env, 2), readouts(env, 1), f"{state} keep {keep}")


SUBPROCESS = r"""
import sys
import numpy as np
from rlfluidcontrol_b200 import AFCCylinderBatch
path, out = sys.argv[1], sys.argv[2]
with AFCCylinderBatch(2, sensors=[("p", 100.0, 96.0)]) as env:
    env.import_states([1], open(path, "rb").read())
    res = {}
    for k in range(6):
        f, pr = env.update2(np.tile(np.float32([[0.4, 0.1]]), (2, 1)) if k == 1 else None, want_probes=True)
        res[f"f{k}"], res[f"pr{k}"], res[f"it{k}"] = f[1], pr[1], env.mg_iters()[1]
    ux, uy, p = env.get_fields(1)
    np.savez(out, ux=ux, uy=uy, p=p, t=env.t[1], dt=env.dt()[1], sensors=env.sensors()[1], **res)
"""


def test_across_processes(rlfc, tmp_path):
    with rlfc.AFCCylinderBatch(3, sensors=[("p", 100.0, 96.0)]) as env:
        warm(env)
        (tmp_path / "state.rec").write_bytes(env.export_states([2]))
        repo = Path(__file__).resolve().parents[1]
        pyenv = dict(os.environ, PYTHONPATH=str(repo) + os.pathsep + os.environ.get("PYTHONPATH", ""))
        res = subprocess.run([sys.executable, "-c", SUBPROCESS, str(tmp_path / "state.rec"), str(tmp_path / "out.npz")],
                             cwd=repo, env=pyenv, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        got = np.load(tmp_path / "out.npz")
        for k in range(6):
            f, pr = env.update2(np.tile(np.float32([[0.4, 0.1]]), (3, 1)) if k == 1 else None, want_probes=True)
            for nm, a in ((f"f{k}", f[2]), (f"pr{k}", pr[2]), (f"it{k}", env.mg_iters()[2])):
                assert got[nm].tobytes() == np.asarray(a).tobytes(), nm
        for nm, a in zip(("ux", "uy", "p"), env.get_fields(2)):
            assert_same(got[nm], a, nm)
        assert got["t"] == env.t[2] and got["dt"] == env.dt()[2]
        assert got["sensors"].tobytes() == env.sensors()[2].tobytes()


@pytest.mark.skipif(device_count() < 2, reason="needs 2 GPUs")
def test_across_devices(rlfc, tmp_path):
    torch = pytest.importorskip("torch")
    with rlfc.AFCCylinderBatch(2, device=0, **CONT) as a, rlfc.AFCCylinderBatch(2, device=1, **CONT) as b:
        warm(a)
        buf = torch.empty(a.record_bytes, dtype=torch.uint8, device="cuda:0")
        ids0 = torch.tensor([1], dtype=torch.int32, device="cuda:0")
        torch.cuda.synchronize(0)
        a.export_states_device(ids0.data_ptr(), 1, buf.data_ptr())
        torch.cuda.synchronize(0)
        buf1 = buf.to("cuda:1")
        ids1 = torch.tensor([0], dtype=torch.int32, device="cuda:1")
        torch.cuda.synchronize(1)
        b.import_states_device(ids1.data_ptr(), 1, buf1.data_ptr(), a.record_bytes)
        torch.cuda.synchronize(1)
        assert_readouts(readouts(b, 0), readouts(a, 1), "right after the import")
        for k in range(5):
            fa = a.update2(full(a, [0.5, 0.5]) if k == 1 else None)
            fb = b.update2(full(b, [0.5, 0.5]) if k == 1 else None)
            assert fa[1].tobytes() == fb[0].tobytes(), k
        assert_readouts(readouts(b, 0), readouts(a, 1), "after 5 steps")


# ---- corrupted records: refused by the device and the host imports, nothing changes ------------------------------------
def set_word(rec, offset, value, dtype="<u4", fix=True):
    rec = bytearray(rec)
    v = np.asarray(value, dtype=dtype).tobytes()
    rec[offset:offset + len(v)] = v
    if fix:
        rec[8:16] = np.uint64(records.checksum(rec)).tobytes()
    return bytes(rec)


def flip(rec, byte, bit=0):
    rec = bytearray(rec)
    rec[byte] ^= 1 << bit
    return bytes(rec)


def corruptions(rec, n, m, K):
    h = records.parse_record(rec)
    fld = 272 + 16 * K
    dt = h["scalars"]["dt"]
    return {
        "flip header field": (flip(rec, 20, 0), "checksum"),       # adaptive_dt: only the checksum covers it
        "flip scalar record": (flip(rec, 80 + 4 * 9, 5), "checksum"),
        "flip sensor table": (flip(rec, 272 + 4, 1), "checksum"),
        "flip sensor value": (flip(rec, 272 + 12 * K + 7, 6), "checksum"),
        "flip ux": (flip(rec, fld + 4 * (3 * m + 7), 0), "checksum"),
        "flip uy": (flip(rec, fld + 4 * n * m + 4 * (5 * m + 1), 7), "checksum"),
        "flip p ghost": (flip(rec, fld + 8 * n * m + 4 * (m - 1), 3), "checksum"),
        "checksum field": (flip(rec, 12, 4), "checksum"),
        "magic": (flip(rec, 0, 1), "magic"),
        "version": (set_word(rec, 16, 2), "version"),
        "length": (set_word(rec, 24, len(rec) + 16, "<u8"), "length"),
        "grid": (set_word(rec, 32, h["resolution"] + 1, "<i4"), "grid"),
        "tuple": (set_word(rec, 52, h["re"] + 1, "<i4"), "parameter tuple"),
        "fixed dt": (set_word(rec, 96, np.nextafter(dt, F(1)), "<f4"), "dt"),
    }


def test_device_and_host_rules(rlfc):
    torch = pytest.importorskip("torch")
    B = 4
    with rlfc.AFCCylinderBatch(B, sensors=SENS) as env:
        warm(env)
        rec0, rec1 = records.split_records(env.export_states([0, 1]), 2)
        rec0, rec1 = bytes(rec0), bytes(rec1)
        assert env.export_states([0, 1]) == rec0 + rec1
        size = len(rec0)
        state = [readouts(env, e) for e in range(B)]
        for what, (bad, check) in corruptions(rec0, env.n, env.m, len(SENS)).items():
            # host: all or nothing, the message names the record and the check
            with pytest.raises(rlfc.RlfcError, match=r"record 1 \(env id 2\): " + check):
                env.import_states([3, 2], rec1 + bad)
            # device: refused, flags bit 3
            d, ids = to_device(torch, bad), dev_ints(torch, [2])
            torch.cuda.synchronize()
            env.import_states_device(ids.data_ptr(), 1, d.data_ptr(), size)
            assert env.flags()[2] == 8, what
            for e in range(B):
                assert_readouts(readouts(env, e), dict(state[e], flags=8 if e == 2 else 0), f"{what}: env {e}")
        # an import that applies clears bit 3; ids out of range are skipped and the last in-range pair wins
        d, ids = to_device(torch, rec0 + rec0 + rec1 + rec0), dev_ints(torch, [7, 2, 2, -1])
        torch.cuda.synchronize()
        env.import_states_device(ids.data_ptr(), 4, d.data_ptr(), size)
        assert env.flags().tolist() == [0, 0, 0, 0]
        assert_readouts(readouts(env, 2), state[1], "env 2 <- record of env 1")
        for e in (0, 1, 3):
            assert_readouts(readouts(env, e), state[e], f"env {e} untouched")
        # an out-of-range export writes a record every import refuses
        out = torch.empty(2 * size, dtype=torch.uint8, device="cuda")
        ids = dev_ints(torch, [-1, B])
        torch.cuda.synchronize()
        env.export_states_device(ids.data_ptr(), 2, out.data_ptr())
        ids = dev_ints(torch, [3, 0])
        torch.cuda.synchronize()
        env.import_states_device(ids.data_ptr(), 2, out.data_ptr(), size)
        assert env.flags().tolist() == [8, 0, 0, 8]
        with pytest.raises(rlfc.RlfcError, match=r"record 0: magic"):
            env.import_states([1], out.cpu().numpy().tobytes()[:size])
        # host argument rules
        for ids_, msg in (([4], "env id 4 out of range"), ([1, 1], "env id 1 listed twice")):
            with pytest.raises(rlfc.RlfcError, match=msg):
                env.import_states(ids_, rec0 * len(ids_))
        with pytest.raises(rlfc.RlfcError, match="env id -1 out of range"):
            env.export_states([-1])
        with pytest.raises(rlfc.RlfcError, match="record_bytes"):
            env.import_states_device(0, 0, 0, size + 4)
    with rlfc.AFCCylinderBatch(2) as env:   # an adaptive record into a fixed-dt handle: only env's own dt passes
        with rlfc.AFCCylinderBatch(1, adaptive_dt=1) as ad:
            warm(ad, 3)
            rec = ad.export_states([0])
        assert records.parse_record(rec)["adaptive_dt"] == 1
        with pytest.raises(rlfc.RlfcError, match=r"record 0 \(env id 0\): dt"):
            env.import_states([0], rec)


def test_format(rlfc):
    torch = pytest.importorskip("torch")
    with rlfc.AFCCylinderBatch(3, sensors=SENS) as env:
        warm(env)
        env.update2(full(env, [0.2, 0.1]))
        blob = env.export_states([0, 1, 2])
        for e, r in enumerate(records.split_records(blob, 3)):
            h = records.parse_record(r)
            assert h["length"] == env.record_bytes == len(r) and h["n_sensors"] == len(SENS)
            assert (h["n"], h["m"], h["resolution"], h["adaptive_dt"]) == (env.n, env.m, 24, 0)
            for nm, a in zip(("ux", "uy", "p"), env.get_fields(e)):
                assert h[nm].tobytes() == a.tobytes(), nm
            sc = h["scalars"]
            assert sc["t"] == env.t[e] and sc["dt"] == env.dt()[e]
            assert sc["iters"].tolist() == env.mg_iters()[e].tolist()
            assert h["sensors"].tobytes() == env.sensors()[e].tobytes()
            assert [tuple(x) for x in h["sensor_table"].tolist()] == [(records_field(f), F(x), F(y)) for f, x, y in SENS]
            lib = rlfc.load_library()
            assert lib.rlfc_record_checksum(bytes(r), len(r)) == h["checksum"] == records.checksum(r)
    # environments in identical states export identical records
    with rlfc.AFCCylinderBatch(2) as env:
        env.update2(full(env, [0.3, 0.3]))
        a, b = records.split_records(env.export_states([0, 1]), 2)
        assert bytes(a) == bytes(b)
    # the sensor rule: values only under a byte-equal table
    with rlfc.AFCCylinderBatch(1, sensors=SENS) as s, rlfc.AFCCylinderBatch(1) as plain, \
            rlfc.AFCCylinderBatch(1, sensors=SENS[:2]) as other, rlfc.AFCCylinderBatch(1, sensors=SENS) as same:
        warm(s)
        for env in (other, same):
            env.update2()
        rec = s.export_states([0])
        keep = other.sensors().copy()
        plain.import_states([0], rec)
        other.import_states([0], rec)
        same.import_states([0], rec)
        assert other.sensors().tobytes() == keep.tobytes()
        assert same.sensors().tobytes() == s.sensors().tobytes()
        for env in (plain, other, same):
            assert_readouts(readouts(env, 0), readouts(s, 0), "sensor rule")
        s.update2(); plain.update2(); other.update2(); same.update2()
        assert_readouts(readouts(plain, 0), readouts(s, 0), "sensor rule, one step later")
        assert other.sensors()[0].tobytes() == s.sensors()[0, :2].tobytes()
        back = plain.export_states([0])           # no sensors -> a handle with sensors keeps its values
        assert records.parse_record(back)["n_sensors"] == 0
        before = same.sensors().copy()
        same.import_states([0], back)
        assert same.sensors().tobytes() == before.tobytes()
        d, ids = to_device(torch, back), dev_ints(torch, [0])
        torch.cuda.synchronize()
        same.import_states_device(ids.data_ptr(), 1, d.data_ptr(), len(back))
        assert same.flags()[0] == 0 and same.sensors().tobytes() == before.tobytes()


def records_field(name):
    return {"p": 0, "ux": 1, "uy": 2}[name]


@pytest.mark.skipif(device_count() < 2, reason="needs 2 GPUs")
def test_slab_mode_rejected(rlfc):
    with rlfc.AFCCylinderBatch(1, init_state=None, resolution=64, n_devices=2) as env:
        for call in (lambda: env.export_states([0]), lambda: env.import_states([0], bytes(env.record_bytes)),
                     lambda: env.export_states_device(0, 0, 0), lambda: env.import_states_device(0, 0, 0, env.record_bytes)):
            with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*slab mode"):
                call()
