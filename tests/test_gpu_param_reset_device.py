"""Device parameter resets (rlfc_env_reset_params_device): an environment reset into any parameter set on the device is
held to rlfc_env_reset_params with the same set and to a lone CPU-oracle environment built with it.  Bar: bit-exact (==),
as in test_gpu_param_sets.  Also: the device's sin / cos against the host's on every float they can receive."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from test_gpu_env_params import (DEFAULT, MIXED, PI, F, assert_fields, assert_hierarchy, hetero_actions, oracle_for,
                                 random_params, step_and_compare)
from test_gpu_param_sets import (NEW, assert_handles_equal, assert_readouts, device_ints, readouts, same_params,
                                 solver_steps_equal)
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu

HERE = Path(__file__).resolve().parent
TWO_PI = F(6.2831855)
# the arguments whose sin / cos lies within 4 double ulps of a float rounding midpoint
NEAR_MIDPOINT = {"sin": [0x3dcf5597, 0x3ef3830f], "cos": [0x39800000, 0x3c107fe6, 0x3a544395]}

# the edges of the valid range on the default grid, and a seeded spread over the ranges bench_env_params draws from
# (re = 1 with a t_step small enough for its viscosity: at dt = 0.18 its explicit diffusion diverges on the host as well)
EDGE_SETS = [dict(DEFAULT), dict(DEFAULT, dR=F(1.0)), dict(DEFAULT, dR=F(0.02)), dict(DEFAULT, gR=F(0.0)),
             dict(DEFAULT, theta=F(0.0)), dict(DEFAULT, theta=PI / F(2)), dict(DEFAULT, theta=-PI / F(2)),
             dict(DEFAULT, theta=TWO_PI), dict(DEFAULT, theta=-TWO_PI), dict(DEFAULT, re=1, t_step=F(0.0004)),
             dict(DEFAULT, re=100000), dict(DEFAULT, t_step=F(0.005)), dict(DEFAULT, t_step=F(0.01)), dict(DEFAULT, t_step=F(0.0025))]
SETS = EDGE_SETS + random_params(10, 77)
ABOVE_TWO_PI = np.nextafter(TWO_PI, F(np.inf))
# one set per rule of build_env_geometries, and the device's theta range
INVALID = [dict(DEFAULT, re=0), dict(DEFAULT, dR=F(0)), dict(DEFAULT, dR=F(1.5)), dict(DEFAULT, dR=F(np.nan)),
           dict(DEFAULT, gR=F(-0.1)), dict(DEFAULT, gR=F(np.inf)), dict(DEFAULT, theta=F(np.nan)),
           dict(DEFAULT, t_step=F(0)), dict(DEFAULT, t_step=F(np.inf)),
           dict(re=500, dR=F(0.5), gR=F(3.3), theta=F(1.5707964), t_step=F(0.0075)),   # the band reaches row n-2
           dict(DEFAULT, theta=ABOVE_TWO_PI), dict(DEFAULT, theta=-ABOVE_TWO_PI)]


def full(p):
    return {k: p.get(k, DEFAULT[k]) for k in DEFAULT}


def pack(torch, sets):
    """(n, 5) int32 on the device: re, then the bits of dR, gR, theta, t_step (rlfc_env_params, 20 bytes a set)."""
    sets = [full(p) for p in sets]
    re = torch.tensor([int(p["re"]) for p in sets], dtype=torch.int32)
    cols = [torch.from_numpy(np.array([p[k] for p in sets], F)).view(torch.int32) for k in ("dR", "gR", "theta", "t_step")]
    return torch.stack([re] + cols, 1).contiguous().cuda()


def device_reset(torch, env, ids, sets, reset_accumulators=False):
    d_ids, d_par = device_ints(torch, ids), pack(torch, sets)
    torch.cuda.synchronize()
    env.reset_params_device(d_ids.data_ptr(), d_par.data_ptr(), len(ids), reset_accumulators)
    env.running()                          # (synchronises the handle's stream while the arrays are alive)


# ---- 1. the device's sin / cos -----------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def trig():
    from rlfluidcontrol_b200 import build as _b
    src = HERE / "trig_dev.cu"
    hdrs = [_b.CSRC / h for h in ("geometry_device.cuh", "param_sets.cuh", "snapshot.cuh", "solver.h")]
    lib = HERE / "_build" / "libtrig_dev.so"
    if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
        lib.parent.mkdir(exist_ok=True)
        flags = [f for f in _b.NVCC_FLAGS if f not in ("-lineinfo",)]
        subprocess.run([_b.nvcc_path(), *flags, "-o", str(lib), str(src)], check=True, capture_output=True)
    L = C.CDLL(str(lib))
    L.trig_check.argtypes = [C.c_uint, C.c_uint, C.POINTER(C.c_longlong), C.POINTER(C.c_uint)]
    L.trig_at.argtypes = [C.c_float, C.POINTER(C.c_float)]
    return L


def test_trig_equals_host_on_every_float_up_to_two_pi(trig):
    """fsin_dev / fcos_dev against (float)std::sin / cos((double)x) on all ~2.2e9 floats of [-2 pi, 2 pi]."""
    hi = int(np.array(TWO_PI).view(np.uint32))
    for lo_b, hi_b in ((0, hi), (0x80000000, 0x80000000 | hi)):
        st, first = (C.c_longlong * 3)(), (C.c_uint * 8)()
        assert trig.trig_check(lo_b, hi_b, st, first) == 0
        bad = [hex(x) for x in first if x != 0xffffffff]
        assert st[0] == 0 and st[1] == 0, f"range {lo_b:#x}..{hi_b:#x}: {st[0]} sin / {st[1]} cos mismatches, e.g. {bad}"
        assert st[2] == hi_b - lo_b + 1
        for xs in NEAR_MIDPOINT.values():
            for x in xs:
                assert x <= hi, "the near-midpoint arguments lie in the range"
    out = (C.c_float * 4)()
    for x in sum(NEAR_MIDPOINT.values(), []):
        for s in (0, 0x80000000):
            assert trig.trig_at(F(np.uint32(x | s).view(F)), out) == 0
            assert np.array(out[:2], F).tobytes() == np.array(out[2:], F).tobytes(), hex(x | s)


# ---- 2. against rlfc_env_reset_params ------------------------------------------------------------------------------------

@pytest.mark.parametrize("envvar,value,adaptive", [(None, None, 0), ("RLFC_NO_GRAPH", "1", 0), ("RLFC_GROUPS", "3", 0),
                                                   (None, None, 1)])
def test_device_reset_equals_host_reset(rlfc, monkeypatch, envvar, value, adaptive):
    """Twin handles: A resets through rlfc_env_reset_params, B through rlfc_env_reset_params_device, with the edges of
    the valid range and a random spread.  Same read-outs (coefficients at every level, del, fields, dt, t, flags), then the
    same solver and RL steps under heterogeneous actions."""
    torch = pytest.importorskip("torch")
    if envvar:
        monkeypatch.setenv(envvar, value)
    B = 8
    acts = hetero_actions(B, 31)
    own = [MIXED[e % len(MIXED)] for e in range(B)]
    kw = dict(env_params=own, init_time=0.05, adaptive_dt=adaptive)
    with rlfc.AFCCylinderBatch(B, **kw) as a, rlfc.AFCCylinderBatch(B, **kw) as b:
        solver_steps_equal(a, b, 2, acts, "before: ")
        for r0 in range(0, len(SETS), B):
            sets = SETS[r0:r0 + B]
            ids = list(range(len(sets)))[::-1]
            a.reset(ids, params=sets, reset_accumulators=True)
            device_reset(torch, b, ids, sets, reset_accumulators=True)
            for e, p in zip(ids, sets):
                assert same_params(b, e, full(p)), (e, p)
            assert_handles_equal(a, b, range(B), f"sets {r0}: ")
            solver_steps_equal(a, b, 2, acts, f"sets {r0}: ")
            for k in range(2):
                oa, ra, da = a.step(acts * F(0.5 * (k + 1)))
                ob, rb, db = b.step(acts * F(0.5 * (k + 1)))
                assert_same(ob, oa, f"sets {r0} obs call {k}")
                assert_same(rb, ra, f"sets {r0} reward call {k}")
                assert (db == da).all()
            assert_handles_equal(a, b, range(B), f"sets {r0} end: ")


def test_device_reset_on_a_fine_grid(rlfc):
    """64 cells per diameter."""
    torch = pytest.importorskip("torch")
    kw = dict(resolution=64, x_lengths=4, y_lengths=2, init_state=None, init_time=-1.0)
    sets = [MIXED[1], NEW[0], dict(DEFAULT, theta=F(-1.0), t_step=F(0.005))]
    with rlfc.AFCCylinderBatch(3, env_params=[{}] * 3, **kw) as a, rlfc.AFCCylinderBatch(3, env_params=[{}] * 3, **kw) as b:
        solver_steps_equal(a, b, 2, hetero_actions(3, 2), "before: ")
        a.reset([0, 1, 2], params=sets)
        device_reset(torch, b, [0, 1, 2], sets)
        assert_handles_equal(a, b, range(3))
        solver_steps_equal(a, b, 3, hetero_actions(3, 5), "after: ")


# ---- 3. against the oracle -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("adaptive", [0, 1])
def test_device_reset_against_oracle(rlfc, oracle, init_state, adaptive):
    """Skipped (-1), out-of-range and duplicated pairs: the skipped environments are untouched, the last pair wins, and
    every environment then matches a lone oracle built with its final set."""
    torch = pytest.importorskip("torch")
    own = [MIXED[0], MIXED[1], MIXED[3], MIXED[4], MIXED[5], MIXED[2]]
    B = len(own)
    acts = hetero_actions(B, 9)
    refs = {e: oracle_for(oracle, init_state, p) for e, p in enumerate(own)}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    envs = [0, 1, 2, 3, 2, -1, 5, 7, 5, 6]
    sets = [NEW[2], NEW[0], NEW[1], EDGE_SETS[7], EDGE_SETS[13], NEW[0], EDGE_SETS[2], NEW[1], EDGE_SETS[10], NEW[0]]
    applied = {0: NEW[2], 1: NEW[0], 2: EDGE_SETS[13], 3: EDGE_SETS[7], 5: EDGE_SETS[10]}
    with rlfc.AFCCylinderBatch(B, env_params=own, adaptive_dt=adaptive) as env:
        step_and_compare(env, refs, 3, acts, adaptive=bool(adaptive), tag="before: ")
        before = {e: readouts(env, e) for e in range(B) if e not in applied}
        device_reset(torch, env, envs, sets)
        for e, want in before.items():
            assert_readouts(readouts(env, e), want, f"skipped env {e} ")
        for e, p in applied.items():
            assert same_params(env, e, full(p)), e
            assert env.t[e] == 0 and env.dt()[e] == F(full(p)["t_step"]) * F(24)
            refs[e] = oracle_for(oracle, init_state, full(p))
            assert_hierarchy(oracle, env, e, refs[e])
        step_and_compare(env, refs, 20, adaptive=bool(adaptive), tag="after: ")
        assert_fields(env, refs)
        for e in applied:
            assert_hierarchy(oracle, env, e, refs[e])
        assert (env.flags() == 0).all()


# ---- 4. refusals -------------------------------------------------------------------------------------------------------------

def test_invalid_sets_change_nothing(rlfc):
    """Each invalid class leaves its environment unchanged bit for bit with flags bit 2, while the call's other pair applies;
    a last invalid pair beats an earlier valid one; a later valid reset clears bit 2."""
    torch = pytest.importorskip("torch")
    with rlfc.AFCCylinderBatch(3, env_params=[MIXED[0], MIXED[3], MIXED[4]]) as env:
        env.update2(hetero_actions(3, 8))
        for k, bad in enumerate(INVALID):
            before = readouts(env, 1)
            good = NEW[k % len(NEW)]
            device_reset(torch, env, [0, 1], [good, bad])
            assert env.flags()[1] == 4, bad
            assert_readouts(readouts(env, 1), dict(before, flags=4), f"invalid {bad}: ")
            assert same_params(env, 0, good) and env.t[0] == 0 and env.flags()[0] == 0
            env.update2()
        before = readouts(env, 2)
        device_reset(torch, env, [2, 2], [NEW[1], INVALID[4]])
        assert_readouts(readouts(env, 2), dict(before, flags=4), "last pair invalid: ")
        device_reset(torch, env, [2], [NEW[1]])
        assert env.flags()[2] == 0 and same_params(env, 2, NEW[1])
        # rejected calls
        d = device_ints(torch, [0])
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*bad pair count"):
            env.reset_params_device(d.data_ptr(), d.data_ptr(), -1)
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*null argument"):
            env.reset_params_device(0, d.data_ptr(), 1)
        env.reset_params_device(0, 0, 0)       # nothing to do
    with rlfc.AFCCylinderBatch(1) as env:
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*needs a handle created with env_params or param_sets"):
            env.reset_params_device(0, 0, 0)


# ---- 5. interplay -----------------------------------------------------------------------------------------------------------

def test_library_and_arbitrary_sets_alternate(rlfc, oracle, init_state):
    torch = pytest.importorskip("torch")
    lib = [NEW[0], MIXED[5]]
    with rlfc.AFCCylinderBatch(3, param_sets=lib) as env:
        env.update2(hetero_actions(3, 4))
        d_e, d_s = device_ints(torch, [0]), device_ints(torch, [1])
        torch.cuda.synchronize()
        env.reset_sets_device(d_e.data_ptr(), d_s.data_ptr(), 1)
        assert same_params(env, 0, lib[1])
        p = SETS[-1]
        device_reset(torch, env, [0], [p])
        assert same_params(env, 0, full(p))
        refs = {0: oracle_for(oracle, init_state, full(p))}
        assert_hierarchy(oracle, env, 0, refs[0])
        step_and_compare(env, refs, 3, tag="arbitrary: ")
        env.reset_sets_device(d_e.data_ptr(), d_s.data_ptr(), 1)
        refs = {0: oracle_for(oracle, init_state, lib[1])}
        assert same_params(env, 0, lib[1])
        assert_hierarchy(oracle, env, 0, refs[0])
        step_and_compare(env, refs, 3, tag="library again: ")


def test_host_copies_follow_a_device_reset(rlfc, tmp_path):
    """get_params, reset, load_bdim's dt check and host restore headers read the set a device reset gave, without a sync."""
    torch = pytest.importorskip("torch")
    p = dict(NEW[1], t_step=F(0.005))
    with rlfc.AFCCylinderBatch(3, env_params=[MIXED[0], MIXED[3], MIXED[4]], n_snapshots=2) as env:
        env.update2(hetero_actions(3, 6))
        d_ids, d_par = device_ints(torch, [1]), pack(torch, [p])
        torch.cuda.synchronize()
        env.reset_params_device(d_ids.data_ptr(), d_par.data_ptr(), 1)
        assert same_params(env, 1, p)
        env.update2()
        d_par2 = pack(torch, [p])
        torch.cuda.synchronize()
        env.reset_params_device(d_ids.data_ptr(), d_par2.data_ptr(), 1)
        env.update2()
        env.reset([1])                         # rlfc_env_reset keeps the new set's dt
        assert env.dt()[1] == F(0.005) * F(24) and env.t[1] == 0
        env.update2()
        path = tmp_path / "dev.bdim"
        env.save_bdim(1, path)
        assert F(path.read_text().splitlines()[1]) == F(0.005) * F(24)
        d_par3 = pack(torch, [dict(MIXED[0], t_step=F(0.01))])
        torch.cuda.synchronize()
        env.reset_params_device(d_ids.data_ptr(), d_par3.data_ptr(), 1)
        with pytest.raises(rlfc.RlfcError, match=r"\(-4\).*does not match"):
            env.load_bdim(1, path)
        device_reset(torch, env, [1], [p])
        env.load_bdim(1, path)
        # host restore headers: a slot of env 1's tuple goes into env 0 once a device reset gave env 0 that tuple
        env.snapshot([1], [0])
        with pytest.raises(rlfc.RlfcError, match="another parameter set"):
            env.restore([0], [0])
        d0, d_par4 = device_ints(torch, [0]), pack(torch, [p])
        torch.cuda.synchronize()
        env.reset_params_device(d0.data_ptr(), d_par4.data_ptr(), 1)
        env.restore([0], [0])
        assert env.flags()[0] == 0


def test_snapshots_across_a_parameter_change(rlfc):
    torch = pytest.importorskip("torch")
    with rlfc.AFCCylinderBatch(2, env_params=[MIXED[0], MIXED[2]], n_snapshots=1) as env:
        env.update2(hetero_actions(2, 3))
        env.snapshot([0], [0])
        device_reset(torch, env, [0], [NEW[0]])
        d = device_ints(torch, [0])
        torch.cuda.synchronize()
        before = readouts(env, 0)
        env.restore_device(d.data_ptr(), d.data_ptr(), 1)          # another tuple: refused
        assert env.flags()[0] == 2
        assert_readouts(readouts(env, 0), dict(before, flags=2), "refused restore: ")
        device_reset(torch, env, [0], [MIXED[0]])                  # the slot's tuple again: accepted
        env.restore_device(d.data_ptr(), d.data_ptr(), 1)
        assert env.flags()[0] == 0


def test_sensors_are_left_alone(rlfc):
    torch = pytest.importorskip("torch")
    sensors = [("p", 150.0, 96.0), ("ux", 200.5, 90.25), ("uy", 300.0, 100.0)]
    with rlfc.AFCCylinderBatch(2, env_params=[{}, {}], sensors=sensors) as env:
        env.update2(hetero_actions(2, 3))
        before = env.sensors()
        device_reset(torch, env, [0, 1], [NEW[0], NEW[2]])
        assert_same(env.sensors(), before, "sensors")
        assert env.t.tolist() == [0, 0]


def test_rl_step_after_a_device_reset_to_half_the_t_step(rlfc):
    """rlfc_env_step bounds its rounds by the smallest t_step, including one a device reset gave."""
    torch = pytest.importorskip("torch")
    init_time = 0.3
    with rlfc.AFCCylinderBatch(2, env_params=[{}, {}], init_time=init_time) as env:
        d_ids, d_par = device_ints(torch, [1]), pack(torch, [dict(t_step=F(0.00375))])
        torch.cuda.synchronize()
        env.reset_params_device(d_ids.data_ptr(), d_par.data_ptr(), 1, reset_accumulators=True)
        env.reset([0], reset_accumulators=True)
        obs, rew, done = env.step(np.zeros((2, 2), F))
        assert env.running() == 0 and not done.any()
        t = env.t
        assert t[0] > init_time and t[1] > init_time and np.isfinite(obs).all()


# ---- 6. a device-only loop -----------------------------------------------------------------------------------------------

def test_device_only_loop(rlfc):
    """step_device + reset_params_device(where(done, arange, -1), fresh random sets) on the handle's stream against a
    second handle driven through the same schedule with host rlfc_env_reset_params."""
    torch = pytest.importorskip("torch")
    B, calls = 6, 14
    kw = dict(init_time=-1.0, episode_time=0.4)
    rng = np.random.default_rng(11)
    schedule = [random_params(B, 100 + k) for k in range(calls)]
    acts = np.clip(rng.normal(0, 0.6, size=(calls, B, 2)), -1, 1).astype(F)
    stream = torch.cuda.Stream()
    resets = 0
    with rlfc.AFCCylinderBatch(B, env_params=[{}] * B, stream=stream.cuda_stream, **kw) as dev, \
            rlfc.AFCCylinderBatch(B, env_params=[{}] * B, **kw) as host:
        ar = device_ints(torch, np.arange(B))
        d_sched = [pack(torch, s) for s in schedule]
        d_acts = torch.from_numpy(acts).cuda()
        obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
        rew = torch.empty(B, dtype=torch.float32, device="cuda")
        done = torch.zeros(B, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        for k in range(calls):
            with torch.cuda.stream(stream):
                dev.step_device(d_acts[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr())
                ids = torch.where(done != 0, ar, torch.full_like(ar, -1))
                dev.reset_params_device(ids.data_ptr(), d_sched[k].data_ptr(), B, reset_accumulators=True)
                got = (obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy())
            o, r, dn = host.step(acts[k])
            assert_same(got[0], o, f"obs call {k}")
            assert_same(got[1], r, f"reward call {k}")
            assert (got[2] == dn).all(), f"done call {k}"
            fin = np.flatnonzero(dn)
            if len(fin):
                resets += len(fin)
                host.reset(fin, params=[schedule[k][e] for e in fin], reset_accumulators=True)
        stream.synchronize()
        assert resets >= B, "too few episode ends for the test to mean anything"
        assert (dev.params() == host.params()).all()
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), dev.get_fields(e), host.get_fields(e)):
                assert_same(x, y, f"{nm} env {e}")
            for nm in ("del.x", "del.y", "c.x", "c.y"):
                assert_same(dev.get_coeffs(e, nm), host.get_coeffs(e, nm), f"{nm} env {e}")


# ---- 7. nothing changes without the call ---------------------------------------------------------------------------------

def test_launches_per_step_unchanged(rlfc):
    torch = pytest.importorskip("torch")
    with rlfc.AFCCylinderBatch(2, env_params=[{}, {}]) as a, rlfc.AFCCylinderBatch(2, env_params=[{}, {}]) as b:
        device_reset(torch, b, [1], [NEW[0]])
        a.update2(); b.update2()
        la, lb = a.launch_count, b.launch_count
        a.update2(); b.update2()
        assert a.launch_count - la == b.launch_count - lb
