"""Flow sensors (rlfc_config.sensors, rlfc_env_get_sensors[_device]): every value is the reference's Field.linear of its field
at its point on the state the environment's next solver step starts from, on every execution path, through RL steps and
snapshots; and a handle with sensors computes exactly what a handle without them does.  Bar: every float compared with ==,
as in test_gpu_parity."""
import numpy as np
import pytest

from test_gpu_parity import assert_same, make_oracle

pytestmark = pytest.mark.gpu

F = np.float32
FIELDS = ("p", "ux", "uy")
BTYPE = {"p": 0, "ux": 1, "uy": 2}


def save_scalar_points(res, xl, yl):
    """The 32 SaveScalar probe points (SaveScalar.pde:61-72), in the reference's float arithmetic."""
    r, cx, cy = F(res), F(xl) * F(res) / F(4), F(yl) * F(res) / F(2)
    pts = []
    for i in range(32):
        a = F(i) / F(32) * F(3.1415927) * F(2)
        pts.append((float(F(np.cos(np.float64(a))) * r / F(2) + cx), float(F(np.sin(np.float64(a))) * r / F(2) + cy)))
    return pts


def sensor_set(res=24, xl=16, yl=8, seed=7):
    """A few hundred sensors of all three fields, K not a multiple of 128: the SaveScalar points as p; exact nodes of each
    btype (Field.linear's s == t == 0 branch); points outside the domain on every side and corner (clamped; for u.x / u.y on
    the far side the shift gives s or t = 1); points inside the main and the control cylinders; random wake points."""
    n, m = xl * res + 2, yl * res + 2
    s = [("p", x, y) for x, y in save_scalar_points(res, xl, yl)]
    for k, l in [(5, 7), (n // 2, m // 3), (n - 3, m - 3), (n - 2, m - 2)]:
        s += [("p", k, l), ("ux", k - 0.5, l), ("uy", k, l - 0.5)]
    outside = [(-5.0, m / 2), (n + 40.0, m / 2 + 0.3), (n / 2, -3.0), (n / 2 + 0.7, m + 17.0),
               (-1e6, -1e6), (1e6, 1e6), (-1e6, 1e6), (1e6, -1e6)]
    s += [(f, x, y) for x, y in outside for f in FIELDS]
    cx, cy = xl * res / 4, yl * res / 2
    r = res / 2 + 0.2 * res + 0.125 * res / 2                      # control-cylinder centres at theta = pi/3
    inside = [(cx, cy), (cx + 3.3, cy - 2.1), (cx + r * 0.5, cy - r * 0.866), (cx + r * 0.5 + 0.4, cy + r * 0.866)]
    s += [(f, x, y) for x, y in inside for f in FIELDS]
    rng = np.random.default_rng(seed)
    wake = 299 - len(s)
    xs, ys = rng.uniform(cx + 13, n - 2, wake), rng.uniform(1, m - 2, wake)
    s += [(FIELDS[i % 3], float(x), float(y)) for i, (x, y) in enumerate(zip(xs, ys))]
    assert len(s) == 299 and len(s) % 128
    return s


SENSORS = sensor_set()


def expected(oracle, fields, sensors):
    """Field.linear (Field.pde:175-190, the oracle's restatement) of each sensor's field on (ux, uy, p)."""
    ux, uy, p = fields
    n, m = p.shape
    fl = {"p": oracle.Field(n, m, 0, values=p), "ux": oracle.Field(n, m, 1, values=ux), "uy": oracle.Field(n, m, 2, values=uy)}
    return np.array([fl[f].linear(x, y) for f, x, y in sensors], F)


def assert_sensors_match_fields(oracle, env, what, sensors=SENSORS):
    got = env.sensors()
    assert got.shape == (env.n_envs, len(sensors))
    for e in range(env.n_envs):
        assert_same(got[e], expected(oracle, env.get_fields(e), sensors), f"{what}: env {e}")
    return got


def hetero_actions(B, seed):
    return np.clip(np.random.default_rng(seed).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)


# ---- 1. oracle parity over solver steps ------------------------------------------------------------------------------
def test_oracle_parity_update2(rlfc, oracle, init_state):
    B = 3
    acts = [hetero_actions(B, s) for s in (1, 2, 3)]
    for a in acts:
        a[0] = 0                                                   # env 0: uncontrolled
    refs = [make_oracle(oracle, init_state) for _ in range(B)]
    pidx = list(range(32))                                         # the p sensors at the SaveScalar points
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS) as env:
        assert env.n_sensors == len(SENSORS)
        for k in range(100):
            a = acts[k // 40] if k % 40 == 0 else None
            _, probes = env.update2(a, want_probes=True)
            got = env.sensors()
            for e, ref in enumerate(refs):
                if a is not None:
                    ref.set_xi(*a[e])
                ref.update2()
                assert_same(got[e], expected(oracle, ref.get_state(), SENSORS), f"step {k} env {e}")
            assert np.array_equal(got[:, pidx], probes), f"step {k}: p sensors at the SaveScalar points vs probes"


# ---- 2. RL steps -----------------------------------------------------------------------------------------------------
def test_rl_step_emission(rlfc, oracle, init_state):
    """Default init_time (the uncontrolled start and the catch-up rounds): after every call each environment holds the
    sample of the step that completed its window, the oracle driver's state at its emission."""
    B = 2
    acts = [np.array([[0, 0], [0, 0]], F), np.array([[0.6, -0.4], [-0.9, 0.2]], F), np.array([[0.1, 0.8], [0.5, -0.5]], F)]
    refs = [make_oracle(oracle, init_state) for _ in range(B)]
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS) as env:
        for k, a in enumerate(acts):
            obs, _, _ = env.step(a)
            got = assert_sensors_match_fields(oracle, env, f"call {k}")
            for e, ref in enumerate(refs):
                ref.set_xi(*a[e])
                o = None
                while o is None:
                    o = ref.driver_step(init_time=1.0)
                assert_same(obs[e], np.array(o, F), f"call {k} env {e}: obs")
                assert_same(got[e], expected(oracle, ref.get_state(), SENSORS), f"call {k} env {e}: oracle at emission")


def test_rl_step_episode_over_keeps_sensors(rlfc, oracle):
    B = 2
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS, init_time=0.2, episode_time=0.6) as env:
        last, k = None, 0
        while True:
            _, _, done = env.step(hetero_actions(B, k))
            got = assert_sensors_match_fields(oracle, env, f"call {k}")
            k += 1
            if done.all():
                break
            last = got
        assert not np.array_equal(got, last)                       # the step that ended the episode was sampled
        for j in range(2):
            env.step(hetero_actions(B, 100 + j))
            assert_same(env.sensors(), got, f"finished environments, call {j}")


def test_rl_step_device(rlfc, oracle):
    """step_device + sensors_device == step + sensors(); an environment still running after a device round holds its latest
    step's sample."""
    torch = pytest.importorskip("torch")
    B, K = 3, len(SENSORS)
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS) as a, rlfc.AFCCylinderBatch(B, sensors=SENSORS) as b:
        act = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        obs = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        sens = torch.full((B, K), float("nan"), dtype=torch.float32, device="cuda")
        for k in range(3):
            h = hetero_actions(B, 40 + k) if k else np.zeros((B, 2), F)
            act.copy_(torch.from_numpy(h))
            torch.cuda.synchronize()
            rounds = 0
            while True:
                a.step_device(act.data_ptr(), obs.data_ptr())
                a.sensors_device(sens.data_ptr())
                torch.cuda.synchronize()
                rounds += 1
                running = a.running()
                assert_same(sens.cpu().numpy(), assert_sensors_match_fields(oracle, a, f"call {k} round {rounds}"),
                            f"call {k} round {rounds}: sensors_device vs sensors")
                if running == 0:
                    break
            assert rounds > 1 or k > 0, "the first call must catch up over several rounds"
            ob, _, _ = b.step(h)
            assert_same(obs.cpu().numpy(), ob, f"call {k}: obs")
            assert_same(sens.cpu().numpy(), b.sensors(), f"call {k}: device vs host variant")


# ---- 3. execution paths ------------------------------------------------------------------------------------------------
MIXED = [dict(), dict(re=300, dR=F(0.2), gR=F(0.3), theta=F(0.9), t_step=F(0.005)), dict(re=100), dict(), dict(theta=F(1.2)),
         dict(t_step=F(0.005))]

PATHS = {
    "no_graph": (dict(), ("RLFC_NO_GRAPH", "1")),
    "groups3": (dict(), ("RLFC_GROUPS", "3")),
    "resid_tile": (dict(), ("RLFC_RESID", "tile")),
    "psum_serial": (dict(), ("RLFC_PSUM", "serial")),
    "smoother_chain": (dict(), ("RLFC_SMOOTHER", "chain")),
    "smoother_wave": (dict(), ("RLFC_SMOOTHER", "wave")),
    "adaptive": (dict(adaptive_dt=1), None),
    "env_params": (dict(env_params=MIXED), None),
    "wide_grid": (dict(n_envs=2, resolution=64, init_state=None), None),
}


@pytest.mark.parametrize("case", list(PATHS))
def test_execution_paths(rlfc, oracle, monkeypatch, case):
    kw, envvar = PATHS[case]
    if envvar:
        monkeypatch.setenv(*envvar)
    kw = dict(kw)
    B = kw.pop("n_envs", 6)
    sensors = sensor_set(res=kw.get("resolution", 24))
    with rlfc.AFCCylinderBatch(B, sensors=sensors, **kw) as env:
        for k in range(6):
            env.update2(hetero_actions(B, k) if k % 3 == 0 else None)
            assert_sensors_match_fields(oracle, env, f"{case} step {k}", sensors)


# ---- 4. no perturbation -------------------------------------------------------------------------------------------------
def test_sensors_change_nothing_else(rlfc, monkeypatch):
    monkeypatch.setenv("RLFC_GROUPS", "2")
    B = 4
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS) as a, rlfc.AFCCylinderBatch(B) as b:
        assert b.n_sensors == 0
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*n_sensors = 0"):
            b.sensors()
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*n_sensors = 0"):
            b.sensors_device(1)
        for k in range(3):
            h = hetero_actions(B, k) if k else np.zeros((B, 2), F)
            for x, y, nm in zip(a.step(h), b.step(h), ("obs", "reward", "done")):
                assert_same(x, y, f"call {k}: {nm}")
        la, lb = a.launch_count, b.launch_count
        steps = 5
        for k in range(steps):
            fa, pa = a.update2(hetero_actions(B, 10 + k) if k == 0 else None, want_probes=True)
            fb, pb = b.update2(hetero_actions(B, 10 + k) if k == 0 else None, want_probes=True)
            assert_same(fa, fb, f"step {k}: force")
            assert_same(pa, pb, f"step {k}: probes")
        assert (a.launch_count - la) - (b.launch_count - lb) == 2 * steps, "one k_sensors launch per group and solver step"
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), a.get_fields(e), b.get_fields(e)):
                assert_same(x, y, f"env {e}: {nm}")
        for nm in ("t", "dt", "mg_iters"):
            x, y = getattr(a, nm), getattr(b, nm)
            x, y = (x(), y()) if callable(x) else (x, y)
            assert np.array_equal(x, y), nm


# ---- 5. snapshots ---------------------------------------------------------------------------------------------------------
def test_snapshots_carry_sensors(rlfc):
    torch = pytest.importorskip("torch")
    B = 4
    with rlfc.AFCCylinderBatch(B, sensors=SENSORS, n_snapshots=2) as env:
        for k in range(3):
            env.update2(hetero_actions(B, k) if k == 0 else None)
        env.snapshot([0], [0])
        at_snap = env.sensors()[0].copy()
        after = []
        for _ in range(3):
            env.update2()
            after.append(env.sensors()[0].copy())
        before = env.sensors()
        # a skipped device restore (slot 1 never written; a pair with -1) leaves the destination's sensors as they are
        e_ = torch.tensor([2, -1], dtype=torch.int32, device="cuda")
        s_ = torch.tensor([1, 0], dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        env.restore_device(e_.data_ptr(), s_.data_ptr(), 2)
        assert env.flags().tolist() == [0, 0, 2, 0]
        assert_same(env.sensors(), before, "after the skipped restores")
        # keep_accumulators does not concern sensors: they come with the state
        env.restore([1], [0], keep_accumulators=True)
        env.restore([0, 3], [0, 0])
        got = env.sensors()
        for e in (0, 1, 3):
            assert_same(got[e], at_snap, f"env {e} right after the restore")
        assert_same(got[2], before[2], "env 2 is not restored")
        for k, want in enumerate(after):
            env.update2()
            got = env.sensors()
            for e in (0, 1, 3):
                assert_same(got[e], want, f"step {k} env {e} after the restore")
