"""GPU parity tests: the CUDA path, called through the C ABI (librlfc.so), against the CPU oracle on
the same seeded inputs.  Bar: bit-exact (==) on every float the path produces -- fields incl. ghost
cells, raw forces, probes, observations.  (-0.0 == 0.0 is accepted; NaNs are not.)"""
import numpy as np
import pytest

from conftest import config1_actions

pytestmark = pytest.mark.gpu


def assert_same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert not np.isnan(a).any(), f"{what}: NaN in device result"
    if not np.array_equal(a, b):
        bad = np.argwhere(a != b)
        k = tuple(bad[0])
        raise AssertionError(f"{what}: {len(bad)} of {a.size} values differ; first at {k}: gpu={a[k]!r} oracle={b[k]!r} "
                             f"max|diff|={np.abs(a.astype(np.float64) - b.astype(np.float64)).max():.3e}")


def make_oracle(oracle, init_state, **kw):
    e = oracle.OracleEnv(literal=False, **kw)
    if init_state is not None:
        e.set_state(init_state["ux"], init_state["uy"], init_state["p"])
    return e


def test_single_env_zero_action_three_steps(rlfc, oracle, init_state):
    ref = make_oracle(oracle, init_state)
    with rlfc.AFCCylinderBatch(1) as env:
        for k in range(3):
            f, pr = env.update2(want_probes=True)
            ref.update2()
            assert_same(f[0], np.array(ref.force(), np.float32), f"force step {k}")
            assert_same(pr[0], ref.probes(32), f"probes step {k}")
            assert tuple(env.mg_iters()[0]) == ref.mg_iters()
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(0), ref.get_state()):
            assert_same(a, b, nm)


def test_survey_drift_values(rlfc):
    """SURVEY 8c restatement-derived values: raw force of the first three steps from init.bdim."""
    with rlfc.AFCCylinderBatch(1) as env:
        f = [env.update2()[0].copy() for _ in range(3)]
    expect = [(13.6044025, 0.103305936), (13.6054707, 0.104807034), (13.6061077, 0.10624747)]
    for got, exp in zip(f, expect):
        assert got[0] == np.float32(exp[0]) and got[1] == np.float32(exp[1])


def test_hundred_steps_with_action(rlfc, oracle, init_state):
    """north_star: u, p relative L2 <= 1e-4 after 100 steps -- here required to be exactly equal."""
    ref = make_oracle(oracle, init_state)
    ref.set_xi(0.5, -0.3)
    act = np.array([[0.5, -0.3]], np.float32)
    with rlfc.AFCCylinderBatch(1) as env:
        for k in range(100):
            f = env.update2(act if k == 0 else None)
            ref.update2()
            assert_same(f[0], np.array(ref.force(), np.float32), f"force step {k}")
        ux, uy, p = env.get_fields(0)
    rux, ruy, rp = ref.get_state()
    assert_same(ux, rux, "ux"); assert_same(uy, ruy, "uy"); assert_same(p, rp, "p")
    n2 = lambda a: float(np.sqrt(np.sum(a.astype(np.float64) ** 2)))
    assert abs(n2(ux) - 286.21613) < 1e-4 and abs(n2(uy) - 51.1349241) < 1e-5 and abs(n2(p) - 47.1899691) < 1e-5


def test_batch_heterogeneous_actions(rlfc, oracle, init_state):
    """Every env of a batch evolves exactly like a lone oracle env fed the same actions."""
    B = 6
    rng = np.random.default_rng(1234)
    acts = np.clip(rng.normal(0, 0.6, size=(3, B, 2)), -1, 1).astype(np.float32)
    acts[:, 0, :] = 0  # env 0: uncontrolled
    refs = {e: make_oracle(oracle, init_state) for e in (0, 1, B - 1)}
    with rlfc.AFCCylinderBatch(B) as env:
        for k in range(3):
            for s in range(4):
                f = env.update2(acts[k] if s == 0 else None)
                for e, ref in refs.items():
                    if s == 0:
                        ref.set_xi(*acts[k, e])
                    ref.update2()
                    assert_same(f[e], np.array(ref.force(), np.float32), f"force env {e} step {k}.{s}")
        for e, ref in refs.items():
            for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(e), ref.get_state()):
                assert_same(a, b, f"{nm} env {e}")


def test_env_step_observations_config1(rlfc, oracle, init_state):
    """rlfc_env_step == 16 frames of clientCFD.draw(): (Cl, Cd) incl. the carry-over quirk, reward, done."""
    ref = make_oracle(oracle, init_state)
    with rlfc.AFCCylinderBatch(2, init_time=-1.0) as env:
        for k in range(4):
            a = config1_actions(k)
            obs, rew, done = env.step(np.stack([a, np.zeros(2, np.float32)]))
            o = ref.env_step(a)
            assert_same(obs[0], np.array(o, np.float32), f"obs step {k}")
            assert abs(float(rew[0]) - oracle.reference_reward(o[1], a)) < 1e-6
            assert done.tolist() == [0, 0]
    # first uncontrolled observation from init.bdim (SURVEY 8c): env 1 saw zero actions throughout


def test_first_observation_value(rlfc):
    with rlfc.AFCCylinderBatch(1, init_time=-1.0) as env:
        obs, _, _ = env.step(np.zeros((1, 2), np.float32))
    assert abs(float(obs[0, 0]) - 0.009605) < 5e-7 and abs(float(obs[0, 1]) - 1.133926) < 5e-7


def test_uniform_start_mg_iterations(rlfc, oracle):
    """Impulsive start (no checkpoint): the data-dependent MG loop takes several iterations at first;
    iteration counts and fields must match the oracle."""
    ref = make_oracle(oracle, None)
    with rlfc.AFCCylinderBatch(2, init_state=None) as env:
        its = []
        for k in range(3):
            f = env.update2()
            ref.update2()
            assert tuple(env.mg_iters()[1]) == ref.mg_iters()
            its.append(ref.mg_iters())
            assert_same(f[1], np.array(ref.force(), np.float32), f"force step {k}")
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(1), ref.get_state()):
            assert_same(a, b, nm)
    assert max(max(i) for i in its) > 1, "expected more than one MG iteration from an impulsive start"


def test_reset_and_field_roundtrip(rlfc, init_state, tmp_path):
    with rlfc.AFCCylinderBatch(3) as env:
        f0 = env.update2().copy()
        env.update2()
        env.reset([1])
        ux, uy, p = env.get_fields(1)
        assert_same(ux, init_state["ux"], "ux after reset"); assert_same(p, init_state["p"], "p after reset")
        assert env.t[1] == 0 and env.t[0] > 0
        env.reset()
        f1 = env.update2()
        assert_same(f1, f0, "force after full reset")
        # BDIM.write / BDIM.resume text round trip
        path = tmp_path / "ck.bdim"
        env.save_bdim(0, path)
        a = env.get_fields(0)
        env.load_bdim(2, path)
        b = env.get_fields(2)
        for nm, x, y in zip(("ux", "uy", "p"), a, b):
            assert_same(y, x, f"{nm} text checkpoint round trip")
        lines = path.read_text().splitlines()
        assert len(lines) == 2 + env.n * env.m and lines[2].count(",") == 2
        # BDIM.t round trip: resume sets t = line 0, every solver step adds dt (BDIM.pde:106,242); one step was taken
        t_file = np.float32(lines[0])
        assert t_file == np.float32(np.float32(init_state["t"]) + np.float32(init_state["dt"]))
        env.update2()
        env.save_bdim(2, path)                       # env 2 resumed from the file: its clock continues from the file's
        assert np.float32(path.read_text().splitlines()[0]) == np.float32(t_file + np.float32(init_state["dt"]))
        # a checkpoint of another grid is rejected, not reinterpreted
        bad = tmp_path / "bad.bdim"
        bad.write_text("\n".join(lines + ["1.0, 0.0, 0.0"]) + "\n")
        with pytest.raises(rlfc.RlfcError):
            env.load_bdim(0, bad)


# (resolution, x_lengths, y_lengths) besides the default (24, 16, 8); tests/test_gpu_shapes.py holds the ragged ones
OTHER_GRIDS = [(16, 16, 8), (8, 16, 8), (12, 8, 4), (24, 8, 4)]


@pytest.mark.parametrize("resolution,xl,yl", OTHER_GRIDS)
def test_other_grids(rlfc, oracle, resolution, xl, yl):
    """Other AFCCylinder grids (different columns-per-lane of the row smoother, different MG depths): impulsive
    start, non-zero actions, every float equal to the oracle's."""
    ref = oracle.OracleEnv(literal=False, resolution=resolution, xLengths=xl, yLengths=yl)
    ref.set_xi(0.4, -0.7)
    act = np.array([[0.4, -0.7], [0.0, 0.0]], np.float32)
    with rlfc.AFCCylinderBatch(2, init_state=None, resolution=resolution, x_lengths=xl, y_lengths=yl) as env:
        assert (env.n, env.m) == (ref.n, ref.m)
        for k in range(4):
            f = env.update2(act if k == 0 else None)
            ref.update2()
            assert_same(f[0], np.array(ref.force(), np.float32), f"force step {k}")
            assert tuple(env.mg_iters()[0]) == ref.mg_iters()
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(0), ref.get_state()):
            assert_same(a, b, nm)


@pytest.mark.parametrize("envvar,value", [("RLFC_SMOOTHER", "wave"), ("RLFC_SMOOTHER", "chain"),
                                          ("RLFC_NO_GRAPH", "1"),
                                          ("RLFC_GROUPS", "3"), ("RLFC_GROUPS", "4"), ("RLFC_FAST_BC", "0"), ("RLFC_PSUM", "serial"),
                                          ("RLFC_RESID", "tile"), ("RLFC_RESID", "march"), ("RLFC_TINY", "0")])
def test_alternative_execution_paths(rlfc, oracle, init_state, monkeypatch, envvar, value):
    """The wavefront fallback smoother, the chained smoother, eager launches, odd env-group splits, the literal setBC kernels and the plain
    serial Field.sum chain are different
    schedules of the same arithmetic: all must reproduce the oracle bit for bit."""
    monkeypatch.setenv(envvar, value)
    ref = make_oracle(oracle, init_state)
    ref.set_xi(-0.6, 0.9)
    B = 7
    act = np.zeros((B, 2), np.float32)
    act[3] = (-0.6, 0.9)
    with rlfc.AFCCylinderBatch(B) as env:
        for k in range(3):
            f = env.update2(act if k == 0 else None)
            ref.update2()
            assert_same(f[3], np.array(ref.force(), np.float32), f"force step {k}")
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(3), ref.get_state()):
            assert_same(a, b, nm)


@pytest.mark.parametrize("resolution,dims", [(64, (1026, 514)), (128, (2050, 1026)), (256, (4098, 2050))])
def test_wide_grid(rlfc, oracle, resolution, dims):
    """Single-domain-style grids wider than the row pipeline's 256 columns: BASELINE config 3 (2048x1024, SURVEY 8d:
    resolution 128, t_step = 0.18/128 so dt stays 0.18 grid units) and its half-scale version.  The wide levels fall
    back to the wavefront smoother, setBC to the literal kernels.  Impulsive start, a non-zero action, every float
    equal to the oracle's.  The 4096x2048 case (8 Mi cells) also runs the three-pass Field.sum of very large domains;
    its oracle needs ~20 s."""
    kw = dict(resolution=resolution, x_lengths=16, y_lengths=8)
    t_step = np.float32(0.18) / np.float32(resolution)
    ref = oracle.OracleEnv(literal=False, resolution=resolution, xLengths=16, yLengths=8, tStep=float(t_step))
    ref.set_xi(0.5, -0.5)
    act = np.array([[0.5, -0.5]], np.float32)
    with rlfc.AFCCylinderBatch(1, init_state=None, t_step=float(t_step), **kw) as env:
        assert (env.n, env.m) == (ref.n, ref.m) == dims
        for k in range(2):
            f = env.update2(act if k == 0 else None)
            ref.update2()
            assert_same(f[0], np.array(ref.force(), np.float32), f"force step {k}")
            assert tuple(env.mg_iters()[0]) == ref.mg_iters()
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(0), ref.get_state()):
            assert_same(a, b, nm)


def test_check_cfl(rlfc, oracle, init_state):
    """BDIM.checkCFL (adaptive-dt variant of the reference, BDIM.pde:217-219): the device maximum == the oracle's, on the
    developed wake and after a few steps of two differently driven environments."""
    refs = [make_oracle(oracle, init_state) for _ in range(2)]
    refs[1].set_xi(0.9, -0.9)
    with rlfc.AFCCylinderBatch(2) as env:
        assert_same(env.check_cfl(), np.array([r.check_cfl() for r in refs], np.float32), "checkCFL at t = 0")
        for k in range(3):
            env.update2(np.array([[0, 0], [0.9, -0.9]], np.float32) if k == 0 else None)
            for r in refs:
                r.update2()
        assert_same(env.check_cfl(), np.array([r.check_cfl() for r in refs], np.float32), "checkCFL after 3 steps")
