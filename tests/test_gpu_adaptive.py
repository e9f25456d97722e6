"""Adaptive time stepping (rlfc_config.adaptive_dt = 1, AFCCylinder.update, AFCCylinder.pde:63-84) against the CPU
oracle's update_adaptive(): every environment takes dt = min(CFL, 1) of its own velocity before each step, and its
Poisson hierarchy is rebuilt on the device from c = del*dt.  Bar: bit-exact (==), as in test_gpu_parity."""
import numpy as np
import pytest

from adaptive_driver import DrawDriver
from test_gpu_parity import assert_same, make_oracle

pytestmark = pytest.mark.gpu

F = np.float32


def oracle_hierarchy(oracle, env, dt):
    """Poisson(c).restrict()... of the oracle for c = del*(1*dt) (BDIM.pde:59-61,81)."""
    dx, dy = env.get_static("del.x"), env.get_static("del.y")
    c = oracle.VField(env.n, env.m)
    c.x[...] = dx * (F(1) * F(dt))
    c.y[...] = dy * (F(1) * F(dt))
    levels = [oracle.Poisson(c)]
    while len(levels) < env.num_levels:
        levels.append(levels[-1].restrict())
    return c, levels


def assert_hierarchy(oracle, env, e, dt):
    c, levels = oracle_hierarchy(oracle, env, dt)
    assert_same(env.get_coeffs(e, "c.x"), c.x, f"c.x env {e}")
    assert_same(env.get_coeffs(e, "c.y"), c.y, f"c.y env {e}")
    for l, A in enumerate(levels):
        for nm, ref in (("lower.x", A.lx), ("lower.y", A.ly), ("inv", A.inv), ("diag", A.diag)):
            assert_same(env.get_coeffs(e, nm, l), ref, f"{nm} level {l} env {e}")


def run_parity(rlfc, oracle, init_state, B, acts, check, steps, **kw):
    """`steps` adaptive solver steps of a batch (actions `acts` taken on the first) against one oracle env per checked env."""
    refs = {e: make_oracle(oracle, init_state, **kw.get("oracle_kw", {})) for e in check}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    with rlfc.AFCCylinderBatch(B, adaptive_dt=1, **kw.get("env_kw", {})) as env:
        for k in range(steps):
            f, pr = env.update2(acts if k == 0 else None, want_probes=True)
            dts, ts, its = env.dt(), env.t, env.mg_iters()
            for e, r in refs.items():
                r.update_adaptive()
                assert dts[e] == r.dt, f"dt env {e} step {k}: {dts[e]!r} vs {r.dt!r}"
                assert_same(f[e], np.array(r.force(), F), f"force env {e} step {k}")
                assert_same(pr[e], r.probes(32), f"probes env {e} step {k}")
                assert tuple(its[e]) == r.mg_iters(), f"mg iters env {e} step {k}"
                assert ts[e] == F(r.t), f"t env {e} step {k}"
        for e, r in refs.items():
            for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(e), r.get_state()):
                assert_same(a, b, f"{nm} env {e}")
        return env.dt(), {e: r.mg_iters() for e, r in refs.items()}


def hetero_actions(B, seed=1234):
    acts = np.clip(np.random.default_rng(seed).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)
    acts[0] = 0
    return acts


def test_hierarchy_per_environment(rlfc, oracle, init_state):
    """After create the per-environment hierarchy is the host's static one; after a few steps each environment's hierarchy
    is the oracle's for its own dt, at every level."""
    acts = np.array([[0, 0], [0.9, -0.9]], F)
    with rlfc.AFCCylinderBatch(2, init_state=None, adaptive_dt=1) as env:
        for nm in ("lower.x", "lower.y", "inv", "diag"):
            for l in range(env.num_levels):
                assert_same(env.get_coeffs(1, nm, l), env.get_static(nm, l), f"initial {nm} level {l}")
        assert_same(env.dt(), np.full(2, F(0.0075) * F(24), F), "initial dt")
        for k in range(3):
            env.update2(acts if k == 0 else None)
        dts = env.dt()
        assert dts[0] != dts[1]
        for e in (0, 1):
            assert_hierarchy(oracle, env, e, dts[e])


def test_batch_heterogeneous_actions(rlfc, oracle, init_state):
    B = 6
    dts, _ = run_parity(rlfc, oracle, init_state, B, hetero_actions(B), (0, 3, 5), 20)
    assert len(set(dts.tolist())) > 1


def test_impulsive_start(rlfc, oracle):
    """Uniform flow start: dt swings widely and solves take several MG iterations (the WHILE node of the step graph)."""
    acts = np.array([[0.5, -0.5], [0, 0], [0.5, -0.5]], F)
    _, its = run_parity(rlfc, oracle, None, 3, acts, (0, 2), 20, env_kw=dict(init_state=None))


def test_impulsive_start_iterations(rlfc, oracle):
    ref = make_oracle(oracle, None)
    ref.set_xi(0.5, -0.5)
    with rlfc.AFCCylinderBatch(1, init_state=None, adaptive_dt=1) as env:
        its = []
        for k in range(3):
            env.update2(np.array([[0.5, -0.5]], F) if k == 0 else None)
            ref.update_adaptive()
            its.append(tuple(env.mg_iters()[0]))
            assert its[-1] == ref.mg_iters()
    assert max(max(i) for i in its) > 1


@pytest.mark.parametrize("resolution,xl,yl", [(16, 16, 8), (8, 16, 8), (12, 8, 4), (24, 8, 4)])
def test_other_grids(rlfc, oracle, resolution, xl, yl):
    ref = oracle.OracleEnv(literal=False, resolution=resolution, xLengths=xl, yLengths=yl)
    ref.set_xi(0.4, -0.7)
    act = np.array([[0.4, -0.7], [0.0, 0.0]], F)
    with rlfc.AFCCylinderBatch(2, init_state=None, resolution=resolution, x_lengths=xl, y_lengths=yl, adaptive_dt=1) as env:
        for k in range(6):
            f = env.update2(act if k == 0 else None)
            ref.update_adaptive()
            assert env.dt()[0] == ref.dt
            assert_same(f[0], np.array(ref.force(), F), f"force step {k}")
            assert tuple(env.mg_iters()[0]) == ref.mg_iters()
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(0), ref.get_state()):
            assert_same(a, b, nm)


@pytest.mark.parametrize("envvar,value", [("RLFC_RESID", "tile"), ("RLFC_RESID", "march"), ("RLFC_NO_GRAPH", "1"),
                                          ("RLFC_GROUPS", "3"), ("RLFC_FAST_BC", "0"), ("RLFC_PSUM", "serial"),
                                          ("RLFC_TINY", "0")])
def test_alternative_execution_paths(rlfc, oracle, init_state, monkeypatch, envvar, value):
    monkeypatch.setenv(envvar, value)
    B = 7
    acts = np.zeros((B, 2), F)
    acts[3] = (-0.6, 0.9)
    acts[6] = (0.8, 0.8)
    run_parity(rlfc, oracle, init_state, B, acts, (3, 6), 4)


def test_large_batch(rlfc, oracle, init_state):
    """256 environments: the marching residual kernel and two environment groups."""
    B = 256
    run_parity(rlfc, oracle, init_state, B, hetero_actions(B, 7), (0, 127, 255), 3)


def test_device_entry_point(rlfc):
    """substep_device runs the same adaptive step as substep."""
    torch = pytest.importorskip("torch")
    B = 3
    acts = hetero_actions(B, 3)
    with rlfc.AFCCylinderBatch(B, adaptive_dt=1) as a, rlfc.AFCCylinderBatch(B, adaptive_dt=1) as b:
        d_acts = torch.from_numpy(acts).cuda()
        torch.cuda.synchronize()
        for k in range(5):
            a.update2(acts if k == 0 else None)
            b.update2_device(d_acts.data_ptr() if k == 0 else 0)
        assert_same(b.dt(), a.dt(), "dt")
        assert_same(b.t, a.t, "t")
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), b.get_fields(e), a.get_fields(e)):
                assert_same(x, y, f"{nm} env {e}")


def test_rl_step(rlfc, oracle, init_state):
    """rlfc_env_step with adaptive steps from a reset (default init_time) to the end of a short episode, against the
    draw() accumulation around update_adaptive."""
    episode_time = 1.6
    ref = DrawDriver(make_oracle(oracle, init_state), episode_time=episode_time)
    with rlfc.AFCCylinderBatch(2, adaptive_dt=1, episode_time=episode_time) as env:
        done = np.zeros(2, np.int32)
        k = 0
        while not done[0]:
            a = np.array([0.8 * np.sin(0.7 * k), -0.8 * np.sin(0.7 * k + 1)], F)
            obs, rew, done = env.step(np.stack([a, -a]))
            o, d = ref.rl_step(a)
            assert_same(obs[0], np.array(o, F), f"obs call {k}")
            assert bool(done[0]) == d, f"done call {k}"
            assert env.t[0] == ref.t and env.dt()[0] == ref.env.dt, f"t / dt call {k}"
            k += 1
            assert k < 40
        assert k >= 2
        for nm, a_, b_ in zip(("ux", "uy", "p"), env.get_fields(0), ref.env.get_state()):
            assert_same(a_, b_, nm)


def test_checkpoint_and_reset(rlfc, init_state, tmp_path):
    with rlfc.AFCCylinderBatch(2, adaptive_dt=1) as env:
        for _ in range(3):
            env.update2()
        dt0 = env.dt()[0]
        assert dt0 != F(0.0075) * F(24)
        path = tmp_path / "ck.bdim"
        env.save_bdim(0, path)
        assert F(path.read_text().splitlines()[1]) == dt0
        env.load_bdim(1, path)
        assert env.dt()[1] == dt0
        for nm, x, y in zip(("ux", "uy", "p"), env.get_fields(1), env.get_fields(0)):
            assert_same(x, y, f"{nm} after load")
        env.reset([0])
        assert env.dt().tolist() == [F(0.0075) * F(24), dt0]
    with rlfc.AFCCylinderBatch(1) as fixed:              # fixed mode: dt and coefficients are the static ones
        assert fixed.dt()[0] == F(0.0075) * F(24)
        assert_same(fixed.get_coeffs(0, "inv", 2), fixed.get_static("inv", 2), "fixed-mode coefficients")


@pytest.mark.parametrize("kw,envvar", [(dict(n_devices=2), None), (dict(), ("RLFC_SMOOTHER", "chain")),
                                       (dict(), ("RLFC_SMOOTHER", "wave")),
                                       (dict(resolution=64, init_state=None), None)])
def test_rejected_configurations(rlfc, monkeypatch, kw, envvar):
    """Slab mode and the chained / wavefront smoothers have no per-environment hierarchy: RLFC_EINVAL (-1)."""
    if envvar:
        monkeypatch.setenv(*envvar)
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*adaptive_dt"):
        rlfc.AFCCylinderBatch(1, adaptive_dt=1, **kw)
