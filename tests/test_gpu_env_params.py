"""Per-environment constructor arguments (rlfc_config.env_params, rlfc_env_reset_params): every environment of a mixed
batch is held to a lone CPU-oracle environment built with that environment's own (Re, dR, gR, theta, tStep).  Bar:
bit-exact (==), as in test_gpu_parity and test_gpu_adaptive."""
import numpy as np
import pytest

from adaptive_driver import DrawDriver
from test_gpu_parity import assert_same, make_oracle

pytestmark = pytest.mark.gpu

F = np.float32
PI = F(3.1415927)
DEFAULT = dict(re=500, dR=F(0.125), gR=F(0.2), theta=PI / F(3), t_step=F(0.0075))
# one environment per varied parameter, plus one default environment
MIXED = [dict(DEFAULT), dict(DEFAULT, re=100), dict(DEFAULT, dR=F(0.25)), dict(DEFAULT, gR=F(0.5)),
         dict(DEFAULT, theta=F(1.2)), dict(DEFAULT, t_step=F(0.005))]


def oracle_for(oracle, init_state, p, **kw):
    return make_oracle(oracle, init_state, Re=int(p["re"]), dR=float(p["dR"]), gR=float(p["gR"]), theta=float(p["theta"]),
                       tStep=float(p["t_step"]), **kw)


def random_params(n, seed):
    rng = np.random.default_rng(seed)
    return [dict(re=int(rng.integers(100, 1001)), dR=F(rng.uniform(0.1, 0.25)), gR=F(rng.uniform(0.1, 0.5)),
                 theta=F(rng.uniform(np.pi / 6, np.pi / 2)), t_step=F(rng.choice([0.005, 0.0075]))) for _ in range(n)]


def hetero_actions(B, seed=1234):
    acts = np.clip(np.random.default_rng(seed).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)
    acts[0] = 0
    return acts


def assert_hierarchy(oracle, env, e, ref):
    """Environment e's del and Poisson hierarchy (every level) against the oracle's for its own del and dt."""
    dx, dy = ref.coeff("del.x"), ref.coeff("del.y")
    assert_same(env.get_coeffs(e, "del.x"), dx, f"del.x env {e}")
    assert_same(env.get_coeffs(e, "del.y"), dy, f"del.y env {e}")
    c = oracle.VField(env.n, env.m)
    c.x[...] = dx * (F(1) * ref.dt)
    c.y[...] = dy * (F(1) * ref.dt)
    assert_same(env.get_coeffs(e, "c.x"), c.x, f"c.x env {e}")
    assert_same(env.get_coeffs(e, "c.y"), c.y, f"c.y env {e}")
    A = oracle.Poisson(c)
    for l in range(env.num_levels):
        for nm, want in (("lower.x", A.lx), ("lower.y", A.ly), ("inv", A.inv), ("diag", A.diag)):
            assert_same(env.get_coeffs(e, nm, l), want, f"{nm} level {l} env {e}")
        if l + 1 < env.num_levels:
            A = A.restrict()


def step_and_compare(env, refs, steps, acts=None, adaptive=False, tag=""):
    """`steps` solver steps of the handle and of every oracle in refs {e: oracle}, compared after each."""
    for k in range(steps):
        f, pr = env.update2(acts if (acts is not None and k == 0) else None, want_probes=True)
        dts, ts, its = env.dt(), env.t, env.mg_iters()
        for e, r in refs.items():
            r.update_adaptive() if adaptive else r.update2()
            assert dts[e] == r.dt, f"{tag}dt env {e} step {k}: {dts[e]!r} vs {r.dt!r}"
            assert_same(f[e], np.array(r.force(), F), f"{tag}force env {e} step {k}")
            assert_same(pr[e], r.probes(32), f"{tag}probes env {e} step {k}")
            assert tuple(its[e]) == r.mg_iters(), f"{tag}mg iters env {e} step {k}"
            assert ts[e] == F(r.t), f"{tag}t env {e} step {k}"


def assert_fields(env, refs, tag=""):
    for e, r in refs.items():
        for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(e), r.get_state()):
            assert_same(a, b, f"{tag}{nm} env {e}")


def test_mixed_batch(rlfc, oracle, init_state):
    B = len(MIXED)
    acts = hetero_actions(B)
    refs = {e: oracle_for(oracle, init_state, p) for e, p in enumerate(MIXED)}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    with rlfc.AFCCylinderBatch(B, env_params=MIXED) as env:
        got = env.params()
        for e, p in enumerate(MIXED):
            assert [got[k][e] for k in p] == [F(v) if k != "re" else v for k, v in p.items()]
        for e, r in refs.items():
            assert_hierarchy(oracle, env, e, r)
        step_and_compare(env, refs, 20, acts)
        assert_fields(env, refs)
        for e, r in refs.items():
            assert_hierarchy(oracle, env, e, r)


def test_all_default_equals_shared(rlfc):
    """A per-environment handle whose sets are all the scalar config's computes what the shared handle computes."""
    B = 4
    acts = hetero_actions(B, 5)
    with rlfc.AFCCylinderBatch(B, init_time=-1.0) as a, \
            rlfc.AFCCylinderBatch(B, init_time=-1.0, env_params=[{}] * B) as b:
        for k in range(3):
            fa, fb = a.update2(acts if k == 0 else None), b.update2(acts if k == 0 else None)
            assert_same(fb, fa, f"force step {k}")
        for k in range(3):
            oa, ra, da = a.step(acts * F(0.5 + 0.1 * k))
            ob, rb, db = b.step(acts * F(0.5 + 0.1 * k))
            assert_same(ob, oa, f"obs call {k}")
            assert_same(rb, ra, f"reward call {k}")
            assert (db == da).all()
        assert_same(b.dt(), a.dt(), "dt")
        assert_same(b.t, a.t, "t")
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), b.get_fields(e), a.get_fields(e)):
                assert_same(x, y, f"{nm} env {e}")


def test_adaptive_dt(rlfc, oracle, init_state):
    """adaptive_dt = 1 with per-environment parameters: update_adaptive() per environment, its own nu in the CFL."""
    params = [MIXED[1], MIXED[0], MIXED[2], MIXED[5]]
    acts = hetero_actions(len(params), 11)
    refs = {e: oracle_for(oracle, init_state, p) for e, p in enumerate(params)}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    with rlfc.AFCCylinderBatch(len(params), adaptive_dt=1, env_params=params) as env:
        cfl = env.check_cfl()
        for e, r in refs.items():
            assert cfl[e] == r.check_cfl(), f"check_cfl env {e}"
        step_and_compare(env, refs, 10, acts, adaptive=True)
        assert_fields(env, refs)
        assert_hierarchy(oracle, env, 0, refs[0])


@pytest.mark.parametrize("envvar,value", [(None, None), ("RLFC_NO_GRAPH", "1"), ("RLFC_GROUPS", "3"), ("RLFC_FAST_BC", "0"),
                                          ("RLFC_RESID", "tile"), ("RLFC_RESID", "march"), ("RLFC_PSUM", "serial"),
                                          ("RLFC_TINY", "0")])
def test_reset_params_mid_run(rlfc, oracle, init_state, monkeypatch, envvar, value):
    """One environment switched to a new parameter set mid-run matches a fresh oracle built with it; the others keep
    matching their own."""
    if envvar:
        monkeypatch.setenv(envvar, value)
    params = [MIXED[0], MIXED[3], MIXED[4], MIXED[1]]
    B = len(params)
    acts = hetero_actions(B, 3)
    refs = {e: oracle_for(oracle, init_state, p) for e, p in enumerate(params)}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    new = dict(re=300, dR=F(0.2), gR=F(0.3), theta=F(0.9), t_step=F(0.005))
    with rlfc.AFCCylinderBatch(B, env_params=params) as env:
        step_and_compare(env, refs, 3, acts, tag="before: ")
        env.reset([2], params=[new])
        refs[2] = oracle_for(oracle, init_state, new)       # xi = 0 after the reset, as the fresh oracle has it
        assert env.params()["re"].tolist() == [500, 500, 300, 100]
        assert env.dt()[2] == F(0.005) * F(24) and env.t[2] == 0
        assert_hierarchy(oracle, env, 2, refs[2])
        step_and_compare(env, refs, 4, tag="after: ")
        assert_fields(env, refs)


def test_rejected_reset_params_changes_nothing(rlfc, init_state):
    B = 3
    with rlfc.AFCCylinderBatch(B, env_params=MIXED[:B]) as env:
        env.update2(hetero_actions(B))
        before = ([env.get_fields(e) for e in range(B)], env.params(), env.dt(), env.t,
                  [env.get_coeffs(e, "inv", 1) for e in range(B)])
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*env_params\[1\].*gR"):
            env.reset([0, 2], params=[dict(re=200), dict(gR=-1.0)])
        after = ([env.get_fields(e) for e in range(B)], env.params(), env.dt(), env.t,
                 [env.get_coeffs(e, "inv", 1) for e in range(B)])
        for e in range(B):
            for x, y in zip(before[0][e], after[0][e]):
                assert_same(y, x, f"fields env {e}")
            assert_same(after[4][e], before[4][e], f"inv env {e}")
        assert (after[1] == before[1]).all()
        assert_same(after[2], before[2], "dt")
        assert_same(after[3], before[3], "t")
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*listed twice"):
            env.reset([1, 1], params=[{}, {}])


def test_rl_step_per_environment_t_step(rlfc, oracle, init_state):
    """rlfc_env_step with different t_step: the environments cross init_time and episode_time at different solver steps."""
    init_time, episode_time = 0.3, 0.62
    params = [dict(t_step=F(0.0075)), dict(t_step=F(0.005), re=250, theta=F(0.8))]
    full = [dict(DEFAULT, **p) for p in params]
    drv = [DrawDriver(oracle_for(oracle, init_state, p), init_time=init_time, episode_time=episode_time, adaptive=False)
           for p in full]
    with rlfc.AFCCylinderBatch(2, env_params=params, init_time=init_time, episode_time=episode_time) as env:
        done = np.zeros(2, np.int32)
        k = 0
        while not done.all():
            a = np.array([[0.8 * np.sin(0.7 * k), -0.8 * np.sin(0.7 * k + 1)], [0.3, -0.6 * np.cos(k)]], F)
            obs, rew, done = env.step(a)
            for e, d in enumerate(drv):
                o, fin = d.rl_step(a[e])
                assert_same(obs[e], np.array(o, F), f"obs env {e} call {k}")
                assert bool(done[e]) == fin, f"done env {e} call {k}"
                assert env.t[e] == d.t, f"t env {e} call {k}"
            k += 1
            assert k < 40
        assert drv[0].solver_steps != drv[1].solver_steps
        for e, d in enumerate(drv):
            for nm, a_, b_ in zip(("ux", "uy", "p"), env.get_fields(e), d.env.get_state()):
                assert_same(a_, b_, f"{nm} env {e}")


def test_large_batch(rlfc, oracle, init_state):
    """256 environments with random parameters: the marching residual kernel and two environment groups."""
    B = 256
    params = random_params(B, 42)
    acts = hetero_actions(B, 7)
    check = (0, 127, 255)
    refs = {e: oracle_for(oracle, init_state, params[e]) for e in check}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    with rlfc.AFCCylinderBatch(B, env_params=params) as env:
        step_and_compare(env, refs, 3, acts)
        assert_fields(env, refs)


def test_device_entry_point(rlfc):
    torch = pytest.importorskip("torch")
    B = 3
    acts = hetero_actions(B, 3)
    params = [MIXED[5], MIXED[2], MIXED[1]]
    with rlfc.AFCCylinderBatch(B, env_params=params) as a, rlfc.AFCCylinderBatch(B, env_params=params) as b:
        d_acts = torch.from_numpy(acts).cuda()
        torch.cuda.synchronize()
        for k in range(4):
            a.update2(acts if k == 0 else None)
            b.update2_device(d_acts.data_ptr() if k == 0 else 0)
        assert_same(b.t, a.t, "t")
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), b.get_fields(e), a.get_fields(e)):
                assert_same(x, y, f"{nm} env {e}")


def test_checkpoints_carry_each_environments_dt(rlfc, tmp_path):
    params = [dict(t_step=F(0.0075)), dict(t_step=F(0.005)), dict(t_step=F(0.005), re=200)]
    with rlfc.AFCCylinderBatch(3, env_params=params) as env:
        env.update2()
        assert env.dt().tolist() == [F(0.0075) * F(24), F(0.005) * F(24), F(0.005) * F(24)]
        path = tmp_path / "ck1.bdim"
        env.save_bdim(1, path)
        assert F(path.read_text().splitlines()[1]) == F(0.005) * F(24)
        with pytest.raises(rlfc.RlfcError, match=r"\(-4\).*does not match"):
            env.load_bdim(0, path)
        env.load_bdim(2, path)
        for nm, x, y in zip(("ux", "uy", "p"), env.get_fields(2), env.get_fields(1)):
            assert_same(x, y, f"{nm} after load")
        env.reset([1])
        assert env.params()["t_step"][1] == F(0.005) and env.dt()[1] == F(0.005) * F(24)


@pytest.mark.parametrize("kw,envvar", [(dict(), ("RLFC_SMOOTHER", "chain")), (dict(), ("RLFC_SMOOTHER", "wave")),
                                       (dict(resolution=64, init_state=None), None)])
def test_rejected_configurations(rlfc, monkeypatch, kw, envvar):
    if envvar:
        monkeypatch.setenv(*envvar)
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*env_params"):
        rlfc.AFCCylinderBatch(1, env_params=[{}], **kw)


def test_reset_params_needs_a_per_environment_handle(rlfc):
    with rlfc.AFCCylinderBatch(1) as env:
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*env_params"):
            env.reset([0], params=[{}])
        assert env.params()["re"].tolist() == [500]


class FakePeer:
    """The agent side of the batch protocol: constant actions, records the calls."""

    def __init__(self, B):
        self.B = B
        self.finished = []

    def init(self, _):
        return True

    def start_episode(self, _):
        return True

    def request_batch_action(self, payload):
        return ";".join(["0.25_-0.5"] * self.B)

    def finish_envs(self, ids):
        self.finished.append([int(e) for e in ids.split(";")])
        return True

    def train(self, _):
        return True

    def save(self, _):
        return True


def test_driver_samples_parameters_at_auto_reset(rlfc):
    from rlfluidcontrol_b200.driver import BatchedEpisodeDriver
    B = 2
    drawn = []

    def sample(rng, env_ids):
        out = [dict(re=int(rng.integers(100, 1001)), dR=float(rng.uniform(0.1, 0.25))) for _ in env_ids]
        drawn.append((list(env_ids), out))
        return out

    with rlfc.AFCCylinderBatch(B, env_params=[{}, dict(t_step=0.005)], init_time=-1.0, episode_time=0.25) as env:
        peer = FakePeer(B)
        drv = BatchedEpisodeDriver(env, proxy=peer, sample_params=sample, seed=7)
        drv.start()
        for _ in range(4):
            drv.step()
            if drawn:
                break
        assert drawn, "no environment finished"
        ids, sets = drawn[0]
        assert peer.finished[0] == ids
        got = env.params()
        for e, p in zip(ids, sets):
            assert got["re"][e] == p["re"] and got["dR"][e] == F(p["dR"])
            assert got["t_step"][e] == F(env.cfg.t_step) and env.t[e] == 0
