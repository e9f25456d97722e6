"""Parameter library (rlfc_config.param_sets, rlfc_env_reset_sets / rlfc_env_reset_sets_device): a reset into library set
s is held to rlfc_env_reset_params with param_sets[s] and to a lone CPU-oracle environment built with that set.  Bar:
bit-exact (==), as in test_gpu_env_params."""
import numpy as np
import pytest

from test_gpu_env_params import (DEFAULT, MIXED, F, assert_fields, assert_hierarchy, hetero_actions, oracle_for,
                                 step_and_compare)
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu

LEVEL0 = ("c.x", "c.y", "del.x", "del.y")
ANY_LEVEL = ("lower.x", "lower.y", "inv", "diag")
NEW = [dict(re=300, dR=F(0.2), gR=F(0.3), theta=F(0.9), t_step=F(0.005)),
       dict(re=800, dR=F(0.15), gR=F(0.25), theta=F(1.3), t_step=F(0.0075)),
       dict(re=150, dR=F(0.1), gR=F(0.4), theta=F(0.7), t_step=F(0.006))]


def params_of(env, e):
    got = env.params()
    return {k: got[k][e] for k in DEFAULT}


def same_params(env, e, p):
    got = params_of(env, e)
    return all(got[k] == (int(p[k]) if k == "re" else F(p[k])) for k in DEFAULT)


def coeffs(env, e):
    out = {nm: env.get_coeffs(e, nm) for nm in LEVEL0}
    for l in range(env.num_levels):
        for nm in ANY_LEVEL:
            out[f"{nm}/{l}"] = env.get_coeffs(e, nm, l)
    return out


def readouts(env, e):
    """Every read-out of environment e that a reset could touch, without stepping."""
    r = dict(zip(("ux", "uy", "p"), env.get_fields(e)))
    r.update(coeffs(env, e))
    r["t"], r["dt"], r["iters"], r["flags"] = env.t[e], env.dt()[e], env.mg_iters()[e], env.flags()[e]
    r["params"] = np.array(list(params_of(env, e).values()), np.float64)
    return r


def assert_readouts(got, want, tag):
    for k in want:
        assert_same(np.asarray(got[k]), np.asarray(want[k]), f"{tag}{k}")


def assert_handles_equal(a, b, envs, tag=""):
    assert (a.params() == b.params()).all(), f"{tag}params"
    for e in envs:
        assert_readouts(readouts(b, e), readouts(a, e), f"{tag}env {e} ")


def solver_steps_equal(a, b, steps, acts=None, tag=""):
    for k in range(steps):
        x = acts if (acts is not None and k == 0) else None
        fa, pa = a.update2(x, want_probes=True)
        fb, pb = b.update2(x, want_probes=True)
        assert_same(fb, fa, f"{tag}force step {k}")
        assert_same(pb, pa, f"{tag}probes step {k}")
        assert_same(b.t, a.t, f"{tag}t step {k}")
        assert_same(b.dt(), a.dt(), f"{tag}dt step {k}")
        assert (b.mg_iters() == a.mg_iters()).all(), f"{tag}mg iters step {k}"


def device_ints(torch, values):
    return torch.tensor(np.asarray(values, np.int32), dtype=torch.int32, device="cuda")


@pytest.mark.parametrize("envvar,value", [(None, None), ("RLFC_NO_GRAPH", "1"), ("RLFC_GROUPS", "3")])
def test_reset_sets_equals_reset_params(rlfc, monkeypatch, envvar, value):
    """Handle A resets through rlfc_env_reset_params, handle B through the library: the same state, coefficients at every
    level and read-outs, then the same solver and RL steps."""
    if envvar:
        monkeypatch.setenv(envvar, value)
    own = [MIXED[0], MIXED[3], MIXED[4], MIXED[1], MIXED[2]]
    B = len(own)
    acts = hetero_actions(B, 21)
    ids, idx = [4, 0, 2, 3], [5, 1, 5, 0]
    with rlfc.AFCCylinderBatch(B, env_params=own, init_time=0.05) as a, \
            rlfc.AFCCylinderBatch(B, env_params=own, param_sets=MIXED, init_time=0.05) as b:
        assert b.n_param_sets == len(MIXED) and a.n_param_sets == 0
        solver_steps_equal(a, b, 3, acts, "before: ")
        a.reset(ids, params=[MIXED[s] for s in idx], reset_accumulators=True)
        b.reset_sets(ids, idx, reset_accumulators=True)
        for e, s in zip(ids, idx):
            assert same_params(b, e, MIXED[s])
        assert_handles_equal(a, b, range(B), "after reset: ")
        solver_steps_equal(a, b, 4, acts, "after: ")
        for k in range(3):
            x = acts * F(0.3 * (k + 1))
            oa, ra, da = a.step(x)
            ob, rb, db = b.step(x)
            assert_same(ob, oa, f"obs call {k}")
            assert_same(rb, ra, f"reward call {k}")
            assert (db == da).all(), f"done call {k}"
        assert_handles_equal(a, b, range(B), "end: ")


def test_reset_sets_on_a_scalar_handle(rlfc):
    """A handle created with a library but without env_params holds the scalar config's set in every environment, as a
    handle with env_params = B copies of it does; a 64-cells-per-diameter grid."""
    kw = dict(resolution=64, x_lengths=4, y_lengths=2, init_state=None, init_time=-1.0)
    lib = [MIXED[1], NEW[0]]
    with rlfc.AFCCylinderBatch(3, env_params=[{}] * 3, **kw) as a, rlfc.AFCCylinderBatch(3, param_sets=lib, **kw) as b:
        assert (a.params() == b.params()).all()
        solver_steps_equal(a, b, 2, hetero_actions(3, 2), "before: ")
        a.reset([1, 2], params=[lib[1], lib[0]])
        b.reset_sets([1, 2], [1, 0])
        assert_handles_equal(a, b, range(3))
        solver_steps_equal(a, b, 3, tag="after: ")


@pytest.mark.parametrize("adaptive", [0, 1])
def test_device_reset_against_oracle(rlfc, oracle, init_state, adaptive):
    """reset_sets_device with skipped pairs (-1, out of range) and a duplicated environment: the skipped environments are
    untouched, the last pair wins, and every environment then matches a lone oracle built with its final set."""
    torch = pytest.importorskip("torch")
    own = [MIXED[0], MIXED[1], MIXED[3], MIXED[4], MIXED[5], MIXED[2]]
    lib = [NEW[0], NEW[1], MIXED[2], NEW[2], NEW[0]]    # sets 0 and 4 share a geometry slot
    B = len(own)
    acts = hetero_actions(B, 9)
    refs = {e: oracle_for(oracle, init_state, p) for e, p in enumerate(own)}
    for e, r in refs.items():
        r.set_xi(*acts[e])
    envs = [0, 1, 2, 3, 2, 4, 5, -1, 7, 5]
    sets = [3, -1, 0, 4, 1, 99, 0, 1, 1, -5]
    applied = {0: 3, 2: 1, 3: 4, 5: 0}          # env 2: the last pair wins; the last pair of env 5 is skipped
    with rlfc.AFCCylinderBatch(B, env_params=own, param_sets=lib, adaptive_dt=adaptive) as env:
        step_and_compare(env, refs, 3, acts, adaptive=bool(adaptive), tag="before: ")
        before = {e: readouts(env, e) for e in range(B) if e not in applied}
        d_env, d_set = device_ints(torch, envs), device_ints(torch, sets)
        torch.cuda.synchronize()
        env.reset_sets_device(d_env.data_ptr(), d_set.data_ptr(), len(envs))
        for e, want in before.items():
            assert_readouts(readouts(env, e), want, f"skipped env {e} ")
        for e, s in applied.items():
            assert same_params(env, e, lib[s]), e
            assert env.t[e] == 0 and env.dt()[e] == F(lib[s]["t_step"]) * F(24)
            refs[e] = oracle_for(oracle, init_state, lib[s])
            assert_hierarchy(oracle, env, e, refs[e])
        step_and_compare(env, refs, 20, adaptive=bool(adaptive), tag="after: ")
        assert_fields(env, refs)
        for e in applied:
            assert_hierarchy(oracle, env, e, refs[e])


def test_host_copies_follow_a_device_switch(rlfc, oracle, init_state, tmp_path):
    torch = pytest.importorskip("torch")
    own = [MIXED[0], MIXED[3], MIXED[4]]
    lib = [MIXED[5], NEW[1]]                     # set 0: t_step .005 against the own sets' .0075
    with rlfc.AFCCylinderBatch(3, env_params=own, param_sets=lib) as env:
        env.update2(hetero_actions(3, 4))
        d_env, d_set = device_ints(torch, [1]), device_ints(torch, [0])
        torch.cuda.synchronize()
        env.reset_sets_device(d_env.data_ptr(), d_set.data_ptr(), 1)
        ref = oracle_for(oracle, init_state, lib[0])
        assert same_params(env, 1, lib[0])
        assert_same(env.get_coeffs(1, "del.x"), ref.coeff("del.x"), "del.x")
        assert_same(env.get_coeffs(1, "del.y"), ref.coeff("del.y"), "del.y")
        env.update2()
        # rlfc_env_reset keeps the set's dt
        env.reset([1])
        assert env.dt()[1] == F(0.005) * F(24) and env.t[1] == 0
        env.update2()
        # checkpoints: the dt line and the fixed-dt check follow the set
        path = tmp_path / "set.bdim"
        env.save_bdim(1, path)
        assert F(path.read_text().splitlines()[1]) == F(0.005) * F(24)
        env.load_bdim(1, path)
        with pytest.raises(rlfc.RlfcError, match=r"\(-4\).*does not match"):
            env.load_bdim(0, path)
        # a host reset_params of another environment leaves the switched one on its set
        env.reset([2], params=[NEW[0]])
        env.reset([1])
        assert same_params(env, 1, lib[0]) and same_params(env, 2, NEW[0])
        refs = {1: oracle_for(oracle, init_state, lib[0]), 2: oracle_for(oracle, init_state, NEW[0])}
        assert_hierarchy(oracle, env, 1, refs[1])
        step_and_compare(env, refs, 5, tag="after reset_params of env 2: ")
        assert_fields(env, refs)
        # reset_params of the switched environment takes it back to its own slot
        env.reset([1], params=[own[1]])
        refs = {1: oracle_for(oracle, init_state, own[1])}
        assert same_params(env, 1, own[1])
        assert_hierarchy(oracle, env, 1, refs[1])
        step_and_compare(env, refs, 5, tag="back on its own slot: ")


def test_rl_step_reaches_the_observation_after_a_smaller_t_step(rlfc):
    """rlfc_env_step bounds its rounds by the smallest dt of the own and the library sets."""
    init_time = 0.3
    with rlfc.AFCCylinderBatch(2, param_sets=[dict(t_step=F(0.002))], init_time=init_time) as env:
        env.reset_sets([1], [0], reset_accumulators=True)
        env.reset([0], reset_accumulators=True)
        obs, rew, done = env.step(np.zeros((2, 2), F))
        assert env.running() == 0 and not done.any()
        t = env.t
        assert t[0] > init_time and t[1] > init_time and np.isfinite(obs).all()


def test_snapshots_follow_the_set(rlfc):
    torch = pytest.importorskip("torch")
    own = [MIXED[0], MIXED[1], MIXED[2]]
    lib = [MIXED[2], MIXED[3]]
    acts = hetero_actions(3, 17)
    with rlfc.AFCCylinderBatch(3, env_params=own, param_sets=lib, n_snapshots=3) as env:
        for k in range(3):
            env.update2(acts if k == 0 else None)
        env.snapshot([2, 1], [0, 1])             # slot 0: tuple MIXED[2], slot 1: tuple MIXED[1]
        d = lambda v: device_ints(torch, v)      # noqa: E731
        e0, s0 = d([0]), d([0])
        torch.cuda.synchronize()
        env.reset_sets_device(e0.data_ptr(), s0.data_ptr(), 1)     # env 0 now holds MIXED[2]
        # a slot of another tuple: skipped, flag bit 1, nothing changes
        before = readouts(env, 0)
        s1 = d([1])
        torch.cuda.synchronize()
        env.restore_device(e0.data_ptr(), s1.data_ptr(), 1)
        assert env.flags()[0] == 2
        assert_readouts(readouts(env, 0), dict(before, flags=2), "refused restore: ")
        with pytest.raises(rlfc.RlfcError, match="another parameter set"):
            env.restore([0], [1])
        # a slot of the set it now holds: accepted, and env 0 continues as env 2 does from the snapshot
        env.restore_device(e0.data_ptr(), s0.data_ptr(), 1)
        assert env.flags()[0] == 0
        env.restore([2], [0])
        for k in range(5):
            f, pr = env.update2(want_probes=True)
            assert_same(f[0], f[2], f"force step {k}")
            assert_same(pr[0], pr[2], f"probes step {k}")
        for nm, x, y in zip(("ux", "uy", "p"), env.get_fields(0), env.get_fields(2)):
            assert_same(x, y, nm)
        # a snapshot of the switched environment goes into an environment that holds the set as its own
        env.snapshot([0], [2])
        env.restore([2], [2])
        assert env.flags()[2] == 0


def test_sensors_keep_their_values(rlfc):
    torch = pytest.importorskip("torch")
    sensors = [("p", 150.0, 96.0), ("ux", 200.5, 90.25), ("uy", 300.0, 100.0)]
    with rlfc.AFCCylinderBatch(2, param_sets=[NEW[0]], sensors=sensors) as env:
        env.update2(hetero_actions(2, 3))
        before = env.sensors()
        d_env, d_set = device_ints(torch, [0, 1]), device_ints(torch, [0, 0])
        torch.cuda.synchronize()
        env.reset_sets_device(d_env.data_ptr(), d_set.data_ptr(), 2)
        assert_same(env.sensors(), before, "sensors")
        assert env.t.tolist() == [0, 0]


def test_device_only_loop(rlfc):
    """step_device + reset_sets_device(where(done, schedule, -1)) on the handle's stream against a second handle driven
    through the same schedule with host rlfc_env_reset_params."""
    torch = pytest.importorskip("torch")
    B, calls = 6, 14
    lib = [NEW[0], NEW[1], NEW[2], MIXED[1]]
    kw = dict(init_time=-1.0, episode_time=0.4)
    rng = np.random.default_rng(5)
    schedule = rng.integers(0, len(lib), size=(calls, B)).astype(np.int32)
    acts = np.clip(rng.normal(0, 0.6, size=(calls, B, 2)), -1, 1).astype(F)
    stream = torch.cuda.Stream()
    resets = 0
    with rlfc.AFCCylinderBatch(B, param_sets=lib, stream=stream.cuda_stream, **kw) as dev, \
            rlfc.AFCCylinderBatch(B, env_params=[{}] * B, **kw) as host:
        ids = device_ints(torch, np.arange(B))
        d_sched = device_ints(torch, schedule)
        d_acts = torch.from_numpy(acts).cuda()
        obs = torch.empty((B, 2), dtype=torch.float32, device="cuda")
        rew = torch.empty(B, dtype=torch.float32, device="cuda")
        done = torch.zeros(B, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        for k in range(calls):
            with torch.cuda.stream(stream):
                dev.step_device(d_acts[k].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr())
                sets = torch.where(done != 0, d_sched[k], torch.full_like(d_sched[k], -1))
                dev.reset_sets_device(ids.data_ptr(), sets.data_ptr(), B, reset_accumulators=True)
                got = (obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy())
            o, r, dn = host.step(acts[k])
            assert_same(got[0], o, f"obs call {k}")
            assert_same(got[1], r, f"reward call {k}")
            assert (got[2] == dn).all(), f"done call {k}"
            fin = np.flatnonzero(dn)
            if len(fin):
                resets += len(fin)
                host.reset(fin, params=[lib[schedule[k][e]] for e in fin], reset_accumulators=True)
        assert resets >= B, "too few episode ends for the test to mean anything"
        assert (dev.params() == host.params()).all()
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), dev.get_fields(e), host.get_fields(e)):
                assert_same(x, y, f"{nm} env {e}")


def test_host_reset_sets_rejections_change_nothing(rlfc):
    with rlfc.AFCCylinderBatch(3, param_sets=[NEW[0], NEW[1]]) as env:
        env.update2(hetero_actions(3))
        before = {e: readouts(env, e) for e in range(3)}
        for ids, sets, msg in (([0, 3], [0, 0], "env id 3 out of range"), ([0, 1], [0, 2], "set 2 out of range"),
                               ([1, 1], [0, 1], "env id 1 listed twice"), ([2], [-1], "set -1 out of range")):
            with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*" + msg):
                env.reset_sets(ids, sets)
        for e in range(3):
            assert_readouts(readouts(env, e), before[e], f"env {e} ")
    with rlfc.AFCCylinderBatch(1) as env:
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*no parameter library"):
            env.reset_sets([0], [0])


def test_library_rejected_with_chained_levels(rlfc):
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*param_sets is not available with the (chained|wavefront)"):
        rlfc.AFCCylinderBatch(1, param_sets=[{}], resolution=64, init_state=None)


def test_no_library_launches_what_it_did(rlfc):
    """A handle without a library launches the same kernels per step as before (the library adds nothing to a step)."""
    with rlfc.AFCCylinderBatch(2, env_params=[{}, {}]) as a, rlfc.AFCCylinderBatch(2, param_sets=[NEW[0]]) as b:
        a.update2(); b.update2()
        la, lb = a.launch_count, b.launch_count
        a.update2(); b.update2()
        assert a.launch_count - la == b.launch_count - lb
