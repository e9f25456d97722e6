"""Flow statistics (rlfc_config.stats_every, rlfc_env_get_stats, rlfc_env_stats_reset[_device]): the device's sums equal, bit
for bit, the same sums taken on the host from rlfc_env_get_fields after every sampled step, on every execution path, through
RL steps and resets; and a handle with statistics computes exactly what a handle without them does."""
import numpy as np
import pytest

from test_flow_stats_host import add_sample
from test_gpu_parity import assert_same, make_oracle
from test_gpu_sensors import MIXED, PATHS, hetero_actions

pytestmark = pytest.mark.gpu

F = np.float32


class Mirror:
    """The statistics of every environment of `env`, kept on the host from get_fields: call after() after every solver step
    (single solver steps: every environment takes part)."""

    def __init__(self, env, k):
        self.k = k
        self.S = np.zeros((env.n_envs, 7, env.n, env.m))
        self.count = np.zeros(env.n_envs, np.int64)
        self.step = np.zeros(env.n_envs, np.int64)

    def after(self, env):
        for e in range(env.n_envs):
            self.step[e] += 1
            if self.step[e] == self.k:
                self.step[e] = 0
                self.count[e] += 1
                add_sample(self.S[e], *env.get_fields(e))

    def reset(self, ids):
        for e in ids:
            self.S[e] = 0
            self.count[e] = self.step[e] = 0

    def check(self, env, what):
        for e in range(env.n_envs):
            count, sums = env.stats_sums(e)
            assert count == self.count[e], f"{what}: env {e} count {count} != {self.count[e]}"
            assert_same(sums, self.S[e], f"{what}: env {e} sums")


def all_sums(env):
    return [env.stats_sums(e) for e in range(env.n_envs)]


def assert_sums_equal(a, b, what):
    for e, ((ca, sa), (cb, sb)) in enumerate(zip(a, b)):
        assert ca == cb, f"{what}: env {e} count {ca} != {cb}"
        assert_same(sa, sb, f"{what}: env {e} sums")


# ---- 1. exact sums --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3])
def test_exact_sums(rlfc, oracle, init_state, k):
    B, steps = 3, 40
    acts = [hetero_actions(B, s) for s in range(4)]
    for a in acts:
        a[0] = 0                                                   # env 0: uncontrolled
    with rlfc.AFCCylinderBatch(B, stats_every=k) as env:
        mirror = Mirror(env, k)
        mirror.check(env, "before any step")
        ref, S_ref = make_oracle(oracle, init_state), np.zeros((7, env.n, env.m))
        for s in range(steps):
            a = acts[s // 10] if s % 10 == 0 else None
            env.update2(a)
            mirror.after(env)
            if k == 1 and s < 5:                                   # the oracle's own fields, accumulated directly
                ref.update2()
                add_sample(S_ref, *ref.get_state())
                if s == 4:
                    count, sums = env.stats_sums(0)
                    assert count == 5
                    assert_same(sums, S_ref, "env 0 vs the oracle's fields over 5 steps")
            if s % 13 == 12:
                mirror.check(env, f"step {s}")
        mirror.check(env, f"after {steps} steps")
        assert mirror.count.tolist() == [steps // k] * B
        st = env.flow_stats(1)
        assert st["count"] == steps // k and np.isfinite(st["var_p"]).all() and st["uv_cov"][1:-1, 1:-1].any()


# ---- 2. execution paths ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", list(PATHS))
def test_execution_paths(rlfc, monkeypatch, case):
    kw, envvar = PATHS[case]
    if envvar:
        monkeypatch.setenv(*envvar)
    kw = dict(kw)
    B = kw.pop("n_envs", 6)
    with rlfc.AFCCylinderBatch(B, stats_every=2, **kw) as env:
        mirror = Mirror(env, 2)
        for s in range(7):
            env.update2(hetero_actions(B, s) if s % 3 == 0 else None)
            mirror.after(env)
            if s in (3, 6):
                mirror.check(env, f"{case} step {s}")


# ---- 3. RL steps ------------------------------------------------------------------------------------------------------------
def test_rl_step_participation(rlfc):
    """step and step_device with the uncontrolled catch-up (default init_time) and a short episode: each environment samples
    every k-th solver step it takes, the finished ones none.  Environment 1 is reset mid-episode (its statistics stay).  After
    that reset step_device rounds are no longer step() calls: an environment at its boundary runs a window in every round
    while environment 1 catches up, so each handle is held to its own solver-step counts."""
    torch = pytest.importorskip("torch")
    B, k, dt = 3, 5, F(0.0075)
    kw = dict(episode_time=1.6)
    with rlfc.AFCCylinderBatch(B, stats_every=1, **kw) as a, rlfc.AFCCylinderBatch(B, stats_every=k, **kw) as b, \
            rlfc.AFCCylinderBatch(B, stats_every=k, **kw) as c:
        act = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        obs = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        before_reset = {h: np.zeros(B, np.int64) for h in "abc"}
        call, done_calls = 0, 0
        while done_calls < 3:
            h = hetero_actions(B, 70 + call) if call else np.zeros((B, 2), F)
            _, _, done = a.step(h)
            b.step(h)
            act.copy_(torch.from_numpy(h))
            torch.cuda.synchronize()
            rounds = 0
            while True:
                c.step_device(act.data_ptr(), obs.data_ptr())
                rounds += 1
                if c.running() == 0:
                    break
            assert rounds > 1 or call > 0, "the first call catches up over several rounds"
            steps = {nm: before_reset[nm] + np.rint(env.t / dt).astype(np.int64)   # solver steps each environment took
                     for nm, env in zip("abc", (a, b, c))}
            assert np.array_equal(steps["a"], steps["b"])
            for nm, env, kk in (("a", a, 1), ("b", b, k), ("c", c, k)):
                count = [env.stats_sums(e)[0] for e in range(B)]
                assert count == (steps[nm] // kk).tolist(), f"call {call}: handle {nm}"
            if call <= 2:                                          # the same steps so far
                assert_sums_equal(all_sums(c), all_sums(b), f"call {call}: step_device vs step")
            if call == 2:
                for nm, env in zip("abc", (a, b, c)):
                    before_reset[nm][1] = steps[nm][1]
                    env.reset([1])
            if done.all():
                if done_calls == 0:
                    finished = all_sums(a), all_sums(b), all_sums(c)
                done_calls += 1
            call += 1
        # two more calls after every episode ended: no environment took a step or a sample
        assert_sums_equal(all_sums(a), finished[0], "finished episodes (k = 1)")
        assert_sums_equal(all_sums(b), finished[1], "finished episodes (k = 5)")
        assert_sums_equal(all_sums(c), finished[2], "finished episodes (k = 5, step_device)")


# ---- 4. resets -----------------------------------------------------------------------------------------------------------
def test_stats_resets(rlfc):
    torch = pytest.importorskip("torch")
    B, k = 4, 2
    with rlfc.AFCCylinderBatch(B, stats_every=k) as env:
        mirror = Mirror(env, k)

        def run(n, seed):
            for s in range(n):
                env.update2(hetero_actions(B, seed + s) if s == 0 else None)
                mirror.after(env)

        run(5, 0)
        env.stats_reset([1, 3])
        mirror.reset([1, 3])
        mirror.check(env, "right after stats_reset([1, 3])")
        run(3, 10)
        mirror.check(env, "3 steps after stats_reset([1, 3])")
        env.stats_reset()
        mirror.reset(range(B))
        run(1, 20)
        mirror.check(env, "1 step after stats_reset(): no sample yet")
        assert not mirror.count.any()
        run(2, 30)
        mirror.check(env, "3 steps after stats_reset()")
        before = all_sums(env)
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*env id 9 out of range"):
            env.stats_reset([0, 9])
        assert_sums_equal(all_sums(env), before, "a refused host reset changes nothing")
        ids = torch.tensor([2, -1, 7, 0], dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        env.stats_reset_device(ids.data_ptr(), 4)
        mirror.reset([2, 0])
        mirror.check(env, "after stats_reset_device([2, -1, 7, 0])")
        run(3, 40)
        mirror.check(env, "3 steps after the device reset")
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\)"):
            env.stats_reset_device(0, -1)


def test_state_changes_leave_statistics_alone(rlfc):
    """Every kind of environment reset, restore and import changes the state the next samples are taken from, never the
    statistics themselves."""
    torch = pytest.importorskip("torch")
    B, k = 4, 1
    lib = [MIXED[1], MIXED[2]]
    with rlfc.AFCCylinderBatch(B, stats_every=k, n_snapshots=1, param_sets=lib) as env:
        mirror = Mirror(env, k)

        def run(n, seed):
            for s in range(n):
                env.update2(hetero_actions(B, seed + s) if s == 0 else None)
                mirror.after(env)

        def dev(a, dtype=torch.int32):
            t = torch.tensor(np.asarray(a), dtype=dtype, device="cuda")
            torch.cuda.synchronize()
            return t

        run(3, 0)
        env.snapshot([0], [0])
        rec = env.export_states([3])
        run(2, 5)
        params = np.zeros(1, dtype=[("re", np.int32), ("dR", F), ("gR", F), ("theta", F), ("t_step", F)])
        params[0] = (250, 0.2, 0.3, 0.9, 0.005)
        packed = dev(params.view(np.int32).reshape(1, 5))
        changes = [   # (restores and imports first: they need the environment's original parameter tuple)
            ("reset", lambda: env.reset([1])),
            ("restore", lambda: env.restore([2], [0])),
            ("restore_device", lambda: env.restore_device(dev([0]).data_ptr(), dev([0]).data_ptr(), 1)),
            ("import_states", lambda: env.import_states([3], rec)),
            ("reset(params=...)", lambda: env.reset([2], params=[dict(re=400)])),
            ("reset_sets", lambda: env.reset_sets([0], [1])),
            ("reset_sets_device", lambda: env.reset_sets_device(dev([3, -1]).data_ptr(), dev([0, 1]).data_ptr(), 2)),
            ("reset_params_device", lambda: env.reset_params_device(dev([1]).data_ptr(), packed.data_ptr(), 1)),
        ]
        for j, (what, change) in enumerate(changes):
            before = all_sums(env)
            change()
            torch.cuda.synchronize()
            assert_sums_equal(all_sums(env), before, what)
            run(2, 100 + 10 * j)
            mirror.check(env, f"2 steps after {what}")
        assert not env.flags().any()
        # the device import: environment 0's record back into environment 0
        buf = torch.empty(len(rec), dtype=torch.uint8, device="cuda")
        env.export_states_device(dev([0]).data_ptr(), 1, buf.data_ptr())
        before = all_sums(env)
        env.import_states_device(dev([0]).data_ptr(), 1, buf.data_ptr(), len(rec))
        torch.cuda.synchronize()
        assert_sums_equal(all_sums(env), before, "import_states_device")
        assert not env.flags().any()


# ---- 5. no perturbation -------------------------------------------------------------------------------------------------
def test_statistics_change_nothing_else(rlfc, monkeypatch):
    monkeypatch.setenv("RLFC_GROUPS", "2")
    B = 4
    sens = [("p", 100.5, 97.0), ("ux", 200.0, 90.5), ("uy", 150.25, 120.0)]
    with rlfc.AFCCylinderBatch(B, stats_every=1, sensors=sens) as a, rlfc.AFCCylinderBatch(B, sensors=sens) as b:
        assert b.cfg.stats_every == 0
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*stats_every = 0"):
            b.stats_sums(0)
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*stats_every = 0"):
            b.stats_reset()
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*out of range"):
            a.stats_sums(B)
        for k in range(3):
            h = hetero_actions(B, k) if k else np.zeros((B, 2), F)
            for x, y, nm in zip(a.step(h), b.step(h), ("obs", "reward", "done")):
                assert_same(x, y, f"call {k}: {nm}")
            assert_same(a.sensors(), b.sensors(), f"call {k}: sensors")
        la, lb = a.launch_count, b.launch_count
        steps = 5
        for k in range(steps):
            fa, pa = a.update2(hetero_actions(B, 10 + k) if k == 0 else None, want_probes=True)
            fb, pb = b.update2(hetero_actions(B, 10 + k) if k == 0 else None, want_probes=True)
            assert_same(fa, fb, f"step {k}: force")
            assert_same(pa, pb, f"step {k}: probes")
            assert_same(a.sensors(), b.sensors(), f"step {k}: sensors")
        assert (a.launch_count - la) - (b.launch_count - lb) == 2 * steps, "one k_flow_stats launch per group and solver step"
        for e in range(B):
            for nm, x, y in zip(("ux", "uy", "p"), a.get_fields(e), b.get_fields(e)):
                assert_same(x, y, f"env {e}: {nm}")
        for nm in ("t", "dt", "mg_iters"):
            x, y = getattr(a, nm), getattr(b, nm)
            x, y = (x(), y()) if callable(x) else (x, y)
            assert np.array_equal(x, y), nm
        # the profile reports the kernel's algorithmic bytes: 3 floats read, 7 doubles read and written per cell
        a.set_profiling(True)
        a.update2()
        prof = {p["name"]: p for p in a.get_profile()}
        assert prof["k_flow_stats"]["launches"] == 1
        assert prof["k_flow_stats"]["bytes_per_launch"] == pytest.approx(124.0 * a.n * a.m * B, rel=1e-12)


def test_create_rejects_bad_stats_every(rlfc):
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*stats_every must be >= 0"):
        rlfc.AFCCylinderBatch(1, stats_every=-1)
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*stats_every is not available in slab mode"):
        rlfc.AFCCylinderBatch(1, stats_every=16, n_devices=2, init_state=None)
