"""Snapshot slots (rlfc_config.n_snapshots, rlfc_env_snapshot / rlfc_env_restore and their _device variants): a restored
environment continues bit-identically to the one the slot was taken from, on every execution path and through every
read-out.  Bar: every float compared with ==, as in test_gpu_parity."""
import numpy as np
import pytest

from test_gpu_adaptive import assert_hierarchy as assert_adaptive_hierarchy
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu

F = np.float32
X = dict(re=300, dR=F(0.2), gR=F(0.3), theta=F(0.9), t_step=F(0.005))


def hetero_actions(B, seed):
    return np.clip(np.random.default_rng(seed).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)


def readouts(env, e, tmp_path=None, tag=""):
    """Everything the read-outs return for environment e (the fields, t, dt, MG iterations, flags, checkpoint text)."""
    out = dict(fields=env.get_fields(e), t=env.t[e], dt=env.dt()[e], iters=tuple(env.mg_iters()[e]), flags=env.flags()[e])
    if tmp_path is not None:
        path = tmp_path / f"{tag}_{e}.bdim"
        env.save_bdim(e, path)
        out["bdim"] = path.read_bytes()
    return out


def assert_readouts(got, want, what):
    for nm, a, b in zip(("ux", "uy", "p"), got["fields"], want["fields"]):
        assert_same(a, b, f"{what}: {nm}")
    for k in ("t", "dt", "iters", "flags"):
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), f"{what}: {k} {got[k]!r} vs {want[k]!r}"
    if "bdim" in want:
        assert got["bdim"] == want["bdim"], f"{what}: save_bdim text differs"


def record(env, envs, steps, acts_at):
    """`steps` solver steps; acts_at(k) = the action array of step k or None.  Per step and environment of `envs`: force,
    probes, t, dt and MG iterations."""
    out = []
    for k in range(steps):
        f, pr = env.update2(acts_at(k), want_probes=True)
        t, dt, it = env.t, env.dt(), env.mg_iters()
        out.append([(f[e].copy(), pr[e].copy(), t[e], dt[e], tuple(it[e])) for e in envs])
    return out


MIXED = [dict(), X, X, dict(re=100), X, dict(theta=F(1.2))]   # envs 1, 2 and 4 share a parameter set

ROUND_TRIP = {
    "default": (dict(), None),
    "no_graph": (dict(), ("RLFC_NO_GRAPH", "1")),
    "groups3": (dict(), ("RLFC_GROUPS", "3")),          # 2 environments per group: 1 -> 4 and 4 -> 2 cross groups
    "resid_tile": (dict(), ("RLFC_RESID", "tile")),
    "resid_march": (dict(), ("RLFC_RESID", "march")),
    "psum_serial": (dict(), ("RLFC_PSUM", "serial")),
    "smoother_chain": (dict(), ("RLFC_SMOOTHER", "chain")),
    "smoother_wave": (dict(), ("RLFC_SMOOTHER", "wave")),
    "adaptive": (dict(adaptive_dt=1), None),
    "env_params": (dict(env_params=MIXED), None),
    "wide_grid": (dict(n_envs=2, resolution=64, init_state=None), None),
}


@pytest.mark.parametrize("case", list(ROUND_TRIP))
def test_round_trip(rlfc, monkeypatch, tmp_path, case):
    kw, envvar = ROUND_TRIP[case]
    if envvar:
        monkeypatch.setenv(*envvar)
    kw = dict(kw)
    B = kw.pop("n_envs", 6)
    src, dst = ([1, 4], [4, 2]) if B == 6 else ([1, 0], [0, 1])
    acts = hetero_actions(B, 1234)
    later = hetero_actions(B, 99)                       # an action change in the middle of the recorded steps
    replay = later.copy()
    for s, d in zip(src, dst):
        replay[d] = later[s]
    with rlfc.AFCCylinderBatch(B, n_snapshots=2, **kw) as env:
        for k in range(5):
            env.update2(acts if k == 0 else None)
        env.snapshot(src, [0, 1])
        at_snap = [readouts(env, e, tmp_path, "src") for e in src]
        rec = record(env, src, 10, lambda k: later if k == 4 else None)
        rec_end = [readouts(env, e) for e in src]
        env.restore(dst, [0, 1])
        for i, e in enumerate(dst):
            assert_readouts(readouts(env, e, tmp_path, "dst"), at_snap[i], f"env {e} right after the restore")
        got = record(env, dst, 10, lambda k: replay if k == 4 else None)
        for k, (r, g) in enumerate(zip(rec, got)):
            for i in range(len(src)):
                for nm, a, b in zip(("force", "probes", "t", "dt", "mg iters"), g[i], r[i]):
                    assert np.array_equal(np.asarray(a), np.asarray(b)), f"{nm} step {k}: env {dst[i]} vs env {src[i]}"
        for i, e in enumerate(dst):
            assert_readouts(readouts(env, e), rec_end[i], f"env {e} after the replay")


# ---- RL steps -------------------------------------------------------------------------------------------------------
RL = dict(init_time=0.2, episode_time=0.6)    # first observation after 43 solver steps, episode over after 80


def rl_actions(k, B):
    return np.tile(np.array([0.8 * np.sin(0.7 * k), -0.8 * np.sin(0.7 * k + 1)], F), (B, 1))


class DeviceRL:
    """rlfc_env_step_device on torch buffers, on the handle's own stream."""

    def __init__(self, torch, env):
        self.torch, self.env, B = torch, env, env.n_envs
        self.act = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        self.obs = torch.zeros((B, 2), dtype=torch.float32, device="cuda")
        self.rew = torch.zeros(B, dtype=torch.float32, device="cuda")
        self.done = torch.zeros(B, dtype=torch.int32, device="cuda")

    def round(self, a):
        self.act.copy_(self.torch.from_numpy(a))
        self.torch.cuda.synchronize()
        self.env.step_device(self.act.data_ptr(), self.obs.data_ptr(), self.rew.data_ptr(), self.done.data_ptr())
        self.torch.cuda.synchronize()
        return self.obs.cpu().numpy(), self.rew.cpu().numpy(), self.done.cpu().numpy(), self.env.running()


def rl_sequence(env, dev, k0):
    """One device round, then three rlfc_env_step calls: obs, reward, done, running() and t of every call."""
    B = env.n_envs
    seq = [dev.round(rl_actions(k0, B)) + (env.t,)]
    for k in range(k0 + 1, k0 + 4):
        o, r, d = env.step(rl_actions(k, B))
        seq.append((o, r, d, env.running(), env.t))
    return seq


@pytest.mark.parametrize("state", ["uncontrolled_start", "mid_window", "boundary", "after_done"])
def test_rl_step_states(rlfc, state):
    """Snapshots taken at the four kinds of RL-step state, restored into another environment: the obs, reward and done
    sequences of the RL steps that follow, and running(), are the source's."""
    torch = pytest.importorskip("torch")
    B = 2
    with rlfc.AFCCylinderBatch(B, n_snapshots=1, **RL) as env:
        dev = DeviceRL(torch, env)
        k = 0
        rounds = {"uncontrolled_start": 1, "mid_window": 2, "boundary": 3, "after_done": 3}[state]
        for _ in range(rounds):
            *_, running = dev.round(rl_actions(k, B))
            k += 1
        if state == "after_done":
            while not env.step(rl_actions(k, B))[2].all():
                k += 1
            k += 1
        t = env.t[0]
        assert {"uncontrolled_start": t <= RL["init_time"], "mid_window": t > RL["init_time"] and running == B,
                "boundary": running == 0, "after_done": t >= RL["episode_time"]}[state], (state, t, running)
        env.snapshot([0], [0])
        want = rl_sequence(env, dev, k)
        env.restore([1, 0], [0, 0])               # env 1 takes env 0's state; env 0 its own, so running() counts both
        got = rl_sequence(env, dev, k)
        for c, (g, w) in enumerate(zip(got, want)):
            for nm, a, b in zip(("obs", "reward", "done", "running", "t"), g, w):
                a, b = np.asarray(a), np.asarray(b)
                assert np.array_equal(a, b), f"{state}: {nm} call {c}: {a!r} vs {b!r}"


# ---- restore from S0 == reset -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("keep", [0, 1])
def test_restore_is_reset(rlfc, keep):
    """restore(S0, keep_accumulators=k) == reset(reset_accumulators=!k), also after a finished episode (where the kept
    accumulators are in the middle of a window)."""
    B = 3
    with rlfc.AFCCylinderBatch(B, n_snapshots=1, **RL) as a, rlfc.AFCCylinderBatch(B, **RL) as b:
        a.reset(None, reset_accumulators=True)
        a.snapshot([0], [0])
        k = 0
        while not a.step(rl_actions(k, B))[2].all():
            b.step(rl_actions(k, B))
            k += 1
        b.step(rl_actions(k, B))
        k += 1
        for which in ([1], [0, 1]):               # finished episodes, then one in progress and one finished
            a.restore(which, [0] * len(which), keep_accumulators=keep)
            b.reset(which, reset_accumulators=not keep)
            for _ in range(4):
                oa, ra, da = a.step(rl_actions(k, B))
                ob, rb, db = b.step(rl_actions(k, B))
                assert_same(oa, ob, f"obs call {k}")
                assert_same(ra, rb, f"reward call {k}")
                assert (da == db).all() and np.array_equal(a.t, b.t), f"done / t call {k}"
                k += 1
        for e in range(B):
            assert_readouts(readouts(a, e), readouts(b, e), f"env {e}")


def test_device_auto_reset_loop(rlfc):
    """step_device + restore_device(arange(B), where(done, S, -1)) == step_device + a host reset of the done ids, with no
    host synchronisation in the first loop.  Environments of two time steps finish at different rounds; each restores its
    own parameter set's slot."""
    torch = pytest.importorskip("torch")
    B = 4
    params = [dict(), dict(t_step=F(0.005)), dict(), dict(t_step=F(0.005))]
    kw = dict(init_time=-1.0, episode_time=0.3, env_params=params)
    stream = torch.cuda.Stream()                  # torch and both handles on one stream: no events needed
    with torch.cuda.stream(stream), rlfc.AFCCylinderBatch(B, n_snapshots=B, stream=stream.cuda_stream, **kw) as a, \
            rlfc.AFCCylinderBatch(B, stream=stream.cuda_stream, **kw) as b:
        a.reset(None, reset_accumulators=True)
        a.snapshot(np.arange(B), np.arange(B))
        ids = torch.arange(B, dtype=torch.int32, device="cuda")
        bufs = [[torch.zeros((B, 2), device="cuda"), torch.zeros(B, device="cuda"), torch.zeros(B, dtype=torch.int32, device="cuda")]
                for _ in range(2)]
        finished = 0
        for k in range(12):
            act = torch.from_numpy(hetero_actions(B, k)).cuda()
            for env, (o, r, d) in zip((a, b), bufs):
                env.step_device(act.data_ptr(), o.data_ptr(), r.data_ptr(), d.data_ptr())
            slots = torch.where(bufs[0][2] != 0, ids, torch.full_like(ids, -1))
            a.restore_device(ids.data_ptr(), slots.data_ptr(), B)
            done_b = bufs[1][2].cpu().numpy()         # (the host reset side synchronises)
            if done_b.any():
                b.reset(np.flatnonzero(done_b), reset_accumulators=True)
                finished += int(done_b.sum())
            for nm, x, y in zip(("obs", "reward", "done"), bufs[0], bufs[1]):
                assert torch.equal(x, y), f"{nm} round {k}"
        # one more round, so that the MG iteration counts and probes (which a reset leaves alone) are rewritten
        for env, (o, r, d) in zip((a, b), bufs):
            env.step_device(act.data_ptr(), o.data_ptr(), r.data_ptr(), d.data_ptr())
        torch.cuda.synchronize()
        assert finished >= B + 1
        assert not a.flags().any()
        for e in range(B):
            assert_readouts(readouts(a, e), readouts(b, e), f"env {e}")


# ---- the rules of the device variants and the host checks -------------------------------------------------------------
def dev_ints(torch, v):
    return torch.tensor(v, dtype=torch.int32, device="cuda")


def all_readouts(env):
    return [readouts(env, e) for e in range(env.n_envs)]


def assert_unchanged(env, before, what):
    for e, r in enumerate(all_readouts(env)):
        assert_readouts(r, before[e], f"{what}: env {e}")


def test_device_rules(rlfc):
    torch = pytest.importorskip("torch")
    B = 4
    with rlfc.AFCCylinderBatch(B, n_snapshots=3) as env:
        env.update2(hetero_actions(B, 5))
        env.update2()
        state = all_readouts(env)
        # out-of-range entries: only the pair (0 -> slot 0) is in range
        e_, s_ = dev_ints(torch, [0, -1, 7, 2, 1]), dev_ints(torch, [0, 1, 1, -5, 3])
        torch.cuda.synchronize()
        env.snapshot_device(e_.data_ptr(), s_.data_ptr(), 5)
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*slot 1 has never been written"):
            env.restore([3], [1])
        # duplicate destinations: the last in-range pair wins
        e_, s_ = dev_ints(torch, [1, 2, 3]), dev_ints(torch, [1, 1, -1])
        torch.cuda.synchronize()
        env.snapshot_device(e_.data_ptr(), s_.data_ptr(), 3)       # slot 1 = env 2
        e_, s_ = dev_ints(torch, [3, 3, 3, -1, 3]), dev_ints(torch, [0, 1, 2, 0, -1])
        torch.cuda.synchronize()
        env.restore_device(e_.data_ptr(), s_.data_ptr(), 5)        # env 3 <- slot 2 (never written): skipped, bit 1
        assert env.flags().tolist() == [0, 0, 0, 2]
        assert_unchanged(env, [*state[:3], dict(state[3], flags=2)], "after a skipped restore")
        e_, s_ = dev_ints(torch, [3, 0, 3]), dev_ints(torch, [2, 4, 1])
        torch.cuda.synchronize()
        env.restore_device(e_.data_ptr(), s_.data_ptr(), 3)        # env 3 <- slot 1 (= env 2); clears bit 1
        assert env.flags().tolist() == [0, 0, 0, 0]
        assert_readouts(readouts(env, 3), state[2], "env 3 after the restore of slot 1")
        env.restore([1], [0])                                      # slot 0 = env 0
        assert_readouts(readouts(env, 1), state[0], "env 1 after the restore of slot 0")
        state = all_readouts(env)
        # host calls that fail change no environment and no slot
        for args, msg in [(([0, 1], [0, 0]), "slot 0 listed twice"), (([4], [0]), "env id 4 out of range"),
                          (([0], [3]), "slot 3 out of range"), (([-1], [0]), "env id -1 out of range")]:
            with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*" + msg):
                env.snapshot(*args)
        for args, msg in [(([2, 2], [0, 1]), "env id 2 listed twice"), (([0, 1], [0, 2]), "slot 2 has never been written"),
                          (([0], [5]), "slot 5 out of range")]:
            with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*" + msg):
                env.restore(*args)
        assert_unchanged(env, state, "after the refused host calls")
        env.restore([0, 2], [1, 0])
        assert_readouts(readouts(env, 0), state[3], "slot 1 after the refused host calls")
        assert_readouts(readouts(env, 2), state[1], "slot 0 after the refused host calls")
    with rlfc.AFCCylinderBatch(1) as env:
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*n_snapshots = 0"):
            env.snapshot([0], [0])
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*n_snapshots = 0"):
            env.restore_device(0, 0, 0)


def test_parameter_mismatch(rlfc):
    torch = pytest.importorskip("torch")
    params = [dict(), X, dict(), X]
    with rlfc.AFCCylinderBatch(4, n_snapshots=2, env_params=params) as env:
        env.update2(hetero_actions(4, 8))
        env.snapshot([0, 1], [0, 1])
        snap1 = readouts(env, 1)
        env.update2()
        state = all_readouts(env)
        with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*slot 0 holds a state of another parameter set than env 1"):
            env.restore([2, 1], [0, 0])
        assert_unchanged(env, state, "after the refused host restore")
        e_, s_ = dev_ints(torch, [1, 2, 3]), dev_ints(torch, [0, 1, 1])
        torch.cuda.synchronize()
        env.restore_device(e_.data_ptr(), s_.data_ptr(), 3)     # 1 <- default set, 2 <- X: skipped; 3 <- X: applies
        assert env.flags().tolist() == [0, 2, 2, 0]
        assert_unchanged(env, [state[0], dict(state[1], flags=2), dict(state[2], flags=2), snap1], "after skipped restores")
        # rlfc_env_reset_params moves the environment to another parameter set: its slots follow what it is now
        env.reset([2], params=[X])
        env.restore([2], [1])
        assert env.flags().tolist() == [0, 2, 0, 0]


def test_adaptive_hierarchy(rlfc, oracle):
    """After a restore the destination's Poisson hierarchy at every level is the source's, and the oracle's
    Poisson(del*dt).restrict()... for the restored dt."""
    B = 3
    with rlfc.AFCCylinderBatch(B, adaptive_dt=1, n_snapshots=1) as env:
        acts = np.array([[0, 0], [0.9, -0.9], [-0.7, 0.2]], F)
        for k in range(4):
            env.update2(acts if k == 0 else None)
        dts = env.dt()
        assert dts[1] != dts[2]
        env.snapshot([1], [0])
        env.restore([2], [0])
        assert env.dt()[2] == dts[1]
        for l in range(env.num_levels):
            for nm in ("lower.x", "lower.y", "inv", "diag"):
                assert_same(env.get_coeffs(2, nm, l), env.get_coeffs(1, nm, l), f"{nm} level {l}")
        assert_adaptive_hierarchy(oracle, env, 2, dts[1])
