"""The device against the oracle at the grid shapes and batches its kernels specialise on.  Bar: bit-exact (==) on every
float, as in test_gpu_parity.

(a) SHAPES reaches every columns-per-lane count C = ceil(columns/32) of the level-0 row smoother (1..8) and of the coarse
    row pipeline (1..4), lanes that own fewer than C columns, fewer than 32 lanes and row counts that are not multiples
    of 16 or 32 (the partial last chunk of k_advdif, k_mg_up0_blk and the residual kernels); tests/test_grid_rules.py
    checks that the table keeps doing so.  Every grid runs in shared mode (default paths, the marching residual kernel,
    the row pipeline on the small coarse levels) and with adaptive_dt, whose device-built hierarchy is compared level
    by level.
(b) A batch whose environments need different numbers of MG iterations in the same solve.
(c) Batches of at least 8 Mi cells on ragged grids: the production kernels (48-row k_advdif, marching residual, two and
    four environment groups, segment-summary and serial Field.sum) with mixed states and actions."""
import numpy as np
import pytest

from test_gpu_adaptive import assert_hierarchy
from test_gpu_parity import assert_same, make_oracle

pytestmark = pytest.mark.gpu

F = np.float32

# (resolution, x_lengths, y_lengths): interior rows x columns = x_lengths*resolution x y_lengths*resolution
SHAPES = [
    (4, 16, 8),     # 64x32: level-0 C = 1 with 32 lanes; every coarse level tiny
    (4, 9, 7),      # 36x28: C = 1 with 28 lanes; rows = 4 mod 16; coarsest 9x7
    (2, 20, 4),     # 40x8: 8 lanes; body band next to the boundary (literal setBC kernels); up to 10 MG iterations
    (8, 9, 5),      # 72x40: C = 2 with 20 lanes; rows = 8 mod 16
    (8, 28, 7),     # 224x56: tall, C = 2
    (8, 7, 17),     # 56x136: C = 5, last lane 1 column; level 1 C = 3, last lane 2 columns
    (16, 7, 9),     # 112x144: C = 5, last lane 4 columns; rows = 16 mod 32
    (20, 16, 8),    # 320x160: C = 5, full lanes; level 1 27 lanes, last lane 2 columns
    (16, 4, 13),    # 64x208: C = 7, 30 lanes, last lane 5 columns; level 1 104 columns (coarse C = 4)
    (28, 8, 8),     # 224x224: C = 7, full lanes; level 1 coarse C = 4; two marching windows (196 + 28 columns)
    (8, 8, 30),     # 64x240: C = 8, 30 lanes; level 1 120 columns (coarse C = 4)
    (4, 14, 58),    # 56x232: C = 8, 29 lanes; rows = 8 mod 16; coarsest 7x29
    (32, 8, 8),     # 256x256: C = 8, full lanes; coarse C = 4 with 32 lanes; 8 levels down to 2x2
]
ACT = F([0.4, -0.7])


def grid_kw(g):
    return dict(resolution=g[0], x_lengths=g[1], y_lengths=g[2]), dict(resolution=g[0], xLengths=g[1], yLengths=g[2])


def assert_fields(env, e, ref, what):
    for nm, a, b in zip(("ux", "uy", "p"), env.get_fields(e), ref.get_state()):
        assert_same(a, b, f"{nm} {what}")


def assert_step(f, pr, its, e, ref, what):
    assert_same(f[e], np.array(ref.force(), F), f"force {what}")
    assert_same(pr[e], ref.probes(32), f"probes {what}")
    assert tuple(its[e]) == ref.mg_iters(), f"mg iters {what}: {tuple(its[e])} vs {ref.mg_iters()}"


@pytest.mark.parametrize("envvar", [None, ("RLFC_RESID", "march"), ("RLFC_TINY", "0")], ids=["default", "march", "notiny"])
@pytest.mark.parametrize("grid", SHAPES, ids=[f"{r}-{x}-{y}" for r, x, y in SHAPES])
def test_shape_shared(rlfc, oracle, monkeypatch, grid, envvar):
    """Impulsive start, a batch of two (a non-zero action on env 0, none on env 1), 4 solver steps."""
    if envvar:
        monkeypatch.setenv(*envvar)
    kw, okw = grid_kw(grid)
    refs = [oracle.OracleEnv(literal=False, **okw) for _ in range(2)]
    refs[0].set_xi(*ACT)
    act = np.stack([ACT, F([0, 0])])
    with rlfc.AFCCylinderBatch(2, init_state=None, **kw) as env:
        assert (env.n, env.m) == (refs[0].n, refs[0].m)
        for k in range(4):
            f, pr = env.update2(act if k == 0 else None, want_probes=True)
            its = env.mg_iters()
            for e, ref in enumerate(refs):
                ref.update2()
                assert_step(f, pr, its, e, ref, f"env {e} step {k}")
        for e, ref in enumerate(refs):
            assert_fields(env, e, ref, f"env {e}")


@pytest.mark.parametrize("grid", SHAPES, ids=[f"{r}-{x}-{y}" for r, x, y in SHAPES])
def test_shape_adaptive(rlfc, oracle, grid):
    """adaptive_dt = 1: 6 steps, then env 0's device-built hierarchy (every level's lower.x/lower.y/inv/diag, ragged
    lanes included) against the oracle's for its dt."""
    kw, okw = grid_kw(grid)
    refs = [oracle.OracleEnv(literal=False, **okw) for _ in range(2)]
    refs[0].set_xi(*ACT)
    act = np.stack([ACT, F([0, 0])])
    with rlfc.AFCCylinderBatch(2, init_state=None, adaptive_dt=1, **kw) as env:
        for k in range(6):
            f, pr = env.update2(act if k == 0 else None, want_probes=True)
            its, dts = env.mg_iters(), env.dt()
            for e, ref in enumerate(refs):
                ref.update_adaptive()
                assert dts[e] == ref.dt, f"dt env {e} step {k}: {dts[e]!r} vs {ref.dt!r}"
                assert_step(f, pr, its, e, ref, f"env {e} step {k}")
        for e, ref in enumerate(refs):
            assert_fields(env, e, ref, f"env {e}")
        assert_hierarchy(oracle, env, 0, env.dt()[0])


@pytest.mark.parametrize("envvar,adaptive", [(None, 0), (("RLFC_NO_GRAPH", "1"), 0), (("RLFC_GROUPS", "3"), 0), (None, 1)],
                         ids=["graph", "eager", "groups3", "adaptive"])
def test_mixed_mg_iterations(rlfc, oracle, init_state, monkeypatch, envvar, adaptive):
    """Default grid, 7 environments: 1, 2, 4, 6 resume the developed wake (one MG iteration per solve), 0, 3, 5 start
    from rest (several), each with its own action.  The MG loop must keep iterating the environments that still need
    it and leave the converged ones untouched."""
    if envvar:
        monkeypatch.setenv(*envvar)
    B = 7
    developed = (1, 2, 4, 6)
    acts = np.clip(np.random.default_rng(77).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)
    refs = [make_oracle(oracle, init_state if e in developed else None) for e in range(B)]
    for e, r in enumerate(refs):
        r.set_xi(*acts[e])
    mixed = False
    with rlfc.AFCCylinderBatch(B, init_state=None, adaptive_dt=adaptive) as env:
        for e in developed:
            env.set_fields(e, init_state["ux"], init_state["uy"], init_state["p"])
        for k in range(4):
            f, pr = env.update2(acts if k == 0 else None, want_probes=True)
            its, dts = env.mg_iters(), env.dt()
            mixed |= len({tuple(r) for r in its}) > 1
            for e, r in enumerate(refs):
                r.update_adaptive() if adaptive else r.update2()
                if adaptive:
                    assert dts[e] == r.dt, f"dt env {e} step {k}"
                assert_step(f, pr, its, e, r, f"env {e} step {k}")
        for e, r in enumerate(refs):
            assert_fields(env, e, r, f"env {e}")
    assert mixed, "the batch never had environments with different MG iteration counts in one step"


@pytest.mark.parametrize("grid,B,envvar", [((28, 8, 8), 168, None), ((16, 7, 9), 521, None),
                                           ((16, 7, 9), 521, ("RLFC_NO_GRAPH", "1"))],
                         ids=["224x224-B168", "112x144-B521", "112x144-B521-eager"])
def test_production_thresholds(rlfc, oracle, monkeypatch, grid, B, envvar):
    """B x cells >= 8 Mi on ragged grids: 48-row k_advdif with a 32- or 16-row tail, the marching residual kernel over
    partial windows and row tails, two groups with segment-summary Field.sum (B = 168) or four groups with the serial
    Field.sum chain (B = 521).  Six classes {rest, developed} x three actions, spread over the batch by a seeded
    permutation so that neighbouring environments, CTA rows and groups mix states and MG iteration counts."""
    if envvar:
        monkeypatch.setenv(*envvar)
    kw, okw = grid_kw(grid)
    assert B * grid[0] ** 2 * grid[1] * grid[2] >= 8 << 20
    dev = oracle.OracleEnv(literal=False, **okw)
    for _ in range(40):
        dev.update2()
    dev_state = dev.get_state()
    actions = F([[0, 0], [0.6, -0.4], [-0.9, 0.8]])
    classes = [(developed, a) for developed in (False, True) for a in range(3)]
    refs = []
    for developed, a in classes:
        r = oracle.OracleEnv(literal=False, **okw)
        if developed:
            r.set_state(*dev_state)
        r.set_xi(*actions[a])
        refs.append(r)
    cls = np.random.default_rng(2024).permutation(np.arange(B) % len(classes))
    acts = actions[[classes[c][1] for c in cls]]
    with rlfc.AFCCylinderBatch(B, init_state=None, **kw) as env:
        for e in np.flatnonzero([classes[c][0] for c in cls]):
            env.set_fields(int(e), *dev_state)
        mixed = False
        for k in range(3):
            f = env.update2(acts if k == 0 else None)
            its = env.mg_iters()
            for r in refs:
                r.update2()
            want_f = np.array([r.force() for r in refs], F)[cls]
            want_its = np.array([r.mg_iters() for r in refs])[cls]
            assert_same(f, want_f, f"forces step {k}")
            assert np.array_equal(its, want_its), f"mg iters step {k}: first env {np.argwhere(its != want_its)[0][0]}"
            mixed |= len({tuple(i) for i in its}) > 1
        for e in range(B):
            assert_fields(env, e, refs[cls[e]], f"env {e} (class {cls[e]})")
    assert mixed, "the batch never had environments with different MG iteration counts in one step"
