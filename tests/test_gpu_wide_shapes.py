"""The device against the oracle on the solver family that runs levels wider than the row pipeline: the chained strip
smoother (smooth_chain3.cuh, smooth_chain.cuh), the wavefront fallback (smooth_wave.cuh) and the large-domain Field.sum
(exact_sum_kernels.cuh).  Bar: bit-exact (==) on every float, as in test_gpu_parity and test_gpu_shapes.

(a) WIDE_SHAPES: grids of more than 256 columns whose levels have partial last strips (1-4, 5-15, 16, 17-31 columns),
    odd and even strip counts, row counts that are not multiples of 32 or 16 or are below 32, five chained levels and a
    coarsest level wider than 128 columns (wave_smooth<1>), on the graph, eager and RLFC_CHAIN_MIN_COLS=1 paths; the
    row-pipeline SHAPES under RLFC_SMOOTHER=chain / wave; and a check that the levels the product chains are the ones
    tests/test_wide_plan.py predicts (which also holds the coverage guard of these tables).
(b) Batches on the natural chained path: mixed MG iteration counts (converged environments' CTAs take their ticket and
    return) and a batch of 128 in two environment groups (two ticket counters and launch tags).
(c) Field.sum of domains of at least 256 record batches (the condensed-block pass) with B > 1 under every switch of that
    path, the natural three-pass case, and solver steps whose environment groups use the per-group offsets.
(d) The profiled launch sequence (rlfc_env_set_profiling) computes what the graph computes.
(e) Slab mode with strip counts that do not split evenly over the devices (skipped with fewer devices)."""
import numpy as np
import pytest

from test_exact_sum import adversarial
from test_gpu_parity import assert_same, make_oracle
from test_gpu_shapes import ACT, SHAPES, assert_fields, assert_step, grid_kw
from test_gpu_slab import device_count

pytestmark = pytest.mark.gpu

F = np.float32

# (resolution, x_lengths, y_lengths); interior rows x columns per level, NS = strips of 32 columns, "last" = columns of
# the last strip.  Every level but the coarsest is chained (the coarsest runs in the one-CTA kernel).
WIDE_SHAPES = [
    (4, 6, 65),     # 24x260 (NS 9, last 4, 24 rows), 12x130 (NS 5, last 2); coarsest 6x65 on the row pipeline (C = 3)
    (8, 7, 33),     # 56x264 (NS 9, last 8, rows 24 mod 32), 28x132 (last 4), 14x66 (NS 3, last 2); coarsest 7x33
    (8, 6, 34),     # 48x272 (NS 9, last 16, rows 16 mod 32), 24x136, 12x68, 6x34 (NS 2, last 2); coarsest 3x17
    (8, 7, 131),    # 56x1048 (NS 33, last 24), 28x524, 14x262; coarsest 7x131 smoothed by wave_smooth<1>
    (16, 4, 66),    # 64x1056 (NS 33, full strips), five chained levels down to 4x66 (NS 3, last 2); coarsest 2x33
    (20, 16, 16),   # 320x320 (NS 10), 160x160 (NS 5), 80x80 (NS 3, last 16), 40x40 (NS 2, last 8); 20x20, 10x10 chained
                    # (NS 1) with RLFC_CHAIN_MIN_COLS=1
]
WIDE_IDS = [f"{r}-{x}-{y}" for r, x, y in WIDE_SHAPES]
# the path switches the wide shapes run under (tests/test_wide_plan.py mirrors what each one chains)
MODES = {"default": None, "eager": ("RLFC_NO_GRAPH", "1"), "mincols1": ("RLFC_CHAIN_MIN_COLS", "1")}
MIXED = ((8, 6, 34), 7)                 # grid and batch of test_wide_mixed_mg_iterations
PRODUCTION = ((8, 7, 33), 128)          # grid and batch of test_wide_production_batch: two environment groups
SUM_GRIDS = [((32, 16, 16), 5), ((256, 16, 8), 2)]   # test_large_domain_field_sum: 512x512 = 256 record batches, 4096x2048
GROUPS_GRID = ((32, 16, 16), 2)         # test_large_domain_groups


def run_impulsive(rlfc, oracle, grid, steps=4):
    """Impulsive start, a batch of two (ACT on env 0, none on env 1): forces, probes and MG iteration counts after every
    step, all fields including ghosts at the end, == the oracle's."""
    kw, okw = grid_kw(grid)
    refs = [oracle.OracleEnv(literal=False, **okw) for _ in range(2)]
    refs[0].set_xi(*ACT)
    act = np.stack([ACT, F([0, 0])])
    with rlfc.AFCCylinderBatch(2, init_state=None, **kw) as env:
        assert (env.n, env.m) == (refs[0].n, refs[0].m)
        for k in range(steps):
            f, pr = env.update2(act if k == 0 else None, want_probes=True)
            its = env.mg_iters()
            for e, ref in enumerate(refs):
                ref.update2()
                assert_step(f, pr, its, e, ref, f"env {e} step {k}")
        for e, ref in enumerate(refs):
            assert_fields(env, e, ref, f"env {e}")


# ---- (a) shapes -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("grid", WIDE_SHAPES, ids=WIDE_IDS)
def test_wide_shape(rlfc, oracle, monkeypatch, grid, mode):
    if MODES[mode]:
        monkeypatch.setenv(*MODES[mode])
    run_impulsive(rlfc, oracle, grid)


@pytest.mark.parametrize("smoother", ["chain", "wave"])
@pytest.mark.parametrize("grid", SHAPES, ids=[f"{r}-{x}-{y}" for r, x, y in SHAPES])
def test_forced_smoothers_on_row_shapes(rlfc, oracle, monkeypatch, grid, smoother):
    """The row-pipeline shape table through the chained smoother (every level but the coarsest: one-strip levels, 28-
    and 36-row levels, partial strips of every width class) and through the wavefront smoother on every level."""
    monkeypatch.setenv("RLFC_SMOOTHER", smoother)
    run_impulsive(rlfc, oracle, grid)


def sweep_kernels(levels):
    """Profile names of the chained sweep kernels of the chained levels `levels` (rlfc_api.cu project_eager)."""
    return {f"k_chain_sweeps_L{l}" if l < 4 else "k_chain_sweeps_L4+" for l in levels}


@pytest.mark.parametrize("mode", ["default", "mincols1"])
@pytest.mark.parametrize("grid", WIDE_SHAPES, ids=WIDE_IDS)
def test_plan_matches_product(rlfc, monkeypatch, grid, mode):
    """One profiled step lists a chained sweep kernel for exactly the levels test_wide_plan.plan() chains, so the
    coverage the CPU guard reasons about is the coverage the product runs."""
    from test_wide_plan import plan
    if MODES[mode]:
        monkeypatch.setenv(*MODES[mode])
    kw, _ = grid_kw(grid)
    want = sweep_kernels(l for l, lv in enumerate(plan(*grid, mode)) if lv["chained"])
    with rlfc.AFCCylinderBatch(1, init_state=None, **kw) as env:
        env.set_profiling(True)
        env.update2(np.array([ACT]))
        got = {p["name"] for p in env.get_profile() if p["launches"] > 0 and p["name"].startswith("k_chain_sweeps_L")}
    assert got == want, f"chained sweep kernels {sorted(got)}, the plan predicts {sorted(want)}"


# ---- (b) batches on the chained path ------------------------------------------------------------------------------------

def developed_state(oracle, okw, steps=40):
    dev = oracle.OracleEnv(literal=False, **okw)
    for _ in range(steps):
        dev.update2()
    return dev.get_state()


@pytest.mark.parametrize("envvar", [None, ("RLFC_NO_GRAPH", "1"), ("RLFC_GROUPS", "3")], ids=["graph", "eager", "groups3"])
def test_wide_mixed_mg_iterations(rlfc, oracle, monkeypatch, envvar):
    """48x272, 7 environments: 1, 2, 4, 6 resume a developed wake (few MG iterations), 0, 3, 5 start from rest (many),
    each with its own action.  Environments that converge early leave the chained sweeps while the others go on."""
    if envvar:
        monkeypatch.setenv(*envvar)
    grid, B = MIXED
    kw, okw = grid_kw(grid)
    developed = (1, 2, 4, 6)
    dev_state = developed_state(oracle, okw)
    acts = np.clip(np.random.default_rng(78).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)
    refs = []
    for e in range(B):
        r = oracle.OracleEnv(literal=False, **okw)
        if e in developed:
            r.set_state(*dev_state)
        r.set_xi(*acts[e])
        refs.append(r)
    mixed = False
    with rlfc.AFCCylinderBatch(B, init_state=None, **kw) as env:
        for e in developed:
            env.set_fields(e, *dev_state)
        for k in range(4):
            f, pr = env.update2(acts if k == 0 else None, want_probes=True)
            its = env.mg_iters()
            mixed |= len({tuple(i) for i in its}) > 1
            for e, r in enumerate(refs):
                r.update2()
                assert_step(f, pr, its, e, r, f"env {e} step {k}")
        for e, r in enumerate(refs):
            assert_fields(env, e, r, f"env {e}")
    assert mixed, "the batch never had environments with different MG iteration counts in one step"


def test_wide_production_batch(rlfc, oracle):
    """56x264 x 128 environments (about 1.9 Mi cells): two environment groups by default, each with its own ticket
    counters and launch tags on four chained levels.  Six classes {rest, developed} x three actions, spread over the batch
    by a seeded permutation; the oracle runs once per class."""
    grid, B = PRODUCTION
    kw, okw = grid_kw(grid)
    dev_state = developed_state(oracle, okw)
    actions = F([[0, 0], [0.6, -0.4], [-0.9, 0.8]])
    classes = [(developed, a) for developed in (False, True) for a in range(3)]
    refs = []
    for developed, a in classes:
        r = oracle.OracleEnv(literal=False, **okw)
        if developed:
            r.set_state(*dev_state)
        r.set_xi(*actions[a])
        refs.append(r)
    cls = np.random.default_rng(2025).permutation(np.arange(B) % len(classes))
    acts = actions[[classes[c][1] for c in cls]]
    mixed = False
    with rlfc.AFCCylinderBatch(B, init_state=None, **kw) as env:
        for e in np.flatnonzero([classes[c][0] for c in cls]):
            env.set_fields(int(e), *dev_state)
        for k in range(3):
            f, pr = env.update2(acts if k == 0 else None, want_probes=True)
            its = env.mg_iters()
            for r in refs:
                r.update2()
            assert_same(f, np.array([r.force() for r in refs], F)[cls], f"forces step {k}")
            assert_same(pr, np.array([r.probes(32) for r in refs])[cls], f"probes step {k}")
            want_its = np.array([r.mg_iters() for r in refs])[cls]
            assert np.array_equal(its, want_its), f"mg iters step {k}: first env {np.argwhere(its != want_its)[0][0]}"
            mixed |= len({tuple(i) for i in its}) > 1
        for e in range(B):
            assert_fields(env, e, refs[cls[e]], f"env {e} (class {cls[e]})")
    assert mixed, "the batch never had environments with different MG iteration counts in one step"


# ---- (c) large-domain Field.sum --------------------------------------------------------------------------------------

def wide_t_step(resolution):
    """t_step = 0.18/resolution keeps dt at 0.18 grid units, as in test_gpu_parity.test_wide_grid."""
    return float(F(0.18) / F(resolution))


def interior_field(n, m, values, ghost):
    """A pressure field whose interior holds `values` in Field.sum's order and whose ghost cells hold `ghost` (Field.sum
    must not read them)."""
    p = np.full((n, m), ghost, F)
    p[1:-1, 1:-1] = np.asarray(values, F).reshape(n - 2, m - 2)
    return p


def family(kind, N, rng):
    """test_exact_sum.adversarial(kind), or "parked2": test_device_field_sum_large_domain's case 6, the accumulator
    parked next to 2.0 by its first addend, then tiny signed addends."""
    if kind != "parked2":
        return adversarial(kind, N, rng)
    a = (1e-6 * rng.standard_normal(N)).astype(F)
    a[0] = 2.0
    return a


def assert_sums(env, oracle, fields, what):
    got = env.field_sum()
    for e, p in enumerate(fields):
        want = F(oracle.Field(env.n, env.m, values=p).sum())
        assert got[e].tobytes() == want.tobytes() or (np.isnan(got[e]) and np.isnan(want)), \
            (what, e, got[e], want, env.field_sum_stats()[e].tolist())


@pytest.mark.parametrize("envvar", [None, ("RLFC_GROUPS", "2"), ("RLFC_XS_PASSES", "3"), ("RLFC_XS_REFINE", "0"),
                                    ("RLFC_XS_REDO", "serial")],
                         ids=["default", "groups2", "passes3", "norefine", "redo-serial"])
def test_large_domain_field_sum_batch(rlfc, oracle, monkeypatch, envvar):
    """512x512 (exactly the 256 record batches from which the condensed-block pass runs), 5 environments, each a
    different adversarial family; NaN, huge and zero ghost cells.  Every environment's sum == the oracle's serial loop."""
    if envvar:
        monkeypatch.setenv(*envvar)
    (res, xl, yl), B = SUM_GRIDS[0]
    rng = np.random.default_rng(31)
    with rlfc.AFCCylinderBatch(B, init_state=None, resolution=res, x_lengths=xl, y_lengths=yl,
                               t_step=wide_t_step(res)) as env:
        n, m = env.n, env.m
        N = (n - 2) * (m - 2)
        assert N >= 256 * 1024
        for rnd, kinds in enumerate([(1, 5, 8, 9, 12), (2, 3, 7, 11, "parked2"), (0, 4, 6, 13, "parked2")]):
            fields = []
            for e, kind in enumerate(kinds):
                fields.append(interior_field(n, m, family(kind, N, rng), [np.nan, 1e30, 0.0, -7.0, np.inf][e]))
                env.set_fields(e, None, None, fields[-1])
            assert_sums(env, oracle, fields, f"round {rnd}")


def test_large_domain_field_sum_three_pass(rlfc, oracle):
    """4096x2048 (8 Mi cells: the three-pass tables and the helper-warp kernel by default), 2 environments, families that
    park the accumulator next to a power of two."""
    (res, xl, yl), B = SUM_GRIDS[1]
    rng = np.random.default_rng(32)
    with rlfc.AFCCylinderBatch(B, init_state=None, resolution=res, x_lengths=xl, y_lengths=yl,
                               t_step=wide_t_step(res)) as env:
        n, m = env.n, env.m
        N = (n - 2) * (m - 2)
        for rnd, kinds in enumerate([(5, 8), (9, "parked2")]):
            fields = [interior_field(n, m, family(k, N, rng), np.nan) for k in kinds]
            for e, p in enumerate(fields):
                env.set_fields(e, None, None, p)
            assert_sums(env, oracle, fields, f"round {rnd}")


@pytest.mark.parametrize("groups", [1, 2])
def test_large_domain_groups(rlfc, oracle, monkeypatch, groups):
    """512x512 with 2 environments in one or two groups: the projection's Field.sum (condensed blocks) and the chained
    levels of group 1 work at their per-group offsets.  Impulsive start, ACT on env 0, 2 steps."""
    monkeypatch.setenv("RLFC_GROUPS", str(groups))
    (res, xl, yl), B = GROUPS_GRID
    t_step = wide_t_step(res)
    refs = [oracle.OracleEnv(literal=False, resolution=res, xLengths=xl, yLengths=yl, tStep=t_step) for _ in range(B)]
    refs[0].set_xi(*ACT)
    act = np.stack([ACT, F([0, 0])])
    with rlfc.AFCCylinderBatch(B, init_state=None, resolution=res, x_lengths=xl, y_lengths=yl, t_step=t_step) as env:
        for k in range(2):
            f, pr = env.update2(act if k == 0 else None, want_probes=True)
            its = env.mg_iters()
            for e, ref in enumerate(refs):
                ref.update2()
                assert_step(f, pr, its, e, ref, f"env {e} step {k}")
        for e, ref in enumerate(refs):
            assert_fields(env, e, ref, f"env {e}")


# ---- (d) the profiled launch path ---------------------------------------------------------------------------------------

def record(env, steps, acts):
    out = []
    for k in range(steps):
        f, pr = env.update2(acts if k == 0 else None, want_probes=True)
        out.append((f.copy(), pr.copy(), env.mg_iters().copy()))
    return out, [env.get_fields(e) for e in range(env.n_envs)]


@pytest.mark.parametrize("grid,B", [(None, 7), ((8, 6, 34), 2), ((16, 4, 66), 2)],
                         ids=["default-B7", "48x272-B2", "64x1056-B2"])
def test_profiled_path_equals_oracle(rlfc, oracle, init_state, grid, B):
    """rlfc_env_set_profiling(1) before any step (the launch sequence bench.py times kernel by kernel): 3 steps == the
    oracle and == an unprofiled run of the same batch."""
    kw, okw = grid_kw(grid) if grid else ({}, {})
    acts = np.clip(np.random.default_rng(79).normal(0, 0.6, size=(B, 2)), -1, 1).astype(F)
    start = None if grid else init_state
    runs = []
    for profiled in (True, False):
        with rlfc.AFCCylinderBatch(B, init_state=None if grid else "default", **kw) as env:
            if profiled:
                env.set_profiling(True)
            runs.append(record(env, 3, acts))
            if profiled:
                names = {p["name"] for p in env.get_profile() if p["launches"] > 0}
                assert names, "profiling recorded no launch"
                assert ("k_chain_sweeps_L0" in names) == (grid is not None), sorted(names)
    refs = [make_oracle(oracle, start, **okw) for _ in range(B)]
    for e, r in enumerate(refs):
        r.set_xi(*acts[e])
    (steps, fields), (steps_g, fields_g) = runs
    for k, ((f, pr, its), (fg, prg, itsg)) in enumerate(zip(steps, steps_g)):
        for r in refs:
            r.update2()
        for e, r in enumerate(refs):
            assert_step(f, pr, its, e, r, f"env {e} step {k}")
        assert_same(f, fg, f"forces step {k} (profiled vs graph)")
        assert_same(pr, prg, f"probes step {k} (profiled vs graph)")
        assert np.array_equal(its, itsg), f"mg iters step {k} (profiled vs graph)"
    for e, r in enumerate(refs):
        for nm, a, b, c in zip(("ux", "uy", "p"), fields[e], fields_g[e], r.get_state()):
            assert_same(a, c, f"{nm} env {e}")
            assert_same(a, b, f"{nm} env {e} (profiled vs graph)")


# ---- (e) slab mode with uneven splits -------------------------------------------------------------------------------------

def slab_run(rlfc, grid, n_devices):
    kw, _ = grid_kw(grid)
    with rlfc.AFCCylinderBatch(1, init_state=None, n_devices=n_devices, **kw) as env:
        out = []
        for k in range(2):
            f, pr = env.update2(np.array([ACT]) if k == 0 else None, want_probes=True)
            out.append((f.copy(), pr.copy(), env.mg_iters().copy()))
        return out, env.get_fields(0)


@pytest.mark.parametrize("n_devices", [2, 3])
@pytest.mark.parametrize("grid", [(8, 6, 34), (8, 7, 131)], ids=["48x272", "56x1048"])
def test_slab_uneven_splits(rlfc, oracle, grid, n_devices):
    """48x272 (NS 9, 5, 3, 2: uneven splits, and on 3 devices a device without a strip of the 2-strip level) and 56x1048
    (NS 33, 17, 9) on 2 and 3 devices: == the oracle and == the single-device run, impulsive start, ACT, 2 steps."""
    if device_count() < n_devices:
        pytest.skip(f"needs {n_devices} GPUs")
    _, okw = grid_kw(grid)
    ref = oracle.OracleEnv(literal=False, **okw)
    ref.set_xi(*ACT)
    single, single_fields = slab_run(rlfc, grid, 1)
    got, got_fields = slab_run(rlfc, grid, n_devices)
    for k, ((f, pr, its), (fs, prs, itss)) in enumerate(zip(got, single)):
        ref.update2()
        assert_step(f, pr, its, 0, ref, f"step {k}")
        assert_same(f, fs, f"force step {k} (vs one device)")
        assert_same(pr, prs, f"probes step {k} (vs one device)")
        assert np.array_equal(its, itss), f"mg iters step {k} (vs one device)"
    for nm, a, b, c in zip(("ux", "uy", "p"), got_fields, single_fields, ref.get_state()):
        assert_same(a, c, nm)
        assert_same(a, b, f"{nm} (vs one device)")
