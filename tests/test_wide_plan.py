"""Which levels the solver smooths with the chained strip smoother or the wavefront fallback, and which of their kernel
specialisations the GPU tests of tests/test_gpu_wide_shapes.py reach.

plan() mirrors the smoother selection of rlfc_env_create (rlfc_api.cu, the pre-skewed coefficient tables of the
multigrid hierarchy); test_gpu_wide_shapes.test_plan_matches_product checks it against the chained sweep kernels a
profiled step of the product launches.  The coverage guard keeps WIDE_SHAPES and the batches of that file reaching every
strip, row and batch case it was chosen for, and keeps each wide grid carrying at least one case no other grid carries."""
import pytest

from rlfluidcontrol_b200.env import geometry_static
from test_gpu_shapes import SHAPES
from test_gpu_wide_shapes import GROUPS_GRID, MIXED, PRODUCTION, SUM_GRIDS, WIDE_SHAPES
from test_grid_rules import levels, mg_failure

CHAIN_MIN_COLS = 33          # default of RLFC_CHAIN_MIN_COLS


def plan(resolution, xl, yl, mode="default"):
    """Every multigrid level: interior rows and columns, strips of 32 columns (NS) and the columns of the last strip,
    whether it is chained and whether it is a wavefront level.  mode: "default" / "eager" (the same plan),
    "mincols1" (RLFC_CHAIN_MIN_COLS=1), "chain" / "wave" (RLFC_SMOOTHER)."""
    lv = levels(resolution, xl, yl)
    min_cols = 1 if mode == "mincols1" else CHAIN_MIN_COLS
    out, chain_levels = [], 0
    for l, (rows, cols) in enumerate(lv):
        C = -(-cols // 32)                                 # columns per lane of the row pipeline
        wave = C > (8 if l == 0 else 4) or mode == "wave"  # too wide for the row pipeline
        prefer = chain_levels > 0 and l >= 1 and cols >= min_cols
        chained = (mode != "wave" and l < len(lv) - 1 and (mode == "chain" or wave or prefer) and chain_levels == l)
        if chained:
            wave = False
            chain_levels += 1
        ns = -(-cols // 32)
        out.append(dict(rows=rows, cols=cols, NS=ns, last=cols - 32 * (ns - 1), chained=chained, wave=wave,
                        coarsest=l == len(lv) - 1))
    return out


def test_plan_examples():
    """The selection on grids whose plan is known: the default grid chains nothing, 2048x1024 chains every level of at
    least 33 columns, RLFC_SMOOTHER=chain every level but the coarsest."""
    assert not any(lv["chained"] or lv["wave"] for lv in plan(24, 16, 8))
    p = plan(128, 16, 8)
    assert [lv["cols"] for lv in p if lv["chained"]] == [1024, 512, 256, 128, 64]
    assert [lv["chained"] for lv in plan(4, 16, 8, "chain")] == [True] * (len(levels(4, 16, 8)) - 1) + [False]
    assert all(lv["wave"] and not lv["chained"] for lv in plan(8, 7, 33, "wave"))
    p = plan(8, 7, 131)
    assert p[-1]["wave"] and p[-1]["cols"] == 131 and not p[-1]["chained"]


@pytest.mark.parametrize("grid", WIDE_SHAPES + [g for g, _ in SUM_GRIDS])
def test_wide_grids_accepted(rlfc, grid):
    """Every wide grid is one the reference runs and the product builds (MG rules, convexity of the bodies)."""
    assert mg_failure(*grid) is None, grid
    geometry_static("inv", 0, resolution=grid[0], x_lengths=grid[1], y_lengths=grid[2])


def cells(grid):
    return grid[0] ** 2 * grid[1] * grid[2]


def features(wide_shapes):
    """The named cases the GPU tests reach, given the wide shape table (the other tables are fixed)."""
    got = set()
    runs = [(g, "default") for g in wide_shapes] + [(g, "mincols1") for g in wide_shapes]
    runs += [(g, "chain") for g in SHAPES]
    for g, mode in runs:
        p = plan(*g, mode)
        chained = [lv for lv in p if lv["chained"]]
        if any(lv["NS"] == 1 for lv in chained):
            got.add("a chained level with NS = 1")
        if mode != "default":
            continue
        # the natural chained path of the wide grids
        l0 = p[0]
        assert l0["chained"], (g, "level 0 of a wide grid is chained")
        last = l0["last"]
        got.add("level-0 last strip of " + ("1-4" if last <= 4 else "5-15" if last < 16 else "16" if last == 16 else
                                            "17-31" if last < 32 else "32") + " columns")
        got.add("level-0 NS " + ("odd" if l0["NS"] % 2 else "even"))
        r = l0["rows"] % 32
        got.add("level-0 rows " + ("= 0" if r == 0 else "= 16" if r == 16 else "neither 0 nor 16") + " mod 32")
        if any(lv["NS"] == 2 and lv["last"] <= 2 for lv in chained):
            got.add("a chained level with NS = 2 and at most 2 columns in its last strip")
        if any(lv["rows"] < 32 for lv in chained):
            got.add("a chained level with fewer than 32 rows")
        if any(lv["rows"] % 16 for lv in chained):
            got.add("a chained level with rows not a multiple of 16")
        if len(chained) >= 5:
            got.add("five or more chained levels (k_chain_*_L4+)")
        if p[-1]["wave"] and p[-1]["cols"] > 128:
            got.add("a coarsest level wider than 128 columns (wave_smooth<1>)")
    for g, B in SUM_GRIDS + [GROUPS_GRID]:
        if B >= 2 and cells(g) >= 1 << 18:
            got.add("B >= 2 at 262144 cells or more")
    for g, B in (PRODUCTION, MIXED):
        if B >= 128 and plan(*g)[0]["chained"]:
            got.add("B >= 128 on a chained grid")
    return got


REQUIRED = {
    "level-0 last strip of 1-4 columns", "level-0 last strip of 5-15 columns", "level-0 last strip of 16 columns",
    "level-0 last strip of 17-31 columns", "level-0 last strip of 32 columns",
    "level-0 NS odd", "level-0 NS even",
    "a chained level with NS = 2 and at most 2 columns in its last strip", "a chained level with NS = 1",
    "level-0 rows = 0 mod 32", "level-0 rows = 16 mod 32", "level-0 rows neither 0 nor 16 mod 32",
    "a chained level with fewer than 32 rows", "a chained level with rows not a multiple of 16",
    "five or more chained levels (k_chain_*_L4+)", "a coarsest level wider than 128 columns (wave_smooth<1>)",
    "B >= 2 at 262144 cells or more", "B >= 128 on a chained grid",
}


@pytest.mark.parametrize("feature", sorted(REQUIRED))
def test_wide_coverage(feature):
    assert feature in features(WIDE_SHAPES), f"no GPU test reaches: {feature}"


@pytest.mark.parametrize("grid", WIDE_SHAPES, ids=[f"{r}-{x}-{y}" for r, x, y in WIDE_SHAPES])
def test_every_wide_grid_carries_a_case(grid):
    """Without this grid the tables miss a named case: no wide grid is redundant, and deleting one makes
    test_wide_coverage name what is lost."""
    lost = REQUIRED & features(WIDE_SHAPES) - features([g for g in WIDE_SHAPES if g != grid])
    assert lost, f"{grid} carries no case that another grid does not"
