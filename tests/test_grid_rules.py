"""Which grids the solver accepts, and which kernel specialisations the GPU shape tests reach.

The reference's multigrid (MG.pde) can only run some grids.  The product (`rlfc_geometry_static`, the same
`build_geometry` as `rlfc_env_create`) must reject exactly those with RLFC_EGRID, and the oracle must refuse them
instead of running into undefined behaviour or exit().  The coverage guard keeps the shape table of
tests/test_gpu_shapes.py reaching every columns-per-lane instantiation of the row smoothers and every ragged lane and
row tail it was chosen for."""
import itertools

import pytest

from rlfluidcontrol_b200.env import geometry_static
from test_gpu_parity import OTHER_GRIDS
from test_gpu_shapes import SHAPES

RLFC_EGRID = -6


def mg_failure(resolution, xl, yl):
    """How the reference's first solve fails on the grid: None (it runs), "exit" or "odd".  Level sizes n x m include
    the ghosts (AFCCylinder.pde:12-13, BDIM.pde:42)."""
    n, m = xl * resolution + 2, yl * resolution + 2
    odd = (n - 2) % 2 or (m - 2) % 2
    # MG.vCycle (MG.pde:68-77) always restricts the finest level and recurses into a coarse level while it is divisible;
    # MG.divisible exits on the first coarse level that is not, with both sides > 9 -- before any increment
    while True:
        n, m = (n - 2) // 2 + 2, (m - 2) // 2 + 2                          # MG.restrict, MG.pde:108-122
        if (n - 2) % 2 == 0 and (m - 2) % 2 == 0 and n > 4 and m > 4:      # MG.divisible, MG.pde:99-100
            continue
        if n > 9 and m > 9:                                                  # MG.pde:101-104: exit()
            return "exit"
        break
    # back on level 0, MG.prolongate (MG.pde:139-152) returns an even-sized correction and MG.increment (MG.pde:94-97)
    # adds it over the whole fine field: level 0 must be even
    return "odd" if odd else None


def mg_rejects(resolution, xl, yl):
    return mg_failure(resolution, xl, yl) is not None


MESSAGE = {"exit": "MultiGrid requires", "odd": "MG.prolongate / MG.increment"}


def product_result(rlfc, resolution, xl, yl):
    """(return code, error message) of rlfc_geometry_static."""
    try:
        geometry_static("inv", 0, resolution=resolution, x_lengths=xl, y_lengths=yl)
    except rlfc.RlfcError as e:
        return int(str(e).split("(")[1].split(")")[0]), str(e)
    return 0, ""


def product_rc(rlfc, resolution, xl, yl):
    return product_result(rlfc, resolution, xl, yl)[0]


def oracle_refuses(oracle, resolution, xl, yl):
    try:
        oracle.OracleEnv(literal=False, resolution=resolution, xLengths=xl, yLengths=yl).close()
    except ValueError:
        return True
    return False


def test_acceptance_sweep(rlfc, oracle):
    """resolution 2..12 x x_lengths 1..20 x y_lengths 1..20: RLFC_EGRID exactly where the oracle refuses, and both
    exactly where MG.pde cannot run, with the message of the failure the reference would meet first.  Grids whose
    bodies fail the convexity test (RLFC_EINVAL, tiny resolutions) are another rule and are not compared."""
    seen = {None: 0, "exit": 0, "odd": 0}
    for res, xl, yl in itertools.product(range(2, 13), range(1, 21), range(1, 21)):
        rc, msg = product_result(rlfc, res, xl, yl)
        if rc not in (0, RLFC_EGRID):
            continue
        want = mg_failure(res, xl, yl)
        seen[want] += 1
        assert (rc == RLFC_EGRID) == (want is not None), (res, xl, yl, rc)
        assert want is None or MESSAGE[want] in msg, (res, xl, yl, msg)
        assert oracle_refuses(oracle, res, xl, yl) == (want is not None), (res, xl, yl)
    assert min(seen.values()) > 100, seen


@pytest.mark.parametrize("grid", [(5, 7, 3), (3, 9, 5)])
def test_odd_level0_rejected(rlfc, oracle, grid):
    """35x15 and 27x15 interiors: odd level 0, whose coarse levels (17x7, 13x7) stop the recursion without exit()."""
    with pytest.raises(rlfc.RlfcError, match=r"\(-6\).*even.*MG.prolongate / MG.increment"):
        geometry_static("inv", 0, resolution=grid[0], x_lengths=grid[1], y_lengths=grid[2])
    assert oracle_refuses(oracle, *grid)


@pytest.mark.parametrize("grid", [(50, 3, 3), (7, 5, 3), (25, 3, 3)])
def test_coarse_rule_rejected(rlfc, oracle, grid):
    """150x150 coarsens to 75x75, and the odd 35x21 and 75x75 to 17x10 and 37x37: a coarse level that is not divisible
    with both sides > 9, where MG.divisible (MG.pde:101-104) exits before any increment reaches level 0."""
    with pytest.raises(rlfc.RlfcError, match=r"\(-6\).*MultiGrid requires"):
        geometry_static("inv", 0, resolution=grid[0], x_lengths=grid[1], y_lengths=grid[2])
    assert oracle_refuses(oracle, *grid)


@pytest.mark.parametrize("grid", [(4, 9, 7), (24, 16, 8)])
def test_accepted(rlfc, oracle, grid):
    """36x28 (coarsest level 9x7 stops the recursion without exit()) and the default 384x192 grid."""
    assert product_rc(rlfc, *grid) == 0 and not oracle_refuses(oracle, *grid)


# ---- coverage guard for the shape table ----------------------------------------------------------------------------

def levels(resolution, xl, yl):
    """Interior (rows, columns) of every multigrid level the reference builds for the grid."""
    r, c = xl * resolution, yl * resolution
    out = [(r, c)]
    while True:
        r, c = r // 2, c // 2
        out.append((r, c))
        if not (r % 2 == 0 and c % 2 == 0 and r > 2 and c > 2):
            return out


def lanes(cols):
    """(columns per lane C = ceil(cols/32), lane count ceil(cols/C), columns of the last lane)."""
    C = -(-cols // 32)
    nl = -(-cols // C)
    return C, nl, cols - (nl - 1) * C


def test_shape_table_coverage():
    """Level 0's C = 3, 4 and 6 come from the default grid and test_gpu_parity's other grids; everything else from
    SHAPES alone.  A coarse level of at most 32 columns is smoothed by the single-warp kernel unless RLFC_TINY=0."""
    lvl0, coarse = [], []
    for g in SHAPES:
        assert not mg_rejects(*g), g
        L = levels(*g)
        lvl0.append((L[0][0],) + lanes(L[0][1]))
        coarse += [(lanes(c), c <= 32) for _, c in L[1:]]
    suite_c = {lanes(yl * res)[0] for res, _, yl in [(24, 16, 8)] + OTHER_GRIDS}
    assert {C for _, C, _, _ in lvl0} | suite_c >= set(range(1, 9)), "level-0 row smoother C = 1..8"
    assert {C for _, C, _, _ in lvl0} >= {1, 5, 7, 8}, "level-0 C = 1, 5, 7, 8 (only SHAPES runs them)"
    assert {C for (C, _, _), tiny in coarse if not tiny} >= {2, 3, 4}, "coarse row pipeline C = 2..4"
    assert any(C == 1 for (C, _, _), tiny in coarse), "coarse C = 1 (rows_smooth<1> with RLFC_TINY=0)"
    assert any(last < C for _, C, _, last in lvl0), "level 0: a last lane with fewer than C columns"
    assert any(last < C for (C, _, last), tiny in coarse if not tiny), "coarse level: a last lane with fewer than C columns"
    assert any(nl < 32 for _, _, nl, _ in lvl0), "fewer than 32 lanes"
    assert any(rows % 16 for rows, _, _, _ in lvl0), "level-0 rows not a multiple of 16"
    assert any(rows % 32 == 16 for rows, _, _, _ in lvl0), "level-0 rows a multiple of 16 but not of 32"
