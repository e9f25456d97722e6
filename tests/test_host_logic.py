"""CPU tests of the product's host side: the C-ABI library loads and exports every symbol include/rlfc.h
declares, the host-side geometry precompute (csrc/geometry.cpp) reproduces the oracle's coefficient fields bit
for bit on every multigrid level, error behaviour without a GPU, Java float formatting, sharding helpers."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol(rlfc):
    L = rlfc.load_library()
    hdr = (ROOT / "include" / "rlfc.h").read_text()
    names = sorted(set(re.findall(r"\b(rlfc_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, f"librlfc.so lacks {missing}"


def test_default_config_matches_reference_constants(rlfc):
    from rlfluidcontrol_b200.env import Config
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    # clientCFD.pde:5-14,94-96
    assert (c.resolution, c.x_lengths, c.y_lengths, c.re, c.substeps, c.mg_max_iters) == (24, 16, 8, 500, 16, 20)
    assert np.float32(c.dR) == np.float32(0.125) and np.float32(c.gR) == np.float32(0.2)
    assert np.float32(c.theta) == np.float32(np.float32(3.1415927) / np.float32(3))
    assert np.float32(c.t_step) == np.float32(0.0075) and c.action_scale == 5.0
    assert c.init_time == 1.0 and c.episode_time == 50.0


def test_no_cpu_fallback(rlfc):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(rlfc.RlfcError, match="no CUDA device"):
        rlfc.AFCCylinderBatch(1)


def test_bad_config_rejected(rlfc):
    from rlfluidcontrol_b200.env import Config
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    c.n_envs = 0
    h = C.c_void_p()
    assert L.rlfc_env_create(C.byref(c), C.byref(h)) == -1 and b"n_envs" in L.rlfc_last_error()
    assert L.rlfc_env_create(None, C.byref(h)) == -1


@pytest.mark.parametrize("name", ["del.x", "del.y", "del1.x", "del1.y", "wnx.x", "wnx.y", "wny.x", "wny.y", "c.x", "c.y"])
def test_geometry_fields_match_oracle(rlfc, oracle, name):
    from rlfluidcontrol_b200.env import geometry_static
    got, nlev = geometry_static(name)
    e = oracle.OracleEnv(literal=False)
    assert nlev == 7
    assert np.array_equal(got, e.coeff(name)), name


def test_multigrid_hierarchy_matches_oracle(rlfc, oracle):
    """lower/diag/inv of all seven levels vs PoissonMatrix + MG.restrict of the oracle (386x194 ... 8x5)."""
    from rlfluidcontrol_b200.env import geometry_static
    e = oracle.OracleEnv(literal=False)
    c = oracle.VField(386, 194, 0, 0)
    c.x[...] = e.coeff("del.x") * np.float32(np.float32(0.0075) * 24)
    c.y[...] = e.coeff("del.y") * np.float32(np.float32(0.0075) * 24)
    A = oracle.Poisson(c)
    dims = []
    for lev in range(7):
        for nm, ref in (("lower.x", A.lx), ("lower.y", A.ly), ("diag", A.diag), ("inv", A.inv)):
            got, _ = geometry_static(nm, lev)
            assert got.shape == ref.shape and np.array_equal(got, ref), (lev, nm)
        dims.append(A.lx.shape)
        if lev < 6:
            A = A.restrict()
    assert dims == [(386, 194), (194, 98), (98, 50), (50, 26), (26, 14), (14, 8), (8, 5)]


def test_velocity_basis(rlfc, oracle):
    """ub = (0 + u1*w1) + u2*w2 from the static basis equals BodyUnion.velocity of the oracle for a rotating pair."""
    from rlfluidcontrol_b200.env import geometry_static
    e = oracle.OracleEnv(literal=True)
    e.set_xi(0.6, -0.9)
    e.update2()                                     # literal: get_coeffs evaluates ub with the current dphi
    ubx, uby = e.coeff("ub.x"), e.coeff("ub.y")
    dt = np.float32(np.float32(0.0075) * 24)
    dRD = np.float32(np.float32(0.125) * np.float32(24))
    dphi = [np.float32(np.float32(np.float32(2) * np.float32(np.float32(5) * np.float32(x)) * dt) / dRD) for x in (0.6, -0.9)]
    w1, _ = geometry_static("w1.x"); w2, _ = geometry_static("w2.x")
    r1, _ = geometry_static("ry1.x"); r2, _ = geometry_static("ry2.x")
    f = np.float32
    u1 = ((f(0) - r1 * dphi[0]).astype(f) / dt).astype(f)
    u2 = ((f(0) - r2 * dphi[1]).astype(f) / dt).astype(f)
    mine = ((f(0) + (u1 * w1).astype(f)).astype(f) + (u2 * w2).astype(f)).astype(f)
    assert np.array_equal(mine, ubx)
    w1, _ = geometry_static("w1.y"); w2, _ = geometry_static("w2.y")
    r1, _ = geometry_static("rx1.y"); r2, _ = geometry_static("rx2.y")
    u1 = ((f(0) + r1 * dphi[0]).astype(f) / dt).astype(f)
    u2 = ((f(0) + r2 * dphi[1]).astype(f) / dt).astype(f)
    mine = ((f(0) + (u1 * w1).astype(f)).astype(f) + (u2 * w2).astype(f)).astype(f)
    assert np.array_equal(mine, uby)


def test_grid_not_divisible_is_an_error(rlfc):
    from rlfluidcontrol_b200.env import geometry_static
    with pytest.raises(rlfc.RlfcError, match="MultiGrid requires"):
        geometry_static("inv", 0, resolution=25, x_lengths=3, y_lengths=3)     # 75 = 3*5^2: coarsens to 37 -> odd and > 9


def test_java_float_format(rlfc):
    """java.lang.Float.toString forms seen in init.bdim and the RPC payloads."""
    L = rlfc.load_library()
    L.rlfc_format_float_java.argtypes = [C.c_float, C.c_char_p, C.c_int]
    cases = {1.0: "1.0", 0.0: "0.0", -7.902107e-4: "-7.902107E-4", -0.0015798381: "-0.0015798381", 0.17233936: "0.17233936",
             2400.2554: "2400.2554", 0.17999999: "0.17999999", 1.0e7: "1.0E7", 123456.7: "123456.7", 1e-3: "0.001", 9.999e-4: "9.999E-4"}
    buf = C.create_string_buffer(64)
    for v, s in cases.items():
        L.rlfc_format_float_java(np.float32(v), buf, 64)
        assert buf.value.decode() == s, (v, buf.value)
        assert np.float32(float(buf.value.decode().replace("E", "e"))) == np.float32(v)


def test_shard_ranges():
    from rlfluidcontrol_b200.sharding import shard_range
    for world in (1, 2, 4, 8):
        edges = [shard_range(4096, r, world) for r in range(world)]
        assert edges[0][0] == 0 and edges[-1][1] == 4096
        assert all(a[1] == b[0] for a, b in zip(edges, edges[1:]))
        assert len({e1 - e0 for e0, e1 in edges}) == 1
    with pytest.raises(ValueError):
        shard_range(10, 3, 2)


def test_bench_actions_are_deterministic_and_sharded():
    import bench
    a0 = bench.make_actions(5, 8, 0)
    a1 = bench.make_actions(5, 8, 1)
    assert a0.shape == (5, 8, 2) and a0.dtype == np.float32 and np.abs(a0).max() <= 1
    assert np.array_equal(a0, bench.make_actions(5, 8, 0)) and not np.array_equal(a0, a1)
    k = np.arange(5)
    assert np.array_equal(a0[:, 0, 0], (0.8 * np.sin(2 * np.pi * k / 25.0)).astype(np.float32))     # env 0: config-1 sequence


def test_bench_dump_outputs_float32_within_budget(tmp_path):
    """--dump-outputs: small arrays are written whole as float32, a field too large for the 64 MB budget is replaced by the
    same sample of its elements in every run."""
    import bench
    done = np.array([0, 1, 0], np.int32)
    big = np.arange(3 * 2000 * 2000, dtype=np.float32).reshape(3, 2000, 2000)          # 48 MB: over the share of one of two
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"done": done, "p": big})
    got = {f.name: np.load(f) for f in sorted((tmp_path / "a").iterdir())}
    assert sorted(got) == ["done.npy", "p.npy"] and all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["done.npy"], done.astype(np.float32))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    p = got["p.npy"]                                      # element values = flat indices: distinct, in storage order
    assert 1000 < p.size < big.size and np.all(np.diff(p) > 0) and np.all(p == np.floor(p)) and p[-1] < big.size
    assert np.array_equal(p, np.load(tmp_path / "b" / "p.npy"))
