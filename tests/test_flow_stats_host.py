"""CPU tests of flow statistics (include/rlfc.h "Flow statistics"): the ctypes mirror of rlfc_config against the header as a C
compiler lays it out, the argument checks that run before any device call, and the derivation of the statistics from the
sums (flow_stats_from_sums)."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from rlfluidcontrol_b200.env import STAT_NAMES, Config, flow_stats_from_sums

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    exe = tmp_path_factory.mktemp("layout") / "config_layout"
    subprocess.run([cc, "-std=c99", "-I", str(ROOT / "include"), "-o", str(exe), str(ROOT / "tests" / "config_layout.c")],
                   check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    return {k: int(v) for k, v in (line.split() for line in out.splitlines())}


def test_config_mirror_matches_the_header(c_layout):
    assert C.sizeof(Config) == c_layout["sizeof"]
    assert Config.stats_every.offset == c_layout["stats_every"]
    for name, _ in Config._fields_:
        assert getattr(Config, name).offset == c_layout[name], name
    # stats_every is appended: every earlier field keeps its offset
    assert [n for n, _ in Config._fields_][-1] == "stats_every"


def test_stat_indices_match_the_header(c_layout):
    assert c_layout["RLFC_NUM_STATS"] == len(STAT_NAMES) == 7
    for i, nm in enumerate(("UX", "UY", "P", "UXUX", "UYUY", "PP", "UV")):
        assert c_layout[f"RLFC_STAT_{nm}"] == i
        assert STAT_NAMES[i] == nm.lower()


def test_default_config_has_no_statistics(rlfc):
    c = Config()
    c.stats_every = 99
    rlfc.load_library().rlfc_default_config(C.byref(c))
    assert c.stats_every == 0


def test_entry_points_reject_bad_handles(rlfc):
    L = rlfc.load_library()
    cnt = C.c_longlong()
    assert L.rlfc_env_get_stats(None, 0, C.byref(cnt), None) == -1
    assert L.rlfc_env_stats_reset(None, None, 0) == -1
    assert L.rlfc_env_stats_reset_device(None, None, 0) == -1


def test_create_rejects_negative_stats_every(rlfc):
    """Checked before any device call, so also without a GPU."""
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    c.stats_every = -1
    h = C.c_void_p()
    assert L.rlfc_env_create(C.byref(c), C.byref(h)) == -1
    assert "stats_every" in L.rlfc_last_error().decode()
    c.stats_every, c.n_devices = 4, 2
    assert L.rlfc_env_create(C.byref(c), C.byref(h)) == -1
    assert "slab mode" in L.rlfc_last_error().decode()


def synthetic_samples(N=5, n=6, m=8, seed=3):
    rng = np.random.default_rng(seed)
    return [tuple(rng.normal(size=(n, m)).astype(np.float32) for _ in range(3)) for _ in range(N)]


def add_sample(S, ux, uy, p):
    """S[7, n, m] += the terms of one sample as rlfc.h defines them: float64 sums, the cross term's ucc and vcc in float32."""
    for i, x in enumerate((ux, uy, p)):
        x = np.asarray(x, np.float32).astype(np.float64)
        S[i] += x
        S[3 + i] += x * x
    ux, uy = np.asarray(ux, np.float32), np.asarray(uy, np.float32)
    ucc = (ux[1:-1, 1:-1] + ux[2:, 1:-1]) * np.float32(0.5)
    vcc = (uy[1:-1, 1:-1] + uy[1:-1, 2:]) * np.float32(0.5)
    S[6, 1:-1, 1:-1] += ucc.astype(np.float64) * vcc.astype(np.float64)


def sums_of(samples):
    """The sums of a sequence of samples, accumulated in sample order."""
    n, m = samples[0][0].shape
    S = np.zeros((7, n, m))
    for ux, uy, p in samples:
        add_sample(S, ux, uy, p)
    return S


def test_flow_stats_derivation():
    samples = synthetic_samples()
    N = len(samples)
    st = flow_stats_from_sums(N, sums_of(samples))
    assert st["count"] == N
    stack = {k: np.stack([s[i].astype(np.float64) for s in samples]) for i, k in enumerate(("ux", "uy", "p"))}
    for k, a in stack.items():
        np.testing.assert_allclose(st[f"mean_{k}"], a.mean(0), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(st[f"var_{k}"], a.var(0), rtol=1e-9, atol=1e-12)
        assert st[f"mean_{k}"].dtype == np.float64
    # the covariance of the cell-centred velocities over the samples (each sample's ucc, vcc formed in float, as summed)
    ucc = np.stack([((ux[1:-1, 1:-1] + ux[2:, 1:-1]) * np.float32(0.5)).astype(np.float64) for ux, _, _ in samples])
    vcc = np.stack([((uy[1:-1, 1:-1] + uy[1:-1, 2:]) * np.float32(0.5)).astype(np.float64) for _, uy, _ in samples])
    want = (ucc * vcc).mean(0) - ucc.mean(0) * vcc.mean(0)
    np.testing.assert_allclose(st["uv_cov"][1:-1, 1:-1], want, rtol=1e-6, atol=1e-7)
    assert not st["uv_cov"][0].any() and not st["uv_cov"][-1].any()
    assert not st["uv_cov"][:, 0].any() and not st["uv_cov"][:, -1].any()


def test_flow_stats_of_a_steady_flow():
    """A flow sampled N times unchanged: means are the field, variances and the covariance vanish."""
    ux, uy, p = synthetic_samples(N=1)[0]
    for N in (1, 7):
        st = flow_stats_from_sums(N, sums_of([(ux, uy, p)] * N))
        np.testing.assert_allclose(st["mean_p"], p.astype(np.float64), rtol=1e-15)
        for k in ("ux", "uy", "p"):
            np.testing.assert_allclose(st[f"var_{k}"], 0, atol=1e-12)
        # (the sums hold ucc, vcc rounded to float, the means are formed in double: they differ by float rounding)
        np.testing.assert_allclose(st["uv_cov"], 0, atol=1e-6)


def test_flow_stats_without_samples():
    with pytest.raises(ValueError, match="no samples"):
        flow_stats_from_sums(0, np.zeros((7, 4, 4)))
