"""CPU tests of per-environment constructor arguments (rlfc_config.env_params): the host geometry away from the default
parameters against the CPU oracle, the validation of parameter sets (before any device call, so it is observable
without a GPU), and the ctypes mirror of the new structs."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
F = np.float32

# (re, dR, gR, theta, t_step): each varies what the defaults (500, .125, .2, PI/3, .0075) keep fixed
PARAM_SETS = [
    (100, 0.125, 0.2, F(3.1415927) / F(3), 0.0075),
    (500, 0.25, 0.2, F(3.1415927) / F(3), 0.0075),
    (500, 0.125, 0.5, F(3.1415927) / F(3), 0.0075),
    (500, 0.125, 0.2, 1.2, 0.0075),
    (500, 0.125, 0.2, F(3.1415927) / F(3), 0.005),
    (1000, 0.2, 0.4, F(3.1415927) / F(6), 0.005),
]


@pytest.mark.parametrize("ps", PARAM_SETS, ids=lambda p: "re%d_dR%g_gR%g_th%.3f_ts%g" % tuple(float(v) for v in p))
def test_geometry_matches_oracle_away_from_defaults(rlfc, oracle, ps):
    from rlfluidcontrol_b200.env import geometry_static
    re_, dR, gR, theta, ts = ps
    e = oracle.OracleEnv(literal=False, Re=re_, dR=dR, gR=gR, theta=theta, tStep=ts)
    for name in ("del.x", "del.y", "del1.x", "del1.y", "wnx.x", "wnx.y", "wny.x", "wny.y", "c.x", "c.y"):
        got, _ = geometry_static(name, re=re_, dR=dR, gR=gR, theta=theta, t_step=ts)
        assert np.array_equal(got, e.coeff(name)), name


def _create(rlfc, params, n_envs=None, **cfg_kw):
    from rlfluidcontrol_b200.env import Config, EnvParams
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    for k, v in cfg_kw.items():
        setattr(c, k, v)
    arr = (EnvParams * len(params))(*[EnvParams(*p) for p in params])
    c.n_envs = len(params) if n_envs is None else n_envs
    c.env_params = C.cast(arr, C.POINTER(EnvParams))
    h = C.c_void_p()
    rc = L.rlfc_env_create(C.byref(c), C.byref(h))
    if rc == 0:
        L.rlfc_env_destroy(h)
    return rc, L.rlfc_last_error().decode()


GOOD = (500, 0.125, 0.2, 1.0471976, 0.0075)


@pytest.mark.parametrize("bad,msg", [
    ((0, 0.125, 0.2, 1.0, 0.0075), "re must be >= 1"),
    ((500, 0.0, 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, 1.5, 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, float("nan"), 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, 0.125, -0.1, 1.0, 0.0075), "gR must be finite"),
    ((500, 0.125, float("inf"), 1.0, 0.0075), "gR must be finite"),
    ((500, 0.125, 0.2, float("nan"), 0.0075), "theta must be finite"),
    ((500, 0.125, 0.2, 1.0, 0.0), "t_step must be finite and > 0"),
    ((500, 0.125, 0.2, 1.0, float("inf")), "t_step must be finite and > 0"),
    # a control cylinder pushed against the lower wall: the band reaches the lines next to the boundary
    ((500, 0.5, 3.3, 1.5707964, 0.0075), "body band reaches the lines next to the domain boundary"),
])
def test_invalid_parameter_set_rejected_without_gpu(rlfc, bad, msg):
    """Each invalid set fails with RLFC_EINVAL and names the entry, also in a batch whose other entries are valid: the
    validation runs before any device call."""
    rc, err = _create(rlfc, [GOOD, bad, GOOD])
    assert rc == -1, (rc, err)
    assert "env_params[1]" in err and re.search(msg, err), err


def test_env_params_rejected_in_slab_mode(rlfc):
    rc, err = _create(rlfc, [GOOD], n_devices=2)
    assert rc == -1 and "slab mode" in err, err


def test_python_env_params_validation(rlfc):
    from rlfluidcontrol_b200.env import _env_params_array, Config
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    arr = _env_params_array([{"re": 200}, {"dR": 0.2, "theta": 0.5}], c)
    assert (arr[0].re, F(arr[0].dR), F(arr[0].t_step)) == (200, F(0.125), F(0.0075))
    assert (arr[1].re, F(arr[1].dR), F(arr[1].theta)) == (500, F(0.2), F(0.5))
    st = np.zeros(2, dtype=[("re", np.int32), ("gR", np.float32)])
    st["re"] = (300, 400)
    st["gR"] = (0.3, 0.4)
    arr = _env_params_array(st, c)
    assert [a.re for a in arr] == [300, 400] and F(arr[1].gR) == F(0.4) and F(arr[1].dR) == F(0.125)
    with pytest.raises(TypeError, match="unknown environment parameter"):
        _env_params_array([{"Re": 100}], c)


def _header_fields(struct):
    hdr = (ROOT / "include" / "rlfc.h").read_text()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    body = re.search(r"typedef struct \{([^{}]*)\}\s*" + struct + ";", hdr).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        # "float dR, gR" / "const char *init_bdim_path" -> the declarator names
        head, *rest = decl.split(",")
        names.append(re.findall(r"\w+", head)[-1])
        names += [re.findall(r"\w+", r)[-1] for r in rest]
    return names


def test_ctypes_mirror_has_header_field_order():
    from rlfluidcontrol_b200.env import Config, EnvParams
    assert [n for n, _ in EnvParams._fields_] == _header_fields("rlfc_env_params")
    assert [n for n, _ in Config._fields_] == _header_fields("rlfc_config")
