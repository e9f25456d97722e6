"""CPU tests of the parameter library (rlfc_config.n_param_sets / param_sets): the configuration checks run before any
device call, so they are observable without a GPU, and the Python mirror's argument handling."""
import ctypes as C
import re

import numpy as np
import pytest

F = np.float32
GOOD = (500, 0.125, 0.2, 1.0471976, 0.0075)
# the invalid sets of test_env_params_host, each with the message that names its fault
BAD = [
    ((0, 0.125, 0.2, 1.0, 0.0075), "re must be >= 1"),
    ((500, 0.0, 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, 1.5, 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, float("nan"), 0.2, 1.0, 0.0075), r"dR must be in \(0, 1\]"),
    ((500, 0.125, -0.1, 1.0, 0.0075), "gR must be finite"),
    ((500, 0.125, float("inf"), 1.0, 0.0075), "gR must be finite"),
    ((500, 0.125, 0.2, float("nan"), 0.0075), "theta must be finite"),
    ((500, 0.125, 0.2, 1.0, 0.0), "t_step must be finite and > 0"),
    ((500, 0.125, 0.2, 1.0, float("inf")), "t_step must be finite and > 0"),
    ((500, 0.5, 3.3, 1.5707964, 0.0075), "body band reaches the lines next to the domain boundary"),
]


def _create(rlfc, sets=None, n_param_sets=None, **cfg_kw):
    from rlfluidcontrol_b200.env import Config, EnvParams
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    for k, v in cfg_kw.items():
        setattr(c, k, v)
    if sets is not None:
        arr = (EnvParams * len(sets))(*[EnvParams(*p) for p in sets])
        c.param_sets = C.cast(arr, C.POINTER(EnvParams))
        c.n_param_sets = len(sets)
    if n_param_sets is not None:
        c.n_param_sets = n_param_sets
    h = C.c_void_p()
    rc = L.rlfc_env_create(C.byref(c), C.byref(h))
    if rc == 0:
        L.rlfc_env_destroy(h)
    return rc, L.rlfc_last_error().decode()


def test_default_has_no_library(rlfc):
    from rlfluidcontrol_b200.env import Config
    c = Config()
    rlfc.load_library().rlfc_default_config(C.byref(c))
    assert c.n_param_sets == 0 and not c.param_sets


def test_negative_count_rejected_without_gpu(rlfc):
    rc, err = _create(rlfc, n_param_sets=-1)
    assert rc == -1 and "n_param_sets must be >= 0" in err, (rc, err)


def test_null_table_rejected_without_gpu(rlfc):
    rc, err = _create(rlfc, n_param_sets=3)
    assert rc == -1 and "param_sets is NULL with n_param_sets > 0" in err, (rc, err)


@pytest.mark.parametrize("bad,msg", BAD)
def test_invalid_set_rejected_without_gpu(rlfc, bad, msg):
    """An invalid set inside an otherwise valid library fails with RLFC_EINVAL and the message names the entry."""
    rc, err = _create(rlfc, [GOOD, GOOD, bad, GOOD])
    assert rc == -1, (rc, err)
    assert "param_sets[2]" in err and re.search(msg, err), err


def test_invalid_set_rejected_with_env_params(rlfc):
    """The library is checked in a per-environment handle too, and named as the library, not as env_params."""
    from rlfluidcontrol_b200.env import EnvParams
    arr = (EnvParams * 2)(EnvParams(*GOOD), EnvParams(*GOOD))
    rc, err = _create(rlfc, [GOOD, BAD[4][0]], env_params=C.cast(arr, C.POINTER(EnvParams)), n_envs=2)
    assert rc == -1 and "param_sets[1]" in err and "gR must be finite" in err, err


def test_library_rejected_in_slab_mode(rlfc):
    rc, err = _create(rlfc, [GOOD], n_devices=2)
    assert rc == -1 and "param_sets is not available in slab mode" in err, (rc, err)


def test_python_param_sets_argument(rlfc):
    """AFCCylinderBatch(param_sets=...) takes dicts or a structured array as env_params does; an invalid entry fails at
    create, before any device call, naming the library entry."""
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*param_sets\[1\].*gR must be finite"):
        rlfc.AFCCylinderBatch(2, param_sets=[{"re": 200}, {"gR": -1.0}])
    st = np.zeros(2, dtype=[("re", np.int32), ("theta", np.float32)])
    st["re"] = (300, 0)
    with pytest.raises(rlfc.RlfcError, match=r"\(-1\).*param_sets\[1\].*re must be >= 1"):
        rlfc.AFCCylinderBatch(1, param_sets=st)
    with pytest.raises(TypeError, match="unknown environment parameter"):
        rlfc.AFCCylinderBatch(1, param_sets=[{"Re": 100}])


def test_python_reset_sets_pairs(rlfc):
    """reset_sets checks that ids and sets pair up before it calls the library."""
    env = object.__new__(rlfc.AFCCylinderBatch)
    with pytest.raises(ValueError, match="2 environment ids for 1 sets"):
        env.reset_sets([0, 1], [0])


def test_null_handle_rejected(rlfc):
    L = rlfc.load_library()
    ids = (C.c_int * 1)(0)
    assert L.rlfc_env_reset_sets(None, ids, ids, 1, 0) == -1
    assert L.rlfc_env_reset_sets_device(None, None, None, 0, 0) == -1
