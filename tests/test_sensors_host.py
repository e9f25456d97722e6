"""CPU tests of flow sensors (rlfc_config.n_sensors / sensors): the configuration checks run before any device call, so they
are observable without a GPU, and the Python mirror's argument handling."""
import ctypes as C

import pytest


def _create(rlfc, sensors=None, **cfg_kw):
    from rlfluidcontrol_b200.env import Config, Sensor
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    for k, v in cfg_kw.items():
        setattr(c, k, v)
    if sensors is not None:
        arr = (Sensor * len(sensors))(*[Sensor(f, x, y) for f, x, y in sensors])
        c.sensors = C.cast(arr, C.POINTER(Sensor))
    h = C.c_void_p()
    rc = L.rlfc_env_create(C.byref(c), C.byref(h))
    if rc == 0:
        L.rlfc_env_destroy(h)
    return rc, L.rlfc_last_error().decode()


def test_default_has_no_sensors(rlfc):
    from rlfluidcontrol_b200.env import Config
    c = Config()
    rlfc.load_library().rlfc_default_config(C.byref(c))
    assert c.n_sensors == 0 and not c.sensors


GOOD = [(0, 100.0, 96.0)]


@pytest.mark.parametrize("kw,msg", [
    (dict(n_sensors=-1), "n_sensors must be >= 0"),
    (dict(n_sensors=2), "sensors is NULL with n_sensors > 0"),
    (dict(n_sensors=1, sensors=[(3, 10.0, 10.0)]), "sensors[0]: field must be 0 (p), 1 (u.x) or 2 (u.y)"),
    (dict(n_sensors=2, sensors=[(0, 10.0, 10.0), (-1, 10.0, 10.0)]), "sensors[1]: field must be"),
    (dict(n_sensors=1, sensors=[(1, float("nan"), 10.0)]), "sensors[0]: coordinates must be finite"),
    (dict(n_sensors=1, sensors=[(2, 10.0, float("inf"))]), "sensors[0]: coordinates must be finite"),
    (dict(n_sensors=1, sensors=[(0, float("-inf"), 0.0)]), "sensors[0]: coordinates must be finite"),
    (dict(n_sensors=1, sensors=GOOD, n_devices=2), "n_sensors is not available in slab mode"),
])
def test_bad_configuration_rejected_without_gpu(rlfc, kw, msg):
    rc, err = _create(rlfc, **kw)
    assert rc == -1 and msg in err, (rc, err)


def test_null_handle_rejected(rlfc):
    L = rlfc.load_library()
    out = (C.c_float * 1)()
    assert L.rlfc_env_get_sensors(None, out) == -1
    assert L.rlfc_env_get_sensors_device(None, None) == -1


def test_python_sensor_names(rlfc):
    from rlfluidcontrol_b200.env import _sensor_array
    arr = _sensor_array([("p", 1, 2.5), ("ux", -3.0, 4), ("uy", 5.25, 1e9)])
    assert [(s.field, s.x, s.y) for s in arr] == [(0, 1.0, 2.5), (1, -3.0, 4.0), (2, 5.25, 1e9)]
    assert len(_sensor_array([])) == 0
    for bad in ("P", "u.x", "vorticity", 0):
        with pytest.raises(ValueError, match="sensor 1: unknown field"):
            _sensor_array([("p", 0, 0), (bad, 1, 1)])
