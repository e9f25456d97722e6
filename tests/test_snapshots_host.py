"""CPU tests of snapshot slots (rlfc_config.n_snapshots): the configuration checks run before any device call, so they are
observable without a GPU, and the Python mirror's argument handling."""
import ctypes as C

import numpy as np
import pytest


def _create(rlfc, **cfg_kw):
    from rlfluidcontrol_b200.env import Config
    L = rlfc.load_library()
    c = Config()
    L.rlfc_default_config(C.byref(c))
    for k, v in cfg_kw.items():
        setattr(c, k, v)
    h = C.c_void_p()
    rc = L.rlfc_env_create(C.byref(c), C.byref(h))
    if rc == 0:
        L.rlfc_env_destroy(h)
    return rc, L.rlfc_last_error().decode()


def test_default_has_no_slots(rlfc):
    from rlfluidcontrol_b200.env import Config
    c = Config()
    rlfc.load_library().rlfc_default_config(C.byref(c))
    assert c.n_snapshots == 0


@pytest.mark.parametrize("n", [-1, -1000])
def test_negative_n_snapshots_rejected_without_gpu(rlfc, n):
    rc, err = _create(rlfc, n_snapshots=n)
    assert rc == -1 and "n_snapshots must be >= 0" in err, (rc, err)


def test_n_snapshots_rejected_in_slab_mode(rlfc):
    rc, err = _create(rlfc, n_snapshots=1, n_devices=2)
    assert rc == -1 and "n_snapshots" in err and "slab mode" in err, (rc, err)


def test_null_handle_rejected(rlfc):
    L = rlfc.load_library()
    ids = (C.c_int * 1)(0)
    assert L.rlfc_env_snapshot(None, ids, ids, 1) == -1
    assert L.rlfc_env_restore(None, ids, ids, 1, 0) == -1
    assert L.rlfc_env_snapshot_device(None, None, None, 0) == -1
    assert L.rlfc_env_restore_device(None, None, None, 0, 0) == -1


def test_python_pairs_must_have_equal_length(rlfc):
    from rlfluidcontrol_b200.env import AFCCylinderBatch
    ids, sl = AFCCylinderBatch._pairs([0, 1], np.array([2, 3], np.int64))
    assert ids.dtype == np.int32 and sl.dtype == np.int32 and sl.tolist() == [2, 3]
    with pytest.raises(ValueError, match="2 environment ids for 1 slots"):
        AFCCylinderBatch._pairs([0, 1], [0])
