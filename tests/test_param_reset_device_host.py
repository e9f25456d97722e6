"""CPU tests of rlfc_env_reset_params_device's interface: the packed parameter layout a device array must have, and the
argument handling of the C entry point and of its Python mirror, which are observable without a GPU."""
import ctypes as C

import numpy as np
import pytest

F = np.float32


def test_packed_layout_is_rlfc_env_params(rlfc):
    """20 bytes per set: int32 re, then float32 dR, gR, theta, t_step, at the offsets of rlfc_env_params."""
    from rlfluidcontrol_b200.env import EnvParams
    assert C.sizeof(EnvParams) == 20
    assert [getattr(EnvParams, k).offset for k in ("re", "dR", "gR", "theta", "t_step")] == [0, 4, 8, 12, 16]


def test_int32_stack_packs_like_the_struct(rlfc):
    """The (n, 5) int32 packing of INTEGRATION.md -- re as int32 and the float32 fields' bits -- is byte for byte an array
    of rlfc_env_params."""
    from rlfluidcontrol_b200.env import EnvParams
    re = np.array([500, 1, 100000], np.int32)
    fl = [np.array(v, F) for v in ([0.125, 1.0, 0.01], [0.2, 0.0, 0.5], [1.0471976, -6.2831855, 0.0], [0.0075, 0.005, 0.01])]
    packed = np.stack([re] + [f.view(np.int32) for f in fl], 1)
    assert packed.shape == (3, 5) and packed.dtype == np.int32
    arr = (EnvParams * 3)(*[EnvParams(int(re[k]), *[float(f[k]) for f in fl]) for k in range(3)])
    assert packed.tobytes() == bytes(arr)


def test_null_handle_rejected(rlfc):
    L = rlfc.load_library()
    assert L.rlfc_env_reset_params_device(None, None, None, 0, 0) == -1
    assert "null handle" in L.rlfc_last_error().decode()


def test_python_wrapper_passes_pointers_and_raises(rlfc):
    """reset_params_device takes data_ptr() ints and raises RlfcError with the library's message on a failure."""
    env = object.__new__(rlfc.AFCCylinderBatch)
    env._L = rlfc.load_library()
    env._h = None
    with pytest.raises(rlfc.RlfcError, match=r"rlfc_env_reset_params_device failed \(-1\): null handle"):
        env.reset_params_device(0x1000, 0x2000, 3, reset_accumulators=True)
