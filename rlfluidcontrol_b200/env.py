"""ctypes mirror of include/rlfc.h.

`AFCCylinderBatch` plays the role of the reference's `AFCCylinder` object (AFCCylinder.pde:1-61) for a
whole batch of environments: `update2()` is one solver step, `step(actions)` is one RL step as
clientCFD.draw() drives it (clientCFD.pde:35-55).  All numerics run in librlfc.so on the GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
# RLFC_LIBRARY selects another build of the same library (e.g. an instrumented one made by tools/); never a fallback
_LIB_PATH = Path(os.environ["RLFC_LIBRARY"]).resolve() if os.environ.get("RLFC_LIBRARY") else _PKG / "librlfc.so"
NUM_PROBES = 32
# rlfc.h "Flow statistics": the sums of rlfc_env_get_stats, in this order (RLFC_STAT_UX .. RLFC_STAT_UV)
STAT_NAMES = ("ux", "uy", "p", "uxux", "uyuy", "pp", "uv")


class RlfcError(RuntimeError):
    pass


class EnvParams(C.Structure):
    """rlfc_env_params: the per-environment arguments of the AFCCylinder constructor."""
    _fields_ = [("re", C.c_int), ("dR", C.c_float), ("gR", C.c_float), ("theta", C.c_float), ("t_step", C.c_float)]


ENV_PARAM_KEYS = tuple(name for name, _ in EnvParams._fields_)


class Sensor(C.Structure):
    """rlfc_sensor: Field.linear of one field at one point (grid coordinates, one unit = one cell)."""
    _fields_ = [("field", C.c_int), ("x", C.c_float), ("y", C.c_float)]


SENSOR_FIELDS = {"p": 0, "ux": 1, "uy": 2}   # RLFC_SENSOR_P, _UX, _UY


class Config(C.Structure):
    _fields_ = [
        ("resolution", C.c_int), ("x_lengths", C.c_int), ("y_lengths", C.c_int), ("re", C.c_int),
        ("dR", C.c_float), ("gR", C.c_float), ("theta", C.c_float), ("t_step", C.c_float),
        ("action_scale", C.c_float), ("substeps", C.c_int), ("init_time", C.c_float),
        ("episode_time", C.c_float), ("n_envs", C.c_int), ("device", C.c_int), ("exact", C.c_int),
        ("mg_max_iters", C.c_int), ("init_bdim_path", C.c_char_p), ("stream", C.c_void_p),
        ("n_groups", C.c_int), ("n_devices", C.c_int), ("adaptive_dt", C.c_int),
        ("env_params", C.POINTER(EnvParams)), ("n_snapshots", C.c_int),
        ("n_sensors", C.c_int), ("sensors", C.POINTER(Sensor)),
        ("n_param_sets", C.c_int), ("param_sets", C.POINTER(EnvParams)),
        ("stats_every", C.c_int),
    ]


_lib = None


def library_path() -> Path:
    return _LIB_PATH


def default_init_state() -> Path:
    """The developed-wake state every reference episode resumes from (saved/init/init.bdim,
    AFCCylinder.pde:35-37), shipped here in binary form."""
    return _PKG / "data" / "init_state.bdimb"


def load_library():
    """dlopen librlfc.so; fails loudly if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RlfcError(f"{_LIB_PATH} is missing: build it with `python -m rlfluidcontrol_b200.build` "
                        "(there is no CPU fallback)")
    L = C.CDLL(str(_LIB_PATH))
    fp, ip, vp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.c_void_p
    L.rlfc_default_config.argtypes = [C.POINTER(Config)]
    L.rlfc_default_config.restype = None
    L.rlfc_env_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.rlfc_env_destroy.argtypes = [vp]
    L.rlfc_env_destroy.restype = None
    L.rlfc_env_reset.argtypes = [vp, ip, C.c_int, C.c_int]
    L.rlfc_env_reset_params.argtypes = [vp, ip, C.c_int, C.POINTER(EnvParams), C.c_int]
    L.rlfc_env_get_params.argtypes = [vp, C.POINTER(EnvParams)]
    L.rlfc_env_reset_sets.argtypes = [vp, ip, ip, C.c_int, C.c_int]
    L.rlfc_env_reset_sets_device.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    L.rlfc_env_reset_params_device.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    L.rlfc_env_step.argtypes = [vp, fp, fp, fp, ip]
    L.rlfc_env_step_device.argtypes = [vp, vp, vp, vp, vp]
    L.rlfc_env_substep.argtypes = [vp, fp, fp, fp]
    L.rlfc_env_substep_device.argtypes = [vp, vp]
    L.rlfc_env_get_fields.argtypes = [vp, C.c_int, fp, fp, fp]
    L.rlfc_env_set_fields.argtypes = [vp, C.c_int, fp, fp, fp]
    L.rlfc_env_save_bdim.argtypes = [vp, C.c_int, C.c_char_p]
    L.rlfc_env_load_bdim.argtypes = [vp, C.c_int, C.c_char_p]
    L.rlfc_env_dims.argtypes = [vp, ip, ip, ip]
    L.rlfc_env_get_time.argtypes = [vp, fp]
    L.rlfc_env_get_mg_iters.argtypes = [vp, ip]
    L.rlfc_env_check_cfl.argtypes = [vp, fp]
    L.rlfc_env_get_dt.argtypes = [vp, fp]
    L.rlfc_env_get_coeffs.argtypes = [vp, C.c_int, C.c_char_p, C.c_int, fp, ip, ip]
    L.rlfc_env_running.argtypes = [vp, ip]
    L.rlfc_env_get_flags.argtypes = [vp, ip]
    L.rlfc_env_snapshot.argtypes = [vp, ip, ip, C.c_int]
    L.rlfc_env_restore.argtypes = [vp, ip, ip, C.c_int, C.c_int]
    L.rlfc_env_snapshot_device.argtypes = [vp, vp, vp, C.c_int]
    L.rlfc_env_restore_device.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    L.rlfc_record_bytes.argtypes = [C.POINTER(Config), C.POINTER(C.c_size_t)]
    L.rlfc_record_checksum.argtypes = [vp, C.c_size_t]
    L.rlfc_record_checksum.restype = C.c_ulonglong
    L.rlfc_env_export.argtypes = [vp, ip, C.c_int, vp]
    L.rlfc_env_import.argtypes = [vp, ip, C.c_int, vp, C.c_int]
    L.rlfc_env_export_device.argtypes = [vp, vp, C.c_int, vp]
    L.rlfc_env_import_device.argtypes = [vp, vp, C.c_int, vp, C.c_size_t, C.c_int]
    L.rlfc_env_get_sensors.argtypes = [vp, fp]
    L.rlfc_env_get_sensors_device.argtypes = [vp, vp]
    L.rlfc_env_get_stats.argtypes = [vp, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_double)]
    L.rlfc_env_stats_reset.argtypes = [vp, ip, C.c_int]
    L.rlfc_env_stats_reset_device.argtypes = [vp, vp, C.c_int]
    L.rlfc_env_field_sum.argtypes = [vp, fp]
    L.rlfc_env_field_sum_stats.argtypes = [vp, ip]
    L.rlfc_env_get_static.argtypes = [vp, C.c_char_p, C.c_int, fp, ip, ip]
    L.rlfc_geometry_static.argtypes = [C.POINTER(Config), C.c_char_p, C.c_int, fp, ip, ip, ip]
    L.rlfc_env_num_levels.argtypes = [vp]
    L.rlfc_env_set_profiling.argtypes = [vp, C.c_int]
    L.rlfc_env_get_profile.argtypes = [vp, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_double),
                                       C.POINTER(C.c_longlong), C.POINTER(C.c_double)]
    L.rlfc_env_stream.argtypes = [vp]
    L.rlfc_env_stream.restype = vp
    L.rlfc_env_slab_info.argtypes = [vp, ip, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.rlfc_env_launch_count.argtypes = [vp]
    L.rlfc_env_launch_count.restype = C.c_longlong
    L.rlfc_env_model_bytes_per_solver_step.argtypes = [vp]
    L.rlfc_env_model_bytes_per_solver_step.restype = C.c_double
    L.rlfc_last_error.restype = C.c_char_p
    L.rlfc_version.restype = C.c_char_p
    _lib = L
    return L


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _env_params_array(params, cfg):
    """A sequence of dicts (or a structured array with some of the fields re, dR, gR, theta, t_step) -> EnvParams[n]; a
    missing key takes the scalar config's value."""
    if isinstance(params, np.ndarray) and params.dtype.names:
        params = [{k: params[k][i] for k in params.dtype.names} for i in range(len(params))]
    params = list(params)
    arr = (EnvParams * len(params))()
    for i, p in enumerate(params):
        unknown = set(p) - set(ENV_PARAM_KEYS)
        if unknown:
            raise TypeError(f"unknown environment parameter(s) {sorted(unknown)}")
        for k in ENV_PARAM_KEYS:
            setattr(arr[i], k, int(p[k]) if k == "re" and k in p else p.get(k, getattr(cfg, k)))
    return arr


def _sensor_array(sensors):
    """A sequence of (field, x, y) with field "p", "ux" or "uy" -> rlfc_sensor[n]."""
    sensors = list(sensors)
    arr = (Sensor * len(sensors))()
    for i, (field, x, y) in enumerate(sensors):
        if field not in SENSOR_FIELDS:
            raise ValueError(f"sensor {i}: unknown field {field!r} (expected one of {sorted(SENSOR_FIELDS)})")
        arr[i].field, arr[i].x, arr[i].y = SENSOR_FIELDS[field], float(x), float(y)
    return arr


def flow_stats_from_sums(count, sums):
    """The flow statistics of one environment from its sample count and sums[7, n, m] (`AFCCylinderBatch.stats_sums`), in
    float64: the means of ux, uy and p; their variances sum(x^2)/N - mean^2; and uv_cov = sum(ucc*vcc)/N - mean(ucc)*mean(vcc)
    on the interior cells (zero on the ghost cells), the cell-centred means taken from the face means as ucc and vcc are from
    the faces: mean(ucc)[i][j] = (mean(ux)[i][j] + mean(ux)[i+1][j]) / 2, mean(vcc)[i][j] = (mean(uy)[i][j] + mean(uy)[i][j+1]) / 2.
    Returns a dict of (n, m) arrays and the count."""
    if count <= 0:
        raise ValueError("no samples: the statistics were reset and no sampled step has run since")
    S = np.asarray(sums, np.float64)
    N = float(count)
    mean = {k: S[i] / N for i, k in enumerate(("ux", "uy", "p"))}
    out = dict(count=int(count))
    for i, k in enumerate(("ux", "uy", "p")):
        out[f"mean_{k}"] = mean[k]
        out[f"var_{k}"] = S[3 + i] / N - mean[k] * mean[k]
    cov = np.zeros_like(S[6])
    ucc = (mean["ux"][1:-1, 1:-1] + mean["ux"][2:, 1:-1]) * 0.5
    vcc = (mean["uy"][1:-1, 1:-1] + mean["uy"][1:-1, 2:]) * 0.5
    cov[1:-1, 1:-1] = S[6][1:-1, 1:-1] / N - ucc * vcc
    out["uv_cov"] = cov
    return out


class AFCCylinderBatch:
    """A batch of AFCCylinder environments on one GPU."""

    def __init__(self, n_envs=1, init_state="default", device=-1, stream=None, env_params=None, sensors=None, param_sets=None,
                 **overrides):
        """env_params: None (every environment uses the scalar config's re, dR, gR, theta, t_step), or n_envs entries, dicts
        or a structured array, each environment's own constructor arguments (missing keys: the scalar config's).
        sensors: None, or a sequence of (field, x, y), field "p", "ux" or "uy", (x, y) in grid coordinates: the flow
        sampled in every environment after each of its solver steps (`sensors()`).
        param_sets: None, or a library of constructor arguments given like env_params (any number of entries), built at
        create; `reset_sets` / `reset_sets_device` switch environments to its entries on the device.
        stats_every (a config keyword): 0 (default) = no flow statistics; k >= 1 = every environment accumulates the sums of
        `stats_sums` / `flow_stats` from a sample after every k-th solver step it takes part in."""
        self._L = load_library()
        cfg = Config()
        self._L.rlfc_default_config(C.byref(cfg))
        cfg.n_envs = int(n_envs)
        cfg.device = int(device)
        if init_state == "default":
            init_state = default_init_state()
        self._init_path = None if init_state is None else str(init_state).encode()
        cfg.init_bdim_path = self._init_path
        if stream is not None:
            cfg.stream = C.c_void_p(int(stream))
        for k, v in overrides.items():
            if not hasattr(cfg, k):
                raise TypeError(f"unknown config field {k}")
            setattr(cfg, k, v)
        if env_params is not None:
            self._env_params = _env_params_array(env_params, cfg)
            if len(self._env_params) != cfg.n_envs:
                raise ValueError(f"env_params has {len(self._env_params)} entries for {cfg.n_envs} environments")
            cfg.env_params = C.cast(self._env_params, C.POINTER(EnvParams))
        if param_sets is not None:
            self._param_sets = _env_params_array(param_sets, cfg)
            cfg.n_param_sets = len(self._param_sets)
            cfg.param_sets = C.cast(self._param_sets, C.POINTER(EnvParams))
        if sensors is not None:
            self._sensors = _sensor_array(sensors)
            cfg.n_sensors = len(self._sensors)
            cfg.sensors = C.cast(self._sensors, C.POINTER(Sensor))
        self.n_sensors = cfg.n_sensors
        self.n_param_sets = cfg.n_param_sets
        self.cfg = cfg
        h = C.c_void_p()
        rc = self._L.rlfc_env_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise RlfcError(f"rlfc_env_create failed ({rc}): {self._L.rlfc_last_error().decode()}")
        self._h = h
        n, m, b = C.c_int(), C.c_int(), C.c_int()
        self._L.rlfc_env_dims(h, C.byref(n), C.byref(m), C.byref(b))
        self.n, self.m, self.n_envs = n.value, m.value, b.value

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.rlfc_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            raise RlfcError(f"{what} failed ({rc}): {self._L.rlfc_last_error().decode()}")

    # -- reference-facing interface ---------------------------------------------------------
    def reset(self, env_ids=None, reset_accumulators=False, params=None):
        """setUpNewSim for the listed environments (None = all).  params (per-environment handles only): one entry per
        listed environment, dicts or a structured array; the environment takes these constructor arguments (missing keys:
        the scalar config's) with its geometry and Poisson hierarchy.  An invalid entry changes no environment."""
        if params is not None:
            ids = np.arange(self.n_envs, dtype=np.int32) if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
            arr = _env_params_array(params, self.cfg)
            if len(arr) != len(ids):
                raise ValueError(f"{len(arr)} parameter sets for {len(ids)} environments")
            rc = self._L.rlfc_env_reset_params(self._h, ids.ctypes.data_as(C.POINTER(C.c_int)), len(ids), arr,
                                               int(reset_accumulators))
            self._check(rc, "rlfc_env_reset_params")
            return
        if env_ids is None:
            rc = self._L.rlfc_env_reset(self._h, None, self.n_envs, int(reset_accumulators))
        else:
            ids = np.ascontiguousarray(env_ids, dtype=np.int32)
            rc = self._L.rlfc_env_reset(self._h, ids.ctypes.data_as(C.POINTER(C.c_int)), len(ids), int(reset_accumulators))
        self._check(rc, "rlfc_env_reset")

    def reset_sets(self, env_ids, sets, reset_accumulators=False):
        """setUpNewSim into the parameter library: environment env_ids[k] takes param_sets[sets[k]] with its geometry and
        Poisson hierarchy, bit for bit what `reset([e], params=[param_sets[s]])` gives, without building anything on the
        host.  All or nothing: an id or set out of range or an environment listed twice raises and changes nothing."""
        ids, st = self._pairs(env_ids, sets, "sets")
        self._check(self._L.rlfc_env_reset_sets(self._h, _ip(ids), _ip(st), len(ids), int(reset_accumulators)),
                    "rlfc_env_reset_sets")

    def reset_sets_device(self, d_env_ids, d_sets, n, reset_accumulators=False):
        """reset_sets() with device int32 arrays of length n (data_ptr() ints), asynchronous on the handle's stream:
        reset_sets_device(arange(B), where(done, draw, -1), B) gives the finished environments new parameter sets without
        the host.  Pairs with an entry out of range (e.g. -1) are skipped; of pairs with the same environment the last wins."""
        self._check(self._L.rlfc_env_reset_sets_device(self._h, C.c_void_p(d_env_ids), C.c_void_p(d_sets), int(n),
                                                       int(reset_accumulators)), "rlfc_env_reset_sets_device")

    def reset_params_device(self, d_env_ids, d_params, n, reset_accumulators=False):
        """reset(params=...) with the parameter sets built on the device: device arrays of length n (data_ptr() ints),
        int32 environment ids and packed rlfc_env_params (20 bytes each: int32 re, float32 dR, gR, theta, t_step, e.g. an
        (n, 5) int32 tensor torch.stack([re.int(), dR.view(torch.int32), ...], 1)), asynchronous on the handle's stream.
        Pairs whose id is out of range (e.g. -1) are skipped; of pairs with the same environment the last wins.  An
        invalid set, or |theta| > 2 pi, leaves its environment unchanged and sets flags() bit 2."""
        self._check(self._L.rlfc_env_reset_params_device(self._h, C.c_void_p(d_env_ids), C.c_void_p(d_params), int(n),
                                                         int(reset_accumulators)), "rlfc_env_reset_params_device")

    def params(self):
        """Each environment's constructor arguments: a structured array with the fields re, dR, gR, theta, t_step."""
        arr = (EnvParams * self.n_envs)()
        self._check(self._L.rlfc_env_get_params(self._h, arr), "rlfc_env_get_params")
        out = np.zeros(self.n_envs, dtype=[("re", np.int32), ("dR", np.float32), ("gR", np.float32), ("theta", np.float32),
                                           ("t_step", np.float32)])
        for i in range(self.n_envs):
            for k in ENV_PARAM_KEYS:
                out[k][i] = getattr(arr[i], k)
        return out

    def step(self, actions, want_reward=True, want_done=True):
        """One RL step: actions (n_envs, 2) in [-1, 1] -> obs (n_envs, 2) = (Cl, Cd), reward, done."""
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n_envs, 2)
        obs = np.empty((self.n_envs, 2), np.float32)
        rew = np.empty(self.n_envs, np.float32) if want_reward else None
        done = np.empty(self.n_envs, np.int32) if want_done else None
        rc = self._L.rlfc_env_step(self._h, _fp(a), _fp(obs), _fp(rew),
                                   done.ctypes.data_as(C.POINTER(C.c_int)) if done is not None else None)
        self._check(rc, "rlfc_env_step")
        return obs, rew, done

    def step_device(self, d_actions, d_obs, d_reward=0, d_done=0):
        """Asynchronous RL step on device pointers (ints, e.g. torch.Tensor.data_ptr())."""
        rc = self._L.rlfc_env_step_device(self._h, C.c_void_p(d_actions), C.c_void_p(d_obs),
                                          C.c_void_p(d_reward) if d_reward else None,
                                          C.c_void_p(d_done) if d_done else None)
        self._check(rc, "rlfc_env_step_device")

    def snapshot(self, env_ids, slots):
        """Environment env_ids[k]'s complete state -> snapshot slot slots[k] (AFCCylinderBatch(n, n_snapshots=K) has K
        slots).  All or nothing: an id or slot out of range or a slot listed twice raises and changes nothing."""
        ids, sl = self._pairs(env_ids, slots)
        self._check(self._L.rlfc_env_snapshot(self._h, _ip(ids), _ip(sl), len(ids)), "rlfc_env_snapshot")

    def restore(self, env_ids, slots, keep_accumulators=False):
        """Slot slots[k] -> environment env_ids[k], which then continues bit-identically to the environment the slot was
        taken from.  keep_accumulators: the destination keeps its own callLearn, Cd, Cl and obs.  All or nothing: also
        raises for a slot never written or taken from an environment with another parameter set."""
        ids, sl = self._pairs(env_ids, slots)
        self._check(self._L.rlfc_env_restore(self._h, _ip(ids), _ip(sl), len(ids), int(keep_accumulators)), "rlfc_env_restore")

    def snapshot_device(self, d_env_ids, d_slots, n):
        """snapshot() with device int32 arrays of length n (data_ptr() ints), asynchronous on the handle's stream.  Pairs
        with an entry out of range (e.g. -1) are skipped; of pairs with the same slot the last wins."""
        self._check(self._L.rlfc_env_snapshot_device(self._h, C.c_void_p(d_env_ids), C.c_void_p(d_slots), int(n)),
                    "rlfc_env_snapshot_device")

    def restore_device(self, d_env_ids, d_slots, n, keep_accumulators=False):
        """restore() with device int32 arrays, asynchronous: restore_device(arange(B), where(done, S0, -1), B) resets the
        finished environments without the host.  Pairs out of range are skipped, the last pair per environment wins, and a
        restore from an unwritten slot or one of another parameter set is skipped and sets flags() bit 1."""
        self._check(self._L.rlfc_env_restore_device(self._h, C.c_void_p(d_env_ids), C.c_void_p(d_slots), int(n),
                                                    int(keep_accumulators)), "rlfc_env_restore_device")

    @property
    def record_bytes(self):
        """Bytes of one state record of this handle (rlfc_record_bytes)."""
        n = C.c_size_t()
        self._check(self._L.rlfc_record_bytes(C.byref(self.cfg), C.byref(n)), "rlfc_record_bytes")
        return n.value

    def export_states(self, env_ids):
        """The complete states of environments env_ids as len(env_ids) consecutive state records (include/rlfc.h "State
        records"; `records.parse_record` reads one).  Any handle of the same grid imports them, on any device or process."""
        ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        out = bytearray(len(ids) * self.record_bytes)
        buf = (C.c_char * len(out)).from_buffer(out) if out else None
        self._check(self._L.rlfc_env_export(self._h, _ip(ids), len(ids), buf), "rlfc_env_export")
        return bytes(out)

    def import_states(self, env_ids, records, keep_accumulators=False):
        """Record k of `records` (bytes of consecutive equal-size records) -> environment env_ids[k]; all or nothing: a
        record that fails a check raises RlfcError naming it, and nothing changes.  keep_accumulators: as in restore()."""
        ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        data = np.frombuffer(memoryview(records).cast("B"), np.uint8)
        if len(ids) and data.size < len(ids) * 16:
            raise ValueError(f"{data.size} bytes cannot hold {len(ids)} records")
        self._check(self._L.rlfc_env_import(self._h, _ip(ids), len(ids), data.ctypes.data if data.size else None,
                                            int(keep_accumulators)), "rlfc_env_import")

    def export_states_device(self, d_env_ids, n, d_records):
        """export_states() into a 16-byte aligned device buffer of n * record_bytes (data_ptr() ints), asynchronous on the
        handle's stream.  A pair whose id is out of range writes a record every import refuses."""
        self._check(self._L.rlfc_env_export_device(self._h, C.c_void_p(d_env_ids), int(n), C.c_void_p(d_records)),
                    "rlfc_env_export_device")

    def import_states_device(self, d_env_ids, n, d_records, record_bytes, keep_accumulators=False):
        """import_states() from a device buffer of n records of record_bytes each, asynchronous.  Ids out of range are
        skipped, the last in-range pair per environment wins; a record that fails a check leaves its environment
        unchanged and sets flags() bit 3."""
        self._check(self._L.rlfc_env_import_device(self._h, C.c_void_p(d_env_ids), int(n), C.c_void_p(d_records),
                                                   int(record_bytes), int(keep_accumulators)), "rlfc_env_import_device")

    def sensors(self):
        """(n_envs, n_sensors) float32: each environment's sensors, sampled after its most recent solver step from the
        state `get_fields` returns.  `step(a)` followed by `sensors()` gives the sensor observation of each environment."""
        out = np.empty((self.n_envs, self.n_sensors), np.float32)
        self._check(self._L.rlfc_env_get_sensors(self._h, _fp(out)), "rlfc_env_get_sensors")
        return out

    def sensors_device(self, d_out):
        """sensors() into a device float32 buffer of n_envs * n_sensors (data_ptr() int), asynchronous on the handle's
        stream: after `step_device` it gives a GPU-resident policy its observation without the host."""
        self._check(self._L.rlfc_env_get_sensors_device(self._h, C.c_void_p(d_out)), "rlfc_env_get_sensors_device")

    def stats_sums(self, e):
        """(count, sums[7, n, m] float64) of environment e's flow statistics (rlfc.h "Flow statistics"; the sums in the
        order of STAT_NAMES).  Synchronises the handle's stream."""
        count = C.c_longlong()
        sums = np.empty((len(STAT_NAMES), self.n, self.m), np.float64)
        self._check(self._L.rlfc_env_get_stats(self._h, int(e), C.byref(count), sums.ctypes.data_as(C.POINTER(C.c_double))),
                    "rlfc_env_get_stats")
        return count.value, sums

    def flow_stats(self, e):
        """Environment e's mean flow, variances and Reynolds shear stress from its sums (`flow_stats_from_sums`).  Samples
        are per step: in adaptive mode they are not weighted by dt."""
        return flow_stats_from_sums(*self.stats_sums(e))

    def stats_reset(self, env_ids=None):
        """Start new statistics for the listed environments (None = all); the next sample comes stats_every steps later.
        All or nothing: an id out of range raises and changes nothing."""
        if env_ids is None:
            rc = self._L.rlfc_env_stats_reset(self._h, None, self.n_envs)
        else:
            ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
            rc = self._L.rlfc_env_stats_reset(self._h, _ip(ids), len(ids))
        self._check(rc, "rlfc_env_stats_reset")

    def stats_reset_device(self, d_env_ids, n):
        """stats_reset() with a device int32 array of length n (data_ptr() int), asynchronous on the handle's stream: ids out
        of range are skipped, so stats_reset_device(where(done, arange(B), -1), B) restarts the finished episodes' statistics."""
        self._check(self._L.rlfc_env_stats_reset_device(self._h, C.c_void_p(d_env_ids), int(n)), "rlfc_env_stats_reset_device")

    @staticmethod
    def _pairs(env_ids, slots, what="slots"):
        ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        sl = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
        if len(ids) != len(sl):
            raise ValueError(f"{len(ids)} environment ids for {len(sl)} {what}")
        return ids, sl

    def update2(self, actions=None, want_probes=False):
        """One solver step.  Returns force (n_envs, 2) [, probes (n_envs, 32)].

        The step is the one the handle was created for: AFCCylinder.update2 with the fixed dt = t_step*resolution
        (adaptive_dt=0, the default), or AFCCylinder.update (adaptive_dt=1): every environment first takes
        dt = min(CFL, 1) of its own velocity (`check_cfl`) and then the update2 statements with it (see `dt`)."""
        a = None if actions is None else np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n_envs, 2)
        force = np.empty((self.n_envs, 2), np.float32)
        probes = np.empty((self.n_envs, NUM_PROBES), np.float32) if want_probes else None
        rc = self._L.rlfc_env_substep(self._h, _fp(a), _fp(force), _fp(probes))
        self._check(rc, "rlfc_env_substep")
        return (force, probes) if want_probes else force

    def update2_device(self, d_actions=0):
        """One solver step, asynchronous on the handle's stream; d_actions = device pointer (int) or 0 to keep xi."""
        self._check(self._L.rlfc_env_substep_device(self._h, C.c_void_p(d_actions) if d_actions else None), "rlfc_env_substep_device")

    # -- state / introspection --------------------------------------------------------------
    def get_fields(self, e=0):
        ux, uy, p = (np.empty((self.n, self.m), np.float32) for _ in range(3))
        self._check(self._L.rlfc_env_get_fields(self._h, e, _fp(ux), _fp(uy), _fp(p)), "rlfc_env_get_fields")
        return ux, uy, p

    def set_fields(self, e, ux=None, uy=None, p=None):
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float32).reshape(self.n, self.m) for a in (ux, uy, p)]
        self._check(self._L.rlfc_env_set_fields(self._h, e, *[_fp(a) for a in arrs]), "rlfc_env_set_fields")

    def save_bdim(self, e, path):
        self._check(self._L.rlfc_env_save_bdim(self._h, e, str(path).encode()), "rlfc_env_save_bdim")

    def load_bdim(self, e, path):
        self._check(self._L.rlfc_env_load_bdim(self._h, e, str(path).encode()), "rlfc_env_load_bdim")

    @property
    def t(self):
        t = np.empty(self.n_envs, np.float32)
        self._check(self._L.rlfc_env_get_time(self._h, _fp(t)), "rlfc_env_get_time")
        return t

    def check_cfl(self):
        """BDIM.checkCFL per environment: min(1/(max(|ux|+|uy|) + 3 nu), 1)."""
        dt = np.empty(self.n_envs, np.float32)
        self._check(self._L.rlfc_env_check_cfl(self._h, _fp(dt)), "rlfc_env_check_cfl")
        return dt

    def dt(self):
        """dt (grid units) of each environment's last solver step: t_step*resolution in fixed mode, the environment's
        own CFL step in adaptive mode (t_step*resolution after create / reset, the checkpoint's after load_bdim)."""
        dt = np.empty(self.n_envs, np.float32)
        self._check(self._L.rlfc_env_get_dt(self._h, _fp(dt)), "rlfc_env_get_dt")
        return dt

    def get_coeffs(self, e, name, level=0):
        """Environment e's Poisson coefficients as its last step used them ("lower.x", "lower.y", "inv", "diag" at any
        level, "c.x", "c.y", "del.x", "del.y" at level 0), reference layout.  Fixed mode without env_params: the same as
        `get_static`."""
        n, m = C.c_int(), C.c_int()
        self._check(self._L.rlfc_env_get_coeffs(self._h, e, name.encode(), level, None, C.byref(n), C.byref(m)), "rlfc_env_get_coeffs")
        out = np.empty((n.value, m.value), np.float32)
        self._check(self._L.rlfc_env_get_coeffs(self._h, e, name.encode(), level, _fp(out), None, None), "rlfc_env_get_coeffs")
        return out

    def running(self):
        """Environments that had not emitted their observation when the last RL-step round ended."""
        n = C.c_int()
        self._check(self._L.rlfc_env_running(self._h, C.byref(n)), "rlfc_env_running")
        return n.value

    def flags(self):
        """Per-environment health flags (bit 0: a non-finite force was produced since the last reset; bit 1: the last
        restore aimed at the environment was skipped, its slot unwritten or of another parameter set; bit 2: the last
        device parameter reset aimed at the environment was refused, its set invalid; bit 3: the last device import aimed
        at the environment was refused, its record failing a check)."""
        f = np.empty(self.n_envs, np.int32)
        self._check(self._L.rlfc_env_get_flags(self._h, f.ctypes.data_as(C.POINTER(C.c_int))), "rlfc_env_get_flags")
        return f

    def mg_iters(self):
        it = np.empty((self.n_envs, 2), np.int32)
        self._check(self._L.rlfc_env_get_mg_iters(self._h, it.ctypes.data_as(C.POINTER(C.c_int))), "rlfc_env_get_mg_iters")
        return it

    def field_sum(self):
        """Field.sum() of every env's pressure field (Field.pde:311-318), evaluated on the device."""
        s = np.empty(self.n_envs, np.float32)
        self._check(self._L.rlfc_env_field_sum(self._h, _fp(s)), "rlfc_env_field_sum")
        return s

    def field_sum_stats(self):
        """Counters of the last Field.sum evaluation per env (see rlfc_env_field_sum_stats)."""
        st = np.zeros((self.n_envs, 8), np.int32)
        self._check(self._L.rlfc_env_field_sum_stats(self._h, st.ctypes.data_as(C.POINTER(C.c_int))), "rlfc_env_field_sum_stats")
        return st

    @property
    def num_levels(self):
        return self._L.rlfc_env_num_levels(self._h)

    def get_static(self, name, level=0):
        n, m = C.c_int(), C.c_int()
        self._check(self._L.rlfc_env_get_static(self._h, name.encode(), level, None, C.byref(n), C.byref(m)), "rlfc_env_get_static")
        out = np.empty((n.value, m.value), np.float32)
        self._check(self._L.rlfc_env_get_static(self._h, name.encode(), level, _fp(out), None, None), "rlfc_env_get_static")
        return out

    def set_profiling(self, on=True):
        self._check(self._L.rlfc_env_set_profiling(self._h, int(on)), "rlfc_env_set_profiling")

    def get_profile(self):
        """[{name, ms, launches, bytes_per_launch}] accumulated since profiling was switched on."""
        out, idx = [], 0
        while True:
            name = C.create_string_buffer(64)
            ms, cnt, by = C.c_double(), C.c_longlong(), C.c_double()
            rc = self._L.rlfc_env_get_profile(self._h, idx, name, 64, C.byref(ms), C.byref(cnt), C.byref(by))
            if rc == 1:
                break
            self._check(rc, "rlfc_env_get_profile")
            out.append(dict(name=name.value.decode(), ms=ms.value, launches=cnt.value, bytes_per_launch=by.value))
            idx += 1
        return out

    @property
    def stream(self):
        return self._L.rlfc_env_stream(self._h)

    @property
    def launch_count(self):
        return int(self._L.rlfc_env_launch_count(self._h))

    def slab_info(self):
        """(devices sharing the domain, device-wide barriers executed so far, bytes of the shared address range)."""
        n, b, by = C.c_int(), C.c_longlong(), C.c_longlong()
        self._check(self._L.rlfc_env_slab_info(self._h, C.byref(n), C.byref(b), C.byref(by)), "rlfc_env_slab_info")
        return n.value, b.value, by.value

    def model_bytes_per_solver_step(self):
        return float(self._L.rlfc_env_model_bytes_per_solver_step(self._h))


def geometry_static(name, level=0, **overrides):
    """Host-side static geometry/coefficient field for a configuration (no GPU needed)."""
    L = load_library()
    cfg = Config()
    L.rlfc_default_config(C.byref(cfg))
    for k, v in overrides.items():
        setattr(cfg, k, v)
    n, m, nl = C.c_int(), C.c_int(), C.c_int()
    rc = L.rlfc_geometry_static(C.byref(cfg), name.encode(), level, None, C.byref(n), C.byref(m), C.byref(nl))
    if rc:
        raise RlfcError(f"rlfc_geometry_static failed ({rc}): {L.rlfc_last_error().decode()}")
    out = np.empty((n.value, m.value), np.float32)
    rc = L.rlfc_geometry_static(C.byref(cfg), name.encode(), level, _fp(out), None, None, None)
    if rc:
        raise RlfcError(f"rlfc_geometry_static failed ({rc}): {L.rlfc_last_error().decode()}")
    return out, nl.value
