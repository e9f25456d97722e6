"""ctypes front end of the CPU oracle (oracle/lilypad_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs.  Nothing under rlfluidcontrol_b200/ may import this module.
PARITY UNPINNED -- see the header of lilypad_oracle.h.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = _HERE / "_build" / "liblilypad_oracle.so"
CLI = _HERE / "_build" / "oracle_cli"


def build(force: bool = False) -> Path:
    """Compile the oracle with oracle/Makefile (gcc -O2 -ffp-contract=off)."""
    src_m = max((_HERE / f).stat().st_mtime for f in ("lilypad_oracle.c", "lilypad_oracle.h", "oracle_cli.c"))
    if force or not _LIB.exists() or not CLI.exists() or _LIB.stat().st_mtime < src_m:
        subprocess.run(["make", "-C", str(_HERE), "-s"], check=True, stdout=subprocess.DEVNULL)
    return _LIB


class _Field(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("btype", C.c_int), ("gradientExit", C.c_int),
                ("bval", C.c_float), ("a", C.POINTER(C.c_float))]


class _VField(C.Structure):
    _fields_ = [("x", _Field), ("y", _Field)]


class _Poisson(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("lower", _VField), ("diagonal", _Field), ("inv", _Field)]


class Config(C.Structure):
    _fields_ = [("resolution", C.c_int), ("xLengths", C.c_int), ("yLengths", C.c_int), ("Re", C.c_int),
                ("dR", C.c_float), ("gR", C.c_float), ("theta", C.c_float), ("tStep", C.c_float),
                ("literal", C.c_int)]


class _Driver(C.Structure):
    _fields_ = [("callLearn", C.c_int), ("Cd", C.c_float), ("Cl", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(_LIB))
        fp = C.POINTER(C.c_float)
        L.ora_default_config.restype = Config
        L.ora_env_new.restype = C.c_void_p
        L.ora_env_new.argtypes = [C.POINTER(Config)]
        L.ora_env_free.argtypes = [C.c_void_p]
        for nm in ("ora_env_n", "ora_env_m"):
            getattr(L, nm).restype = C.c_int
            getattr(L, nm).argtypes = [C.c_void_p]
        L.ora_env_set_state.argtypes = [C.c_void_p, fp, fp, fp]
        L.ora_env_get_state.argtypes = [C.c_void_p, fp, fp, fp]
        L.ora_env_set_xi.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.ora_env_update2.argtypes = [C.c_void_p]
        L.ora_env_check_cfl.restype = C.c_float
        L.ora_env_check_cfl.argtypes = [C.c_void_p]
        L.ora_env_dt.restype = C.c_float
        L.ora_env_dt.argtypes = [C.c_void_p]
        L.ora_env_update_adaptive.restype = None
        L.ora_env_update_adaptive.argtypes = [C.c_void_p]
        L.ora_env_t.restype = C.c_float
        L.ora_env_t.argtypes = [C.c_void_p]
        L.ora_env_force.argtypes = [C.c_void_p, fp, fp]
        L.ora_env_probes.argtypes = [C.c_void_p, C.c_int, fp]
        L.ora_env_last_mg_iters.restype = C.c_int
        L.ora_env_last_mg_iters.argtypes = [C.c_void_p, C.c_int]
        L.ora_env_coeff.restype = fp
        L.ora_env_coeff.argtypes = [C.c_void_p, C.c_char_p]
        L.ora_driver_new.restype = _Driver
        L.ora_driver_step.restype = C.c_int
        L.ora_driver_step.argtypes = [C.POINTER(_Driver), C.c_void_p, C.c_float, fp, fp]
        L.ora_read_bdim_text.restype = C.c_int
        L.ora_read_bdim_text.argtypes = [C.c_char_p, C.c_int, C.c_int, fp, fp, fp, fp, fp]
        # operator-level entry points
        L.ora_field_new.restype = _Field
        L.ora_field_new.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float]
        L.ora_field_free.argtypes = [C.POINTER(_Field)]
        L.ora_field_setBC.argtypes = [C.POINTER(_Field)]
        L.ora_field_linear.restype = C.c_float
        L.ora_field_linear.argtypes = [C.POINTER(_Field), C.c_float, C.c_float]
        L.ora_field_inner.restype = C.c_float
        L.ora_field_inner.argtypes = [C.POINTER(_Field), C.POINTER(_Field)]
        L.ora_field_sum.restype = C.c_float
        L.ora_field_sum.argtypes = [C.POINTER(_Field)]
        L.ora_field_Linf.restype = C.c_float
        L.ora_field_Linf.argtypes = [C.POINTER(_Field)]
        L.ora_vfield_new.restype = _VField
        L.ora_vfield_new.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float]
        L.ora_vfield_free.argtypes = [C.POINTER(_VField)]
        L.ora_vfield_setBC.argtypes = [C.POINTER(_VField)]
        L.ora_vfield_AdvDif.argtypes = [C.POINTER(_VField), C.POINTER(_VField), C.c_float, C.c_float]
        L.ora_vfield_divergence.restype = _Field
        L.ora_vfield_divergence.argtypes = [C.POINTER(_VField)]
        L.ora_field_gradient.restype = _VField
        L.ora_field_gradient.argtypes = [C.POINTER(_Field)]
        L.ora_vfield_project.restype = C.c_int
        L.ora_vfield_project.argtypes = [C.POINTER(_VField), C.POINTER(_VField), C.POINTER(_Field), C.c_int, C.c_void_p]
        L.ora_poisson_new.restype = _Poisson
        L.ora_poisson_new.argtypes = [C.POINTER(_VField)]
        L.ora_poisson_free.argtypes = [C.POINTER(_Poisson)]
        L.ora_poisson_times.restype = _Field
        L.ora_poisson_times.argtypes = [C.POINTER(_Poisson), C.POINTER(_Field)]
        L.ora_mg_solve.restype = C.c_int
        L.ora_mg_solve.argtypes = [C.c_float, C.POINTER(_Poisson), C.POINTER(_Field), C.POINTER(_Field),
                                   C.c_void_p, C.c_int, fp, fp]
        L.ora_mg_restrict_matrix.restype = _Poisson
        L.ora_mg_restrict_matrix.argtypes = [C.POINTER(_Poisson)]
        L.ora_mg_restrict_field.restype = _Field
        L.ora_mg_restrict_field.argtypes = [C.POINTER(_Field)]
        L.ora_mg_prolongate.restype = _Field
        L.ora_mg_prolongate.argtypes = [C.POINTER(_Field)]
        L.ora_body_new.restype = C.c_void_p
        L.ora_body_new.argtypes = [C.c_float, C.c_float]
        L.ora_body_add.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.ora_body_end.argtypes = [C.c_void_p]
        L.ora_circle_new.restype = C.c_void_p
        L.ora_circle_new.argtypes = [C.c_float, C.c_float, C.c_float]
        L.ora_body_free.argtypes = [C.c_void_p]
        L.ora_body_distance.restype = C.c_float
        L.ora_body_distance.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.ora_body_wallnormal.argtypes = [C.c_void_p, C.c_float, C.c_float, fp, fp]
        L.ora_bdim_delta0.restype = C.c_float
        L.ora_bdim_delta0.argtypes = [C.c_float, C.c_float]
        L.ora_bdim_delta1.restype = C.c_float
        L.ora_bdim_delta1.argtypes = [C.c_float, C.c_float]
        L.ora_union_delta0.restype = C.c_float
        L.ora_union_delta0.argtypes = [C.c_float]
        _lib = L
    return _lib


def _fp(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags.c_contiguous
    return a.ctypes.data_as(C.POINTER(C.c_float))


# ----------------------------------------------------------------------------------------------
# operator-level helpers working on numpy arrays (n x m, i-major)
# ----------------------------------------------------------------------------------------------
class Field:
    """Owned oracle Field (Field.pde:24-58) with a numpy view `.a` of shape (n, m)."""

    def __init__(self, n, m, btype=0, bval=0.0, gradientExit=False, values=None, _raw=None):
        self._f = _raw if _raw is not None else lib().ora_field_new(n, m, btype, C.c_float(bval))
        self._f.gradientExit = int(gradientExit)
        self.a = np.ctypeslib.as_array(self._f.a, shape=(self._f.n, self._f.m))
        if values is not None:
            self.a[...] = np.asarray(values, dtype=np.float32)

    @property
    def n(self): return self._f.n

    @property
    def m(self): return self._f.m

    def setBC(self): lib().ora_field_setBC(C.byref(self._f))
    def linear(self, x, y): return float(lib().ora_field_linear(C.byref(self._f), x, y))
    def inner(self, o): return float(lib().ora_field_inner(C.byref(self._f), C.byref(o._f)))
    def sum(self): return float(lib().ora_field_sum(C.byref(self._f)))
    def Linf(self): return float(lib().ora_field_Linf(C.byref(self._f)))
    def gradient(self): return VField(_raw=lib().ora_field_gradient(C.byref(self._f)))

    def __del__(self):
        try:
            lib().ora_field_free(C.byref(self._f))
        except Exception:
            pass


class VField:
    """Owned oracle VectorField (VectorField.pde:22-39)."""

    def __init__(self, n=0, m=0, xval=0.0, yval=0.0, _raw=None):
        self._v = _raw if _raw is not None else lib().ora_vfield_new(n, m, C.c_float(xval), C.c_float(yval))
        self.x = np.ctypeslib.as_array(self._v.x.a, shape=(self._v.x.n, self._v.x.m))
        self.y = np.ctypeslib.as_array(self._v.y.a, shape=(self._v.y.n, self._v.y.m))

    def set_gradient_exit(self, flag=True): self._v.x.gradientExit = int(flag)
    def setBC(self): lib().ora_vfield_setBC(C.byref(self._v))
    def AdvDif(self, u0: "VField", dt, nu): lib().ora_vfield_AdvDif(C.byref(self._v), C.byref(u0._v), dt, nu)
    def divergence(self): return Field(0, 0, _raw=lib().ora_vfield_divergence(C.byref(self._v)))

    def project(self, coeffs: "VField", p: Field) -> int:
        return lib().ora_vfield_project(C.byref(self._v), C.byref(coeffs._v), C.byref(p._f), 1, None)

    def __del__(self):
        try:
            lib().ora_vfield_free(C.byref(self._v))
        except Exception:
            pass


class Poisson:
    def __init__(self, lower: VField = None, _raw=None):
        self._A = _raw if _raw is not None else lib().ora_poisson_new(C.byref(lower._v))
        n, m = self._A.n, self._A.m
        self.lx = np.ctypeslib.as_array(self._A.lower.x.a, shape=(n, m))
        self.ly = np.ctypeslib.as_array(self._A.lower.y.a, shape=(n, m))
        self.diag = np.ctypeslib.as_array(self._A.diagonal.a, shape=(n, m))
        self.inv = np.ctypeslib.as_array(self._A.inv.a, shape=(n, m))

    def times(self, x: Field): return Field(0, 0, _raw=lib().ora_poisson_times(C.byref(self._A), C.byref(x._f)))
    def restrict(self): return Poisson(_raw=lib().ora_mg_restrict_matrix(C.byref(self._A)))

    def solve(self, x: Field, b: Field, itmx=20.0):
        rr, tol = C.c_float(), C.c_float()
        it = lib().ora_mg_solve(itmx, C.byref(self._A), C.byref(x._f), C.byref(b._f), None, 0, C.byref(rr), C.byref(tol))
        return it, rr.value, tol.value

    def __del__(self):
        try:
            lib().ora_poisson_free(C.byref(self._A))
        except Exception:
            pass


def restrict_field(a: Field): return Field(0, 0, _raw=lib().ora_mg_restrict_field(C.byref(a._f)))
def prolongate(a: Field): return Field(0, 0, _raw=lib().ora_mg_prolongate(C.byref(a._f)))


# ----------------------------------------------------------------------------------------------
# the environment
# ----------------------------------------------------------------------------------------------
class OracleEnv:
    """One AFCCylinder environment (AFCCylinder.pde) + the clientCFD.draw() accumulation."""

    def __init__(self, literal: bool = False, **kw):
        L = lib()
        cfg = L.ora_default_config()
        cfg.literal = int(literal)
        for k, v in kw.items():
            setattr(cfg, k, v)
        self.cfg = cfg
        self._e = L.ora_env_new(C.byref(cfg))
        if not self._e:
            raise ValueError(f"the reference cannot run the grid resolution={cfg.resolution}, xLengths={cfg.xLengths}, "
                             f"yLengths={cfg.yLengths} (MG.pde:94-104,139-152)")
        self.n, self.m = L.ora_env_n(self._e), L.ora_env_m(self._e)
        self._drv = L.ora_driver_new()

    def close(self):
        if self._e:
            lib().ora_env_free(self._e)
            self._e = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_state(self, ux, uy, p):
        ux, uy, p = (np.ascontiguousarray(a, dtype=np.float32).reshape(self.n, self.m) for a in (ux, uy, p))
        lib().ora_env_set_state(self._e, _fp(ux), _fp(uy), _fp(p))

    def get_state(self):
        ux, uy, p = (np.empty((self.n, self.m), np.float32) for _ in range(3))
        lib().ora_env_get_state(self._e, _fp(ux), _fp(uy), _fp(p))
        return ux, uy, p

    def set_xi(self, xi1, xi2): lib().ora_env_set_xi(self._e, float(xi1), float(xi2))
    def check_cfl(self): return np.float32(lib().ora_env_check_cfl(self._e))          # BDIM.checkCFL
    def update_adaptive(self): lib().ora_env_update_adaptive(self._e)                 # AFCCylinder.update(), one pass
    @property
    def dt(self): return np.float32(lib().ora_env_dt(self._e))
    def update2(self): lib().ora_env_update2(self._e)

    @property
    def t(self): return float(lib().ora_env_t(self._e))

    def force(self):
        fx, fy = C.c_float(), C.c_float()
        lib().ora_env_force(self._e, C.byref(fx), C.byref(fy))
        return np.float32(fx.value), np.float32(fy.value)

    def probes(self, num=32):
        out = np.empty(num, np.float32)
        lib().ora_env_probes(self._e, num, _fp(out))
        return out

    def mg_iters(self): return tuple(lib().ora_env_last_mg_iters(self._e, w) for w in (0, 1))

    def coeff(self, name):
        ptr = lib().ora_env_coeff(self._e, name.encode())
        if not ptr:
            raise KeyError(name)
        return np.ctypeslib.as_array(ptr, shape=(self.n, self.m)).copy()

    def adopt_driver(self, other):
        """Take over another environment's draw() accumulators: callLearn, Cd, Cl are sketch globals that survive
        setUpNewSim (clientCFD.pde:11-13)."""
        self._drv = other._drv

    def driver_step(self, init_time=-1.0):
        """One solver step + clientCFD.draw() accumulation.  Returns (Cl, Cd) when an observation was
        produced on this step, else None."""
        cl, cd = C.c_float(), C.c_float()
        if lib().ora_driver_step(C.byref(self._drv), self._e, init_time, C.byref(cl), C.byref(cd)):
            return np.float32(cl.value), np.float32(cd.value)
        return None

    def env_step(self, action, substeps=16, init_time=-1.0):
        """Apply an action (xi1, xi2) in [-1,1], run `substeps` solver steps, return (Cl, Cd).
        Mirrors one callAction period of clientCFD.draw() once t > initTime."""
        self.set_xi(action[0], action[1])
        obs = None
        for _ in range(substeps):
            obs = self.driver_step(init_time)
        return obs


def read_bdimb(path):
    """Read the committed binary fixture (format in lilypad_oracle.h)."""
    raw = Path(path).read_bytes()
    assert raw[:8] == b"RLFCBDIM"
    n, m = np.frombuffer(raw, np.int32, 2, 8)
    t, dt = np.frombuffer(raw, np.float32, 2, 16)
    N = int(n) * int(m)
    arr = np.frombuffer(raw, np.float32, 3 * N, 24).reshape(3, n, m).copy()
    return dict(n=int(n), m=int(m), t=float(t), dt=float(dt), ux=arr[0], uy=arr[1], p=arr[2])


def reference_reward(cd_next, action):
    """server/server.py:61-65 `_reward_func` restated: -Cd - pi/8*0.0097*3.66**3*sum|a|^3 ... see tests."""
    a = np.abs(np.asarray(action, dtype=np.float64))
    return -float(cd_next) - np.pi / 8 * 0.0097 * 3.66 ** 3 * float(np.sum(a ** 3))
