"""ctypes wrapper around oracle/oracle.c -- TEST INFRASTRUCTURE ONLY (see the header of oracle.c).

`OracleSim` plays the role the pair (`mujoco.MjModel`, `mujoco.MjData`) plays in the reference
(gymnasium_robotics/envs/robot_env.py:292-303): numpy views alias the C arrays.
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this module.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


_NATIVE = False


def use_native_build():
    """bench.py's CPU arm only: build and load liboracle with `-O3 -march=native` for the box it runs on (the default -O2 build is
    what the parity tests use and what travels between machines).  Must be called before the first `lib()`."""
    global _NATIVE
    if _LIB is None:
        _NATIVE = True


def build(force: bool = False) -> str:
    """Compile oracle.c -> oracle/_build/liboracle.so with gcc (idempotent).  The native build goes to a fresh temporary directory,
    removed at exit: bench.py, its only user, runs from a tree it does not write to."""
    src = os.path.join(_HERE, "oracle.c")
    if _NATIVE:
        import atexit
        import shutil
        import tempfile

        out = os.path.join(tempfile.mkdtemp(prefix="liboracle_native_"), "liboracle.so")
        atexit.register(shutil.rmtree, os.path.dirname(out), True)
        subprocess.check_call(["gcc", "-O3", "-march=native", "-fPIC", "-shared", "-o", out, src, "-lm"])
        return out
    out = os.path.join(_HERE, "_build", "liboracle.so")
    hdr = os.path.join(_HERE, "..", "include", "b200sim_model.h")
    if force or not os.path.exists(out) or (os.path.exists(src) and os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(hdr))):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", tmp, src, "-lm"])
        os.replace(tmp, out)
    return out


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        L.oracle_create.restype = ctypes.c_void_p
        L.oracle_create.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
        for f in ("oracle_destroy", "oracle_reset_data", "oracle_forward"):
            getattr(L, f).argtypes = [ctypes.c_void_p]
            getattr(L, f).restype = None
        L.oracle_step.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.oracle_step.restype = None
        L.oracle_jac_site.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.oracle_contact.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        for f in ("oracle_ncon", "oracle_nefc", "oracle_solver_iter", "oracle_overflow"):
            getattr(L, f).argtypes = [ctypes.c_void_p]
            getattr(L, f).restype = ctypes.c_int
        L.oracle_set_noslip.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.oracle_set_noslip.restype = None
        L.oracle_noslip_iter.argtypes = [ctypes.c_void_p]
        L.oracle_cfrc_ext.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.oracle_cfrc_ext.restype = None
        L.oracle_cfrc_rows.argtypes = [ctypes.c_void_p]
        L.oracle_total_newton_iter.argtypes = [ctypes.c_void_p]
        L.oracle_total_newton_iter.restype = ctypes.c_long
        L.oracle_size.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.oracle_size.restype = ctypes.c_int
        _LIB = L
    return _LIB


class OracleSim:
    _FIELDS = {  # name -> shape lambda(model)
        "qpos": lambda m: (m.nq,), "qvel": lambda m: (m.nv,), "ctrl": lambda m: (m.nu,),
        "mocap_pos": lambda m: (m.nmocap, 3), "mocap_quat": lambda m: (m.nmocap, 4),
        "qacc_warmstart": lambda m: (m.nv,), "qacc": lambda m: (m.nv,),
        "xpos": lambda m: (m.nbody, 3), "xquat": lambda m: (m.nbody, 4), "xmat": lambda m: (m.nbody, 9),
        "site_xpos": lambda m: (m.nsite, 3), "site_xmat": lambda m: (m.nsite, 9),
        "geom_xpos": lambda m: (m.ngeom, 3), "geom_xmat": lambda m: (m.ngeom, 9),
        "eq_data": lambda m: (m.neq, 11), "act_gainprm": lambda m: (m.nu, 3), "act_biasprm": lambda m: (m.nu, 3),
        "body_pos": lambda m: (m.nbody, 3), "body_quat": lambda m: (m.nbody, 4), "M": lambda m: (m.nv, m.nv), "qfrc_bias": lambda m: (m.nv,),
        "qfrc_smooth": lambda m: (m.nv,), "qacc_smooth": lambda m: (m.nv,), "qfrc_constraint": lambda m: (m.nv,),
        "qfrc_actuator": lambda m: (m.nv,), "qfrc_passive": lambda m: (m.nv,),
        "sensordata": lambda m: (m.nsensor,), "subtree_com": lambda m: (m.nbody, 3), "cdof": lambda m: (m.nv, 6),
        "time": lambda m: (1,),
    }

    def __init__(self, model):
        """model: gymnasium_robotics_b200.mjcf.Model"""
        self.model = model
        blob = model.to_blob()
        self._L = lib()
        self._h = self._L.oracle_create(blob, len(blob))
        if not self._h:
            raise RuntimeError("oracle_create failed (bad blob)")
        for name, shp in self._FIELDS.items():
            fn = getattr(self._L, "oracle_" + name)
            fn.restype = ctypes.POINTER(ctypes.c_double)
            fn.argtypes = [ctypes.c_void_p]
            shape = shp(model)
            n = int(np.prod(shape))
            if n == 0:
                setattr(self, name, np.zeros(shape))
                continue
            ptr = fn(self._h)
            setattr(self, name, np.ctypeslib.as_array(ptr, shape=(n,)).reshape(shape))

    def __del__(self):
        try:
            if self._h:
                self._L.oracle_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # mj_* equivalents ---------------------------------------------------------------
    def reset_data(self):
        self._L.oracle_reset_data(self._h)

    def forward(self):
        self._L.oracle_forward(self._h)

    def step(self, nstep=1):
        self._L.oracle_step(self._h, int(nstep))

    def jac_site(self, site):
        nv = self.model.nv
        jp, jr = np.zeros((3, nv)), np.zeros((3, nv))
        self._L.oracle_jac_site(self._h, int(site), jp.ctypes.data, jr.ctypes.data)
        return jp, jr

    @property
    def ncon(self):
        return self._L.oracle_ncon(self._h)

    @property
    def nefc(self):
        return self._L.oracle_nefc(self._h)

    @property
    def solver_iter(self):
        return self._L.oracle_solver_iter(self._h)

    def set_noslip(self, on: bool):
        """Switch the noslip post-pass (models with <option noslip_iterations>) on or off; on by default."""
        self._L.oracle_set_noslip(self._h, int(bool(on)))

    @property
    def noslip_iter(self):
        return self._L.oracle_noslip_iter(self._h)

    def cfrc_ext(self):
        """data.cfrc_ext after an explicit mj_rnePostConstraint [ext]: one row per MJCF body, torque | force (contacts only)."""
        out = np.zeros((int(self._L.oracle_cfrc_rows(self._h)), 6))
        self._L.oracle_cfrc_ext(self._h, out.ctypes.data)
        return out

    @property
    def total_newton_iter(self):
        return self._L.oracle_total_newton_iter(self._h)

    @property
    def overflow(self):
        return self._L.oracle_overflow(self._h)

    def contacts(self):
        out = []
        buf = np.zeros(17)
        for k in range(self.ncon):
            self._L.oracle_contact(self._h, k, buf.ctypes.data)
            out.append(dict(dist=buf[0], pos=buf[1:4].copy(), frame=buf[4:13].copy().reshape(3, 3), dim=int(buf[13]),
                            geom1=int(buf[14]), geom2=int(buf[15]), efc_address=int(buf[16])))
        return out

    def efc(self, name):
        fn = getattr(self._L, "oracle_efc_" + name)
        fn.restype = ctypes.POINTER(ctypes.c_double)
        fn.argtypes = [ctypes.c_void_p]
        n = self.nefc * (self.model.nv if name == "J" else 1)
        a = np.ctypeslib.as_array(fn(self._h), shape=(max(n, 1),))[:n].copy()
        return a.reshape(self.nefc, -1) if name == "J" else a
