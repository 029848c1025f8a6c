"""ctypes binding of ``libtrex_emu_dyn.so`` (TEST INFRASTRUCTURE ONLY): the emulator of ``emu.py`` built together with the
dynamics query (``trex_get_dynamics``), which it runs over records passed in.

``EmuDynEnv`` is an ``emu.EmuEnv`` on that library; ``dynamics(rec, envp=None)`` returns the query's three outputs for a
record ``[160]`` or records ``[n, 160]``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

import emu

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libtrex_emu_dyn.so")
_lib = None
NDOF, NB = 31, 26


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("emu_dyn_main.cpp", "emu_main.cpp", "lane_emu.h")] + [
        os.path.join(emu._CSRC, f) for f in ("trex_core.h", "trex_model.h", "trex_topology.h")
    ]
    stale = force or not os.path.isfile(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(s) for s in srcs)
    if stale:
        subprocess.check_call(
            ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-I" + emu._CSRC, "-o", _LIB,
             os.path.join(_HERE, "emu_dyn_main.cpp")]
        )
    return _LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB)
        vp, fp, u8p = ctypes.c_void_p, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint8)
        L.emu_create.restype = vp
        L.emu_create.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                 ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint]
        L.emu_destroy.argtypes = [vp]
        L.emu_last_error.restype = ctypes.c_char_p
        L.emu_state_stride.restype = ctypes.c_int
        L.emu_step.argtypes = [vp, fp, fp, fp, fp, u8p, fp, ctypes.c_int, ctypes.c_longlong]
        L.emu_step4.argtypes = [vp, ctypes.c_int, fp, fp, fp, fp, u8p, fp, ctypes.c_int, ctypes.c_longlong]
        L.emu_set_deferred.argtypes = [vp, ctypes.c_int]
        L.emu_dynamics.argtypes = [vp, ctypes.c_int, fp, fp, fp, fp, fp]
        _lib = L
    return _lib


_fp = emu._fp


class EmuDynEnv(emu.EmuEnv):
    """``EmuEnv`` on the emulator that also holds the dynamics query."""

    def __init__(self, blob: bytes, num_substeps=5, reward_weights=(1.0, 0.005, 0.002), max_episode_steps=0,
                 contacts=True, reset_mode=0, seed=0, env_id=0, deferred=True):
        self._L = lib()
        d, e, k = reward_weights
        self._h = self._L.emu_create(blob, len(blob), num_substeps, d, e, k, max_episode_steps, int(contacts), int(reset_mode), int(seed))
        if not self._h:
            raise RuntimeError(self._L.emu_last_error().decode())
        self.env_id = int(env_id)
        self._L.emu_set_deferred(self._h, int(deferred))
        self.stride = self._L.emu_state_stride()
        self.rec = np.zeros(self.stride, np.float32)
        self.rec[6] = 1.0
        self.aux = np.zeros(8, np.float32)

    def dynamics(self, rec=None, envp=None, outputs="Mbj"):
        """(M [n, 31, 31], b [n, 31], J [n, 26, 6, 31]) of records [n, 160] (or [160]: no leading axis; None: ``self.rec``),
        with the mass scales of parameter rows envp [n, 32] (None: the model's masses).  Outputs whose letter is missing
        from ``outputs`` are passed as NULL and returned as None."""
        r = np.ascontiguousarray(self.rec if rec is None else rec, np.float32)
        one = r.ndim == 1
        r = r.reshape(-1, self.stride)
        n = r.shape[0]
        ep = None if envp is None else np.ascontiguousarray(np.broadcast_to(envp, (n, 32)), np.float32)
        M = np.zeros((n, NDOF, NDOF), np.float32) if "M" in outputs else None
        b = np.zeros((n, NDOF), np.float32) if "b" in outputs else None
        J = np.zeros((n, NB, 6, NDOF), np.float32) if "j" in outputs else None
        self._L.emu_dynamics(self._h, n, _fp(r), None if ep is None else _fp(ep), *(None if x is None else _fp(x) for x in (M, b, J)))
        if one:
            return tuple(None if x is None else x[0] for x in (M, b, J))
        return M, b, J
