"""ctypes binding of ``libtrex_emu_envp.so`` (TEST INFRASTRUCTURE ONLY): the warp emulator of ``emu.py`` built together with
the ENVP instances of the product kernels (per-environment dynamics parameters, ``trex_config.env_params = 1``).

``EmuEnvpEnv`` / ``EmuEnvpWarp4`` behave like ``EmuEnv`` / ``EmuWarp4`` -- bit for bit the uniform path -- until
``set_env_params`` gives the handle parameter rows; from then on they step through the ENVP instances.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

import emu

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libtrex_emu_envp.so")
_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("emu_envp_main.cpp", "emu_main.cpp", "lane_emu.h")] + [
        os.path.join(emu._CSRC, f) for f in ("trex_core.h", "trex_model.h", "trex_topology.h")
    ]
    stale = force or not os.path.isfile(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(s) for s in srcs)
    if stale:
        subprocess.check_call(
            ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-I" + emu._CSRC, "-o", _LIB,
             os.path.join(_HERE, "emu_envp_main.cpp")]
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
        L.emu_shared_bytes.restype = ctypes.c_int
        L.emu_step.argtypes = [vp, fp, fp, fp, fp, u8p, fp, ctypes.c_int, ctypes.c_longlong]
        L.emu_step4.argtypes = [vp, ctypes.c_int, fp, fp, fp, fp, u8p, fp, ctypes.c_int, ctypes.c_longlong]
        L.emu_set_deferred.argtypes = [vp, ctypes.c_int]
        L.emu_set_env_params.argtypes = [vp, fp, ctypes.c_int]
        L.emu_get_env_params.argtypes = [vp, fp, ctypes.c_int]
        L.emu_default_env_params.argtypes = [vp, fp]
        L.emu_set_env_param_ranges.restype = ctypes.c_int
        L.emu_set_env_param_ranges.argtypes = [vp, fp, fp]
        _lib = L
    return _lib


_fp = emu._fp


class EmuEnvpEnv(emu.EmuEnv):
    """``EmuEnv`` on the emulator that also holds the ENVP instances."""

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

    def default_env_params(self):
        row = np.zeros(32, np.float32)
        self._L.emu_default_env_params(self._h, _fp(row))
        return row

    def set_env_params(self, rows):
        """Run the ENVP instances from now on, with these rows ([32] or [n, 32]; element 30 is derived from 29)."""
        r = np.ascontiguousarray(np.atleast_2d(np.asarray(rows, np.float32)))
        self._L.emu_set_env_params(self._h, _fp(r), r.shape[0])

    def get_env_params(self, n=1):
        out = np.zeros((n, 32), np.float32)
        self._L.emu_get_env_params(self._h, _fp(out), n)
        return out

    def set_env_param_ranges(self, lo, hi):
        """Randomizer ranges (None, None: off); raises ValueError on ranges the library rejects."""
        if lo is None and hi is None:
            rc = self._L.emu_set_env_param_ranges(self._h, None, None)
        else:
            lo = np.ascontiguousarray(lo, np.float32)
            hi = np.ascontiguousarray(hi, np.float32)
            rc = self._L.emu_set_env_param_ranges(self._h, _fp(lo), _fp(hi))
        if rc != 0:
            raise ValueError(self._L.emu_last_error().decode())


class EmuEnvpWarp4(emu.EmuWarp4):
    """``EmuWarp4`` on the emulator that also holds the ENVP instances (``self.env`` is an ``EmuEnvpEnv``)."""

    def __init__(self, blob: bytes, n=4, deferred=True, **kw):
        self.env = EmuEnvpEnv(blob, deferred=deferred, **kw)
        self.n = n
        self.stride = self.env.stride
        self.rec = np.zeros((n, self.stride), np.float32)
        self.rec[:, 6] = 1.0
        self.aux = np.zeros((n, 8), np.float32)
