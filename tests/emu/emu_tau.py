"""ctypes binding of ``libtrex_emu_tau.so`` (TEST INFRASTRUCTURE ONLY): the emulator of ``emu_extf.py`` built together with
the TAU instances of the front and tail phases (joint torque control, ``trex_config.actuation = TREX_ACTUATION_TORQUE``).

``EmuTauEnv`` / ``EmuTauWarp4`` behave like ``EmuExtfEnv`` / ``EmuExtfWarp4`` until ``set_torque_mode`` switches the handle;
from then on an action is the joint torque, and they step through the TAU instances (with the ENVP / EXTF instances as well
once the handle has parameter rows / a wrench record).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

import emu
import emu_extf

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libtrex_emu_tau.so")
_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("emu_tau_main.cpp", "emu_extf_main.cpp", "emu_envp_main.cpp", "emu_main.cpp",
                                             "lane_emu.h")] + [
        os.path.join(emu._CSRC, f) for f in ("trex_core.h", "trex_model.h", "trex_topology.h")
    ]
    stale = force or not os.path.isfile(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(s) for s in srcs)
    if stale:
        subprocess.check_call(
            ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-I" + emu._CSRC, "-o", _LIB,
             os.path.join(_HERE, "emu_tau_main.cpp")]
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
        L.emu_tau_step4.argtypes = [vp, ctypes.c_int, fp, fp, fp, fp, u8p, fp, ctypes.c_int, ctypes.c_longlong]
        L.emu_set_deferred.argtypes = [vp, ctypes.c_int]
        L.emu_set_env_params.argtypes = [vp, fp, ctypes.c_int]
        L.emu_get_env_params.argtypes = [vp, fp, ctypes.c_int]
        L.emu_default_env_params.argtypes = [vp, fp]
        L.emu_set_env_param_ranges.restype = ctypes.c_int
        L.emu_set_env_param_ranges.argtypes = [vp, fp, fp]
        L.emu_set_external_forces.argtypes = [vp, fp, ctypes.c_int]
        L.emu_get_external_forces.argtypes = [vp, fp, ctypes.c_int]
        L.emu_set_push_schedule.restype = ctypes.c_int
        L.emu_set_push_schedule.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_float, ctypes.c_float, ctypes.c_float]
        L.emu_body_com.argtypes = [vp, fp]
        L.emu_extf_forget.argtypes = [vp]
        L.emu_set_torque_mode.argtypes = [vp]
        L.emu_tau_forget.argtypes = [vp]
        _lib = L
    return _lib


_fp = emu._fp


def _u8p(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


class EmuTauEnv(emu_extf.EmuExtfEnv):
    """``EmuExtfEnv`` on the emulator that also holds the TAU instances."""

    def __init__(self, blob: bytes, num_substeps=5, reward_weights=(1.0, 0.005, 0.002), max_episode_steps=0,
                 contacts=True, reset_mode=0, seed=0, env_id=0, deferred=True, torque=False):
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
        if torque:
            self.set_torque_mode()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.emu_tau_forget(h)
        super().__del__()

    def set_torque_mode(self):
        """Actions are joint torques from now on (the TAU instances, motors without gain or strength)."""
        self._L.emu_set_torque_mode(self._h)

    def _call(self, n, rec, action, aux, force_reset):
        obs = np.zeros((n, 75), np.float32)
        r = np.zeros(n, np.float32)
        d = np.zeros(n, np.uint8)
        a = None if action is None else _fp(np.ascontiguousarray(action, np.float32))
        self._L.emu_tau_step4(self._h, n, _fp(rec), a, _fp(obs), _fp(r), _u8p(d), _fp(aux), int(force_reset), self.env_id)
        return obs, r, d


class EmuTauWarp4(emu.EmuWarp4):
    """``EmuWarp4`` on the emulator that also holds the TAU instances (``self.env`` is an ``EmuTauEnv``)."""

    def __init__(self, blob: bytes, n=4, deferred=True, **kw):
        self.env = EmuTauEnv(blob, deferred=deferred, **kw)
        self.n = n
        self.stride = self.env.stride
        self.rec = np.zeros((n, self.stride), np.float32)
        self.rec[:, 6] = 1.0
        self.aux = np.zeros((n, 8), np.float32)

    def _call(self, action, force_reset):
        return self.env._call(self.n, self.rec, action, self.aux, force_reset)
