"""The CPU oracle with joint torque control (TEST INFRASTRUCTURE ONLY): ``libtrex_oracle_tau.so``.

pybullet's torque control (``setJointMotorControlArray(controlMode=TORQUE_CONTROL, forces=tau)`` after the motors were turned
off with ``VELOCITY_CONTROL, forces=0``) adds tau to the joint force of the articulated-body pass, where pybullet's joint
damping enters as an explicit joint torque, and the motor rows keep no gain and no strength.  The oracle
(``oracle/trex_oracle.c``) has no such input, and it stays as it is.  This module builds a second library from that source
unchanged, with insertions at fixed anchors (each must occur exactly once, or the build fails):
  - a field of ``struct trex_oracle``: the torque-mode flag, its bound and the commanded torques;
  - in ``trex_oracle_substep``, at the damping line: ``jt[k] += tau[k]`` while torque mode is on and not suppressed;
  - in ``trex_oracle_substep``, behind the motor-impulse read-back: the applied joint torque reported is the command;
  - in ``trex_oracle_reset``: the torques are suppressed for the reset's physics step (its motors are zero-gain already);
  - in ``trex_oracle_step``: in torque mode the action is clipped to +-bound into the commanded torques and the substeps
    run with kp = kd = 0 and motor impulse bound 0.
Everything else -- kinematics, ABA, constraint rows, PGS -- is the oracle's own code.  ``OracleTau`` is
``oracle.oracle.Oracle`` on that library plus ``set_torque_mode``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

from oracle import oracle as _oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_DIR = os.path.normpath(os.path.join(_HERE, "..", "..", "oracle"))
_LIB = os.path.join(_HERE, "libtrex_oracle_tau.so")
_lib = None

_ANCHOR_FIELDS = "  row_t* rows;\n};\n"
_ANCHOR_DAMPING = "  for (int k = 0; k < nd; k++) jt[k] = -o->damping[o->dof_link[k]] * o->qd[k];\n"
_ANCHOR_READBACK = "    if (rows[j].motor_dof >= 0) o->tau[rows[j].motor_dof] = rows[j].lam / dt;\n"
_ANCHOR_RESET = "  trex_oracle_substep(o, zero, 0.0);\n"
_ANCHOR_STEP = ("  o->sig = 0;\n"
                "  for (int s = 0; s < o->n_sub; s++) /* trex_env.py:148-150 ; max impulse = force*dt */\n"
                "    trex_oracle_substep(o, target, o->P[P_MAX_TORQUE] * dt);\n")
_INSERTIONS = (
    (_ANCHOR_FIELDS,
     "  row_t* rows;\n"
     "  int tau_on, tau_off;     /* torque mode; tau_off: suppressed (the physics step of a reset) */\n"
     "  double tau_bound;        /* |command| <= tau_bound */\n"
     "  double jtau[MAXDOF];     /* commanded joint torques of the current step, per dof */\n"
     "};\n"),
    (_ANCHOR_DAMPING,
     _ANCHOR_DAMPING +
     "  if (o->tau_on && !o->tau_off) for (int k = 0; k < nd; k++) jt[k] += o->jtau[k]; /* TORQUE_CONTROL: next to damping */\n"),
    (_ANCHOR_READBACK,
     _ANCHOR_READBACK +
     "  if (o->tau_on && !o->tau_off) for (int k = 0; k < nd; k++) o->tau[k] = o->jtau[k]; /* applied torque = the command */\n"),
    (_ANCHOR_RESET,
     "  o->tau_off = 1; /* no joint torque in the reset's physics step */\n" + _ANCHOR_RESET + "  o->tau_off = 0;\n"),
    (_ANCHOR_STEP,
     "  o->sig = 0;\n"
     "  if (o->tau_on) { /* the action is the joint torque; the motors keep no gain and no strength */\n"
     "    for (int k = 0; k < 25; k++) { int d = o->obs_dof[k]; o->jtau[d] = clampd(action[k], -o->tau_bound, o->tau_bound); target[d] = 0; }\n"
     "    double kp = o->P[P_KP], kd = o->P[P_KD];\n"
     "    o->P[P_KP] = 0; o->P[P_KD] = 0;\n"
     "    for (int s = 0; s < o->n_sub; s++) trex_oracle_substep(o, target, 0.0);\n"
     "    o->P[P_KP] = kp; o->P[P_KD] = kd;\n"
     "  } else\n"
     "  for (int s = 0; s < o->n_sub; s++) /* trex_env.py:148-150 ; max impulse = force*dt */\n"
     "    trex_oracle_substep(o, target, o->P[P_MAX_TORQUE] * dt);\n"),
)
_SETTER = ("\nvoid trex_oracle_set_torque_mode(trex_oracle* o, int on, double bound) {\n"
           "  o->tau_on = on;\n"
           "  o->tau_bound = bound;\n"
           "  memset(o->jtau, 0, sizeof(o->jtau));\n"
           "}\n")


def source() -> str:
    """The oracle's source with torque control inserted."""
    src = open(os.path.join(_ORACLE_DIR, "trex_oracle.c")).read()
    for anchor, replacement in _INSERTIONS:
        if src.count(anchor) != 1:
            raise RuntimeError("oracle_tau: anchor %r occurs %d times in oracle/trex_oracle.c" % (anchor, src.count(anchor)))
        src = src.replace(anchor, replacement)
    return src + _SETTER


def build(force: bool = False) -> str:
    deps = [os.path.join(_ORACLE_DIR, f) for f in ("trex_oracle.c", "trex_oracle.h")] + [os.path.abspath(__file__)]
    stale = force or not os.path.isfile(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps)
    if stale:
        with tempfile.TemporaryDirectory() as tmp:
            c = os.path.join(tmp, "trex_oracle_tau.c")
            with open(c, "w") as f:
                f.write(source())
            # the flags of oracle/Makefile
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-Wall", "-Wextra", "-Wno-unused-parameter",
                                   "-ffp-contract=off", "-I" + _ORACLE_DIR, "-shared", "-o", _LIB, c, "-lm"])
    return _LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB)
        # every entry point of the oracle keeps the signature oracle.oracle declares for it
        for name, f in vars(_oracle.lib()).items():
            if name.startswith("trex_oracle_"):
                g = getattr(L, name)
                g.argtypes, g.restype = f.argtypes, f.restype
        L.trex_oracle_set_torque_mode.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_double]
        _lib = L
    return _lib


class OracleTau(_oracle.Oracle):
    """``Oracle`` with joint torque control (``set_torque_mode``)."""

    def __init__(self, blob: bytes, num_substeps: int | None = None, contacts: bool = True,
                 reward_weights=(1.0, 0.005, 0.002)):
        self._L = lib()
        self._h = self._L.trex_oracle_create(blob, len(blob))
        if not self._h:
            raise RuntimeError("trex_oracle_create: " + self._L.trex_oracle_last_error().decode())
        if num_substeps is not None:
            self._L.trex_oracle_set_substeps(self._h, int(num_substeps))
        self._L.trex_oracle_enable_contacts(self._h, int(bool(contacts)))
        d, e, k = reward_weights
        self._L.trex_oracle_set_reward_weights(self._h, float(d), float(e), float(k))
        self.state_dim = self._L.trex_oracle_state_dim(self._h)
        self.num_candidates = self._L.trex_oracle_num_candidates(self._h)

    def set_torque_mode(self, on: bool, bound: float = 0.0) -> None:
        """On: ``step``'s action is the joint torque (name-sorted), clipped to +-bound; off: motor targets (the oracle)."""
        self._L.trex_oracle_set_torque_mode(self._h, int(bool(on)), float(bound))
