"""The CPU oracle with external wrenches (TEST INFRASTRUCTURE ONLY): ``libtrex_oracle_extf.so``.

pybullet applies an external force / torque on a link (``applyExternalForce(..., linkWorldCOM, WORLD_FRAME)`` /
``applyExternalTorque``) as ``btMultiBody::addLinkForce`` / ``addLinkTorque``: the link's bias force in the articulated-body
pass loses the wrench rotated into the link frame, at the link's COM (the link frame's origin), where gravity enters.  The
oracle (``oracle/trex_oracle.c``) has no such input, and it stays as it is.  This module builds a second library from that
source unchanged, with four insertions at fixed anchors (each must occur exactly once, or the build fails):
  - two fields of ``struct trex_oracle``: the per-link wrenches and their on / suppressed flags;
  - in ``aba``, right behind the gravity term of each link: ``pA[0:3] -= Rw T``, ``pA[3:6] -= Rw F``;
  - in ``trex_oracle_reset``: the wrenches are suppressed for the reset's physics step;
  - ``trex_oracle_set_external_forces(o, link_wrench [n_links + 1][6])``: world force at the link's COM, world torque,
    base first; NULL clears.  They act in every substep of ``trex_oracle_step`` / ``_run`` / ``_substep`` until set again.
Everything else -- kinematics, ABA, constraint rows, PGS -- is the oracle's own code, so agreement with the kernels (which
apply the wrench to merged bodies in their own algebra) stays evidence.  ``OracleExtf`` is ``oracle.oracle.Oracle`` on that
library plus ``set_external_forces``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as _oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_DIR = os.path.normpath(os.path.join(_HERE, "..", "..", "oracle"))
_LIB = os.path.join(_HERE, "libtrex_oracle_extf.so")
_lib = None

# (anchor, what replaces it): the anchor itself stays, with the insertion before or behind it
_ANCHOR_FIELDS = "  row_t* rows;\n};\n"
_ANCHOR_GRAVITY = "    pA[b][3] = -fl[0]; pA[b][4] = -fl[1]; pA[b][5] = -fl[2];\n"
_ANCHOR_RESET = "  trex_oracle_substep(o, zero, 0.0);\n"
_INSERTIONS = (
    (_ANCHOR_FIELDS,
     "  row_t* rows;\n"
     "  double ext[MAXL + 1][6]; /* external wrenches per link, base first: world force at the link's COM, world torque */\n"
     "  int ext_on, ext_off;     /* ext_off: suppressed (the physics step of a reset) */\n"
     "};\n"),
    (_ANCHOR_GRAVITY,
     _ANCHOR_GRAVITY +
     "    if (o->ext_on && !o->ext_off) { /* btMultiBody::addLinkForce / addLinkTorque: world frame, at the link's COM */\n"
     "      v3 fe, te;\n"
     "      m3mulv(fe, o->Rw[b], o->ext[b]);\n"
     "      m3mulv(te, o->Rw[b], o->ext[b] + 3);\n"
     "      for (int k = 0; k < 3; k++) { pA[b][k] -= te[k]; pA[b][3 + k] -= fe[k]; }\n"
     "    }\n"),
    (_ANCHOR_RESET,
     "  o->ext_off = 1; /* external wrenches never act in the reset's physics step */\n" + _ANCHOR_RESET + "  o->ext_off = 0;\n"),
)
_SETTER = ("\nvoid trex_oracle_set_external_forces(trex_oracle* o, const double* w) {\n"
           "  o->ext_on = w != NULL;\n"
           "  if (w) memcpy(o->ext, w, sizeof(double) * 6 * (o->n + 1));\n"
           "}\n")


def source() -> str:
    """The oracle's source with the wrench inserted."""
    src = open(os.path.join(_ORACLE_DIR, "trex_oracle.c")).read()
    for anchor, replacement in _INSERTIONS:
        if src.count(anchor) != 1:
            raise RuntimeError("oracle_extf: anchor %r occurs %d times in oracle/trex_oracle.c" % (anchor, src.count(anchor)))
        src = src.replace(anchor, replacement)
    return src + _SETTER


def build(force: bool = False) -> str:
    deps = [os.path.join(_ORACLE_DIR, f) for f in ("trex_oracle.c", "trex_oracle.h")] + [os.path.abspath(__file__)]
    stale = force or not os.path.isfile(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps)
    if stale:
        with tempfile.TemporaryDirectory() as tmp:
            c = os.path.join(tmp, "trex_oracle_extf.c")
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
        L.trex_oracle_set_external_forces.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
        _lib = L
    return _lib


class OracleExtf(_oracle.Oracle):
    """``Oracle`` with external wrenches (``set_external_forces``)."""

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

    def set_external_forces(self, link_wrench) -> None:
        """[n_links + 1, 6] per link of the full model, base first: world force at the link's COM, world torque (None clears)."""
        if link_wrench is None:
            self._L.trex_oracle_set_external_forces(self._h, None)
            return
        self._ext = np.ascontiguousarray(link_wrench, dtype=np.float64)
        self._L.trex_oracle_set_external_forces(self._h, self._ext.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
