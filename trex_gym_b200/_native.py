"""ctypes binding of ``libtrex_b200.so`` (C ABI: ``include/trex_b200.h``).

There is no Python or CPU fallback: if the CUDA library is missing or no GPU is
present, constructing a simulator raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("TREX_LIB", os.path.join(CSRC, "libtrex_b200.so"))

NUM_JOINTS = 25
OBS_DIM = 75
STATE_DIM = 160
AUX_DIM = 8
ENV_PARAM_DIM = 32  # per-environment parameter row (include/trex_b200.h, trex_set_env_params)
EXT_BODIES = 26  # bodies of the external-wrench layout [N][26][6] (include/trex_b200.h, trex_set_external_forces)
BODY_STATE_DIM = 13  # floats of a body row of trex_get_body_states: p | q | v | w
NUM_DOFS = 31  # generalized coordinates of trex_get_dynamics: base angular | base linear | 25 joints in link order
JACOBIAN_ROWS = 6  # rows of a body Jacobian: v_COM | w

EXPORTED_SYMBOLS = (
    "trex_create", "trex_destroy", "trex_reset", "trex_step", "trex_step_host", "trex_step_host_async", "trex_host_wait",
    "trex_reset_host",
    "trex_get_state", "trex_set_state", "trex_get_aux", "trex_get_joint_limits", "trex_get_action_limits",
    "trex_set_env_params", "trex_get_env_params", "trex_set_env_param_ranges",
    "trex_set_external_forces", "trex_get_external_forces", "trex_set_push_schedule",
    "trex_get_body_states", "trex_get_dynamics",
    "trex_fill_random_actions", "trex_get_stats", "trex_measure_fp32_peak", "trex_gae", "trex_normalize",
    "trex_policy_param_count", "trex_policy_forward", "trex_kernel_launches", "trex_num_envs",
    "trex_last_error", "trex_version",
)


class TrexConfig(ctypes.Structure):
    _fields_ = [
        ("num_substeps", ctypes.c_int32),
        ("distance_weight", ctypes.c_float),
        ("energy_weight", ctypes.c_float),
        ("drift_weight", ctypes.c_float),
        ("max_episode_steps", ctypes.c_int32),
        ("enable_contacts", ctypes.c_int32),
        ("reset_mode", ctypes.c_int32),
        ("seed", ctypes.c_uint32),
        ("env_offset", ctypes.c_int64),
        ("warps_per_block", ctypes.c_int32),
        ("solver_placement", ctypes.c_int32),
        ("heavy_share_div", ctypes.c_int32),
        ("pipelines", ctypes.c_int32),
        ("heavy_memory", ctypes.c_int32),
        ("chunk_envs", ctypes.c_int32),
        ("contact_memory", ctypes.c_int32),
        ("env_params", ctypes.c_int32),
        ("external_forces", ctypes.c_int32),
        ("actuation", ctypes.c_int32),
        ("reserved", ctypes.c_int32 * 4),
    ]


class TrexPushSchedule(ctypes.Structure):
    _fields_ = [
        ("body", ctypes.c_int32),
        ("interval", ctypes.c_int32),
        ("duration", ctypes.c_int32),
        ("first_step", ctypes.c_int32),
        ("probability", ctypes.c_float),
        ("force_min", ctypes.c_float),
        ("force_max", ctypes.c_float),
        ("reserved", ctypes.c_int32 * 9),
    ]


SOLVE_DEFAULT, SOLVE_FRONT, SOLVE_FREE_ONLY, SOLVE_NO_HEAVY = 0, 1, 2, 3  # trex_config.solver_placement
HEAVY_BOTH, HEAVY_SHARED, HEAVY_TENSOR = 0, 1, 2  # trex_config.heavy_memory
CONTACT_TENSOR, CONTACT_SHARED = 0, 1  # trex_config.contact_memory
ACTUATION = {"position": 0, "torque": 1}  # trex_config.actuation: TREX_ACTUATION_POSITION / TREX_ACTUATION_TORQUE


class TrexStats(ctypes.Structure):
    _fields_ = [
        ("env_steps", ctypes.c_int64),
        ("episodes", ctypes.c_int64),
        ("nan_resets", ctypes.c_int64),
        ("mean_solver_iterations", ctypes.c_double),
        ("mean_contacts", ctypes.c_double),
        ("contact_overflow", ctypes.c_int64),
    ]


NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in
            ("trex_capi.cu", "trex_core.h", "trex_model.h", "trex_topology.h", "lane_cuda.h", "trex_policy.h")]
    srcs.append(os.path.join(_HERE, "..", "include", "trex_b200.h"))
    stale = force or not os.path.isfile(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(s) for s in srcs)
    if stale:
        nvcc = os.environ.get("NVCC", "nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, os.path.join(CSRC, "trex_capi.cu")]
        subprocess.check_call(cmd, cwd=CSRC)
    return LIB_PATH


_lib = None


def lib():
    """Load ``libtrex_b200.so``; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            "libtrex_b200.so not found at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(trex_gym_b200 has no CPU fallback)" % LIB_PATH
        )
    L = ctypes.CDLL(LIB_PATH)
    vp, fp, u8p = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p  # raw device/host addresses
    L.trex_create.restype = ctypes.c_int
    L.trex_create.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int32, ctypes.c_int32,
                              ctypes.POINTER(TrexConfig), ctypes.POINTER(ctypes.c_void_p)]
    L.trex_destroy.restype = None
    L.trex_destroy.argtypes = [vp]
    L.trex_reset.restype = ctypes.c_int
    L.trex_reset.argtypes = [vp, u8p, fp, vp]
    L.trex_step.restype = ctypes.c_int
    L.trex_step.argtypes = [vp, fp, fp, fp, u8p, vp]
    L.trex_step_host.restype = ctypes.c_int
    L.trex_step_host.argtypes = [vp, fp, fp, fp, u8p]
    L.trex_step_host_async.restype = ctypes.c_int
    L.trex_step_host_async.argtypes = [vp, fp, fp, fp, u8p]
    L.trex_host_wait.restype = ctypes.c_int
    L.trex_host_wait.argtypes = [vp]
    L.trex_reset_host.restype = ctypes.c_int
    L.trex_reset_host.argtypes = [vp, fp]
    for name in ("trex_get_state", "trex_set_state", "trex_get_aux"):
        f = getattr(L, name)
        f.restype = ctypes.c_int
        f.argtypes = [vp, fp, vp]
    L.trex_set_env_params.restype = ctypes.c_int
    L.trex_set_env_params.argtypes = [vp, fp, u8p, vp]
    L.trex_get_env_params.restype = ctypes.c_int
    L.trex_get_env_params.argtypes = [vp, fp, vp]
    L.trex_set_env_param_ranges.restype = ctypes.c_int
    L.trex_set_env_param_ranges.argtypes = [vp, fp, fp]
    L.trex_set_external_forces.restype = ctypes.c_int
    L.trex_set_external_forces.argtypes = [vp, fp, u8p, vp]
    L.trex_get_external_forces.restype = ctypes.c_int
    L.trex_get_external_forces.argtypes = [vp, fp, vp]
    L.trex_get_body_states.restype = ctypes.c_int
    L.trex_get_body_states.argtypes = [vp, vp, vp, vp]
    L.trex_get_dynamics.restype = ctypes.c_int
    L.trex_get_dynamics.argtypes = [vp, vp, vp, vp, vp]
    L.trex_set_push_schedule.restype = ctypes.c_int
    L.trex_set_push_schedule.argtypes = [vp, ctypes.POINTER(TrexPushSchedule)]
    L.trex_get_joint_limits.restype = ctypes.c_int
    L.trex_get_joint_limits.argtypes = [vp, fp, fp]
    L.trex_get_action_limits.restype = ctypes.c_int
    L.trex_get_action_limits.argtypes = [vp, fp, fp]
    L.trex_fill_random_actions.restype = ctypes.c_int
    L.trex_fill_random_actions.argtypes = [vp, fp, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int64, vp]
    L.trex_get_stats.restype = ctypes.c_int
    L.trex_get_stats.argtypes = [vp, ctypes.POINTER(TrexStats)]
    L.trex_measure_fp32_peak.restype = ctypes.c_int
    L.trex_measure_fp32_peak.argtypes = [ctypes.c_int32, ctypes.POINTER(ctypes.c_double)]
    L.trex_gae.restype = ctypes.c_int
    L.trex_gae.argtypes = [ctypes.c_int32, vp, vp, vp, vp, vp, ctypes.c_float, ctypes.c_float, vp, vp, ctypes.c_int32, ctypes.c_int32, vp]
    L.trex_normalize.restype = ctypes.c_int
    L.trex_normalize.argtypes = [ctypes.c_int32, vp, vp, vp, ctypes.c_float, ctypes.c_float, vp, ctypes.c_int64, ctypes.c_int32, vp]
    L.trex_policy_param_count.restype = ctypes.c_int
    L.trex_policy_param_count.argtypes = []
    L.trex_policy_forward.restype = ctypes.c_int
    L.trex_policy_forward.argtypes = [ctypes.c_int32, vp, vp, vp, ctypes.c_float, ctypes.c_float, vp, ctypes.c_uint32, ctypes.c_uint64,
                                      ctypes.c_int64, ctypes.c_int32, vp, vp, vp, vp, ctypes.c_int64, vp]
    L.trex_kernel_launches.restype = ctypes.c_int64
    L.trex_kernel_launches.argtypes = [vp]
    L.trex_num_envs.restype = ctypes.c_int32
    L.trex_num_envs.argtypes = [vp]
    L.trex_last_error.restype = ctypes.c_char_p
    L.trex_version.restype = ctypes.c_char_p
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().trex_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError("%s: %s" % (what, msg))
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))
