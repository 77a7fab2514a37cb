"""ctypes binding of ``libvfk.so`` (C ABI in ``include/vfk.h``).

There is no fallback: if the shared library is missing or cannot be loaded the import
of any compute entry point raises ``VfkLibraryError`` telling the user to build it
(``python -c "import __graft_entry__ as g; g.build()"`` or ``python -m vfclik_b200.build``).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

VFK_MAX_JOINTS = 17
VFK_N_PORTS = 6
VFK_GOAL_COMPS = 13
VFK_POSE_COMPS = 12
VFK_AUX_COMPS = 12
VFK_TILE = 32
VFK_MAX_SHARED_OBSTACLES = 1024     # largest shared obstacle list (BuffersC.obst_shared = 1 or 2)
# BuffersC.obst_shared: per-instance lists, one list for the whole batch, or both (the mixed fields at the struct's end)
VFK_OBST_PER_INSTANCE, VFK_OBST_SHARED, VFK_OBST_MIXED = 0, 1, 2

VFK_OK = 0
VFK_ERR_INVALID = -1
VFK_ERR_UNSUPPORTED = -2
VFK_ERR_CUDA = -3
VFK_ERR_NO_DEVICE = -4

FLAG_AT_GOAL, FLAG_NS_LIMIT, FLAG_NAN, FLAG_CLAMPED = 1, 2, 4, 8
NS_OFF, NS_PROJECTOR, NS_CONTROL = 0, 1, 2

# VFK_LIB selects an alternative build of the same ABI (kernel tuning experiments); default = in-tree libvfk.so
LIB_PATH = os.environ.get("VFK_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libvfk.so")

# every symbol include/vfk.h declares (tests check the library exports all of them)
EXPORTS = [
    "vfk_version", "vfk_default_params", "vfk_create", "vfk_set_params", "vfk_get_params", "vfk_chain_pattern",
    "vfk_destroy",
    "vfk_last_error", "vfk_step", "vfk_solve", "vfk_field_eval", "vfk_field_eval_scene", "vfk_mix", "vfk_set_vel", "vfk_monitor", "vfk_pack", "vfk_unpack", "vfk_session_create", "vfk_session_set_goal",
    "vfk_session_set_obstacles", "vfk_session_set_shared_obstacles", "vfk_session_use_obstacles", "vfk_session_set_aux", "vfk_session_set_q", "vfk_session_set_jp_ref", "vfk_session_set_jp_limits", "vfk_session_set_ns_input",
    "vfk_session_cycle", "vfk_session_solve", "vfk_session_enable", "vfk_session_read", "vfk_session_buffers", "vfk_session_destroy",
]


class VfkLibraryError(RuntimeError):
    pass


class VfkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("vfk error %d: %s" % (code, msg))
        self.code = code


class ChainDescC(C.Structure):
    _fields_ = [
        ("n_joints", C.c_int32),
        ("joint_type", C.c_int32 * VFK_MAX_JOINTS),
        ("base", C.c_double * 12),
        ("tip", (C.c_double * 12) * VFK_MAX_JOINTS),
        ("q_lo", C.c_double * VFK_MAX_JOINTS),
        ("q_hi", C.c_double * VFK_MAX_JOINTS),
    ]


class ParamsC(C.Structure):
    _fields_ = [
        ("ik_lambda", C.c_double), ("ns_lambda", C.c_double), ("dt", C.c_double), ("speed_scale", C.c_double),
        ("max_vel", C.c_double), ("jp_kp", C.c_double), ("jp_delta", C.c_double), ("ns_gain", C.c_double),
        ("ns_lookahead", C.c_double), ("ns_limit_gain", C.c_double), ("rot_slowdown", C.c_double),
        ("goal_force", C.c_double), ("obst_force", C.c_double), ("obst_safe", C.c_double), ("obst_order", C.c_double),
        ("mixer_w", C.c_double * VFK_N_PORTS), ("w_task", C.c_double * 6), ("w_joint", C.c_double * VFK_MAX_JOINTS),
        ("tool", C.c_double * 12), ("jp_ref", C.c_double * VFK_MAX_JOINTS), ("ns_control", C.c_double * 4),
        ("shoulder_vel", C.c_double * 2), ("ik_eps", C.c_double),
        ("ns_mode", C.c_int32), ("direct_control", C.c_int32), ("integrate", C.c_int32), ("bridge_kind", C.c_int32),
        ("ik_mode", C.c_int32), ("reserved", C.c_int32),
    ]


class BuffersC(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("goal", C.c_void_p), ("obst", C.c_void_p), ("obst_ext", C.c_void_p), ("aux", C.c_void_p),
        ("jp_ref", C.c_void_p),
        ("ns_in", C.c_void_p),
        ("ns_lastvec", C.c_void_p), ("q_cmded", C.c_void_p), ("ext_cmd", C.c_void_p * 3), ("qdot_vf", C.c_void_p),
        ("qdot_ns", C.c_void_p), ("qdot_jp", C.c_void_p), ("qdot", C.c_void_p), ("cmd", C.c_void_p),
        ("pose", C.c_void_p), ("twist", C.c_void_p), ("flags", C.c_void_p), ("n_aux", C.c_int32), ("obst_shared", C.c_int32),
        ("jp_lo", C.c_void_p), ("jp_hi", C.c_void_p),
        # read by the library only when obst_shared == VFK_OBST_MIXED
        ("shared_obst", C.c_void_p), ("shared_obst_ext", C.c_void_p), ("n_shared_obst", C.c_int32), ("reserved2", C.c_int32),
    ]


_lib = None


def load():
    """Load ``libvfk.so`` once; raise loudly when it is absent (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VfkLibraryError(
            "%s not found: build the CUDA library first (python -m vfclik_b200.build). "
            "vfclik_b200 has no CPU fallback." % LIB_PATH)
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise VfkLibraryError("cannot load %s: %s" % (LIB_PATH, e)) from e
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.vfk_version.restype = i32
    lib.vfk_default_params.argtypes = [C.POINTER(ParamsC), i32]
    lib.vfk_default_params.restype = None
    lib.vfk_create.argtypes = [C.POINTER(vp), C.POINTER(ChainDescC), i32, i32]
    lib.vfk_set_params.argtypes = [vp, C.POINTER(ParamsC)]
    lib.vfk_get_params.argtypes = [vp, C.POINTER(ParamsC)]
    lib.vfk_chain_pattern.argtypes = [vp]
    lib.vfk_destroy.argtypes = [vp]
    lib.vfk_destroy.restype = None
    lib.vfk_last_error.argtypes = [vp]
    lib.vfk_last_error.restype = C.c_char_p
    lib.vfk_step.argtypes = [vp, C.POINTER(BuffersC), i64, i32, i32, vp]
    lib.vfk_solve.argtypes = [vp, C.POINTER(BuffersC), i64, i32, i32, C.c_double, C.c_double, vp, vp, vp]
    lib.vfk_field_eval.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, i64, i32, vp]
    lib.vfk_field_eval_scene.argtypes = [vp, vp, C.POINTER(BuffersC), i64, i32, vp, vp]
    lib.vfk_mix.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_double), i32, i32, vp, vp, i64, vp]
    lib.vfk_set_vel.argtypes = [vp, vp, vp, vp, C.c_double, i32, vp, vp, i32, i64, vp]
    lib.vfk_monitor.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    lib.vfk_pack.argtypes = [vp, vp, vp, i32, i32, i64, vp]
    lib.vfk_unpack.argtypes = [vp, vp, vp, i32, i32, i64, vp]
    lib.vfk_session_create.argtypes = [vp, i64, i32, i32, C.POINTER(vp)]
    for name in ("vfk_session_set_goal", "vfk_session_set_q", "vfk_session_set_jp_ref", "vfk_session_set_ns_input"):
        getattr(lib, name).argtypes = [vp, vp]
    lib.vfk_session_set_obstacles.argtypes = [vp, vp, vp]
    lib.vfk_session_set_shared_obstacles.argtypes = [vp, vp, vp, i32]
    lib.vfk_session_use_obstacles.argtypes = [vp, i32]
    lib.vfk_session_set_jp_limits.argtypes = [vp, vp, vp]
    lib.vfk_session_set_aux.argtypes = [vp, vp, i32]
    lib.vfk_session_cycle.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.vfk_session_solve.argtypes = [vp, vp, i32, C.c_double, C.c_double, vp, vp, vp]
    lib.vfk_session_read.argtypes = [vp, C.c_char_p, vp]
    lib.vfk_session_enable.argtypes = [vp, C.c_char_p, i32]
    lib.vfk_session_buffers.argtypes = [vp, C.POINTER(BuffersC)]
    lib.vfk_session_destroy.argtypes = [vp]
    lib.vfk_session_destroy.restype = None
    _lib = lib
    return lib


def chain_to_c(chain) -> ChainDescC:
    c = ChainDescC()
    n = int(chain.n_joints)
    c.n_joints = n
    for j in range(n):
        c.joint_type[j] = int(chain.joint_type[j])
        for k in range(12):
            c.tip[j][k] = float(chain.tip[j, k])
        c.q_lo[j] = float(chain.q_lo[j])
        c.q_hi[j] = float(chain.q_hi[j])
    for k in range(12):
        c.base[k] = float(chain.base[k])
    return c


def np_ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)
