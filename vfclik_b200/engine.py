"""Batch engine: Python face of the fused control-cycle kernel (``libvfk.so``).

``Engine`` wraps a ``vfk_handle`` (chain + per-robot constants); ``Engine.step`` runs K
fused cycles on device buffers (torch CUDA tensors in the tile-blocked layout of
``include/vfk.h``; ``DeviceBatch`` allocates and converts them);
``Engine.session`` opens a host-buffer session (numpy in / numpy out) whose scene
(goal, obstacles) stays resident on the GPU between cycles -- the call the
reference-facing host modules (``vf``, ``nullspace``, ``joint_p_controller``, ``bridge``)
make.  There is no CPU path: constructing an ``Engine`` without ``libvfk.so`` or
without a B200 raises.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import weakref
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import (BuffersC, ParamsC, VfkError, NS_CONTROL, NS_OFF, NS_PROJECTOR,  # noqa: F401
                   VFK_OBST_PER_INSTANCE, VFK_OBST_SHARED, VFK_OBST_MIXED)


BRIDGE_LWR, BRIDGE_POWERCUBE, BRIDGE_ICUB = 0, 1, 2
BRIDGE_KINDS = {"lwr": BRIDGE_LWR, "powercube": BRIDGE_POWERCUBE, "icub": BRIDGE_ICUB}   # config.arm_type (scripts/bridge:102-111)


@dataclasses.dataclass
class Params:
    """Per-robot constants, mirror of ``vfk_params`` (include/vfk.h)."""
    ik_lambda: float = 0.1
    ns_lambda: float = 0.1
    dt: float = 0.01
    speed_scale: float = 0.2
    max_vel: float = 1.0
    jp_kp: float = 1.5
    jp_delta: float = 0.087
    ns_gain: float = 0.5
    ns_lookahead: float = 0.3
    ns_limit_gain: float = 1.0
    rot_slowdown: float = 0.09
    goal_force: float = 1.0
    obst_force: float = -10.0
    obst_safe: float = 0.001
    obst_order: float = 20.0
    mixer_w: Sequence[float] = (1.0, 1.0, 0.0, 0.0, 0.0, 0.0)
    w_task: Sequence[float] = (1.0,) * 6
    w_joint: Optional[Sequence[float]] = None
    tool: Sequence[float] = (1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0)
    jp_ref: Optional[Sequence[float]] = None
    ns_control: Sequence[float] = (0.0, 0.0, 0.0, 0.0)
    ns_mode: int = NS_PROJECTOR
    direct_control: int = -1
    integrate: int = 1
    bridge_kind: int = 0                                   # BRIDGE_LWR / BRIDGE_POWERCUBE / BRIDGE_ICUB
    shoulder_vel: Sequence[float] = (0.0, 0.0)             # Powercube: config.max_vel_shoulder_pos, max_vel_shoulder_neg
    ik_mode: int = 0                                       # 0: north_star's damped least squares; 1: KDL-wdls-style truncated form (FP64)
    ik_eps: float = 1e-5                                   # ik_mode 1: singular values below this are damped, the rest inverted

    @staticmethod
    def from_config(config, **over) -> "Params":
        """Pick the attributes the reference reads from ``config`` (SURVEY.md App. B.5)."""
        kw = {}
        for attr, key in (("speedScale", "speed_scale"), ("jpctrl_kp", "jp_kp"), ("max_vel", "max_vel"),
                          ("rate", "dt"), ("ik_lambda", "ik_lambda"), ("ns_lambda", "ns_lambda"),
                          ("ns_limit_gain", "ns_limit_gain")):
            if hasattr(config, attr):
                kw[key] = float(getattr(config, attr))
        if hasattr(config, "initial_joint_pos"):
            kw["jp_ref"] = tuple(float(v) for v in config.initial_joint_pos)
        kind = BRIDGE_KINDS.get(str(getattr(config, "arm_type", "lwr")).lower())
        if kind is not None:
            kw["bridge_kind"] = kind
        if hasattr(config, "max_vel_shoulder_pos") and hasattr(config, "max_vel_shoulder_neg"):
            kw["shoulder_vel"] = (float(config.max_vel_shoulder_pos), float(config.max_vel_shoulder_neg))
        kw.update(over)
        return Params(**kw)

    def to_c(self, n_joints: int) -> ParamsC:
        p = ParamsC()
        for f in ("ik_lambda", "ns_lambda", "dt", "speed_scale", "max_vel", "jp_kp", "jp_delta", "ns_gain",
                  "ns_lookahead", "ns_limit_gain", "rot_slowdown", "goal_force", "obst_force", "obst_safe",
                  "obst_order"):
            setattr(p, f, float(getattr(self, f)))
        if len(self.mixer_w) != 6 or len(self.w_task) != 6 or len(self.tool) != 12 or len(self.ns_control) != 4:
            raise ValueError("mixer_w/w_task need 6 values, tool 12, ns_control 4")
        for k in range(6):
            p.mixer_w[k] = float(self.mixer_w[k])
            p.w_task[k] = float(self.w_task[k])
        wj = [1.0] * n_joints if self.w_joint is None else list(self.w_joint)
        ref = [0.0] * n_joints if self.jp_ref is None else list(self.jp_ref)
        if len(wj) != n_joints or len(ref) != n_joints:
            raise ValueError("w_joint / jp_ref need n_joints values")
        for j in range(_lib.VFK_MAX_JOINTS):
            p.w_joint[j] = float(wj[j]) if j < n_joints else 1.0
            p.jp_ref[j] = float(ref[j]) if j < n_joints else 0.0
        for k in range(12):
            p.tool[k] = float(self.tool[k])
        for k in range(4):
            p.ns_control[k] = float(self.ns_control[k])
        p.ns_mode, p.direct_control, p.integrate = int(self.ns_mode), int(self.direct_control), int(self.integrate)
        p.bridge_kind = int(self.bridge_kind)
        p.shoulder_vel[0], p.shoulder_vel[1] = float(self.shoulder_vel[0]), float(self.shoulder_vel[1])
        p.ik_mode, p.ik_eps = int(self.ik_mode), float(self.ik_eps)
        return p


def ns_ctrl_vectors(n_joints: int) -> int:
    """Basis vectors the reference's four-float nullspace control interface addresses: ``min(4, N - 6)``
    (``scripts/nullspace:113``); ``ns_lastvec`` holds that many vectors of N components per instance."""
    return max(0, min(4, int(n_joints) - 6))


def round_up(n: int, m: int = 32) -> int:
    return (int(n) + m - 1) // m * m


_BUF_FIELDS = ("q", "goal", "obst", "obst_ext", "aux", "jp_ref", "jp_lo", "jp_hi", "ns_in", "ns_lastvec", "q_cmded", "qdot_vf", "qdot_ns", "qdot_jp",
               "qdot", "cmd", "pose", "twist", "flags")
_PER_CYCLE = ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "twist", "flags")     # outputs vfk_solve does not take


def _dev_ptr(x) -> Optional[int]:
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        if not x.is_cuda:
            raise TypeError("device buffers must be CUDA tensors")
        if not x.is_contiguous():
            raise ValueError("device buffers must be contiguous [comps, ld] tensors")
        return x.data_ptr()
    raise TypeError("expected a CUDA tensor or an integer device pointer, got %r" % type(x))


class Engine:
    def __init__(self, chain, precision: int = 32, device: int = 0, params: Optional[Params] = None):
        self._lib = _lib.load()
        self.chain = chain
        self.n_joints = int(chain.n_joints)
        self.precision = int(precision)
        self.device = int(device)
        self.np_dtype = np.float32 if precision == 32 else np.float64
        self._h = C.c_void_p()
        cdesc = _lib.chain_to_c(chain)
        rc = self._lib.vfk_create(C.byref(self._h), C.byref(cdesc), self.precision, self.device)
        if rc != 0:
            raise VfkError(rc, self._lib.vfk_last_error(None).decode())
        self.launches = 0                       # kernels launched through this engine
        self._sessions = weakref.WeakSet()      # live host-buffer sessions: closed before the handle goes
        self.chain_pattern = {0: "generic", 1: "lwr", 2: "dh"}.get(self._lib.vfk_chain_pattern(self._h), "?")
        self.params = params if params is not None else Params()
        self.set_params(self.params)

    # -- lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            for s in list(getattr(self, "_sessions", ())):
                s.close()
            self._lib.vfk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise VfkError(rc, self._lib.vfk_last_error(self._h).decode())
        return rc

    def _launched(self, rc: int) -> int:
        """``_check`` for a call that returns the number of kernels it launched: counts them in ``launches``."""
        self.launches += self._check(rc)
        return rc

    def set_params(self, params: Optional[Params] = None, **over):
        if params is None:
            params = self.params
        if over:
            params = dataclasses.replace(params, **over)
        pc = params.to_c(self.n_joints)
        self._check(self._lib.vfk_set_params(self._h, C.byref(pc)))
        self.params = params
        return params

    @property
    def torch_dtype(self):
        import torch
        return torch.float32 if self.precision == 32 else torch.float64

    # -- device-buffer path
    def _stream(self, stream):
        if stream is None:
            import torch
            stream = torch.cuda.current_stream(self.device).cuda_stream
        return C.c_void_p(stream)

    @staticmethod
    def _buffers(bufs, ext_cmd, obst_shared, n_shared_obstacles=None) -> BuffersC:
        b = BuffersC()
        for f in _BUF_FIELDS:
            setattr(b, f, _dev_ptr(bufs.get(f)))
        for e in range(3):
            b.ext_cmd[e] = _dev_ptr(ext_cmd[e])
        aux = bufs.get("aux")
        b.n_aux = 0 if aux is None else int(aux.shape[1]) // 12
        b.obst_shared = int(bufs.get("obst_shared", False) if obst_shared is None else obst_shared)
        if b.obst_shared == VFK_OBST_MIXED:
            sh = bufs.get("shared_obst")
            b.shared_obst = _dev_ptr(sh)
            b.shared_obst_ext = _dev_ptr(bufs.get("shared_obst_ext"))
            if n_shared_obstacles is None:
                n_shared_obstacles = bufs.get("n_shared_obst", 0 if sh is None else int(sh.shape[0]))
            b.n_shared_obst = int(n_shared_obstacles)
        return b

    def step(self, bufs: Dict[str, object], n_instances: int, n_obstacles: int, k_cycles: int = 1,
             stream: Optional[int] = None, ext_cmd=(None, None, None), obst_shared: Optional[int] = None,
             n_shared_obstacles: Optional[int] = None) -> int:
        """K fused cycles on blocked device buffers; returns the number of kernels launched.  ``obst_shared`` (default:
        ``bufs["obst_shared"]``, else 0; ``vfk_buffers.obst_shared``, include/vfk.h): 0 (``VFK_OBST_PER_INSTANCE``) per-instance
        lists; 1 (``VFK_OBST_SHARED``, or True) ``obst`` / ``obst_ext`` are one dense ``[M, 4]`` / ``[M, 2]`` list for the whole
        batch; 2 (``VFK_OBST_MIXED``) ``obst`` / ``obst_ext`` are per instance (``n_obstacles`` of them) and
        ``bufs["shared_obst"]`` / ``bufs["shared_obst_ext"]`` one dense list for the whole batch, summed after the own ones.
        Its length is ``n_shared_obstacles``, else ``bufs["n_shared_obst"]``, else the array's."""
        b = self._buffers(bufs, ext_cmd, obst_shared, n_shared_obstacles)
        return self._launched(self._lib.vfk_step(self._h, C.byref(b), int(n_instances), int(n_obstacles), int(k_cycles),
                                                  self._stream(stream)))

    def solve(self, bufs: Dict[str, object], n_instances: int, n_obstacles: int, max_cycles: int, tol_trans: float,
              tol_rot: float, cycles_out, dist_out=None, stream: Optional[int] = None, ext_cmd=(None, None, None),
              obst_shared: Optional[int] = None, n_shared_obstacles: Optional[int] = None) -> int:
        """Run each instance's control loop until its tool frame is within ``tol_trans`` metres and ``tol_rot`` radians of
        its goal (strict), for at most ``max_cycles`` cycles (``vfk_solve``, include/vfk.h): the batched
        ``HandleArm.gotoFrame``.  ``cycles_out`` [1] int32 gets the cycle at which each instance stopped (-1: never),
        ``dist_out`` [2] the distance and angle to the goal at the returned q; q is updated in place.  ``bufs`` may hold
        no per-cycle output; ``obst_shared`` and the shared list as in ``step``.  Returns the number of kernels launched."""
        b = self._buffers(bufs, ext_cmd, obst_shared, n_shared_obstacles)
        return self._launched(self._lib.vfk_solve(self._h, C.byref(b), int(n_instances), int(n_obstacles), int(max_cycles),
                                                   float(tol_trans), float(tol_rot), _dev_ptr(cycles_out), _dev_ptr(dist_out),
                                                   self._stream(stream)))

    def field_eval(self, pose, goal, obst, twist_out, n_instances, n_obstacles, obst_ext=None, aux=None, n_aux=0,
                   stream=None) -> int:
        return self._launched(self._lib.vfk_field_eval(self._h, _dev_ptr(pose), _dev_ptr(goal), _dev_ptr(obst),
                                                        _dev_ptr(obst_ext), _dev_ptr(aux), int(n_aux), _dev_ptr(twist_out),
                                                        int(n_instances), int(n_obstacles), self._stream(stream)))

    def field_eval_scene(self, pose, bufs: Dict[str, object], twist_out, n_instances: int, n_obstacles: int,
                         obst_shared: Optional[int] = None, n_shared_obstacles: Optional[int] = None, stream=None) -> int:
        """The field query (``vfk_field_eval_scene``) at tool poses ``pose`` [12] on the scene of ``bufs`` as ``step`` reads
        it: ``goal``, ``obst`` / ``obst_ext``, ``aux`` and, by ``obst_shared``, the shared list.  ``twist_out`` [6]."""
        b = self._buffers(bufs, (None, None, None), obst_shared, n_shared_obstacles)
        return self._launched(self._lib.vfk_field_eval_scene(self._h, _dev_ptr(pose), C.byref(b), int(n_instances), int(n_obstacles),
                                                              _dev_ptr(twist_out), self._stream(stream)))

    def mix(self, cmds, weights, out, n_channels, n_instances, nan_flags=None, stream=None) -> int:
        n_ports = len(cmds)
        arr = (C.c_void_p * n_ports)(*[_dev_ptr(c) for c in cmds])
        w = (C.c_double * n_ports)(*[float(x) for x in weights])
        return self._launched(self._lib.vfk_mix(self._h, arr, w, n_ports, int(n_channels), _dev_ptr(out),
                                                 _dev_ptr(nan_flags), int(n_instances), self._stream(stream)))

    def set_vel(self, qdot, q, cmd_out, max_vel: float, direct_control: bool, n_channels: int, n_instances: int,
                q_cmded=None, qdot_lim_out=None, stream=None) -> int:
        """``LWR_Bridge.set_vel`` arithmetic (``scripts/bridge:188-203``) on blocked device buffers."""
        return self._launched(self._lib.vfk_set_vel(self._h, _dev_ptr(qdot), _dev_ptr(q), _dev_ptr(q_cmded), float(max_vel),
                                                     int(bool(direct_control)), _dev_ptr(cmd_out), _dev_ptr(qdot_lim_out),
                                                     int(n_channels), int(n_instances), self._stream(stream)))

    def monitor(self, pose, twist, goal, state_f, state_i, n_instances: int, track_out=None, dist_out=None,
                tracking_state_out=None, stream=None) -> int:
        """Tracking diagnostics + distance monitor (``scripts/vf:349-428``, ``scripts/monitor_distance:148-219``)."""
        return self._launched(self._lib.vfk_monitor(self._h, _dev_ptr(pose), _dev_ptr(twist), _dev_ptr(goal), _dev_ptr(state_f),
                                                     _dev_ptr(state_i), _dev_ptr(track_out), _dev_ptr(dist_out),
                                                     _dev_ptr(tracking_state_out), int(n_instances), self._stream(stream)))

    def pack(self, dense, blocked, comps: int, width: int, n_instances: int, stream=None) -> int:
        """dense SoA [comps][n] (x width scalars) -> tile-blocked, on the device."""
        return self._launched(self._lib.vfk_pack(self._h, _dev_ptr(dense), _dev_ptr(blocked), int(comps), int(width),
                                                  int(n_instances), self._stream(stream)))

    def unpack(self, blocked, dense, comps: int, width: int, n_instances: int, stream=None) -> int:
        return self._launched(self._lib.vfk_unpack(self._h, _dev_ptr(blocked), _dev_ptr(dense), int(comps), int(width),
                                                    int(n_instances), self._stream(stream)))

    def alloc(self, comps: int, n_instances: int, width: int = 1, dtype=None):
        """Zeroed blocked device tensor ``[tiles, comps, 32(, width)]`` for ``n_instances`` instances
        (torch's caching allocator returns >= 512-byte aligned blocks).  ``width == 4`` is the obstacle array: rows
        ``2p, 2p + 1`` of a tile hold the pair-interleaved planes of obstacles ``2p, 2p + 1`` (include/vfk.h), not two
        plain ``{x, y, z, radius}`` rows -- use ``pack`` / ``unpack`` (or ``obstacles_of``) to convert."""
        import torch
        tiles = round_up(n_instances, 32) // 32
        if width == 4:
            comps = round_up(comps, 2)          # obstacles are stored in pairs (include/vfk.h): an odd count gets a zero slot
        shape = (tiles, comps, 32) if width == 1 else (tiles, comps, 32, width)
        t = torch.zeros(shape, dtype=dtype or self.torch_dtype, device="cuda:%d" % self.device)
        assert t.data_ptr() % 128 == 0
        return t

    # -- host-buffer path
    def session(self, n_instances: int, n_obstacles: int, obst_ext: bool = False) -> "Session":
        return Session(self, n_instances, n_obstacles, obst_ext)


def _out_ptr(a, shape, dt):
    """Pointer to a host output array the session fills in place (None: not requested)."""
    if a is None:
        return None
    if a.dtype != dt or a.shape != shape or not a.flags.c_contiguous:
        raise ValueError("output array must be contiguous %s %r" % (dt, shape))
    return _lib.np_ptr(a)


class Session:
    """Resident scene + state on the GPU; numpy arrays in and out (dense SoA ``[comps, n]``;
    obstacles ``[M, n, 4]`` and optionally ``[M, n, 2]`` {safe, order})."""

    def __init__(self, engine: Engine, n_instances: int, n_obstacles: int, obst_ext: bool = False):
        self.e = engine
        self.n, self.m, self.ext = int(n_instances), int(n_obstacles), bool(obst_ext)
        self._s = C.c_void_p()
        engine._check(engine._lib.vfk_session_create(engine._h, self.n, self.m, int(self.ext), C.byref(self._s)))
        engine._sessions.add(self)

    def close(self):
        if getattr(self, "_s", None) is not None and self._s:
            self.e._lib.vfk_session_destroy(self._s)
            self._s = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _arr(self, a, rows):
        a = np.ascontiguousarray(a, dtype=self.e.np_dtype)
        if a.shape != (rows, self.n):
            raise ValueError("expected shape (%d, %d), got %r" % (rows, self.n, a.shape))
        return a

    def set_goal(self, goal):
        a = self._arr(goal, 13)
        self.e._check(self.e._lib.vfk_session_set_goal(self._s, _lib.np_ptr(a)))

    def set_obstacles(self, obst, obst_ext=None):
        if self.m == 0:
            return
        a = np.ascontiguousarray(obst, dtype=self.e.np_dtype)
        if a.shape != (self.m, self.n, 4):
            raise ValueError("obstacles must be [M, n, 4], got %r" % (a.shape,))
        x = None
        if self.ext:
            x = np.ascontiguousarray(obst_ext, dtype=self.e.np_dtype)
            if x.shape != (self.m, self.n, 2):
                raise ValueError("obstacle ext must be [M, n, 2], got %r" % (x.shape,))
        self.e._check(self.e._lib.vfk_session_set_obstacles(self._s, _lib.np_ptr(a), None if x is None else _lib.np_ptr(x)))

    def set_shared_obstacles(self, obst, obst_ext=None):
        """One scene for every instance (``vfk_session_set_shared_obstacles``): ``obst`` ``[M, 4]`` {x, y, z, radius},
        ``obst_ext`` ``[M, 2]`` {safe, order} or None (the parameters' values); M <= ``VFK_MAX_SHARED_OBSTACLES``.  Later
        cycles and solves use it until ``set_obstacles`` is called (on a session created with obstacles)."""
        a = np.ascontiguousarray(obst, dtype=self.e.np_dtype)
        if a.ndim != 2 or a.shape[1] != 4:
            raise ValueError("shared obstacles must be [M, 4], got %r" % (a.shape,))
        x = None
        if obst_ext is not None:
            x = np.ascontiguousarray(obst_ext, dtype=self.e.np_dtype)
            if x.shape != (a.shape[0], 2):
                raise ValueError("shared obstacle ext must be [M, 2], got %r" % (x.shape,))
        self.e._check(self.e._lib.vfk_session_set_shared_obstacles(self._s, _lib.np_ptr(a), None if x is None else _lib.np_ptr(x),
                                                                   int(a.shape[0])))

    def use_obstacles(self, mode: int):
        """Which lists later cycles and solves use (``vfk_session_use_obstacles``): ``VFK_OBST_PER_INSTANCE`` (0),
        ``VFK_OBST_SHARED`` (1, needs ``set_shared_obstacles``) or ``VFK_OBST_MIXED`` (2: the per-instance scene and the
        shared list together; needs a session created with obstacles and a shared list).  ``set_obstacles`` and
        ``set_shared_obstacles`` select 0 and 1 themselves, so call this after both."""
        self.e._check(self.e._lib.vfk_session_use_obstacles(self._s, int(mode)))

    def set_aux(self, aux):
        """Auxiliary field records ``[n_aux, 12, n]`` ({type, force, 10 params}; types 4 and 5), or None to clear."""
        if aux is None:
            self.e._check(self.e._lib.vfk_session_set_aux(self._s, None, 0))
            return
        a = np.ascontiguousarray(aux, dtype=self.e.np_dtype)
        if a.ndim != 3 or a.shape[1:] != (12, self.n):
            raise ValueError("aux must be [n_aux, 12, n], got %r" % (a.shape,))
        self.e._check(self.e._lib.vfk_session_set_aux(self._s, _lib.np_ptr(a), int(a.shape[0])))

    def set_q(self, q):
        a = self._arr(q, self.e.n_joints)
        self.e._check(self.e._lib.vfk_session_set_q(self._s, _lib.np_ptr(a)))

    def set_jp_ref(self, ref):
        if ref is None:
            self.e._check(self.e._lib.vfk_session_set_jp_ref(self._s, None))
        else:
            a = self._arr(ref, self.e.n_joints)
            self.e._check(self.e._lib.vfk_session_set_jp_ref(self._s, _lib.np_ptr(a)))

    def set_jp_limits(self, lo, hi):
        """Per-instance limits the joint controller clamps its reference into (``config.updateJntLimits(q)`` evaluated per
        instance, ``scripts/joint_p_controller:79-89``), ``[N, n]`` each; ``None, None`` -> the chain's static limits."""
        if lo is None or hi is None:
            self.e._check(self.e._lib.vfk_session_set_jp_limits(self._s, None, None))
        else:
            a, b = self._arr(lo, self.e.n_joints), self._arr(hi, self.e.n_joints)
            self.e._check(self.e._lib.vfk_session_set_jp_limits(self._s, _lib.np_ptr(a), _lib.np_ptr(b)))

    def set_ns_input(self, x):
        if x is None:
            self.e._check(self.e._lib.vfk_session_set_ns_input(self._s, None))
        else:
            rows = 4 if self.e.params.ns_mode == NS_CONTROL else self.e.n_joints
            a = self._arr(x, rows)
            self.e._check(self.e._lib.vfk_session_set_ns_input(self._s, _lib.np_ptr(a)))

    def cycle(self, q_in=None, k_cycles: int = 1, qdot_out=None, q_out=None, flags_out=None) -> int:
        """One host-facing call: H2D of q (if given), K fused cycles, D2H of the requested outputs.

        Output arrays must be C-contiguous numpy arrays of the engine dtype, shape ``[N, n]``
        (flags: int32 ``[n]``); they are filled in place.
        """
        N = self.e.n_joints

        qp = None
        if q_in is not None:
            q_in = self._arr(q_in, N)
            qp = _lib.np_ptr(q_in)
        return self.e._launched(self.e._lib.vfk_session_cycle(
            self._s, qp, int(k_cycles), _out_ptr(qdot_out, (N, self.n), self.e.np_dtype),
            _out_ptr(q_out, (N, self.n), self.e.np_dtype), _out_ptr(flags_out, (self.n,), np.int32)))

    def solve(self, q_in=None, max_cycles: int = 1000, tol_trans: float = 1e-3, tol_rot: float = 1e-2, q_out=None,
              cycles_out=None, dist_out=None) -> int:
        """``vfk_session_solve``: q from the host (if given), then every instance runs until its tool reaches the goal
        (see ``Engine.solve``).  Outputs are filled in place: q ``[N, n]`` and dist ``[2, n]`` of the engine dtype, cycles
        int32 ``[n]``."""
        N = self.e.n_joints

        qp = None
        if q_in is not None:
            q_in = self._arr(q_in, N)
            qp = _lib.np_ptr(q_in)
        return self.e._launched(self.e._lib.vfk_session_solve(
            self._s, qp, int(max_cycles), float(tol_trans), float(tol_rot), _out_ptr(q_out, (N, self.n), self.e.np_dtype),
            _out_ptr(cycles_out, (self.n,), np.int32), _out_ptr(dist_out, (2, self.n), self.e.np_dtype)))

    def enable(self, *what: str, on: bool = True):
        """Ask the kernel to also write per-controller outputs ("qdot_vf", "qdot_ns", "qdot_jp", "cmd", "pose")."""
        for w in what:
            self.e._check(self.e._lib.vfk_session_enable(self._s, w.encode(), int(on)))

    def read(self, what: str) -> np.ndarray:
        rows = {"pose": 12, "twist": 6, "lastvec": max(1, ns_ctrl_vectors(self.e.n_joints)) * self.e.n_joints}.get(what, self.e.n_joints)
        out = np.empty((rows, self.n), dtype=self.e.np_dtype)
        self.e._check(self.e._lib.vfk_session_read(self._s, what.encode(), _lib.np_ptr(out)))
        return out


class DeviceBatch:
    """Device-resident buffers for one batch: torch CUDA tensors in the tile-blocked layout.

    Convenience for callers that keep everything on the GPU (the benchmark's kernel-only arm,
    the multi-GPU driver).  ``upload`` takes dense numpy arrays (``[comps, n]``; obstacles
    ``[M, n, 4]``, ext ``[M, n, 2]``), moves them to the device and converts them with the
    library's pack kernel; ``download`` converts back.  ``bufs`` is what ``Engine.step`` takes.
    ``shared_obstacles=True``: one scene for the whole batch, ``obst`` dense ``[M, 4]`` and ``obst_ext`` ``[M, 2]`` on the
    device as they are uploaded (``vfk_buffers.obst_shared``).  ``n_shared_obstacles=Ms`` (with ``shared_obstacles``
    False): a mixed scene, the per-instance ``obst`` / ``obst_ext`` of ``n_obstacles`` each plus ``shared_obst`` ``[Ms, 4]``
    and ``shared_obst_ext`` ``[Ms, 2]`` (when ``obst_ext``) for the whole batch, uploaded as they are.
    """

    _ROWS = {"goal": 13, "pose": 12, "flags": 1, "twist": 6, "track": 8, "dist": 2, "mon_f": 32, "solve_dist": 2}

    def __init__(self, engine: Engine, n_instances: int, n_obstacles: int, obst_ext: bool = False,
                 outputs=("qdot",), inputs=(), shared_obstacles: bool = False, n_shared_obstacles: Optional[int] = None):
        self.e, self.n, self.m = engine, int(n_instances), int(n_obstacles)
        self.shared = bool(shared_obstacles)
        self.mixed = n_shared_obstacles is not None
        self.ms = int(n_shared_obstacles or 0)
        if self.shared and self.mixed:
            raise ValueError("shared_obstacles and n_shared_obstacles exclude each other (a mixed scene has both lists)")
        self.t: Dict[str, object] = {}
        self.t["q"] = engine.alloc(engine.n_joints, self.n)
        self.t["goal"] = engine.alloc(13, self.n)
        if self.m and self.shared:
            import torch
            if self.m > _lib.VFK_MAX_SHARED_OBSTACLES:
                raise ValueError("a shared obstacle list holds at most %d obstacles" % _lib.VFK_MAX_SHARED_OBSTACLES)
            dev = "cuda:%d" % engine.device
            self.t["obst"] = torch.zeros((self.m, 4), dtype=engine.torch_dtype, device=dev)
            if obst_ext:
                self.t["obst_ext"] = torch.zeros((self.m, 2), dtype=engine.torch_dtype, device=dev)
        elif self.m:
            self.t["obst"] = engine.alloc(self.m, self.n, width=4)
            if obst_ext:
                self.t["obst_ext"] = engine.alloc(self.m, self.n, width=2)
        if self.mixed:
            import torch
            if not 0 <= self.ms <= _lib.VFK_MAX_SHARED_OBSTACLES:
                raise ValueError("a shared obstacle list holds 0..%d obstacles" % _lib.VFK_MAX_SHARED_OBSTACLES)
            dev = "cuda:%d" % engine.device
            # at least one row, so that the pointer is a real 128-byte aligned block even for an empty list
            self.t["shared_obst"] = torch.zeros((max(self.ms, 1), 4), dtype=engine.torch_dtype, device=dev)
            if obst_ext:
                self.t["shared_obst_ext"] = torch.zeros((max(self.ms, 1), 2), dtype=engine.torch_dtype, device=dev)
        for name in tuple(outputs) + tuple(inputs):
            self._ensure(name)
        self.ext_cmd = [None, None, None]

    def _comps(self, name):
        if name == "ns_in":
            return 4 if self.e.params.ns_mode == NS_CONTROL else self.e.n_joints
        if name == "ns_lastvec":
            return max(1, ns_ctrl_vectors(self.e.n_joints)) * self.e.n_joints
        return self._ROWS.get(name, self.e.n_joints)

    def _ensure(self, name):
        if name in self.t:
            return self.t[name]
        import torch
        if name in ("flags", "mon_i", "tracking_state", "cycles"):
            self.t[name] = self.e.alloc({"flags": 1, "mon_i": 6, "tracking_state": 2, "cycles": 1}[name], self.n, dtype=torch.int32)
        elif name in ("obst", "obst_ext", "shared_obst", "shared_obst_ext"):
            raise KeyError("%s was not allocated (n_obstacles = 0 or obst_ext=False)" % name)
        else:
            self.t[name] = self.e.alloc(self._comps(name), self.n)
        return self.t[name]

    def to_blocked(self, arr: np.ndarray, out=None, width: int = 1):
        """Dense numpy ``[comps, n]`` (or ``[comps, n, width]``) -> new (or given) blocked device tensor."""
        import torch
        a = np.ascontiguousarray(arr, dtype=self.e.np_dtype)
        comps = a.shape[0]
        if a.shape[1] != self.n or (width > 1 and a.shape[2:] != (width,)):
            raise ValueError("expected [%d, %d%s], got %r" % (comps, self.n, ", %d" % width if width > 1 else "", a.shape))
        dense = torch.from_numpy(a).to("cuda:%d" % self.e.device)
        if out is None:
            out = self.e.alloc(comps, self.n, width=width)
        self.e.pack(dense, out, comps, width, self.n)
        torch.cuda.current_stream(self.e.device).synchronize()       # `dense` may be freed after return
        return out

    def set_aux(self, aux: np.ndarray):
        """Auxiliary field records ``[n_aux, 12, n]`` -> blocked ``aux`` buffer of this batch."""
        a = np.ascontiguousarray(aux, dtype=self.e.np_dtype)
        if a.ndim != 3 or a.shape[1:] != (12, self.n):
            raise ValueError("aux must be [n_aux, 12, n], got %r" % (a.shape,))
        self.t["aux"] = self.to_blocked(a.reshape(a.shape[0] * 12, self.n))
        return self.t["aux"]

    def upload(self, name: str, arr: np.ndarray):
        if (self.shared and name in ("obst", "obst_ext")) or name in ("shared_obst", "shared_obst_ext"):   # dense: a plain copy
            import torch
            t = self._ensure(name)
            a = np.ascontiguousarray(arr, dtype=self.e.np_dtype)
            if name.startswith("shared_") and a.shape[0] == 0:
                return t
            if a.shape != tuple(t.shape):
                raise ValueError("%s: expected %r, got %r" % (name, tuple(t.shape), a.shape))
            t.copy_(torch.from_numpy(a))
            return t
        t = self._ensure(name)
        width = {"obst": 4, "obst_ext": 2}.get(name, 1)
        a = np.asarray(arr)
        if width == 1:
            a = a.reshape(-1, self.n)
        have = self.m if name in ("obst", "obst_ext") else t.shape[1]
        if a.shape[0] != have:
            raise ValueError("%s: %d components given, buffer has %d" % (name, a.shape[0], have))
        return self.to_blocked(a, out=t, width=width)

    def download(self, name: str) -> np.ndarray:
        """Blocked device tensor -> dense numpy ``[comps, n]`` (``[M, n, width]`` for obstacles)."""
        import torch
        t = self.t[name]
        if self.shared and name in ("obst", "obst_ext"):
            return t.cpu().numpy()
        if name in ("shared_obst", "shared_obst_ext"):
            return t[:self.ms].cpu().numpy()
        if t.dtype == torch.int32:                                   # int32 arrays: un-block on the host
            a = t.cpu().numpy()                                      # [tiles, comps, 32]
            return np.ascontiguousarray(a.transpose(1, 0, 2).reshape(a.shape[1], -1)[:, :self.n])
        comps = self.m if name in ("obst", "obst_ext") else t.shape[1]
        width = t.shape[3] if t.dim() == 4 else 1
        shape = (comps, self.n) if width == 1 else (comps, self.n, width)
        dense = torch.empty(shape, dtype=t.dtype, device=t.device)
        self.e.unpack(t, dense, comps, width, self.n)
        return dense.cpu().numpy()

    def obstacles_of(self, idx) -> np.ndarray:
        """``{x, y, z, radius}`` of every obstacle of the instances ``idx`` -> numpy ``[M, len(idx), 4]``, gathered from
        the pair-interleaved blocked array on the device (for sampling batches too large to convert as a whole)."""
        import torch
        t = self.t["obst"]
        if self.shared:
            return np.repeat(t.cpu().numpy()[:, None], len(idx), axis=1)
        ti = torch.as_tensor(np.asarray(idx), device=t.device)
        tiles, mp, k = t.shape[0], t.shape[1], int(ti.numel())
        if self.e.precision == 32:       # pair = planes {x0, x1, y0, y1}, {z0, z1, r0, r1} of 32 lanes x float4
            pr = t.reshape(tiles, mp // 2, 2, 32, 2, 2)[ti // 32, :, :, ti % 32]       # [k, pair, plane, component-in-plane, slot]
            o = pr.permute(1, 4, 0, 2, 3).reshape(mp, k, 4)                            # obstacle 2 * pair + slot
        else:                            # pair = planes {x0, x1}, {y0, y1}, {z0, z1}, {r0, r1} of 32 lanes x double2
            pr = t.reshape(tiles, mp // 2, 4, 32, 2)[ti // 32, :, :, ti % 32]          # [k, pair, component, slot]
            o = pr.permute(1, 3, 0, 2).reshape(mp, k, 4)
        return o[:self.m].contiguous().cpu().numpy()

    @property
    def bufs(self) -> Dict[str, object]:
        b = {k: v for k, v in self.t.items() if k in _BUF_FIELDS}
        if self.shared:
            b["obst_shared"] = True
        if self.mixed:
            b["obst_shared"] = VFK_OBST_MIXED
            b["shared_obst"] = self.t["shared_obst"]
            if "shared_obst_ext" in self.t:
                b["shared_obst_ext"] = self.t["shared_obst_ext"]
            b["n_shared_obst"] = self.ms
        return b

    def monitor(self, stream=None) -> int:
        """Run ``vfk_monitor`` on this batch's pose / twist / goal (allocates state and outputs on first use)."""
        for name in ("mon_f", "mon_i", "track", "dist", "tracking_state"):
            self._ensure(name)
        return self.e.monitor(self.t["pose"], self.t["twist"], self.t["goal"], self.t["mon_f"], self.t["mon_i"], self.n,
                              track_out=self.t["track"], dist_out=self.t["dist"], tracking_state_out=self.t["tracking_state"],
                              stream=stream)

    def step(self, k_cycles: int = 1, stream=None) -> int:
        return self.e.step(self.bufs, self.n, self.m, k_cycles, stream=stream, ext_cmd=tuple(self.ext_cmd))

    def solve(self, max_cycles: int, tol_trans: float, tol_rot: float, stream=None):
        """``Engine.solve`` on this batch: q moves in place (``download("q")``); returns ``(cycles [n] int32, dist [2, n])``.
        The batch's per-cycle outputs (qdot, flags, ...) are left out of the call and keep their contents."""
        self._ensure("cycles")
        self._ensure("solve_dist")                                   # metres, radians (the monitor's "dist" is in degrees)
        bufs = {k: v for k, v in self.bufs.items() if k not in _PER_CYCLE}
        self.e.solve(bufs, self.n, self.m, max_cycles, tol_trans, tol_rot, self.t["cycles"], self.t["solve_dist"], stream=stream,
                     ext_cmd=tuple(self.ext_cmd))
        return self.download("cycles")[0], self.download("solve_dist")
