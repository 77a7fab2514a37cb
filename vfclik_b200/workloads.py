"""Synthetic workloads of BASELINE.json's configs (SURVEY.md section 8d), seeded numpy.

Arrays are produced directly in the GPU layout: dense SoA ``[comps, I]``.
"""
from __future__ import annotations

import numpy as np

from .config import ChainDesc


def quat_to_rot_rows(quat: np.ndarray) -> np.ndarray:
    """[I,4] (w,x,y,z) unit quaternions -> [9, I] row-major rotation components."""
    w, x, y, z = quat.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], axis=0)


# Exact arithmetic of one instance-cycle (SURVEY.md section 8d): {(N, M): (FLOPs, transcendentals)}, counted by executing the
# oracle's cycle on a counting scalar type (the `opcount` module of the test oracle; add / sub / mul / div / sqrt = 1 FLOP, FMA = 2; sin, cos,
# atan2, pow counted apart; constant folding and structural 0 / 1 entries free).  Frozen here; tests/test_oracle.py
# re-derives them.  The K-fused roofline (FP32 pipe) in bench.py is computed from these.
ALGORITHMIC_OPS = {(7, 3): (1064, 18), (7, 32): (1644, 47), (7, 256): (6124, 271), (17, 64): (3449, 99)}


def algorithmic_flops(n_joints: int, n_obst: int) -> int:
    """FLOPs per instance-cycle; shapes other than the frozen ones use the per-obstacle slope (20 FLOPs) of the nearest."""
    if (n_joints, n_obst) in ALGORITHMIC_OPS:
        return ALGORITHMIC_OPS[(n_joints, n_obst)][0]
    same = [(abs(m - n_obst), m) for (n, m) in ALGORITHMIC_OPS if n == n_joints]
    if not same:
        raise KeyError("no frozen operation count for %d joints" % n_joints)
    m0 = min(same)[1]
    return ALGORITHMIC_OPS[(n_joints, m0)][0] + 20 * (n_obst - m0)


def random_batch(chain: ChainDesc, n_instances: int, n_obstacles: int, seed: int, dtype=np.float64,
                 obst_ext: bool = False, slowdown: float = 0.05, order: float = 20.0, safe: float = 0.001,
                 shoulder=None, box: float = 0.8):
    """Configs 2-5: q ~ U(0.9 * limits); goal position ~ U(shell 0.3-0.8 m around the shoulder),
    goal rotation ~ Haar (normalised Gaussian quaternion); obstacles ~ U(workspace box),
    radius ~ U(0.03, 0.10); ``numpy.random.default_rng(seed)``.

    Returns dict(q [N,I], goal [13,I], obst [M,I,4] {x,y,z,radius} [, obst_ext [M,I,2] {safe, order}]) of ``dtype``.
    """
    rng = np.random.default_rng(seed)
    I, N, M = int(n_instances), chain.n_joints, int(n_obstacles)
    if shoulder is None:
        shoulder = chain.base[9:12]            # origin of the first joint
    q = rng.uniform((0.9 * chain.q_lo)[:, None], (0.9 * chain.q_hi)[:, None], size=(N, I)).astype(dtype)
    quat = rng.normal(size=(I, 4))
    quat /= np.linalg.norm(quat, axis=1, keepdims=True)
    d = rng.normal(size=(I, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    pg = d * rng.uniform(0.3, 0.8, size=(I, 1)) + np.asarray(shoulder)[None, :]
    goal = np.concatenate([quat_to_rot_rows(quat), pg.T, np.full((1, I), slowdown)], axis=0).astype(dtype)
    obst = np.empty((M, I, 4), dtype=dtype)
    sh = np.asarray(shoulder, dtype=np.float64)
    for m in range(M):                       # per-obstacle draws keep peak memory at O(I)
        obst[m, :, 0:3] = (rng.uniform(-box, box, size=(I, 3)) + sh[None, :]).astype(dtype)
        obst[m, :, 3] = rng.uniform(0.03, 0.10, size=I).astype(dtype)
    out = dict(q=q, goal=goal, obst=obst)
    if obst_ext:
        ext = np.empty((M, I, 2), dtype=dtype)
        ext[:, :, 0] = safe
        ext[:, :, 1] = order
        out["obst_ext"] = ext
    return out


def shared_scene_batch(chain: ChainDesc, n_instances: int, n_obstacles: int, seed: int, dtype=np.float64,
                       obst_ext: bool = False, **kw):
    """One workcell for the whole batch (``vfk_buffers.obst_shared``): per-instance starts and goals, one obstacle list.
    Starts and goals are :func:`random_batch`'s with ``seed``; the scene is the obstacle list :func:`random_batch` draws for
    a single instance with ``seed + 1``, so every distribution is :func:`random_batch`'s.

    Returns dict(q [N,I], goal [13,I], obst [M,4] {x,y,z,radius} [, obst_ext [M,2] {safe, order}]) of ``dtype``."""
    w = random_batch(chain, n_instances, 0, seed, dtype=dtype, **kw)
    scene = random_batch(chain, 1, n_obstacles, seed + 1, dtype=dtype, obst_ext=obst_ext, **kw)
    out = dict(q=w["q"], goal=w["goal"], obst=np.ascontiguousarray(scene["obst"][:, 0]))
    if obst_ext:
        out["obst_ext"] = np.ascontiguousarray(scene["obst_ext"][:, 0])
    return out


def replicate_scene(obst: np.ndarray, n_instances: int) -> np.ndarray:
    """A shared list ``[M, C]`` as the per-instance array ``[M, n, C]`` that gives every instance the same scene."""
    return np.ascontiguousarray(np.broadcast_to(obst[:, None, :], (obst.shape[0], int(n_instances), obst.shape[1])))


def mixed_scene_batch(chain: ChainDesc, n_instances: int, n_own: int, n_shared: int, seed: int, dtype=np.float64,
                      obst_ext: bool = False, **kw):
    """A shared workcell plus obstacles of each instance's own (``vfk_buffers.obst_shared = 2``): per-instance starts, goals
    and ``n_own`` obstacles as :func:`random_batch` draws them with ``seed``, and ``n_shared`` obstacles for the whole batch,
    the list :func:`random_batch` draws for a single instance with ``seed + 1`` (as :func:`shared_scene_batch`).

    Returns dict(q [N,I], goal [13,I], obst [Mi,I,4], shared_obst [Ms,4] [, obst_ext [Mi,I,2], shared_obst_ext [Ms,2]])
    of ``dtype``."""
    w = random_batch(chain, n_instances, n_own, seed, dtype=dtype, obst_ext=obst_ext, **kw)
    scene = random_batch(chain, 1, n_shared, seed + 1, dtype=dtype, obst_ext=obst_ext, **kw)
    out = dict(w, shared_obst=np.ascontiguousarray(scene["obst"][:, 0]))
    if obst_ext:
        out["shared_obst_ext"] = np.ascontiguousarray(scene["obst_ext"][:, 0])
    return out


def concat_scene(own: np.ndarray, shared: np.ndarray, n_instances: int) -> np.ndarray:
    """The per-instance array ``[Mi + Ms, n, C]`` equivalent to a mixed scene: each instance's own list ``[Mi, n, C]``
    followed by the shared list ``[Ms, C]``, in the order the field sums them."""
    own = np.asarray(own)
    shared = np.asarray(shared)
    n = int(n_instances)
    if own.shape[1:] != (n, shared.shape[1]):
        raise ValueError("own list %r does not match %d instances of %d components" % (own.shape, n, shared.shape[1]))
    return np.ascontiguousarray(np.concatenate([own, replicate_scene(shared.astype(own.dtype, copy=False), n)], axis=0))


def random_batch_device(engine, n_instances: int, n_obstacles: int, seed: int, slowdown: float = 0.05, box: float = 0.8):
    """Same distributions as :func:`random_batch`, drawn on the GPU with torch's generator (large shapes:
    config 4's 2M x 256 obstacles per GPU would take minutes and 8 GB of host memory through numpy).
    Returns a ``DeviceBatch`` with q / goal / obst filled (blocked layout)."""
    import torch
    from .engine import DeviceBatch
    chain = engine.chain
    dev = "cuda:%d" % engine.device
    dt = engine.torch_dtype
    g = torch.Generator(device=dev)
    g.manual_seed(int(seed))
    I, N, M = int(n_instances), chain.n_joints, int(n_obstacles)
    lo = torch.tensor(0.9 * chain.q_lo, dtype=dt, device=dev)[:, None]
    hi = torch.tensor(0.9 * chain.q_hi, dtype=dt, device=dev)[:, None]
    q = lo + (hi - lo) * torch.rand((N, I), generator=g, dtype=dt, device=dev)
    quat = torch.randn((4, I), generator=g, dtype=dt, device=dev)
    quat = quat / quat.norm(dim=0, keepdim=True)
    w, x, y, z = quat
    rot = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                       2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                       2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=0)
    d = torch.randn((3, I), generator=g, dtype=dt, device=dev)
    d = d / d.norm(dim=0, keepdim=True)
    sh = torch.tensor(chain.base[9:12], dtype=dt, device=dev)[:, None]
    pg = d * (0.3 + 0.5 * torch.rand((1, I), generator=g, dtype=dt, device=dev)) + sh
    goal = torch.cat([rot, pg, torch.full((1, I), slowdown, dtype=dt, device=dev)], dim=0)
    db = DeviceBatch(engine, I, M, outputs=("qdot",))
    engine.pack(q.contiguous(), db.t["q"], N, 1, I)
    engine.pack(goal.contiguous(), db.t["goal"], 13, 1, I)
    step = max(2, min(M, (1 << 26) // max(I, 1)) & ~1)       # obstacles per slice (whole pairs): bound the dense temporary
    tiles = db.t["obst"].shape[0]
    for m0 in range(0, M, step):
        m1 = min(M, m0 + step)
        o = torch.empty((m1 - m0, I, 4), dtype=dt, device=dev)
        o[:, :, 0:3] = (2 * box) * torch.rand((m1 - m0, I, 3), generator=g, dtype=dt, device=dev) - box + sh.T[None]
        o[:, :, 3] = 0.03 + 0.07 * torch.rand((m1 - m0, I), generator=g, dtype=dt, device=dev)
        blk = engine.alloc(m1 - m0, I, width=4)
        engine.pack(o, blk, m1 - m0, 4, I)
        db.t["obst"][:, m0:m0 + blk.shape[1]] = blk             # pair rows 2p, 2p + 1 <-> obstacles 2p, 2p + 1 (m0 is even)
        del o, blk
    torch.cuda.synchronize(engine.device)
    return db


def config1(chain: ChainDesc, config, seed: int = 0):
    """BASELINE config 1: single LWR, start q and goal of old/system_start.sh.old:234,346,
    three ObstacleP (radius 0.05, order 20: old/README.old:75) seeded between the start
    end-effector position and the goal."""
    rng = np.random.default_rng(seed)
    g = np.asarray(config.initial_vf_pose[2], dtype=np.float64)
    T = g[:16].reshape(4, 4)
    goal = np.concatenate([T[:3, :3].reshape(9), T[:3, 3], [g[16] if g.size > 16 else 0.03]])[:, None]
    q = np.asarray(config.initial_joint_pos, dtype=np.float64)[:, None]
    start_ee = np.array([0.73, 0.28, 0.63])      # approximate EE at the start posture (offset seed only)
    obst = np.zeros((3, 1, 4))
    for m in range(3):
        t = (m + 1) / 4.0
        c = start_ee * (1 - t) + T[:3, 3] * t + rng.uniform(-0.08, 0.08, size=3)
        obst[m, 0, 0:3] = c
        obst[m, 0, 3] = 0.05
    return dict(q=q, goal=goal, obst=obst)


def torso_arm_chain(n_joints: int = 10) -> ChainDesc:
    """The first ``n_joints`` joints of the mixed-axis :func:`dual_arm_torso_chain`; the default 10 = 3-DOF torso + one
    7-joint arm, the shape of the reference's iCub configuration (``scripts/bridge:344-345``: arm 7 + torso 3 -> a 4-D
    nullspace)."""
    return dual_arm_torso_chain(n_joints, dh=False)


def dual_arm_torso_chain(n_joints: int = 17, dh: bool = True) -> ChainDesc:
    """BASELINE config 5: 3-DOF torso + 14 arm joints treated as one 17-joint serial chain
    (6x17 Jacobian).  Synthetic geometry: a 3-axis torso followed by two LWR-like 7-joint
    segments; only the shape (N = 17) matters for the benchmark.

    ``dh=True`` (default): the whole chain in Denavit-Hartenberg form -- revolute Z joints, X-twist tips -- the way humanoid
    models are published (e.g. iCub's iKin tables); such chains take the kernels' ``DhPattern``.  ``dh=False``: the torso's
    third joint is a KDL ``RotX`` joint (yaw-pitch-roll), which the host canonicalises into a general tip rotation and the
    kernels run through ``GenericPattern``."""
    from . import kdl
    from math import pi
    segs = [
        kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame(kdl.Rotation.RotX(pi / 2), kdl.Vector(0, 0, 0.20))),
        kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame(kdl.Rotation.RotX(-pi / 2), kdl.Vector(0, 0, 0.0))),
        (kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame(kdl.Rotation.RotX(pi / 2), kdl.Vector(0.05, 0, 0.25))) if dh else
         kdl.Segment(kdl.Joint(kdl.Joint.RotX), kdl.Frame(kdl.Rotation.Identity(), kdl.Vector(0, 0, 0.25)))),
    ]
    for _ in range(2):
        segs += [
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, pi / 2, 0.0, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, -pi / 2, 0.20, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, -pi / 2, 0.0, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, pi / 2, 0.195, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, pi / 2, 0.0, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame.DH_Craig1989(0.0, -pi / 2, 0.0, 0.0)),
            kdl.Segment(kdl.Joint(kdl.Joint.RotZ), kdl.Frame(kdl.Rotation.Identity(), kdl.Vector(0, 0, 0.05))),
        ]
    deg = pi / 180.0
    limits = [[-60 * deg, 60 * deg], [-30 * deg, 60 * deg], [-30 * deg, 30 * deg]] + \
             ([[-170 * deg, 170 * deg], [-120 * deg, 120 * deg]] * 3 + [[-170 * deg, 170 * deg]]) * 2
    from .config import chain_from_segments
    return chain_from_segments(segs[:n_joints], limits[:n_joints])
