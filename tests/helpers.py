"""Shared helpers for the parity tests (test infrastructure)."""
import numpy as np

FP64_RTOL = 1e-9
FP32_RTOL = 1e-4


def to_oracle(batch_arrays, n_obst):
    """GPU layouts (q [N,I], goal [13,I], obst [M,I,4], obst_ext [M,I,2]) -> the oracle's instance-major arrays."""
    q = batch_arrays["q"].T.astype(np.float64)
    goal = batch_arrays["goal"].T.astype(np.float64)
    obst = None
    if n_obst > 0:
        obst = batch_arrays["obst"].transpose(1, 0, 2).astype(np.float64)
        if "obst_ext" in batch_arrays:
            obst = np.concatenate([obst, batch_arrays["obst_ext"].transpose(1, 0, 2).astype(np.float64)], axis=2)
    return q, goal, obst


def rel_err(a, b, floor=1e-3):
    """Per-instance relative error of joint-velocity vectors: max_i |a_i - b_i| / max(max_i |b_i|, floor).

    a, b: [I, N].  The floor keeps instances whose reference velocity is ~0 from dividing by noise.
    """
    num = np.max(np.abs(a - b), axis=1)
    den = np.maximum(np.max(np.abs(b), axis=1), floor)
    return num / den


def oracle_params(params):
    """vfclik_b200.engine.Params -> oracle.batch.Params (same field names)."""
    import dataclasses
    from oracle import batch
    d = dataclasses.asdict(params)
    for k in ("mixer_w", "w_task", "tool", "ns_control"):
        d[k] = tuple(d[k])
    for k in ("w_joint", "jp_ref"):
        d[k] = None if d[k] is None else tuple(d[k])
    return batch.Params(**d)


# ---------------------------------------------------------------------------------------------- the oracle over all host cores
_PAR = {}


def _oracle_chunk(span):
    """One chunk of instances through oracle.batch.step (runs in a forked worker: the arrays are inherited, not pickled)."""
    from oracle import batch
    i0, i1 = span
    q, goal, obst = to_oracle({k: (v[:, i0:i1] if k != "obst" else v[:, i0:i1, :]) for k, v in _PAR["w"].items()}, _PAR["m"])
    out = batch.step(_PAR["chain"], _PAR["prm"], q, goal, obst, k_cycles=_PAR["k"])
    return i0, {k: out[k] for k in _PAR["keys"]}


def oracle_parallel(chain, params, w, n_obst, k=1, keys=("qdot",), chunk=16384):
    """oracle.batch.step over a large batch, fanned over the host cores in chunks (fork: zero-copy inputs).  The vectorised
    oracle does ~1.7e5 instance-cycles/s per core, so the full 1,048,576-instance configuration takes seconds, not minutes."""
    import multiprocessing as mp
    import os
    n = w["q"].shape[1]
    _PAR.update(chain=chain, prm=oracle_params(params), w=w, m=n_obst, k=k, keys=tuple(keys))
    spans = [(i, min(n, i + chunk)) for i in range(0, n, chunk)]
    procs = max(1, min(len(spans), len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
    with mp.get_context("fork").Pool(procs) as pool:
        parts = pool.map(_oracle_chunk, spans)
    _PAR.clear()
    out = {}
    for key in keys:
        first = parts[0][1][key]
        full = np.empty((n,) + first.shape[1:], dtype=first.dtype)
        for i0, d in parts:
            full[i0:i0 + d[key].shape[0]] = d[key]
        out[key] = full
    return out


# ---------------------------------------------------------------------------------------------- GPU run, oracle run, comparison
def run_gpu(engine, w, n_obst, k=1, outputs=("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "flags"),
            extra=None, aux=None, ext_cmd=None):
    """One launch of K fused cycles on a DeviceBatch filled from the dense arrays of ``w`` (+ ``extra`` inputs, auxiliary
    field records [n_aux, 12, I], extra mixer ports [N, I]); returns the requested outputs instance-major ([I, comps]), the
    final q, the flags as [I], and the nullspace state and joint-controller reference if they were given."""
    from vfclik_b200.engine import DeviceBatch
    n = w["q"].shape[1]
    db = DeviceBatch(engine, n, n_obst, obst_ext="obst_ext" in w, outputs=outputs)
    db.upload("q", w["q"])
    db.upload("goal", w["goal"])
    if n_obst:
        db.upload("obst", w["obst"])
        if "obst_ext" in w:
            db.upload("obst_ext", w["obst_ext"])
    for name, arr in (extra or {}).items():
        db.upload(name, arr)
    if aux is not None:
        db.set_aux(aux)
    for i, x in enumerate(ext_cmd or ()):
        db.ext_cmd[i] = db.to_blocked(x)
    assert db.step(k) == 1
    out = {name: db.download(name).T for name in outputs}
    out["q"] = db.download("q").T
    if "flags" in out:
        out["flags"] = out["flags"][:, 0]
    if "ns_lastvec" in db.t:
        out["lastvec"] = db.download("ns_lastvec").T
    if "jp_ref" in db.t:
        out["jp_ref"] = db.download("jp_ref").T
    return out


def run_oracle(chain, params, w, n_obst, k=1, **kw):
    from oracle import batch
    q, goal, obst = to_oracle(w, n_obst)
    return batch.step(chain, oracle_params(params), q, goal, obst, k_cycles=k, **kw)


def check(out, ref, rtol, keys=("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd"), pose_atol=None):
    for k in keys:
        e = rel_err(out[k].astype(np.float64), ref[k])
        assert e.max() <= rtol, (k, float(e.max()), int(np.argmax(e)))
    if pose_atol is not None:
        assert np.max(np.abs(out["pose"] - ref["pose"])) <= pose_atol


# ---------------------------------------------------------------------------------------------- batches near goals and obstacles
def tool_frame(chain, q, tool=None):
    """Tool frame of the oracle's FK for q [N, I] (dense GPU layout): R [I, 3, 3], p [I, 3]."""
    from oracle import batch
    R, p, _ = batch.fk_jac(chain, np.asarray(q, dtype=np.float64).T)
    if tool is None:
        return R, p
    t = np.asarray(tool, dtype=np.float64)
    return R @ t[:9].reshape(3, 3), p + R @ t[9:12]


def _unit_vectors(rng, n):
    u = rng.normal(size=(n, 3))
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def axis_angle_rotation(axis, theta):
    """Rodrigues: rotations by theta [I] about the unit axes [I, 3] -> [I, 3, 3] (1 - cos written as 2 sin^2 so that tiny
    angles keep their relative precision)."""
    K = np.zeros(axis.shape[:1] + (3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -axis[:, 2], axis[:, 1], -axis[:, 0]
    K[:, 1, 0], K[:, 2, 0], K[:, 2, 1] = axis[:, 2], -axis[:, 1], axis[:, 0]
    s = np.sin(theta)[:, None, None]
    vc = (2.0 * np.sin(0.5 * theta) ** 2)[:, None, None]
    return np.eye(3)[None] + s * K + vc * (K @ K)


SLOWDOWNS = (0.0, 0.01, 0.05, 0.2)


def goal_distances(s):
    """Goal distances tried for the translational slowdown s.  With the slowdown off (s = 0) the field is discontinuous at the
    goal -- full speed along a direction the rounding of the kinematic chain decides within 1e-7 m of it -- so there the
    distances are taken relative to 0.05 m and the two absolute ones are left out."""
    if s > 0:
        return (1e-7, 1e-4, s / 2, s * (1 - 1e-3), s * (1 + 1e-3), 2 * s)
    return (0.025, 0.05 * (1 - 1e-3), 0.05 * (1 + 1e-3), 0.1)


def goal_angles(rot_slowdown):
    """Goal rotation angles tried for ``rot_slowdown``; with it off (0), relative to 0.09 and without the absolute tiny angles
    (the same discontinuity as in :func:`goal_distances`)."""
    rs = rot_slowdown if rot_slowdown > 0 else 0.09
    tail = (rs / 2, rs * (1 - 1e-3), rs * (1 + 1e-3), 0.5, np.pi / 2, np.pi - 1e-3)
    return ((1e-7, 1e-4) + tail) if rot_slowdown > 0 else tail


def near_goal(chain, n, n_obst, seed, rot_slowdown=0.09, dtype=np.float64, tool=None, **kw):
    """``workloads.random_batch`` with every goal moved next to the instance's own tool frame: the goal position at a distance
    d along a random direction from the tool position, the goal rotation R(a, theta) R_tool about a random axis a.  Each
    instance draws its translational slowdown s from SLOWDOWNS (0 = off) and (s, d, theta) from the products of
    ``goal_distances(s)`` and ``goal_angles(rot_slowdown)``, so every combination occurs once n is a few hundred.  The frame
    is the oracle's FK of q as rounded to ``dtype``.  Returns (w, meta) with meta = dict(d, theta, slowdown) [I]."""
    from vfclik_b200 import workloads
    w = workloads.random_batch(chain, n, n_obst, seed, dtype=dtype, **kw)
    rng = np.random.default_rng(seed + 7919)
    combos = [(s, d, t) for s in SLOWDOWNS for d in goal_distances(s) for t in goal_angles(rot_slowdown)]
    pick = np.concatenate([rng.permutation(len(combos)) for _ in range(-(-n // len(combos)))])[:n]
    s, d, theta = (np.array([combos[i][j] for i in pick]) for j in range(3))
    R, p = tool_frame(chain, w["q"], tool)
    pg = p + d[:, None] * _unit_vectors(rng, n)
    Rg = axis_angle_rotation(_unit_vectors(rng, n), theta) @ R
    w["goal"] = np.concatenate([Rg.reshape(n, 9), pg, s[:, None]], axis=1).T.astype(dtype)
    return w, dict(d=d, theta=theta, slowdown=s)


OBST_SAFES = (0.0, 1e-3, 0.02, 0.1)
OBST_ORDERS = (1.0, 2.0, 3.0, 5.0, 7.5, 20.0, 33.0)
FP32_WEIGHT_LIMIT = 1e28           # the FP32 kernels saturate a repeller weight at 1e30 (tested on its own): stay clear of it


def obstacle_distances(safe, radius):
    """Distances of a placed obstacle's centre from the tool: inside, just inside and just outside the safe distance, and
    half, one and three radii.  A safe distance of 0 has no inner band (0.2 safe would put the centre on the tool point,
    the field's singular point), so those become fractions of the radius."""
    if safe > 0:
        return (0.2 * safe, 0.9 * safe, 1.1 * safe, radius / 2, radius, 3 * radius)
    return (0.2 * radius, 0.3 * radius, 0.4 * radius, radius / 2, radius, 3 * radius)


def near_obstacles(chain, n, n_obst, seed, dtype=np.float64, obst_ext=True, safe=1e-3, order=20.0, n_near=2, tool=None, **kw):
    """``workloads.random_batch`` with ``n_near`` obstacles of every instance (in random slots) moved next to its tool point.
    With ``obst_ext`` every obstacle gets its own {safe, order} row drawn from OBST_SAFES x OBST_ORDERS; otherwise the
    uniform ``safe`` / ``order`` (the engine's) apply.  A placed obstacle sits at one of ``obstacle_distances(safe, radius)``
    along a random direction.  In FP32 an obstacle whose weight (radius / max(d, safe))^order / d would pass
    FP32_WEIGHT_LIMIT takes the largest order of OBST_ORDERS that stays below it (ext rows), or is pushed out to where its
    weight does (uniform parameters).  Returns (w, meta): meta = dict(slot [n_near, I], d [n_near, I])."""
    from vfclik_b200 import workloads
    assert n_obst >= n_near
    w = workloads.random_batch(chain, n, n_obst, seed, dtype=dtype, obst_ext=obst_ext, safe=safe, order=order, **kw)
    rng = np.random.default_rng(seed + 104729)
    _, pt = tool_frame(chain, w["q"], tool)
    obst = w["obst"].astype(np.float64)
    if obst_ext:
        ext = np.empty((n_obst, n, 2))
        ext[:, :, 0] = rng.choice(OBST_SAFES, size=(n_obst, n))
        ext[:, :, 1] = rng.choice(OBST_ORDERS, size=(n_obst, n))
    slot = np.argsort(rng.random((n_obst, n)), axis=0)[:n_near]                 # distinct random slots per instance
    cols = np.arange(n)
    dist = np.empty((n_near, n))
    for k in range(n_near):
        sf = ext[slot[k], cols, 0] if obst_ext else np.full(n, float(safe))
        rad = obst[slot[k], cols, 3]
        pick = rng.integers(0, 6, size=n)
        d = np.array([obstacle_distances(sf[i], rad[i])[pick[i]] for i in range(n)])
        if dtype == np.float32 and not obst_ext:
            # push the obstacle out to where its weight fits: inside the safe distance the weight is (r / safe)^o / d,
            # outside it r^o / d^(o + 1)
            o = float(order)
            inner = np.where(sf > 0, (rad / np.where(sf > 0, sf, 1.0)) ** o / FP32_WEIGHT_LIMIT, np.inf)
            outer = (rad ** o / FP32_WEIGHT_LIMIT) ** (1.0 / (o + 1.0))
            d_min = 1.01 * np.where(inner < sf, inner, np.maximum(outer, sf))
            d = np.maximum(d, d_min)
        obst[slot[k], cols, 0:3] = pt + d[:, None] * _unit_vectors(rng, n)
        dist[k] = d
    if dtype == np.float32 and obst_ext:
        # the largest order of OBST_ORDERS, up to the one drawn, whose weight fits
        d = np.linalg.norm(obst[:, :, 0:3].astype(np.float32).astype(np.float64) - pt[None], axis=2)
        ratio = obst[:, :, 3] / np.maximum(d, ext[:, :, 0])
        best = np.full(d.shape, OBST_ORDERS[0])
        for o in OBST_ORDERS:
            best = np.where((ratio ** o / d <= FP32_WEIGHT_LIMIT) & (o <= ext[:, :, 1]), o, best)
        ext[:, :, 1] = best
    w["obst"] = obst.astype(dtype)
    if obst_ext:
        w["obst_ext"] = ext.astype(dtype)
    return w, dict(slot=slot, d=dist)


# ---------------------------------------------------------------------------------------------- batches near singular postures
SINGULAR_LEVELS = (0.0, 1e-12, 1e-9, 1e-6, 1e-3, 1e-1)


def singular_values(chain, q):
    """Singular values [I, 6] (descending) of the oracle's Jacobian at q [N, I] (dense GPU layout), in FP64."""
    from oracle import batch
    J = batch.fk_jac(chain, np.asarray(q, dtype=np.float64).T)[2]
    return np.linalg.svd(J, compute_uv=False)


def near_singular(chain, n, n_obst, seed, dtype=np.float64, kind="home", levels=SINGULAR_LEVELS, **kw):
    """``workloads.random_batch`` with every posture moved next to a kinematic singularity, where J loses rank.

    Base postures: ``home`` is q = 0, rank-deficient on every chain of the suite (LWR: rank 3; torso_arm_chain: 4;
    dual_arm_torso_chain: 5, generic form 4); ``elbow`` (the 7-joint LWR) keeps random_batch's q with the elbow straight,
    q[3] = 0 (rank 5).  The base posture is asserted singular through the oracle's Jacobian: sigma_min / sigma_max < 1e-15.
    Each instance then moves by one of ``levels`` (delta, each drawn about equally often): ``home`` along a random unit
    direction of joint space, ``elbow`` by q[3] = +-delta only.  q is rounded to ``dtype`` (delta = 0 stays exactly singular
    in FP32 too) and stays inside the chain's limits.  Returns (w, meta): meta = dict(delta [I], sigma [I, 6] and cond [I]
    = sigma_max / sigma_min, both of the oracle's Jacobian at q as rounded)."""
    from vfclik_b200 import workloads
    w = workloads.random_batch(chain, n, n_obst, seed, dtype=dtype, **kw)
    rng = np.random.default_rng(seed + 15485863)
    N = w["q"].shape[0]
    if kind == "home":
        base = np.zeros((N, n))
    elif kind == "elbow":
        assert N == 7, "the elbow singularity is the 7-joint LWR's"
        base = w["q"].astype(np.float64).copy()
        base[3] = 0.0
    else:
        raise ValueError(kind)
    s0 = singular_values(chain, base)
    assert np.all(s0[:, -1] <= 1e-15 * s0[:, 0]), "base posture is not singular"
    lv = np.asarray(levels, dtype=np.float64)
    delta = lv[np.concatenate([rng.permutation(len(lv)) for _ in range(-(-n // len(lv)))])[:n]]
    if kind == "home":
        u = rng.normal(size=(N, n))
        step = u / np.linalg.norm(u, axis=0, keepdims=True)
    else:
        step = np.zeros((N, n))
        step[3] = rng.choice((-1.0, 1.0), size=n)
    q = (base + delta[None, :] * step).astype(dtype)
    assert np.all(q >= chain.q_lo[:, None]) and np.all(q <= chain.q_hi[:, None])
    w["q"] = q
    sigma = singular_values(chain, q)
    with np.errstate(divide="ignore"):
        cond = sigma[:, 0] / sigma[:, -1]
    return w, dict(delta=delta, sigma=sigma, cond=cond)
