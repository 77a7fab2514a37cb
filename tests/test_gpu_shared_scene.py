"""One obstacle list for the whole batch (vfk_buffers.obst_shared) on the GPU.

The reference is the per-instance path given the same list replicated to every instance: the shared scene must reproduce it
bit for bit, on q and every output, through vfk_step, vfk_solve and the host-buffer session.  The per-instance reference
runs the one-thread-per-instance kernel (VFK_NO_COOP / VFK_NO_SPLIT), the only shape that has a shared variant.
"""
import dataclasses

import numpy as np
import pytest

from helpers import (FP32_RTOL, FP64_RTOL, OBST_ORDERS, OBST_SAFES, check, near_goal, obstacle_distances, run_oracle,
                     tool_frame)

pytestmark = pytest.mark.gpu

ALL_OUT = ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "twist", "flags")
CAP = 1024


def _chain(lwr, name):
    from vfclik_b200 import workloads
    return {"lwr": lambda: lwr[0],                                          # 7 joints, LwrPattern
            "gen6": lambda: workloads.dual_arm_torso_chain(6),              # GenericPattern, N = 6
            "gen7": lambda: workloads.dual_arm_torso_chain(7),
            "pad8": lambda: workloads.dual_arm_torso_chain(8),              # runs padded in the 10-joint generic kernel
            "dh10": lambda: workloads.dual_arm_torso_chain(10),             # DhPattern
            "gen10": lambda: workloads.torso_arm_chain(10),
            "dh17": lambda: workloads.dual_arm_torso_chain(17),
            "gen17": lambda: workloads.dual_arm_torso_chain(17, dh=False)}[name]()


def _params(lwr, chain, config):
    from vfclik_b200.engine import Params
    base = Params.from_config(lwr[1]) if chain.n_joints == 7 and chain is lwr[0] else Params()
    N = chain.n_joints
    if config == "lean":
        return base
    if config == "order5":          # FP64: the fixed multiplication chain of order 5
        return dataclasses.replace(base, obst_order=5.0)
    if config == "order7.5":        # pow() in both precisions
        return dataclasses.replace(base, obst_order=7.5)
    if config == "general":         # tool frame, task and joint weights, the joint controller observed
        return dataclasses.replace(base, tool=(0, -1, 0, 1, 0, 0, 0, 0, 1, 0.01, 0.02, 0.05), w_task=(1, 1, 1, 0.5, 0.5, 0.5),
                                   w_joint=tuple(np.linspace(0.7, 1.0, N)), mixer_w=(1, 1, 0.2, 0, 0, 0))
    raise KeyError(config)


def _outputs(config):
    return ALL_OUT if config == "general" else ("qdot",)


def _engine(lwr, precision, chain_name, config):
    from vfclik_b200.engine import Engine
    chain = _chain(lwr, chain_name)
    return Engine(chain, precision=precision, params=_params(lwr, chain, config)), chain


def _scene(chain, n, M, seed, dtype, ext):
    from vfclik_b200 import workloads
    w = workloads.shared_scene_batch(chain, n, M, seed, dtype=dtype, obst_ext=ext)
    if ext:                          # per-obstacle {safe, order} across the values the field distinguishes
        rng = np.random.default_rng(seed + 3)
        w["obst_ext"][:, 0] = rng.choice(OBST_SAFES[1:], size=M)
        w["obst_ext"][:, 1] = rng.choice(OBST_ORDERS[:4], size=M)     # FP32: orders that stay clear of the weight limit
    return w


def _replicated(w, n):
    from vfclik_b200 import workloads
    r = dict(q=w["q"], goal=w["goal"])
    for k in ("obst", "obst_ext"):
        if k in w:
            r[k] = workloads.replicate_scene(w[k], n)
    return r


def _batch(e, w, M, shared, outputs=()):
    from vfclik_b200.engine import DeviceBatch
    n = w["q"].shape[1]
    db = DeviceBatch(e, n, M, obst_ext="obst_ext" in w, outputs=outputs, shared_obstacles=shared)
    db.upload("q", w["q"])
    db.upload("goal", w["goal"])
    if M:
        db.upload("obst", w["obst"])
        if "obst_ext" in w:
            db.upload("obst_ext", w["obst_ext"])
    return db


@pytest.fixture
def one_thread(monkeypatch):
    """Run the per-instance reference on the one-thread-per-instance kernel."""
    monkeypatch.setenv("VFK_NO_COOP", "1")
    monkeypatch.setenv("VFK_NO_SPLIT", "1")


def same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def run_step(e, w, M, k, shared, outputs):
    n = w["q"].shape[1]
    db = _batch(e, w if shared else _replicated(w, n), M, shared, outputs)
    assert db.step(k) == 1
    out = {name: db.download(name) for name in outputs}
    out["q"] = db.download("q")
    return out


# ------------------------------------------------------------------------------------------ 1. step: bit-identity
# (chain, config, M, obst_ext, K, n): every pattern and joint count, lean / general / HIOCC (FP32 K = 1 lean, N <= 7), the
# FP64 order specialisations and pow(), odd M, M < 8, M = 0 and M at the cap, ext rows, partial last tiles, K = 1 and 50
STEP_CASES = [
    ("lwr", "lean", 32, False, 1, 1000),
    ("lwr", "lean", 32, False, 50, 1000),
    ("lwr", "order5", 37, False, 50, 1000),
    ("lwr", "order7.5", 21, False, 1, 1000),
    ("lwr", "general", 37, False, 1, 1000),
    ("lwr", "general", 5, True, 50, 1000),
    ("lwr", "lean", 13, True, 50, 1000),
    ("lwr", "lean", 0, False, 50, 1000),
    ("gen6", "lean", 1, False, 1, 1000),
    ("gen6", "general", 7, False, 50, 700),
    ("gen7", "lean", CAP, False, 1, 500),
    ("gen7", "general", CAP, True, 2, 500),
    ("pad8", "general", 40, True, 50, 1000),
    ("pad8", "lean", 40, False, 50, 1000),
    ("dh10", "lean", 24, False, 50, 1000),
    ("gen10", "general", 9, False, 50, 1000),
    ("dh17", "lean", 64, False, 50, 1000),
    ("dh17", "general", 16, True, 1, 1000),
    ("gen17", "general", 33, False, 1, 1000),
]


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("chain_name,config,M,ext,K,n", STEP_CASES)
def test_step_equals_replicated_scene(lwr, built_lib, one_thread, precision, chain_name, config, M, ext, K, n):
    e, chain = _engine(lwr, precision, chain_name, config)
    dtype = np.float32 if precision == 32 else np.float64
    w = _scene(chain, n, M, seed=11 + M + K, dtype=dtype, ext=ext)
    outputs = _outputs(config)
    got = run_step(e, w, M, K, True, outputs)
    want = run_step(e, w, M, K, False, outputs)
    for k in want:
        assert same(got[k], want[k]), (k, np.argwhere(got[k] != want[k])[:5])
    assert np.all(np.isfinite(got["q"]))
    e.close()


# ------------------------------------------------------------------------------------------ 2. solve: bit-identity
def _solve(e, w, M, shared, k, tt, tr):
    n = w["q"].shape[1]
    db = _batch(e, w if shared else _replicated(w, n), M, shared)
    cycles, dist = db.solve(k, tt, tr)
    return dict(cycles=cycles, dist=dist, q=db.download("q"))


SOLVE_CASES = [                      # (chain, config, M, obst_ext, tolerances)
    ("lwr", "lean", 32, False, "mixed"),
    ("lwr", "lean", 32, False, "at_start"),
    ("lwr", "lean", 32, False, "never"),
    ("lwr", "general", 21, True, "mixed"),
    ("dh17", "lean", 40, False, "mixed"),
    ("gen10", "general", 3, False, "mixed"),
]
TOLS = {"mixed": (0.01, 0.05), "at_start": (100.0, 4.0), "never": (0.0, 0.0)}


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("chain_name,config,M,ext,tols", SOLVE_CASES)
def test_solve_equals_replicated_scene(lwr, built_lib, one_thread, precision, chain_name, config, M, ext, tols):
    e, chain = _engine(lwr, precision, chain_name, config)
    dtype = np.float32 if precision == 32 else np.float64
    n, K = 900, 40
    w = _scene(chain, n, M, seed=5, dtype=dtype, ext=ext)
    g, _ = near_goal(chain, n, 0, seed=5, dtype=dtype, tool=e.params.tool)    # some start inside the tolerances, some arrive
    w["q"], w["goal"] = g["q"], g["goal"]
    tt, tr = TOLS[tols]
    got = _solve(e, w, M, True, K, tt, tr)
    want = _solve(e, w, M, False, K, tt, tr)
    for k in ("cycles", "dist", "q"):
        assert same(got[k], want[k]), (k, np.argwhere(got[k] != want[k])[:5])
    c = got["cycles"]
    if tols == "at_start":
        assert np.all(c == 0)
    elif tols == "never":
        assert np.all(c == -1)
    else:
        assert np.count_nonzero(c >= 0) > 0
    e.close()


# ------------------------------------------------------------------------------------------ 3. host-buffer session
def _pinned(shape, dtype):
    import torch
    return torch.zeros(shape, dtype={np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32}[dtype]).pin_memory().numpy()


def _session_run(e, w, M, shared, session_m, n, path, calls=3, k=3):
    """Three vfk_session_cycle calls (chunked path: eager, graph capture, graph replay) -> the outputs of each."""
    s = e.session(n, session_m, obst_ext="obst_ext" in w and not shared)
    s.set_goal(w["goal"])
    if shared:
        s.set_shared_obstacles(w["obst"], w.get("obst_ext"))
    elif M:
        r = _replicated(w, n)
        s.set_obstacles(r["obst"], r.get("obst_ext"))
    N, dt = e.n_joints, e.np_dtype
    mk = _pinned if path == "direct" else (lambda shape, d: np.zeros(shape, dtype=d))
    q_in, qdot, q_out, flags = mk((N, n), dt), mk((N, n), dt), mk((N, n), dt), mk((n,), np.int32)
    q_in[...] = w["q"]
    outs = []
    for _ in range(calls):
        s.cycle(q_in, k, qdot_out=qdot, q_out=q_out, flags_out=flags)
        outs.append((qdot.copy(), q_out.copy(), flags.copy()))
        q_in[...] = q_out
    return s, outs, q_in


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("path", ["direct", "chunked"])
def test_session_equals_replicated_scene(lwr, built_lib, one_thread, precision, path):
    """Direct host I/O (page-locked, tile-aligned batch) and the chunked copy pipeline (pageable, two chunks, a partial last
    tile): the chunk views must keep the shared list un-offset.  The shared session of the chunked case is created with no
    obstacles of its own; the direct one has them, and set_obstacles takes it back to its per-instance scene."""
    e, chain = _engine(lwr, precision, "lwr", "lean")
    dtype = e.np_dtype
    n, M = (4096, 32) if path == "direct" else (2 * 65536 + 40, 19)
    w = _scene(chain, n, M, seed=23, dtype=dtype, ext=False)
    s1, got, q1 = _session_run(e, w, M, True, M if path == "direct" else 0, n, path)
    s0, want, q0 = _session_run(e, w, M, False, M, n, path)
    for c, (a, b) in enumerate(zip(got, want)):
        for name, x, y in zip(("qdot", "q", "flags"), a, b):
            assert same(x, y), (c, name)
    if path == "direct":
        # back to a per-instance scene: a different list, the same in both sessions
        other = _replicated(_scene(chain, n, M, seed=29, dtype=dtype, ext=False), n)
        for s, q in ((s1, q1), (s0, q0)):
            s.set_obstacles(other["obst"])
        o1, o0 = [np.zeros((e.n_joints, n), dtype=dtype) for _ in range(2)]
        s1.cycle(q1, 2, qdot_out=o1)
        s0.cycle(q0, 2, qdot_out=o0)
        assert same(o1, o0)
    e.close()


@pytest.mark.parametrize("precision", [32, 64])
def test_session_solve_equals_replicated_scene(lwr, built_lib, one_thread, precision):
    e, chain = _engine(lwr, precision, "lwr", "lean")
    dtype = e.np_dtype
    n, M, K = 3000, 27, 40
    w = _scene(chain, n, M, seed=31, dtype=dtype, ext=True)
    g, _ = near_goal(chain, n, 0, seed=31, dtype=dtype)
    w["q"], w["goal"] = g["q"], g["goal"]
    res = []
    for shared in (True, False):
        s = e.session(n, 0 if shared else M, obst_ext=not shared)
        s.set_goal(w["goal"])
        if shared:
            s.set_shared_obstacles(w["obst"], w["obst_ext"])
        else:
            r = _replicated(w, n)
            s.set_obstacles(r["obst"], r["obst_ext"])
        q, cyc, dist = np.zeros((e.n_joints, n), dtype), np.zeros(n, np.int32), np.zeros((2, n), dtype)
        s.solve(w["q"], K, 0.01, 0.05, q_out=q, cycles_out=cyc, dist_out=dist)
        res.append((q, cyc, dist))
    for x, y in zip(*res):
        assert same(x, y)
    assert np.count_nonzero(res[0][1] >= 0) > 0
    e.close()


# ------------------------------------------------------------------------------------------ 4. against the oracle
def _near_scene(chain, n, M, seed, dtype, n_near, tool):
    """A shared scene whose first n_near obstacles each sit next to the tool point of one instance (0 .. n_near - 1), at one
    of helpers.obstacle_distances with its own {safe, order} row: the near-obstacle regime inside one workcell."""
    w = _scene(chain, n, M, seed, dtype, ext=True)
    rng = np.random.default_rng(seed + 17)
    _, pt = tool_frame(chain, w["q"], tool)
    for j in range(n_near):
        safe, order = rng.choice(OBST_SAFES), rng.choice(OBST_ORDERS)
        d = obstacle_distances(safe, float(w["obst"][j, 3]))[j % 6]
        u = rng.normal(size=3)
        w["obst"][j, 0:3] = pt[j] + d * u / np.linalg.norm(u)
        w["obst_ext"][j] = (safe, order)
    return w


@pytest.mark.parametrize("precision,regime", [(64, "random"), (64, "near_obstacles"), (32, "random")])
def test_shared_scene_against_oracle(lwr, built_lib, precision, regime):
    e, chain = _engine(lwr, precision, "lwr", "general")
    dtype = e.np_dtype
    n, M = 400, 48
    w = _scene(chain, n, M, 41, dtype, ext=False) if regime == "random" else _near_scene(chain, n, M, 41, dtype, n_near=M, tool=e.params.tool)
    out = {k: v.T for k, v in run_step(e, w, M, 1, True, ALL_OUT).items()}
    ref = run_oracle(chain, e.params, _replicated(w, n), M, k=1)
    check(out, ref, FP64_RTOL if precision == 64 else FP32_RTOL)
    e.close()


# ------------------------------------------------------------------------------------------ 5. refusals
def test_shared_scene_refusals(lwr, built_lib):
    import ctypes as C
    import torch
    from vfclik_b200 import _lib
    from vfclik_b200.engine import VfkError
    e, chain = _engine(lwr, 32, "lwr", "lean")
    n = 64
    db = _batch(e, _scene(chain, n, 8, 3, np.float32, False), 8, True, outputs=("qdot",))
    big = torch.zeros((CAP + 1, 4), dtype=torch.float32, device="cuda")

    def code(fn, *args, **kw):
        with pytest.raises(VfkError) as ei:
            fn(*args, **kw)
        return ei.value.code

    bufs = db.bufs
    cyc = e.alloc(1, n, dtype=torch.int32)
    for run in (lambda b, m: e.step(b, n, m, 1), lambda b, m: e.solve({k: v for k, v in b.items() if k != "qdot"}, n, m, 5, 0.01, 0.05, cyc)):
        assert code(run, dict(bufs, obst_shared=2), 8) == _lib.VFK_ERR_INVALID
        assert code(run, dict(bufs, obst_shared=-1), 8) == _lib.VFK_ERR_INVALID
        assert code(run, dict(bufs, obst=big), CAP + 1) == _lib.VFK_ERR_UNSUPPORTED
        assert code(run, dict(bufs, obst=None), 8) == _lib.VFK_ERR_INVALID
        assert code(run, dict(bufs, obst=bufs["obst"].data_ptr() + 16), 8) == _lib.VFK_ERR_INVALID
        run(dict(bufs, obst=big), CAP)                     # the cap itself is accepted
        run(dict(bufs, obst=None), 0)                      # and so is an empty list
    torch.cuda.synchronize()
    s = e.session(n, 0)
    assert code(s.set_shared_obstacles, np.zeros((CAP + 1, 4))) == _lib.VFK_ERR_UNSUPPORTED
    assert e._lib.vfk_session_set_shared_obstacles(s._s, None, None, 4) == _lib.VFK_ERR_INVALID
    assert e._lib.vfk_session_set_shared_obstacles(s._s, None, None, -1) == _lib.VFK_ERR_INVALID
    # a session created with no obstacles: set_obstacles stays a no-op that returns VFK_OK, and leaves the shared scene on
    s.set_shared_obstacles(np.zeros((3, 4)))
    assert e._lib.vfk_session_set_obstacles(s._s, None, None) == _lib.VFK_OK
    b = _lib.BuffersC()
    assert e._lib.vfk_session_buffers(s._s, C.byref(b)) == _lib.VFK_OK and b.obst_shared == 1
    e.close()
