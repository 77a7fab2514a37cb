"""A mixed scene (vfk_buffers.obst_shared = 2) on the GPU: each instance's own obstacles plus one list for the whole batch.

The reference is the per-instance path on the concatenated list [own ; shared] (workloads.concat_scene).  With an own count
that is a multiple of 8 the mixed scene reproduces it bit for bit, on q and every output, through vfk_step, vfk_solve and the
host-buffer session; other own counts are held to the oracle.  The per-instance reference runs the one-thread-per-instance
kernel (VFK_NO_COOP / VFK_NO_SPLIT), the only shape that has a shared variant.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from helpers import FP32_RTOL, FP64_RTOL, OBST_ORDERS, OBST_SAFES, check, near_goal, oracle_params, run_oracle, to_oracle

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
    if config == "order2":          # FP64: the chain of order 2
        return dataclasses.replace(base, obst_order=2.0)
    if config == "order7.5":        # pow() in both precisions
        return dataclasses.replace(base, obst_order=7.5)
    if config == "general":         # tool frame, task and joint weights, the joint controller observed
        return dataclasses.replace(base, tool=(0, -1, 0, 1, 0, 0, 0, 0, 1, 0.01, 0.02, 0.05), w_task=(1, 1, 1, 0.5, 0.5, 0.5),
                                   w_joint=tuple(np.linspace(0.7, 1.0, N)), mixer_w=(1, 1, 0.2, 0, 0, 0))
    raise KeyError(config)


def _engine(lwr, precision, chain_name, config):
    from vfclik_b200.engine import Engine
    chain = _chain(lwr, chain_name)
    return Engine(chain, precision=precision, params=_params(lwr, chain, config)), chain


def _scene(chain, n, Mi, Ms, seed, dtype, ext):
    from vfclik_b200 import workloads
    w = workloads.mixed_scene_batch(chain, n, Mi, Ms, seed, dtype=dtype, obst_ext=ext)
    if ext:                          # per-obstacle {safe, order} across the values the field distinguishes
        rng = np.random.default_rng(seed + 3)
        w["obst_ext"][:, :, 0] = rng.choice(OBST_SAFES[1:], size=(Mi, n))
        w["obst_ext"][:, :, 1] = rng.choice(OBST_ORDERS[:4], size=(Mi, n))      # FP32: clear of the weight limit
        w["shared_obst_ext"][:, 0] = rng.choice(OBST_SAFES[1:], size=Ms)
        w["shared_obst_ext"][:, 1] = rng.choice(OBST_ORDERS[:4], size=Ms)
    return w


def _concat(w, n):
    from vfclik_b200 import workloads
    r = dict(q=w["q"], goal=w["goal"], obst=workloads.concat_scene(w["obst"], w["shared_obst"], n))
    if "obst_ext" in w:
        r["obst_ext"] = workloads.concat_scene(w["obst_ext"], w["shared_obst_ext"], n)
    return r


def _mixed_batch(e, w, Mi, Ms, outputs=()):
    from vfclik_b200.engine import DeviceBatch
    n = w["q"].shape[1]
    db = DeviceBatch(e, n, Mi, obst_ext="obst_ext" in w, outputs=outputs, n_shared_obstacles=Ms)
    db.upload("q", w["q"])
    db.upload("goal", w["goal"])
    if Mi:
        db.upload("obst", w["obst"])
        if "obst_ext" in w:
            db.upload("obst_ext", w["obst_ext"])
    db.upload("shared_obst", w["shared_obst"])
    if "obst_ext" in w:
        db.upload("shared_obst_ext", w["shared_obst_ext"])
    return db


def _plain_batch(e, w, M, outputs=(), shared=False):
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


def _download(db, outputs):
    out = {name: db.download(name) for name in outputs}
    out["q"] = db.download("q")
    return out


def run_mixed(e, w, Mi, Ms, k, outputs):
    db = _mixed_batch(e, w, Mi, Ms, outputs)
    assert db.step(k) == 1
    return _download(db, outputs)


def run_concat(e, w, Mi, Ms, k, outputs):
    db = _plain_batch(e, _concat(w, w["q"].shape[1]), Mi + Ms, outputs)
    assert db.step(k) == 1
    return _download(db, outputs)


# ------------------------------------------------------------------------------------------ 1. step: bit-identity
# (chain, config, Mi, Ms, obst_ext, K, n): every pattern and joint count, lean / general / HIOCC (FP32 K = 1 lean, N <= 7), the
# FP64 order specialisations and pow(), an own ring that is resident (Mi <= 16) and one that streams (Mi = 32), odd Ms,
# Ms < 8 and Ms at the cap (the 17-joint ext case is the largest shared-memory shape), ext rows, partial tiles, K = 1 and 50
STEP_CASES = [
    ("lwr", "lean", 8, 32, False, 1, 1000),
    ("lwr", "lean", 32, 256, False, 50, 1000),
    ("lwr", "order5", 16, 37, False, 50, 1000),
    ("lwr", "order2", 8, 21, False, 1, 1000),
    ("lwr", "order7.5", 8, 21, False, 1, 1000),
    ("lwr", "general", 16, 37, False, 1, 1000),
    ("lwr", "general", 8, 5, True, 50, 1000),
    ("lwr", "lean", 32, 13, True, 50, 1000),
    ("gen6", "lean", 8, 1, False, 1, 1000),
    ("gen6", "general", 32, 7, False, 50, 700),
    ("gen7", "lean", 8, CAP, False, 1, 500),
    ("gen7", "general", 16, CAP, True, 2, 500),
    ("pad8", "general", 8, 40, True, 50, 1000),
    ("pad8", "lean", 32, 40, False, 50, 1000),
    ("dh10", "lean", 16, 24, False, 50, 1000),
    ("gen10", "general", 8, 9, False, 50, 1000),
    ("dh17", "lean", 32, 64, False, 50, 1000),
    ("dh17", "general", 32, CAP, True, 1, 1000),
    ("gen17", "general", 8, 33, False, 1, 1000),
]


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("chain_name,config,Mi,Ms,ext,K,n", STEP_CASES)
def test_step_equals_concatenated_scene(lwr, built_lib, one_thread, precision, chain_name, config, Mi, Ms, ext, K, n):
    e, chain = _engine(lwr, precision, chain_name, config)
    dtype = np.float32 if precision == 32 else np.float64
    w = _scene(chain, n, Mi, Ms, seed=11 + Mi + Ms + K, dtype=dtype, ext=ext)
    outputs = ALL_OUT if config == "general" else ("qdot",)
    got = run_mixed(e, w, Mi, Ms, K, outputs)
    want = run_concat(e, w, Mi, Ms, K, outputs)
    for k in want:
        assert same(got[k], want[k]), (k, np.argwhere(got[k] != want[k])[:5])
    assert np.all(np.isfinite(got["q"]))
    e.close()


# ------------------------------------------------------------------------------------------ 2. other own counts: the oracle
@pytest.mark.parametrize("precision", [64, 32])
@pytest.mark.parametrize("Mi,Ms,ext", [(1, 24, False), (5, 19, True), (13, 8, False)])
def test_step_odd_own_list_against_oracle(lwr, built_lib, precision, Mi, Ms, ext):
    """An own count that is not a multiple of 8 moves the shared list's chunk boundaries against the concatenated list, so
    the sum's rounding differs: both are held to the oracle on [own ; shared]."""
    e, chain = _engine(lwr, precision, "lwr", "general")
    n = 500
    w = _scene(chain, n, Mi, Ms, seed=7 + Mi, dtype=e.np_dtype, ext=ext)
    out = {k: v.T for k, v in run_mixed(e, w, Mi, Ms, 1, ALL_OUT).items()}
    ref = run_oracle(chain, e.params, _concat(w, n), Mi + Ms, k=1)
    check(out, ref, FP64_RTOL if precision == 64 else FP32_RTOL)
    e.close()


# ------------------------------------------------------------------------------------------ 3. degenerate lists
@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("n", [512, 3000])
def test_no_shared_obstacles_is_the_per_instance_call(lwr, built_lib, precision, n):
    """Ms = 0 runs the per-instance dispatch unchanged, including the FP64 cooperative shape at n <= 4096."""
    e, chain = _engine(lwr, precision, "lwr", "lean")
    Mi = 32
    w = _scene(chain, n, Mi, 0, seed=3, dtype=e.np_dtype, ext=False)
    got = run_mixed(e, w, Mi, 0, 3, ("qdot",))
    db = _plain_batch(e, w, Mi, ("qdot",))
    assert db.step(3) == 1
    want = _download(db, ("qdot",))
    for k in want:
        assert same(got[k], want[k]), k
    e.close()


def test_no_shared_obstacles_lane_split(lwr, built_lib):
    """Ms = 0 on the FP64 17-joint DH chain: the lane-split shape of the per-instance dispatch, unchanged."""
    e, chain = _engine(lwr, 64, "dh17", "lean")
    n, Mi = 5000, 16
    w = _scene(chain, n, Mi, 0, seed=4, dtype=e.np_dtype, ext=False)
    got = run_mixed(e, w, Mi, 0, 2, ("qdot",))
    db = _plain_batch(e, w, Mi, ("qdot",))
    assert db.step(2) == 1
    want = _download(db, ("qdot",))
    for k in want:
        assert same(got[k], want[k]), k
    e.close()


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("ext", [False, True])
def test_no_own_obstacles_is_the_shared_call(lwr, built_lib, precision, ext):
    e, chain = _engine(lwr, precision, "lwr", "general")
    n, Ms = 1000, 29
    w = _scene(chain, n, 0, Ms, seed=9, dtype=e.np_dtype, ext=ext)
    got = run_mixed(e, w, 0, Ms, 4, ALL_OUT)
    sw = dict(q=w["q"], goal=w["goal"], obst=w["shared_obst"])
    if ext:
        sw["obst_ext"] = w["shared_obst_ext"]
    db = _plain_batch(e, sw, Ms, ALL_OUT, shared=True)
    assert db.step(4) == 1
    want = _download(db, ALL_OUT)
    for k in want:
        assert same(got[k], want[k]), k
    e.close()


# ------------------------------------------------------------------------------------------ 4. solve: bit-identity
SOLVE_CASES = [                      # (chain, config, Mi, Ms, obst_ext, tolerances, K)
    ("lwr", "lean", 16, 32, False, "mixed", 40),       # resident own ring
    ("lwr", "lean", 32, 32, False, "mixed", 40),       # streaming own ring
    ("lwr", "lean", 32, 21, False, "at_start", 40),
    ("lwr", "lean", 32, 21, False, "never", 40),
    ("lwr", "lean", 24, 9, False, "mixed", 1),
    ("lwr", "general", 8, 21, True, "mixed", 40),
    ("dh17", "lean", 32, 40, False, "mixed", 40),
    ("gen10", "general", 16, 3, False, "mixed", 40),
]
TOLS = {"mixed": (0.01, 0.05), "at_start": (100.0, 4.0), "never": (0.0, 0.0)}


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("chain_name,config,Mi,Ms,ext,tols,K", SOLVE_CASES)
def test_solve_equals_concatenated_scene(lwr, built_lib, one_thread, precision, chain_name, config, Mi, Ms, ext, tols, K):
    e, chain = _engine(lwr, precision, chain_name, config)
    dtype = np.float32 if precision == 32 else np.float64
    n = 900
    w = _scene(chain, n, Mi, Ms, seed=5, dtype=dtype, ext=ext)
    g, _ = near_goal(chain, n, 0, seed=5, dtype=dtype, tool=e.params.tool)    # some start inside the tolerances, some arrive
    w["q"], w["goal"] = g["q"], g["goal"]
    tt, tr = TOLS[tols]
    res = []
    for db in (_mixed_batch(e, w, Mi, Ms), _plain_batch(e, _concat(w, n), Mi + Ms)):
        cycles, dist = db.solve(K, tt, tr)
        res.append(dict(cycles=cycles, dist=dist, q=db.download("q")))
    got, want = res
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


# ------------------------------------------------------------------------------------------ 5. the field query
@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("Mi,Ms,ext", [(5, 11, False), (3, 7, True)])
def test_field_eval_scene(lwr, built_lib, precision, Mi, Ms, ext):
    """vfk_field_eval_scene in every mode against vfk_field_eval on the concatenated / replicated per-instance list (bit for
    bit: both sum one obstacle at a time in the same order), and against the oracle's field."""
    import torch
    from oracle import batch
    from vfclik_b200 import _lib, workloads
    e, chain = _engine(lwr, precision, "lwr", "lean")
    n = 700
    w = _scene(chain, n, Mi, Ms, seed=13, dtype=e.np_dtype, ext=ext)
    q, goal, _ = to_oracle(w, 0)
    R, p, _ = batch.fk_jac(chain, q)
    db = _mixed_batch(e, w, Mi, Ms)
    pose = db.upload("pose", np.concatenate([R.reshape(n, 9), p], axis=1).T)
    sw = dict(q=w["q"], goal=w["goal"], obst=w["shared_obst"])
    if ext:
        sw["obst_ext"] = w["shared_obst_ext"]
    sdb = _plain_batch(e, sw, Ms, shared=True)
    cases = [                         # (bufs, n_obstacles, per-instance equivalent)
        ({k: v for k, v in db.bufs.items() if k not in ("obst_shared", "shared_obst", "shared_obst_ext", "n_shared_obst")}, Mi,
         {k: w[k] for k in ("q", "goal", "obst", "obst_ext") if k in w}),
        (sdb.bufs, Ms, dict(sw, obst=workloads.replicate_scene(sw["obst"], n),
                             **({"obst_ext": workloads.replicate_scene(sw["obst_ext"], n)} if ext else {}))),
        (db.bufs, Mi, _concat(w, n)),
    ]
    for mode, (bufs, m, per) in enumerate(cases):
        assert bufs.get("obst_shared", 0) == mode
        tw = e.alloc(6, n)
        assert e.field_eval_scene(pose, bufs, tw, n, m) == 1
        ref_db = _plain_batch(e, per, per["obst"].shape[0])
        tw_ref = e.alloc(6, n)
        assert e.field_eval(pose, ref_db.t["goal"], ref_db.t["obst"], tw_ref, n, per["obst"].shape[0],
                            obst_ext=ref_db.t.get("obst_ext")) == 1
        torch.cuda.synchronize()
        assert torch.equal(tw, tw_ref), mode
        _, _, obst = to_oracle(per, per["obst"].shape[0])
        v, om = batch.field_eval(oracle_params(e.params), R, p, goal, obst)
        got = tw.permute(1, 0, 2).reshape(6, -1)[:, :n].cpu().numpy().T.astype(np.float64)
        want = np.concatenate([v, om], axis=1)
        tol = 1e-9 if precision == 64 else 1e-4
        assert np.allclose(got, want, rtol=tol, atol=tol * max(1.0, float(np.max(np.abs(want))))), mode
    assert _lib.VFK_OBST_MIXED == 2
    e.close()


# ------------------------------------------------------------------------------------------ 6. host-buffer session
def _pinned(shape, dtype):
    import torch
    return torch.zeros(shape, dtype={np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32}[dtype]).pin_memory().numpy()


def _session(e, w, Mi, Ms, mixed, n):
    """A session holding the mixed scene (mode 2) or the concatenated per-instance scene."""
    ext = "obst_ext" in w
    if mixed:
        s = e.session(n, Mi, obst_ext=ext)
        s.set_obstacles(w["obst"], w.get("obst_ext"))
        s.set_shared_obstacles(w["shared_obst"], w.get("shared_obst_ext"))
        s.use_obstacles(2)
    else:
        c = _concat(w, n)
        s = e.session(n, Mi + Ms, obst_ext=ext)
        s.set_obstacles(c["obst"], c.get("obst_ext"))
    s.set_goal(w["goal"])
    return s


def _cycles(s, e, w, n, path, calls=3, k=3):
    """Three vfk_session_cycle calls (chunked path: eager, graph capture, graph replay) -> the outputs of each."""
    N, dt = e.n_joints, e.np_dtype
    mk = _pinned if path == "direct" else (lambda shape, d: np.zeros(shape, dtype=d))
    q_in, qdot, q_out, flags = mk((N, n), dt), mk((N, n), dt), mk((N, n), dt), mk((n,), np.int32)
    q_in[...] = w["q"]
    outs = []
    for _ in range(calls):
        s.cycle(q_in, k, qdot_out=qdot, q_out=q_out, flags_out=flags)
        outs.append((qdot.copy(), q_out.copy(), flags.copy()))
        q_in[...] = q_out
    return outs


@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("path", ["direct", "chunked"])
def test_session_equals_concatenated_scene(lwr, built_lib, one_thread, precision, path):
    """Direct host I/O (page-locked, tile-aligned batch) and the chunked copy pipeline (pageable, two chunks, a partial last
    tile): the chunk views must offset the own list and keep the shared list whole."""
    e, chain = _engine(lwr, precision, "lwr", "lean")
    n, Mi, Ms = (4096, 16, 21) if path == "direct" else (2 * 65536 + 40, 8, 19)
    w = _scene(chain, n, Mi, Ms, seed=23, dtype=e.np_dtype, ext=False)
    got = _cycles(_session(e, w, Mi, Ms, True, n), e, w, n, path)
    want = _cycles(_session(e, w, Mi, Ms, False, n), e, w, n, path)
    for c, (a, b) in enumerate(zip(got, want)):
        for name, x, y in zip(("qdot", "q", "flags"), a, b):
            assert same(x, y), (c, name)
    e.close()


@pytest.mark.parametrize("precision", [32, 64])
def test_session_solve_equals_concatenated_scene(lwr, built_lib, one_thread, precision):
    e, chain = _engine(lwr, precision, "lwr", "lean")
    n, Mi, Ms, K = 3000, 16, 27, 40
    w = _scene(chain, n, Mi, Ms, seed=31, dtype=e.np_dtype, ext=True)
    g, _ = near_goal(chain, n, 0, seed=31, dtype=e.np_dtype)
    w["q"], w["goal"] = g["q"], g["goal"]
    res = []
    for mixed in (True, False):
        s = _session(e, w, Mi, Ms, mixed, n)
        q, cyc, dist = np.zeros((e.n_joints, n), e.np_dtype), np.zeros(n, np.int32), np.zeros((2, n), e.np_dtype)
        s.solve(w["q"], K, 0.01, 0.05, q_out=q, cycles_out=cyc, dist_out=dist)
        res.append((q, cyc, dist))
    for x, y in zip(*res):
        assert same(x, y)
    assert np.count_nonzero(res[0][1] >= 0) > 0
    e.close()


def test_session_switches_modes(lwr, built_lib, one_thread):
    """0 -> 2 -> 1 -> 0 on one session, each against a session holding the equivalent per-instance scene; the setters keep
    their side effects (set_obstacles selects mode 0, set_shared_obstacles mode 1), and vfk_session_buffers reports the mode."""
    from vfclik_b200 import _lib, workloads
    e, chain = _engine(lwr, 64, "lwr", "lean")
    n, Mi, Ms = 2048, 8, 13
    w = _scene(chain, n, Mi, Ms, seed=37, dtype=e.np_dtype, ext=False)
    s = e.session(n, Mi)
    s.set_goal(w["goal"])

    def mode():
        b = _lib.BuffersC()
        assert e._lib.vfk_session_buffers(s._s, C.byref(b)) == _lib.VFK_OK
        return b.obst_shared

    def run(sess):
        out = np.zeros((e.n_joints, n), e.np_dtype)
        sess.cycle(w["q"], 2, qdot_out=out)
        return out

    def ref(obst):
        r = e.session(n, obst.shape[0])
        r.set_goal(w["goal"])
        r.set_obstacles(obst)
        return run(r)

    s.set_obstacles(w["obst"])
    assert mode() == 0 and same(run(s), ref(w["obst"]))
    s.set_shared_obstacles(w["shared_obst"])
    assert mode() == 1                                              # set_shared_obstacles selects the shared list
    s.use_obstacles(2)
    assert mode() == 2 and same(run(s), ref(workloads.concat_scene(w["obst"], w["shared_obst"], n)))
    s.use_obstacles(1)
    assert mode() == 1 and same(run(s), ref(workloads.replicate_scene(w["shared_obst"], n)))
    s.use_obstacles(0)
    assert mode() == 0 and same(run(s), ref(w["obst"]))
    s.use_obstacles(2)
    s.set_obstacles(w["obst"])                                      # set_obstacles selects the per-instance list
    assert mode() == 0
    e.close()


# ------------------------------------------------------------------------------------------ 7. refusals
def test_mixed_scene_refusals(lwr, built_lib):
    import torch
    from vfclik_b200 import _lib
    from vfclik_b200.engine import VfkError
    e, chain = _engine(lwr, 32, "lwr", "lean")
    n, Mi, Ms = 64, 8, 8
    db = _mixed_batch(e, _scene(chain, n, Mi, Ms, 3, np.float32, True), Mi, Ms, outputs=("qdot",))
    big = torch.zeros((CAP + 1, 4), dtype=torch.float32, device="cuda")
    cyc = e.alloc(1, n, dtype=torch.int32)
    bufs = db.bufs
    sh, she = bufs["shared_obst"], bufs["shared_obst_ext"]

    def code(fn, *args, **kw):
        with pytest.raises(VfkError) as ei:
            fn(*args, **kw)
        return ei.value.code

    def raw(fn, bufs, **fields):           # set BuffersC fields the Python layer does not expose
        b = e._buffers(bufs, (None, None, None), None)
        for k, v in fields.items():
            setattr(b, k, v)
        return fn(b)

    step = lambda b: e._lib.vfk_step(e._h, C.byref(b), n, Mi, 1, None)
    solve = lambda b: e._lib.vfk_solve(e._h, C.byref(b), n, Mi, 5, 0.01, 0.05, cyc.data_ptr(), None, None)
    solve_bufs = {k: v for k, v in bufs.items() if k != "qdot"}
    for fn, b0 in ((step, bufs), (solve, solve_bufs)):
        assert raw(fn, b0, obst_shared=3) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0, n_shared_obst=-1) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0, reserved2=1) == _lib.VFK_ERR_INVALID
        assert raw(fn, dict(b0, shared_obst=big), n_shared_obst=CAP + 1) == _lib.VFK_ERR_UNSUPPORTED
        assert raw(fn, b0, shared_obst=None) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0, shared_obst=None, n_shared_obst=0) == _lib.VFK_ERR_INVALID     # mode 2 always names its list
        assert raw(fn, b0, shared_obst=sh.data_ptr() + 16) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0, shared_obst_ext=she.data_ptr() + 16) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0, shared_obst_ext=None) == _lib.VFK_ERR_INVALID                  # ext rows: both lists or neither
        assert raw(fn, b0, obst_ext=None) == _lib.VFK_ERR_INVALID
        assert raw(fn, b0) >= 1                                                          # the batch itself is accepted
        assert raw(fn, dict(b0, shared_obst=big), n_shared_obst=CAP, shared_obst_ext=None, obst_ext=None) >= 1
    torch.cuda.synchronize()
    tw = e.alloc(6, n)
    pose = e.alloc(12, n)
    assert code(e.field_eval_scene, pose, dict(bufs, obst_shared=3), tw, n, Mi) == _lib.VFK_ERR_INVALID
    assert code(e.field_eval_scene, pose, bufs, tw, n, Mi, n_shared_obstacles=CAP + 1) == _lib.VFK_ERR_UNSUPPORTED
    assert code(e.field_eval_scene, pose, dict(bufs, shared_obst=None), tw, n, Mi) == _lib.VFK_ERR_INVALID
    # sessions
    s0 = e.session(n, 0)
    assert code(s0.use_obstacles, 1) == _lib.VFK_ERR_INVALID         # no shared list yet
    s0.set_shared_obstacles(np.zeros((3, 4)))
    assert code(s0.use_obstacles, 2) == _lib.VFK_ERR_INVALID         # created without a per-instance scene
    assert code(s0.use_obstacles, 3) == _lib.VFK_ERR_INVALID
    assert code(s0.use_obstacles, -1) == _lib.VFK_ERR_INVALID
    s0.use_obstacles(1)
    s1 = e.session(n, Mi, obst_ext=True)
    assert code(s1.use_obstacles, 2) == _lib.VFK_ERR_INVALID         # no shared list yet
    s1.set_shared_obstacles(np.zeros((3, 4)))
    assert code(s1.use_obstacles, 2) == _lib.VFK_ERR_INVALID         # the shared list has no ext rows
    s1.set_shared_obstacles(np.zeros((3, 4)), np.ones((3, 2)))
    s1.use_obstacles(2)
    assert e._lib.vfk_session_use_obstacles(None, 0) == _lib.VFK_ERR_INVALID
    e.close()
