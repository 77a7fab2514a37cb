"""Which cycle kernel each call runs.

The HIOCC, lean and general instantiations of the cycle kernel give the same bits, and the cooperative and lane-split
shapes match the one-thread kernel too, so a call routed to the wrong instantiation passes every parity test and only
shows in its time.  Each case here runs one call under torch.profiler and checks the template arguments
<T, N, PAT, EXT, LEAN, MINB, G, SOLVE, SHARED> of the cycle kernel it launched (or that it launched the lane-split kernel),
and the launch count the call returns.
"""
import re

import pytest

CYCLE_FIELDS = ("T", "N", "PAT", "EXT", "LEAN", "MINB", "G", "SOLVE", "SHARED")
_MANGLED = re.compile(r"vfk_cycle_kernelI([fd])Li(\d+)ENS_\d+(\w+?Pattern)ELb([01])ELb([01])ELi(\d+)ELi(\d+)ELb([01])ELb([01])E")
_DEMANGLED = re.compile(r"vfk_cycle_kernel<([^<>]*)>")


def _bool(s):
    return {"true": True, "1": True, "false": False, "0": False}[s.strip()]


def parse_kernel(name):
    """A profiler kernel name -> ("split",), a dict of the cycle kernel's template arguments, or None."""
    if "vfk_split_kernel" in name:
        return ("split",)
    m = _MANGLED.search(name)
    if m:
        t, n, pat, ext, lean, minb, g, solve, shared = m.groups()
        vals = ({"f": "float", "d": "double"}[t], int(n), pat, ext == "1", lean == "1", int(minb), int(g), solve == "1",
                shared == "1")
        return dict(zip(CYCLE_FIELDS, vals))
    m = _DEMANGLED.search(name)
    if m:
        args = [a.strip() for a in m.group(1).split(",")]
        assert len(args) == 9, "unexpected cycle-kernel name %r" % name
        vals = (args[0], int(args[1]), args[2].split("::")[-1], _bool(args[3]), _bool(args[4]), int(args[5]), int(args[6]),
                _bool(args[7]), _bool(args[8]))
        return dict(zip(CYCLE_FIELDS, vals))
    assert "vfk_cycle_kernel" not in name, "cannot parse the cycle kernel's template arguments from %r" % name
    return None


def launched(call):
    """Run call() under the profiler; returns (its return value, the cycle / split kernels it launched)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = call()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [k for k in map(parse_kernel, names) if k is not None]
    assert kernels, "no cycle-kernel launch recorded; vfk kernels seen: %r" % sorted({x for x in names if "vfk" in x})
    return rc, kernels


def test_parse_kernel_names():
    a = parse_kernel("void vfk::vfk_cycle_kernel<float, 7, vfk::LwrPattern, false, true, 4, 1, false, false>"
                     "(vfk::KConst<float>, vfk::KArgs<float>)")
    b = parse_kernel("_ZN3vfk16vfk_cycle_kernelIfLi7ENS_10LwrPatternELb0ELb1ELi4ELi1ELb0ELb0EEEvNS_6KConstIT_EENS_5KArgsIS3_EE")
    assert a == b == dict(T="float", N=7, PAT="LwrPattern", EXT=False, LEAN=True, MINB=4, G=1, SOLVE=False, SHARED=False)
    assert parse_kernel("void vfk::vfk_split_kernel<double, 17>(vfk::KConst<double>, vfk::KArgs<double>, vfk::SplitMaps)") == ("split",)
    assert parse_kernel("void vfk::vfk_pack_kernel<float>(float const*, long, float*, int, long, long)") is None


def _chain(lwr, name):
    from vfclik_b200 import workloads
    return {"lwr": lambda: lwr[0], "pad5": lambda: workloads.dual_arm_torso_chain(5),
            "dh10": lambda: workloads.dual_arm_torso_chain(10), "dh17": lambda: workloads.dual_arm_torso_chain(17)}[name]()


def _engine(lwr, chain_name, precision):
    from vfclik_b200.engine import Engine, Params
    chain = _chain(lwr, chain_name)
    params = Params.from_config(lwr[1]) if chain_name == "lwr" else Params()
    return Engine(chain, precision=precision, params=params), chain


def _batch(e, chain, n, M, mode=0, Ms=0, ext=False, outputs=("qdot",)):
    """A DeviceBatch with random starts, goals and obstacles: mode 0 per instance (M each), 1 one shared list of M, 2 M own
    plus Ms shared."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    dt = e.np_dtype
    if mode == 1:
        w = workloads.shared_scene_batch(chain, n, M, seed=5, dtype=dt, obst_ext=ext)
        db = DeviceBatch(e, n, M, obst_ext=ext, outputs=outputs, shared_obstacles=True)
    elif mode == 2:
        w = workloads.mixed_scene_batch(chain, n, M, Ms, seed=5, dtype=dt, obst_ext=ext)
        db = DeviceBatch(e, n, M, obst_ext=ext, outputs=outputs, n_shared_obstacles=Ms)
    else:
        w = workloads.random_batch(chain, n, M, seed=5, dtype=dt, obst_ext=ext)
        db = DeviceBatch(e, n, M, obst_ext=ext, outputs=outputs)
    for k in ("q", "goal", "obst", "obst_ext", "shared_obst", "shared_obst_ext"):
        if k in w and (M > 0 or k not in ("obst", "obst_ext")) and (Ms > 0 or not k.startswith("shared_")):
            db.upload(k, w[k])
    return db


def _cycle(T, N, PAT, EXT=False, LEAN=False, MINB=3, G=1, SOLVE=False, SHARED=False):
    return dict(T=T, N=N, PAT=PAT, EXT=EXT, LEAN=LEAN, MINB=MINB, G=G, SOLVE=SOLVE, SHARED=SHARED)


# (id, chain, precision, n, M, mode, Ms, ext, outputs, K, solve, environment, expected kernel)
CASES = [
    ("f32-lwr-lean-k1", "lwr", 32, 8192, 16, 0, 0, False, ("qdot",), 1, False, {},
     _cycle("float", 7, "LwrPattern", LEAN=True, MINB=4)),
    ("f32-lwr-lean-k10", "lwr", 32, 8192, 16, 0, 0, False, ("qdot",), 10, False, {},
     _cycle("float", 7, "LwrPattern", LEAN=True, MINB=3)),
    ("f32-lwr-pose", "lwr", 32, 8192, 16, 0, 0, False, ("qdot", "pose"), 1, False, {},
     _cycle("float", 7, "LwrPattern", MINB=3)),
    ("f32-lwr-ext", "lwr", 32, 8192, 16, 0, 0, True, ("qdot",), 1, False, {},
     _cycle("float", 7, "LwrPattern", EXT=True, MINB=3)),
    ("f32-pad5", "pad5", 32, 8192, 16, 0, 0, False, ("qdot",), 1, False, {},
     _cycle("float", 6, "GenericPattern", MINB=3)),
    ("f32-dh10", "dh10", 32, 8192, 16, 0, 0, False, ("qdot",), 1, False, {},
     _cycle("float", 10, "DhPattern", LEAN=True, MINB=3)),
    ("f64-coop", "lwr", 64, 1024, 16, 0, 0, False, ("qdot",), 1, False, {},
     _cycle("double", 7, "LwrPattern", MINB=2, G=8)),
    ("f64-no-coop", "lwr", 64, 1024, 16, 0, 0, False, ("qdot",), 1, False, {"VFK_NO_COOP": "1"},
     _cycle("double", 7, "LwrPattern", LEAN=True, MINB=2)),
    ("f64-dh17-split", "dh17", 64, 8192, 16, 0, 0, False, ("qdot",), 1, False, {}, ("split",)),
    ("f64-dh17-no-split", "dh17", 64, 8192, 16, 0, 0, False, ("qdot",), 1, False, {"VFK_NO_SPLIT": "1"},
     _cycle("double", 17, "DhPattern", LEAN=True, MINB=1)),
    ("solve-f64-dh17", "dh17", 64, 8192, 16, 0, 0, False, (), 20, True, {},
     _cycle("double", 17, "DhPattern", LEAN=True, MINB=1, SOLVE=True)),
    ("solve-f32-lwr", "lwr", 32, 8192, 16, 0, 0, False, (), 20, True, {},
     _cycle("float", 7, "LwrPattern", LEAN=True, MINB=3, SOLVE=True)),
    ("shared-on-coop-shape", "lwr", 64, 1024, 16, 1, 0, False, ("qdot",), 1, False, {},
     _cycle("double", 7, "LwrPattern", LEAN=True, MINB=2, SHARED=True)),
    ("shared-empty", "lwr", 64, 1024, 0, 1, 0, False, ("qdot",), 1, False, {},
     _cycle("double", 7, "LwrPattern", LEAN=True, MINB=2)),
    ("mixed-no-shared-coop", "lwr", 64, 1024, 16, 2, 0, False, ("qdot",), 1, False, {},
     _cycle("double", 7, "LwrPattern", MINB=2, G=8)),
    ("mixed-ext", "lwr", 32, 8192, 8, 2, 13, True, ("qdot",), 1, False, {},
     _cycle("float", 7, "LwrPattern", EXT=True, MINB=3, SHARED=True)),
    ("shared-solve-f32-lwr", "lwr", 32, 8192, 16, 1, 0, False, (), 20, True, {},
     _cycle("float", 7, "LwrPattern", LEAN=True, MINB=4, SOLVE=True, SHARED=True)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_route(lwr, built_lib, monkeypatch, case):
    _, chain_name, precision, n, M, mode, Ms, ext, outputs, K, solve, env, want = case
    for k in ("VFK_NO_COOP", "VFK_NO_SPLIT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    e, chain = _engine(lwr, chain_name, precision)
    db = _batch(e, chain, n, M, mode, Ms, ext, outputs)
    if solve:
        cycles = db._ensure("cycles")
        call = lambda: e.solve(db.bufs, n, M, K, 1e-3, 1e-2, cycles)      # noqa: E731
    else:
        call = lambda: db.step(K)                                         # noqa: E731
    call()                                                                # warm: plan caches, module load
    rc, kernels = launched(call)
    assert kernels == [want]
    assert rc == 1
    e.close()


@pytest.mark.gpu
def test_route_session_direct(lwr, built_lib, monkeypatch):
    """A session cycle on the direct host I/O path runs the one-thread kernel, not the lane-split shape it would take from
    device buffers, in a single launch."""
    import torch
    from vfclik_b200 import workloads
    for k in ("VFK_NO_COOP", "VFK_NO_SPLIT", "VFK_SESSION_DIRECT"):
        monkeypatch.delenv(k, raising=False)
    e, chain = _engine(lwr, "dh17", 64)
    n, M = 2048, 8
    w = workloads.random_batch(chain, n, M, seed=5)
    s = e.session(n, M)
    s.set_goal(w["goal"])
    s.set_obstacles(w["obst"])
    q_in = torch.from_numpy(w["q"]).pin_memory().numpy()
    qd = torch.zeros((chain.n_joints, n), dtype=torch.float64).pin_memory().numpy()
    s.cycle(q_in, 1, qdot_out=qd)
    rc, kernels = launched(lambda: s.cycle(q_in, 1, qdot_out=qd))
    assert rc == 1
    assert kernels == [_cycle("double", 17, "DhPattern", LEAN=True, MINB=1)]
    s.close()
    e.close()
