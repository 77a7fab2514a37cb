"""CPU tests of the host-side logic: config loading, chain folding, ports, launcher CLI, sharding (gloo, world 2)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_chain_folds_fixed_segments(lwr):
    chain, cfg = lwr
    assert chain.n_joints == cfg.nJoints == 7
    assert np.allclose(chain.base[9:12], [0.25, 0.0, 0.45 + 0.31])        # mounting * 0.31 m column
    assert np.all(chain.joint_type == 3)                                  # all RotZ
    assert np.allclose(chain.tip[1, 9:12], [0.0, 0.4, 0.0]) and np.allclose(chain.tip[6, 9:12], [0, 0, 0.078])
    assert np.allclose(np.rad2deg(chain.q_hi), [170, 120, 170, 120, 170, 120, 170])


def test_kdl_frame_algebra_matches_conventions():
    from vfclik_b200 import kdl
    a = kdl.Frame(kdl.Rotation.RotZ(0.3), kdl.Vector(1, 2, 3))
    b = kdl.Frame(kdl.Rotation.RotX(-0.7), kdl.Vector(-1, 0.5, 0.25))
    c = a * b
    A = np.eye(4); A[:3, :3] = np.asarray(a.M.m).reshape(3, 3); A[:3, 3] = a.p.v
    B = np.eye(4); B[:3, :3] = np.asarray(b.M.m).reshape(3, 3); B[:3, 3] = b.p.v
    assert np.allclose(np.asarray(c.to_list16()).reshape(4, 4), A @ B)
    assert kdl.Frame.from_list16(c.to_list16()).to_list12() == c.to_list12()
    f = kdl.Frame.DH_Craig1989(0.1, np.pi / 2, 0.4, 0.0)
    assert f.M.m == [1, 0, 0, 0, 0, -1, 0, 1, 0] and np.allclose(f.p.v, [0.1, -0.4, 0.0])


def test_config_errors(tmp_path):
    from vfclik_b200.config import load_config
    with pytest.raises(FileNotFoundError):
        load_config(str(tmp_path / "config-none-right.py"))
    bad = tmp_path / "config-bad-right.py"
    bad.write_text("nJoints = 7\n")
    with pytest.raises(AttributeError):
        load_config(str(bad))


def test_ports_latest_value_and_strict_queue():
    from vfclik_b200 import ports as yarp
    yarp.Network.reset()
    out = yarp.BufferedPortBottle(); out.open("/a/out")
    latest = yarp.BufferedPortBottle(); latest.open("/b/in")
    strict = yarp.BufferedPortBottle(); strict.open("/c/in"); strict.setStrict(True)
    assert yarp.Network.connect("/a/out", "/b/in") and yarp.Network.connect("/a/out", "/c/in")
    for k in range(3):
        yarp.sendListPort(out, [k, k + 0.5])
    assert yarp.readListPort(latest) == [2.0, 2.5] and latest.read(False) is None       # newest only, once
    assert [yarp.readListPort(strict) for _ in range(3)] == [[0.0, 0.5], [1.0, 1.5], [2.0, 2.5]]
    with pytest.raises(RuntimeError):
        strict.read(True)                                                                # would block forever
    # nested bottles: ("add", id, force, type, (params...))  scripts/vf:226-266
    yarp.write_bottle_lists(out, ["add", 1, 1.0, 1, [0.0] * 17])
    b = strict.read(False)
    assert b.size() == 5 and b.get(0).toString() == "add" and b.get(1).asInt() == 1 and b.get(4).asList().size() == 17
    assert b.get(2).isDouble() and b.get(3).isInt() and not b.get(0).isInt()
    yarp.Network.reset()


def test_arcosyarp_naming_and_readiness():
    from vfclik_b200 import ports as yarp
    yarp.Network.reset()
    a = yarp.ArcosYarp(ports_name_prefix="/0", module_name_prefix="/lwr/right/vectorField")
    b = yarp.ArcosYarp(ports_name_prefix="/0", module_name_prefix="/lwr/right/bridge")
    qdot = a.create_yarp_port("/qdotOut", input_port=False)
    assert qdot.getName() == "/0/lwr/right/vectorField/qdotOut"
    a.connect(qdot, "/lwr/right/bridge", "/vectorfieldcmd")
    assert not a.is_ready()                                  # remote port does not exist yet
    cmd = b.create_yarp_port("/vectorfieldcmd", strict=False)
    assert a.is_ready()
    yarp.sendListPort(qdot, [1, 2, 3])
    assert yarp.readListPort(cmd) == [1.0, 2.0, 3.0]
    yarp.Network.reset()


def test_weight_bottle_parsing():
    from vfclik_b200 import ports as yarp
    from vfclik_b200.vf import get_weight_matrix, list16_to_pose12, pose12_to_list16
    b = yarp.Bottle.from_list(["t", 1.0, 1.0, 1.0, 0.5, 0.5, 0.5])
    assert get_weight_matrix(b, 6) == [1.0, 1.0, 1.0, 0.5, 0.5, 0.5]
    assert get_weight_matrix(b, 7) is None                   # wrong size -> ignored (scripts/vf:176-179)
    p12 = list(range(12))
    assert list16_to_pose12(pose12_to_list16(p12)) == p12


def test_launcher_cli(tmp_path):
    from vfclik_b200 import launcher
    opts, _ = launcher.build_parser().parse_args([])
    assert (opts.robot, opts.instance, opts.namespace, opts.config_dir, opts.sim, opts.no_nullspace) == \
        ("lwr", "right", "/0", "../config_data/lwr/", False, False)
    opts, _ = launcher.build_parser().parse_args(["-r", "icub", "-i", "left", "-n", "/1", "-d", "/x/", "-s", "--no_nullspace"])
    assert (opts.robot, opts.instance, opts.namespace, opts.config_dir, opts.sim, opts.no_nullspace) == \
        ("icub", "left", "/1", "/x/", True, True)
    r = subprocess.run([sys.executable, "-m", "vfclik_b200.launcher", "-d", str(tmp_path) + "/", "-r", "nope"], cwd=ROOT,
                       capture_output=True, text=True)
    assert r.returncode == 255 and "not found, exiting" in r.stdout       # sys.exit(-1) (scripts/vfclik:83-85)


def test_shard_range_partitions_exactly():
    from vfclik_b200.distributed import shard_range
    for n, w in ((16 << 20, 8), (1000, 3), (5, 8), (0, 2)):
        ranges = [shard_range(n, r, w) for r in range(w)]
        assert ranges[0][0] == 0 and ranges[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        sizes = [e - b for b, e in ranges]
        assert max(sizes) - min(sizes) <= 1


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from vfclik_b200.distributed import reduce_stats, shard_range
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
b, e = shard_range(1000, r, w)
stats = reduce_stats({"inst_cycles": float(e - b) * 10, "elapsed_ms_max": 1.0 + r, "err_max": 1e-9 * (r + 1), "t_min": 5.0 - r})
if r == 0:
    print("RESULT", stats["inst_cycles"], stats["elapsed_ms_max"], stats["err_max"], stats["t_min"])
dist.destroy_process_group()
"""


def test_stats_reduction_world_size_2_gloo(tmp_path):
    """The N > 1 host path (shard ranges + the final all_reduce) on CPU with the gloo backend."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29577", str(script), ROOT], capture_output=True, text=True, env=env,
                       timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split()
    assert [float(x) for x in line[1:]] == [10000.0, 2.0, 2e-9, 4.0]


def test_module_command_lines_follow_the_launcher_contract(tmp_path, capsys):
    """scripts/vfclik:88-105 starts every module as `<module> -c <config> -n <namespace>` (bridge adds -s); the parser
    keeps arcospyu's ConfigFileParser surface: .parser.add_option(...) and .get_all() -> (options, args, config)."""
    import importlib
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, config_filename
    from vfclik_b200.module_cli import ConfigFileParser
    cfgfile = config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right")
    cp = ConfigFileParser(["bridge", "-c", cfgfile, "-s", "-n", "/7"])
    cp.parser.add_option("-s", "--simulation", action="store_true", dest="sim", default=False, help="Simulation")
    options, args, config = cp.get_all()
    assert options.namespace == "/7" and options.sim is True and args == [] and config.nJoints == 7
    assert ConfigFileParser(["vf", "-c", cfgfile]).get_all()[0].namespace == ""
    with pytest.raises(SystemExit):
        ConfigFileParser(["vf", "-n", "/0"]).get_all()               # no config file
    with pytest.raises(FileNotFoundError):
        ConfigFileParser(["vf", "-c", str(tmp_path / "missing.py")]).get_all()
    for mod in ("vf", "nullspace", "joint_p_controller", "bridge", "object_feeder", "monitor_distance", "launcher"):
        assert callable(importlib.import_module("vfclik_b200." + mod).main), mod
    # a module that needs no GPU runs stand-alone: the feeder publishes config.initial_vf_pose and stops after --cycles
    from vfclik_b200 import object_feeder
    assert object_feeder.main(["object_feeder", "-c", cfgfile, "-n", "/7", "--cycles", "2", "--no_sleep"]) == 0
    assert "iterations: 2" in capsys.readouterr().out


def test_object_feeder_parses_the_reference_example_bottles(capsys):
    """The only input fixtures the reference ships are the example bottles of old/README.old:69-78; fed verbatim through the
    feeder they must come out as the field messages of scripts/object_feeder:229-354 (ids, forces, vfl types, layouts)."""
    from vfclik_b200 import ports as yarp
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, config_filename, load_config
    from vfclik_b200.object_feeder import ObjectFeederModule
    yarp.Network.reset()
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    del cfg.initial_vf_pose                                   # no automatic first goal: the examples set it
    fd = ObjectFeederModule(cfg, "/t")
    sink = yarp.BufferedPortBottle(); sink.open("/t/sink"); sink.setStrict(True)
    yarp.Network.connect(fd.paramPort.getName(), "/t/sink")
    src = yarp.BufferedPortBottle(); src.open("/t/src")
    yarp.Network.connect("/t/src", fd.objectPort.getName())

    def send(*items):
        yarp.write_bottle_lists(src, list(items), strict=True)
        assert fd.update()
        out = []
        while True:
            b = sink.read(False)
            if b is None:
                return out
            row = [b.get(0).asString(), b.get(1).asInt()]
            if row[0] == "add":
                pl = b.get(4).asList()
                row += [b.get(2).asDouble(), b.get(3).asInt(), [pl.get(i).asDouble() for i in range(pl.size())]]
            out.append(row)

    try:
        # an obstacle before any goal is stored but not sent (scripts/object_feeder:216-219)
        obst = [1, 0, 0, 0.0, 0, 1, 0, -0.4, 0, 0, 1, 0.4, 0, 0, 0, 1, 0.05, 20]               # old/README.old:75
        assert send("set", "ObstacleP", 0, [float(v) for v in obst]) == []
        assert "waiting for a goal" in capsys.readouterr().out
        goal = [0, 1, 0, 0, -1, 0, 0, 0.3, 0, 0, 1, 1.1, 0, 0, 0, 1, 0.1]                      # old/README.old:69
        msgs = send("set", "goal", [float(v) for v in goal])
        assert msgs[0] == ["add", 1, 1.0, 1, [float(v) for v in goal]]
        assert msgs[1:3] == [["remove", 2], ["remove", 3]]                                       # no funnel, no near-goal repeller
        assert msgs[3] == ["add", 5, -10.0, 2, [0.0, -0.4, 0.4, 0.05, 0.001, 20.0]]              # id 4 + (n + 1), xyz, radius, safe, order
        table = [1, 0, 0, 0, 0, 1, 0, -0.4, 0, 0, 1, 0.3, 0, 0, 0, 1, 0, 0, 1, 0.001, 5]       # old/README.old:78
        msgs = send("set", "ObstacleH", 1, [float(v) for v in table])
        assert msgs[-1] == ["add", 6, -50.0, 4, [0.0, -0.4, 0.3, 0.0, 0.0, 1.0, 0.001, 5.0]]
        gan = [1, 0, 0, 0.4, 0, -1, 0, -0.4, 0, 0, -1, 0.4, 0, 0, 0, 1, 0, -1, 0, 0.1, 0.15, 0.15]   # old/README.old:72-73
        msgs = send("set", "goalAndNormal", [float(v) for v in gan])
        assert msgs[0] == ["add", 1, 1.0, 1, [float(v) for v in gan[:16]] + [0.15]]              # frame + slowdown (last value)
        assert msgs[1] == ["add", 2, 30.0, 5, [0.4, -0.4, 0.4, 0.0, -1.0, 0.0, 0.1, 10.0, 0.15, 2.0]]      # funnel
        assert msgs[2][:4] == ["add", 3, -10.0, 2] and np.allclose(msgs[2][4], [0.4, -0.45, 0.4, 0.2, 0.001, 5.0])   # near-goal repeller
        # wrong lengths are reported and ignored; unknown actions too
        send("set", "goal", [1.0, 2.0, 3.0])
        send("fly", "goal", [1.0])
        text = capsys.readouterr().out
        assert "Wrong number of values, expected 16" in text and "Action not recognized" in text
        assert send("remove", 0)[0] == ["remove", 5]
        send("remove", 7)
        assert "Object doesn't exist" in capsys.readouterr().out
    finally:
        fd.close(); sink.close(); src.close(); yarp.Network.reset()


def test_object_feeder_matches_the_reference_loop_message_for_message(golden, capsys):
    """tests/golden holds what scripts/object_feeder's own loop body (:93-359), executed by oracle/gen_golden.py:gen_feeder,
    wrote to /param and /objectOut for a scripted message sequence (the README examples, default slowdown, wrong lengths,
    removals, an unknown action).  The host module must write exactly the same messages in the same order."""
    import json
    from vfclik_b200 import ports as yarp
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, config_filename, load_config
    from vfclik_b200.object_feeder import ObjectFeederModule
    yarp.Network.reset()
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    del cfg.initial_vf_pose
    fd = ObjectFeederModule(cfg, "/g")
    sinks = {}
    for name, port in (("param", fd.paramPort), ("objectOut", fd.objectOutPort)):
        p = yarp.BufferedPortBottle(); p.open("/g/sink_" + name); p.setStrict(True)
        yarp.Network.connect(port.getName(), "/g/sink_" + name)
        sinks[name] = p
    src = yarp.BufferedPortBottle(); src.open("/g/src")
    yarp.Network.connect("/g/src", fd.objectPort.getName())
    try:
        for msg, want in zip(golden["feeder_script"], golden["feeder_out"]):
            yarp.write_bottle_lists(src, json.loads(str(msg)), strict=True)
            assert fd.update()
            got = {}
            for name, p in sinks.items():
                got[name] = []
                while True:
                    b = p.read(False)
                    if b is None:
                        break
                    got[name].append(b.to_list())
            assert got == json.loads(str(want)), str(msg)
    finally:
        fd.close(); src.close()
        for p in sinks.values():
            p.close()
        yarp.Network.reset()
    capsys.readouterr()


def test_handlers_send_what_the_reference_handlers_send(golden, capsys):
    """Row f3: every sender of HandleArmNew / HandleArm / HandleBridge / HandleJController, called with the same arguments as
    the reference's own src/handlers.py was when it was executed for tests/golden (oracle/gen_golden.py:gen_handlers), puts
    the same bottles on the same arm-side ports -- including HandleBridge talking to `/bridge/weights` (sic)."""
    import json
    from oracle.gen_golden import HANDLER_SINKS, handler_calls
    from vfclik_b200 import handlers
    from vfclik_b200 import ports as yarp
    yarp.Network.reset()
    prefix = "/0/lwr/right"
    sinks = {}
    for name in HANDLER_SINKS:
        p = yarp.BufferedPortBottle(); p.open(prefix + name); p.setStrict(True)
        sinks[name] = p
    srcs = []
    for name in ("/vectorField/pose", "/dmonitor/distOut", "/bridge/encoders"):
        p = yarp.BufferedPortBottle(); p.open(prefix + name); srcs.append(p)

    def drain():
        got = {}
        for name in HANDLER_SINKS:
            while True:
                b = sinks[name].read(False)
                if b is None:
                    break
                got.setdefault(name, []).append(b.to_list())
        return got
    try:
        rec = handler_calls(handlers, prefix, sinks, drain)
    finally:
        yarp.Network.reset()
    want = json.loads(str(golden["handlers_record"][0]))
    assert [r[0] for r in rec] == [w[0] for w in want]
    for (label, got), (_, exp) in zip(rec, want):
        got = json.loads(json.dumps(got))
        if label.startswith("bridge.") and "/bridge/weights" in got:
            # the reference connects HandleBridge to `/bridge/weights`, a name scripts/bridge never opens (its port is
            # `/weight`, :571), so there its controller switching goes nowhere; this repo's class writes to both
            assert got.pop("/bridge/weight") == got["/bridge/weights"]
        assert got == exp, (label, got, exp)
    capsys.readouterr()


def test_injected_transport():
    """Row f4: the host modules' ports come from ``ArcosYarp``, which creates and connects them through the transport chosen
    with ``ports.use_transport`` -- the real ``yarp`` module where it exists (it does not in this image).  A duck-typed
    stand-in with its OWN port class, bottle class and connection table proves nothing falls through to the in-process
    registry: naming, direction of the links, strictness, and the list helpers all go through the injected objects."""
    import types
    from vfclik_b200 import ports

    calls = {"open": [], "connect": [], "strict": []}

    class Val:
        def __init__(self, v):
            self.v = v

        def asDouble(self):
            return float(self.v)

        def asInt(self):
            return int(self.v)

        def asString(self):
            return str(self.v)

        def asList(self):
            return self.v

    class FBottle:
        def __init__(self):
            self.v = []

        def clear(self):
            self.v = []

        def addDouble(self, x):
            self.v.append(float(x))

        def addInt(self, x):
            self.v.append(int(x))

        def addString(self, x):
            self.v.append(str(x))

        def addList(self):
            b = FBottle()
            self.v.append(b)
            return b

        def size(self):
            return len(self.v)

        def get(self, i):
            return Val(self.v[i])

    wires, inbox = {}, {}

    class FPort:
        __slots__ = ("name", "out")                      # like a SWIG proxy: no foreign attributes

        def __init__(self):
            self.name, self.out = None, FBottle()

        def open(self, name):
            self.name = name
            calls["open"].append(name)
            inbox[name] = []
            return True

        def close(self):
            inbox.pop(self.name, None)

        def getName(self):
            return self.name

        def setStrict(self, strict=True):
            calls["strict"].append((self.name, bool(strict)))

        def prepare(self):
            return self.out

        def write(self, force=False):
            for dst in wires.get(self.name, []):
                b = FBottle()
                b.v = list(self.out.v)
                inbox[dst].append(b)

        writeStrict = write

        def read(self, wait=True):
            q = inbox[self.name]
            return q.pop(0) if q else None

    class FNetwork:
        @staticmethod
        def connect(src, dst, style=None):
            calls["connect"].append((src, dst))
            if dst not in wires.setdefault(src, []):        # connecting twice is a no-op, as in YARP
                wires[src].append(dst)
            return True

        @staticmethod
        def isConnected(src, dst):
            return dst in wires.get(src, [])

    fake = types.SimpleNamespace(BufferedPortBottle=FPort, Network=FNetwork, Bottle=FBottle)
    ports.Network.reset()
    ports.use_transport(fake)
    try:
        assert ports.transport() is fake
        a = ports.ArcosYarp(ports_name_prefix="/0", module_name_prefix="/lwr/right/vectorField")
        b = ports.ArcosYarp(ports_name_prefix="/0", module_name_prefix="/lwr/right/bridge")
        out = a.create_yarp_port("/qdotOut", input_port=False)
        inp = b.create_yarp_port("/vectorfieldcmd", strict=False)
        assert isinstance(out, FPort) and isinstance(inp, FPort)
        assert calls["open"] == ["/0/lwr/right/vectorField/qdotOut", "/0/lwr/right/bridge/vectorfieldcmd"]
        assert calls["strict"] == [("/0/lwr/right/bridge/vectorfieldcmd", False)]
        a.connect(out, "/lwr/right/bridge", "/vectorfieldcmd")           # an output port writes TO the remote
        b.connect(inp, "/lwr/right/vectorField", "/qdotOut")             # an input port reads FROM it: same wire
        assert calls["connect"] == [("/0/lwr/right/vectorField/qdotOut", "/0/lwr/right/bridge/vectorfieldcmd")] * 2
        assert a.is_ready() and b.is_ready()
        ports.sendListPort(out, [0.1, -0.2, 0.3])
        assert ports.readListPort(inp) == [0.1, -0.2, 0.3]
        ports.write_bottle_lists(out, ["add", 7, -10.0, 2, [0.5, 0.25, 1.0, 0.05, 0.001, 20]])
        got = inp.read(False)
        assert got.get(0).asString() == "add" and got.get(1).asInt() == 7 and got.get(4).asList().v == [0.5, 0.25, 1.0, 0.05, 0.001, 20.0]
        assert not ports.Network.exists("/0/lwr/right/vectorField/qdotOut")     # the in-process registry never saw these ports
    finally:
        ports.use_transport(None)
    assert ports.transport() is ports


def test_bench_reference_arm_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) needs no GPU: one JSON line with the GPU
    arm's metric / unit / config, `impl`, a `cpu_baseline` describing this very run and an `e2e` that copies no bytes."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-cycles", "10"], capture_output=True, text=True, timeout=300, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "instance-control-cycles/sec" and d["unit"] == "inst-cycles/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["config"]["workload"].startswith("config3")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] > 0 and "control cycles" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_write_outputs_whole_or_seeded_sample(tmp_path):
    """`bench.py --dump-outputs` writes arrays that fit the budget whole, and larger ones as the same seeded sample of
    instances (columns) in every array and every run, within the budget."""
    import bench
    rng = np.random.default_rng(4)
    arrays = {"q": rng.normal(size=(7, 5000)).astype(np.float32), "qdot": rng.normal(size=(7, 5000))}
    bench.write_outputs(str(tmp_path / "whole"), arrays, budget=1 << 20)
    for name, a in arrays.items():
        got = np.load(tmp_path / "whole" / (name + ".npy"))
        assert got.dtype == a.dtype and np.array_equal(got, a)
    budget = 20000
    for run in ("a", "b"):
        bench.write_outputs(str(tmp_path / run), arrays, budget=budget)
    got = {run: {name: np.load(tmp_path / run / (name + ".npy")) for name in arrays} for run in ("a", "b")}
    assert sum(a.nbytes for a in got["a"].values()) <= budget
    cols = [int(np.flatnonzero(arrays["q"][0] == x)[0]) for x in got["a"]["q"][0]]
    assert len(cols) == budget // (7 * 4 + 7 * 8) and cols == sorted(set(cols))
    for name, a in arrays.items():
        assert got["a"][name].dtype == a.dtype and np.array_equal(got["a"][name], a[:, cols])
        assert np.array_equal(got["a"][name], got["b"][name])
