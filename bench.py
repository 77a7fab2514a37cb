#!/usr/bin/env python
"""Benchmark: instance-control-cycles/s of the fused vfclik control-cycle kernel on N B200s.

Contract: ``python bench.py --gpus N --steps K --warmup W`` (for N > 1 launched under
torch.distributed.run, one rank per GPU).  Rank 0 prints ONE JSON line.

* step      = one pass of the hot path over one batch: one kernel launch advancing every
              instance of the rank's shard by ``--kcycles`` (default 1) control cycles, state and
              scene read from / written to HBM.
* workload  = BASELINE.json configs[2]: 1,048,576 LWR (7-DOF) instances per GPU, 32 obstacles
              each, nullspace joint-limit avoidance on, FP32 mode (the metric's "(7-DOF, 32 obst)").
              ``--workload config2`` selects configs[1] (65,536 instances, FP64).
* value     = whole-job inst-cycles/s with inputs resident in HBM (CUDA events, max over ranks).
* e2e       = same metric through the host-buffer C-ABI session (the reference-facing call): every
              step copies q host->device from pinned memory and the clamped qdot device->host.
* roofline  = HBM: algorithmic bytes (DESIGN.md: s*(3N+13+4M) per instance per launch) / launch time.
* cpu_baseline = oracle/refshape.py (reference-shaped scalar loop) on all host cores, bounded sample.
* ``--impl reference`` = that same CPU loop as the timed arm (the reference itself cannot run:
  python2 + PyKDL/vfl/arcospyu/yarp are absent; see DESIGN.md).
* ``--dump-outputs DIR`` = q and qdot after the last timed step, as .npy files (at most 60 MiB: a seeded sample of the
  instances where the shard is larger); the inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "instance-control-cycles/sec"
UNIT = "inst-cycles/s"

WORKLOADS = {
    # name: (instances per GPU, obstacles, precision, description)
    "config3": (1 << 20, 32, 32, "BASELINE configs[2]: 1M LWR instances/GPU, 32 obstacles, nullspace limit avoidance, FP32"),
    "config2": (1 << 16, 32, 64, "BASELINE configs[1]: 65,536 LWR instances/GPU, 32 obstacles, FP64"),
    "config4": (1 << 21, 256, 32, "BASELINE configs[3] shard: 2M LWR instances/GPU, 256 obstacles, FP32"),
    "config5": (1 << 19, 64, 32, "BASELINE configs[4] shard: 512k 17-DOF instances/GPU, 64 obstacles, FP32"),
    "config5_fp64": (1 << 18, 64, 64, "configs[4]'s chain in the FP64 mode: 256k 17-DOF instances/GPU, 64 obstacles (not a BASELINE config)"),
}


def algorithmic_bytes(n_joints: int, n_obst: int, elem: int) -> int:
    """Compulsory HBM bytes per instance per launch (SURVEY.md 8d): q in/out 2N, qdot out N, goal 13, obstacles 4M."""
    return elem * (3 * n_joints + 13 + 4 * n_obst)


DUMP_BUDGET = 60 << 20      # bytes of array data --dump-outputs writes at most


def write_outputs(out_dir: str, arrays: dict, budget: int = DUMP_BUDGET):
    """Save dense ``[comps, instances]`` arrays as ``out_dir/<name>.npy``.  When they exceed ``budget`` bytes together, the
    same seeded sample of instances (columns, in order) is taken from every array, so that two runs with the same
    arguments write the same instances."""
    os.makedirs(out_dir, exist_ok=True)
    n = next(iter(arrays.values())).shape[1]
    per_instance = sum(a.itemsize * a.shape[0] for a in arrays.values())
    if per_instance * n > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // per_instance, replace=False))
        arrays = {name: a[:, idx] for name, a in arrays.items()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def kernel_source_stamp() -> str:
    """sha256 over the CUDA sources and the ABI header the library is built from (with the compiler version): what a
    profile-derived constant (``profiles/traffic.json``) is stamped with, so that a number measured on other kernels is
    recognised as stale instead of being reported."""
    import glob
    import hashlib
    import re
    h = hashlib.sha256()
    files = sorted(glob.glob(os.path.join(ROOT, "vfclik_b200", "csrc", "*.cu*"))) + [os.path.join(ROOT, "include", "vfk.h")]
    for f in files:
        text = open(f, encoding="utf-8").read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)          # comments and layout do not change the code
        text = re.sub(r"//[^\n]*", "", text)
        h.update(os.path.basename(f).encode())
        h.update("".join(text.split()).encode())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------------------- clocks

class ClockSampler:
    """Samples SM clocks and throttle reasons through NVML (every ~2 ms) while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.gpu, self.sm, self.reasons, self.power = gpu_index, [], set(), []
        self.stop_flag = threading.Event()
        self.thread = None
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if visible:
                try:
                    phys = int(visible.split(",")[gpu_index])
                except (ValueError, IndexError):
                    phys = gpu_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                   # noqa: BLE001
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
            except Exception:                                    # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + self.err]}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                "reasons": sorted(self.reasons), "source": "nvml, sampled during the timed region"}


# ----------------------------------------------------------------------------------------- CPU arm (oracle)

def _cpu_worker_main(conn, seed, n_obst, ns_mode):
    """One host core: builds its own reference-shaped control loop (oracle/refshape.py) once, then advances it by the
    number of control cycles the parent asks for and reports the time the cycles took."""
    from oracle import batch, refshape
    from vfclik_b200 import workloads
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    chain = chain_from_config(cfg)
    w = workloads.random_batch(chain, 1, n_obst, seed=seed)
    g = w["goal"][:, 0]
    g17 = [g[0], g[1], g[2], g[9], g[3], g[4], g[5], g[10], g[6], g[7], g[8], g[11], 0, 0, 0, 1, g[12]]
    prm = batch.Params(ns_mode=ns_mode, jp_ref=tuple(cfg.initial_joint_pos), speed_scale=cfg.speedScale, dt=cfg.rate)
    loop = refshape.ControlLoop(chain, prm, w["q"][:, 0], g17, obstacles=w["obst"][:, 0, :].tolist())
    conn.send("ready")
    while True:
        cycles = conn.recv()
        if cycles is None:
            break
        t0 = time.perf_counter()
        loop.run(cycles)
        conn.send((cycles, time.perf_counter() - t0))


class CpuArm:
    """All host cores, each advancing its own instance (instances are independent, like GPU shards)."""

    def __init__(self, n_obst: int, ns_mode: int = 1):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self.n_obst, self.ns_mode = n_obst, ns_mode
        self.workers = []
        for c in range(self.cores):
            parent, child = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker_main, args=(child, 1000 + c, n_obst, ns_mode), daemon=True)
            p.start()
            self.workers.append((p, parent))
        for _, conn in self.workers:
            assert conn.recv() == "ready"

    def step(self, cycles_per_core: int):
        """Every core advances its instance by `cycles_per_core` control cycles; returns (total cycles, wall seconds)."""
        t0 = time.perf_counter()
        for _, conn in self.workers:
            conn.send(cycles_per_core)
        res = [conn.recv() for _, conn in self.workers]
        wall = time.perf_counter() - t0
        return sum(r[0] for r in res), wall

    def close(self):
        for p, conn in self.workers:
            conn.send(None)
        for p, _ in self.workers:
            p.join(timeout=5)


def cpu_vectorised(n_obst: int, instances: int = 8192):
    """Best-effort CPU: the vectorised numpy oracle (oracle/batch.py), one core, one cycle over a batch."""
    from oracle import batch
    from vfclik_b200 import workloads
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    chain = chain_from_config(cfg)
    w = workloads.random_batch(chain, instances, n_obst, seed=77)
    q, goal = w["q"].T.copy(), w["goal"].T.copy()
    obst = w["obst"].transpose(1, 0, 2).copy()
    prm = batch.Params(jp_ref=tuple(cfg.initial_joint_pos), speed_scale=cfg.speedScale, dt=cfg.rate)
    batch.step(chain, prm, q[:256], goal[:256], obst[:256])
    t0 = time.perf_counter()
    batch.step(chain, prm, q, goal, obst)
    return instances / (time.perf_counter() - t0)


def run_reference_arm(args, rank: int):
    """--impl reference: the reference-shaped CPU loop as the timed arm (rank 0 only)."""
    if rank != 0:
        return
    n_inst, n_obst, precision, desc = WORKLOADS[args.workload]
    arm = CpuArm(n_obst)
    cycles_per_core = args.cpu_cycles
    rate = None
    for _ in range(max(args.warmup, 1)):
        c, t = arm.step(max(1, cycles_per_core // 4))
        rate = c / t / arm.cores                       # control cycles per second per core
    # bound the whole timed run to about a minute whatever --steps is: a step is a fixed number of cycles per core
    budget_s = 60.0
    cycles_per_core = max(1, min(cycles_per_core, int(budget_s * rate / max(args.steps, 1))))
    total, wall = 0, 0.0
    for _ in range(args.steps):
        c, t = arm.step(cycles_per_core)
        total += c
        wall += t
    arm.close()
    value = total / wall
    sample = "%d cores x %d control cycles of one instance each per step (7-DOF, %d obstacles, nullspace on, FP64)" % (
        arm.cores, cycles_per_core, n_obst)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload + ": " + desc, "sample": sample,
                   "note": "reference itself is python2 + PyKDL/vfl/arcospyu/yarp (absent): oracle/refshape.py port timed"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- GPU arm

class _StdoutToStderr:
    """NCCL prints its version banner on stdout; keep rank 0's stdout to the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300,
                    help="timed launches (default 300 = a ~35 ms burst, like the copy that measured the HBM peak; runs of >= 1000 "
                         "launches draw enough power for sw_power_cap to lower the SM clock on some boxes, see DESIGN.md)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS))
    ap.add_argument("--kcycles", type=int, default=1, help="control cycles fused per launch (per step)")
    ap.add_argument("--instances", type=int, default=0, help="override instances per GPU")
    ap.add_argument("--cpu-cycles", type=int, default=1000, help="CPU arm: control cycles per core per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the K-fused and FP64 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the joint positions and velocities of the last timed step (rank 0's "
                         "shard) as DIR/q.npy and DIR/qdot.npy, [joints, instances] in the run's precision, so that two builds "
                         "can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product has no CPU path (use --impl reference for the CPU arm)")
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    from vfclik_b200.distributed import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local_rank)          # before any page-locked allocation: staging memory lands next to the GPU
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        with _StdoutToStderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()

    import __graft_entry__ as ge
    ge.build()
    from vfclik_b200 import workloads
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
    from vfclik_b200.engine import DeviceBatch, Engine, Params

    n_inst, n_obst, precision, desc = WORKLOADS[args.workload]
    if args.instances:
        n_inst = args.instances
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    chain = workloads.dual_arm_torso_chain() if args.workload.startswith("config5") else chain_from_config(cfg)
    params = Params.from_config(cfg) if not args.workload.startswith("config5") else Params()
    N = chain.n_joints
    np_dt = np.float32 if precision == 32 else np.float64
    elem = 4 if precision == 32 else 8

    eng = Engine(chain, precision=precision, device=local_rank, params=params)
    big = n_inst * max(n_obst, 1) > (1 << 26)              # config 4 / 5 shards: draw the batch on the GPU
    if big:
        w = None
        db = workloads.random_batch_device(eng, n_inst, n_obst, seed=1 + rank)
    else:
        w = workloads.random_batch(chain, n_inst, n_obst, seed=1 + rank, dtype=np_dt)   # configs[2]: seed 1 (+rank: shards differ)
        db = DeviceBatch(eng, n_inst, n_obst, outputs=("qdot",))
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
    q0 = db.t["q"].clone()
    # Inputs smaller than the L2 would be served from it on every launch after the first: rotate over enough independent
    # copies of the batch that a launch's inputs were evicted before they are read again (> 3x the 126 MB L2 in flight).
    bytes_per_launch = algorithmic_bytes(N, n_obst, elem) * n_inst
    n_rot = 1 if bytes_per_launch > 400e6 else int(400e6 // bytes_per_launch) + 2
    dbs = [db]
    for _ in range(n_rot - 1):
        d2 = DeviceBatch(eng, n_inst, n_obst, outputs=("qdot",))
        for name in ("q", "goal", "obst"):
            if name in db.t:
                d2.t[name].copy_(db.t[name])
        dbs.append(d2)
    rot = {"i": 0}

    def step_rotating(k):
        d = dbs[rot["i"] % n_rot]
        rot["i"] += 1
        return d.step(k)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        """`steps` back-to-back calls of fn between two CUDA events on torch's current stream -> ms (max over ranks)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- kernel-resident arm (value)
    for _ in range(max(args.warmup, 3)):
        step_rotating(args.kcycles)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.launches
    ms = timed(lambda: step_rotating(args.kcycles), args.steps)
    gpu_launches = eng.launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        last = dbs[(rot["i"] - 1) % n_rot]             # the batch the last timed step advanced: q integrated in place, qdot
        write_outputs(args.dump_outputs, {name: last.download(name) for name in ("q", "qdot")})
    value = world * n_inst * args.kcycles * args.steps / (ms * 1e-3)
    launch_ms = ms / args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu capture on record for this workload"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if args.workload in tj:
            if tj.get(args.workload + "_stamp") == kernel_source_stamp():
                traffic, traffic_note = tj[args.workload], tj.get(args.workload + "_source")
            else:
                traffic_note = "stale: profiles/traffic.json was measured on other kernel sources (stamp %s, now %s)" % (
                    tj.get(args.workload + "_stamp"), kernel_source_stamp())
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                "traffic": traffic, "traffic_source": traffic_note, "peak_source": "measured" if peaks else "fallback",
                "algorithmic_bytes_per_instance": algorithmic_bytes(N, n_obst, elem),
                "kernel": "vfk_cycle_kernel<%s,%d>" % ("float" if precision == 32 else "double", N)}

    # ---- sustained: >= 1000 back-to-back launches (where sw_power_cap, if the box has it, has had time to act), own clock record
    if not args.no_extras:
        sus_steps = max(1000, args.steps)
        sampler2 = ClockSampler(local_rank)
        if rank == 0:
            sampler2.start()
        ms_sus = timed(lambda: step_rotating(args.kcycles), sus_steps) / sus_steps
        clocks2 = sampler2.stop() if rank == 0 else None
        ach2 = bytes_per_launch / (ms_sus * 1e-3) / 1e9
        roofline["sustained"] = {"launches": sus_steps, "ms_per_step": ms_sus, "achieved": ach2, "frac": ach2 / peak_gbs, "clocks": clocks2}

    # ---- end-to-end arm: host buffers through the C-ABI session (H2D q + D2H qdot every step)
    e2e, e2e_launches = None, 0
    if w is not None:
        sess = eng.session(n_inst, n_obst)
        sess.set_goal(w["goal"]); sess.set_obstacles(w["obst"])
        t_dt = torch.float32 if precision == 32 else torch.float64
        q_host = torch.from_numpy(np.ascontiguousarray(w["q"])).pin_memory()
        qd_host = torch.empty((N, n_inst), dtype=t_dt).pin_memory()
        q_np, qd_np = q_host.numpy(), qd_host.numpy()
        e2e_steps = max(3, min(args.steps, 20))
        for _ in range(3):
            sess.cycle(q_in=q_np, k_cycles=args.kcycles, qdot_out=qd_np)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_launches += sess.cycle(q_in=q_np, k_cycles=args.kcycles, qdot_out=qd_np)   # synchronous: returns after the D2H landed
        barrier()
        e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = world * n_inst * args.kcycles * e2e_steps / float(e2e_s.item())
        io_bytes = N * n_inst * elem
        e2e_ms = 1e3 * float(e2e_s.item()) / e2e_steps
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes,
               "steps": e2e_steps, "ms_per_step": e2e_ms, "gpu_launches": e2e_launches,
               "api": "vfk_session_cycle (pinned host q in, pinned host qdot out; scene resident; direct host I/O: the cycle kernel reads q from and writes qdot to the host buffers over PCIe)",
               "numa": numa}
        # The ceiling of this box for this I/O pattern, measured now with every rank doing it at once: the same two buffers
        # moved by the two DMA engines (H2D and D2H concurrently, no kernel), max over ranks.
        d_in = torch.empty((N, n_inst), dtype=t_dt, device="cuda")
        d_out = torch.empty((N, n_inst), dtype=t_dt, device="cuda")
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()

        def dma_pair():
            with torch.cuda.stream(s_up):
                d_in.copy_(q_host, non_blocking=True)
            with torch.cuda.stream(s_dn):
                qd_host.copy_(d_out, non_blocking=True)
            s_up.synchronize(); s_dn.synchronize()
        for _ in range(3):
            dma_pair()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            dma_pair()
        barrier()
        dma_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dma_s, op=dist.ReduceOp.MAX)
        floor_ms = 1e3 * float(dma_s.item()) / e2e_steps
        e2e["roofline"] = {"bound": "pcie", "floor_ms_per_step": floor_ms, "peak_gbs_each_way": io_bytes / (floor_ms * 1e-3) / 1e9,
                           "achieved_gbs_each_way": io_bytes / (e2e_ms * 1e-3) / 1e9, "frac": floor_ms / e2e_ms,
                           "how": "H2D + D2H of the same %d-byte buffers on the two DMA engines concurrently, all %d ranks at once, "
                                  "max over ranks, same run" % (io_bytes, world)}
        # simulated plant (the reference's bridge -s): 100 control cycles per call, one q in and one command out per call
        k_sim = 100
        sess.cycle(q_in=q_np, k_cycles=k_sim, qdot_out=qd_np)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            e2e_launches += sess.cycle(q_in=q_np, k_cycles=k_sim, qdot_out=qd_np)
        barrier()
        sim_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(sim_s, op=dist.ReduceOp.MAX)
        e2e["k100"] = {"kcycles": k_sim, "value": world * n_inst * k_sim * 3 / float(sim_s.item()), "unit": UNIT,
                       "ms_per_step": 1e3 * float(sim_s.item()) / 3}
        del d_in, d_out
        sess.close()
    else:
        e2e = {"value": None, "unit": UNIT, "note": "not measured for the device-generated config 4 / 5 shards"}

    # ---- side measurements (same run, not the headline)
    extras = {}
    if not args.no_extras:
        kf = 100
        db.t["q"].copy_(q0)
        db.step(kf)
        ms_k = timed(lambda: db.step(kf), 3)
        extras["k_fused"] = {"kcycles": kf, "value": world * n_inst * kf * 3 / (ms_k * 1e-3), "unit": UNIT,
                             "ms_per_launch": ms_k / 3}
        try:
            # compute-bound shape: algorithmic FLOPs (frozen exact count, workloads.ALGORITHMIC_OPS) against the FFMA /
            # DFMA rate measured on this pool's B200 by scripts/peaks.cu (profiles/r01_pipe_peaks.json)
            flops = workloads.algorithmic_flops(N, n_obst)
            pk = json.load(open(os.path.join(ROOT, "profiles", "r01_pipe_peaks.json")))
            peak_tf = float(pk["fp32_ffma_tflops" if precision == 32 else "fp64_dfma_tflops"])
            ach = flops * n_inst * kf * 3 / (ms_k * 1e-3) / 1e12
            extras["k_fused"]["roofline"] = {"bound": "fp32 pipe" if precision == 32 else "fp64 pipe", "achieved": ach,
                                             "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                                             "algorithmic_flops_per_instance_cycle": flops,
                                             "peak_source": "profiles/r01_pipe_peaks.json (scripts/peaks.cu)"}
        except Exception as exc:      # the headline line must not depend on a side measurement
            extras["k_fused"]["roofline"] = {"error": str(exc)}
        if args.workload == "config3":
            n2, m2 = WORKLOADS["config2"][0], WORKLOADS["config2"][1]
            e64 = Engine(chain, precision=64, device=local_rank, params=params)
            w2 = workloads.random_batch(chain, n2, m2, seed=0)
            d2 = DeviceBatch(e64, n2, m2, outputs=("qdot",))
            d2.upload("q", w2["q"]); d2.upload("goal", w2["goal"]); d2.upload("obst", w2["obst"])
            # 85 MB per launch fits the L2: rotate over 7 copies (594 MB) so that every launch reads from HBM.  (A 256 MiB fill
            # between launches, the earlier method, leaves the L2 full of DIRTY lines whose write-back the timed launch then
            # pays for: 45 us against 24 us cold-clean under ncu.)
            copies = [d2]
            for _ in range(6):
                dc = DeviceBatch(e64, n2, m2, outputs=("qdot",))
                for name in ("q", "goal", "obst"):
                    dc.t[name].copy_(d2.t[name])
                copies.append(dc)
            for dc in copies:
                dc.step(1)
            reps = 6
            ms2 = timed(lambda: [dc.step(1) for dc in copies], reps) / (reps * len(copies))
            b2 = algorithmic_bytes(N, m2, 8) * n2
            extras["fp64_config2"] = {"instances_per_gpu": n2, "value": world * n2 / (ms2 * 1e-3), "unit": UNIT, "ms_per_launch": ms2,
                                      "l2": "launches rotate over 7 copies of the batch (594 MB): inputs come from HBM",
                                      "roofline": {"bound": "hbm", "achieved": b2 / (ms2 * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                                                   "frac": b2 / (ms2 * 1e-3) / 1e9 / peak_gbs}}
            del copies, d2
            e64.close()
            torch.cuda.empty_cache()

            # BASELINE configs[3] and configs[4] at their per-GPU shard size on 8 GPUs (2 M x 256 obstacles; 512 k x 17-DOF x 64
            # obstacles), drawn on the device: every rank runs its shard, whatever N is, so the scaling run reports them too
            for wname in ("config4", "config5", "config5_generic"):
                n4, m4, p4, d4 = WORKLOADS["config5" if wname == "config5_generic" else wname]
                # config5_generic: the same shape with the mixed-axis torso (a KDL RotX joint -> general tip rotation), which
                # takes GenericPattern instead of DhPattern: reported so that the chain-pattern gain is visible in every record
                ch4 = (workloads.dual_arm_torso_chain(dh=(wname == "config5")) if wname.startswith("config5") else chain)
                if wname == "config5_generic":
                    d4 = d4 + " -- mixed-axis torso variant (GenericPattern)"
                e4 = Engine(ch4, precision=p4, device=local_rank, params=params if wname == "config4" else Params())
                db4 = workloads.random_batch_device(e4, n4, m4, seed=2 + rank if wname == "config4" else 3 + rank)
                for _ in range(3):
                    db4.step(1)
                st4 = 30
                ms4 = timed(lambda: db4.step(1), st4) / st4
                b4 = algorithmic_bytes(ch4.n_joints, m4, 4) * n4
                extras[wname] = {"workload": d4, "instances_per_gpu": n4, "value": world * n4 / (ms4 * 1e-3), "unit": UNIT, "ms_per_launch": ms4,
                                 "chain_pattern": e4.chain_pattern,
                                 "roofline": {"bound": "hbm", "achieved": b4 / (ms4 * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                                              "frac": b4 / (ms4 * 1e-3) / 1e9 / peak_gbs,
                                              "algorithmic_bytes_per_instance": algorithmic_bytes(ch4.n_joints, m4, 4)}}
                del db4
                e4.close()
                torch.cuda.empty_cache()

        if world == 1 and args.workload == "config3":
            # BASELINE configs[0] on the GPU: ONE LWR, the reference's first goal, 3 obstacles, 1000 control cycles fused
            # into one launch (the latency-bound opposite corner of the design space; the CPU reference loop does ~10^3/s)
            e1 = Engine(chain, precision=64, device=local_rank, params=params)
            w1 = workloads.config1(chain, cfg)
            d1 = DeviceBatch(e1, 1, 3, outputs=("qdot",))
            d1.upload("q", w1["q"]); d1.upload("goal", w1["goal"]); d1.upload("obst", w1["obst"])
            d1.step(1000)
            ms1 = timed(lambda: d1.step(1000), 3) / 3
            extras["config1_single_robot_fp64"] = {"instances": 1, "kcycles": 1000, "value": 1000 / (ms1 * 1e-3), "unit": UNIT,
                                                   "us_per_cycle": ms1}
            e1.close()

    # ---- final stats gather (the only collective: NCCL all_reduce of a few scalars)
    stats = torch.tensor([float(n_inst * args.kcycles * args.steps), float(gpu_launches + e2e_launches)],
                         device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)

    if rank == 0:
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            if all_cpus is not None:
                os.sched_setaffinity(0, all_cpus)        # the CPU arm uses every core of the box, not only the GPU's NUMA node
            arm = CpuArm(n_obst)
            arm.step(20)                       # warm the pool (imports)
            c, t = arm.step(max(1000, args.cpu_cycles))
            arm.close()
            cpu_baseline = {"value": c / t, "unit": UNIT, "cores": arm.cores, "kind": "port",
                            "sample": "%d cores x %d control cycles of one instance each (oracle/refshape.py, 7-DOF, %d obstacles, FP64)"
                                      % (arm.cores, max(1000, args.cpu_cycles), n_obst),
                            "vectorised_numpy_1core": cpu_vectorised(n_obst)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if precision == 32 else "f64", "data": "synthetic",
            "config": {"workload": args.workload + ": " + desc, "instances_per_gpu": n_inst, "n_joints": N,
                       "n_obstacles": n_obst, "kcycles_per_step": args.kcycles,
                       "precision_note": ("FP32 mode is mixed precision: everything that touches HBM and the whole field / IK / nullspace is FP32, "
                                          "the kinematic chain (sin, cos, frame products) runs in FP64 (DESIGN.md section 2)") if precision == 32
                                         else "FP64 throughout", "parallelism": "instances sharded x%d, no collective" % world,
                       "l2": "inputs per launch (%.0f MB) exceed the 126 MB L2" % (bytes_per_launch / 1e6)
                             if n_rot == 1 else "launches rotate over %d independent copies of the batch (%.0f MB in all, > 3x the 126 MB L2): "
                                                "no launch finds its inputs in L2" % (n_rot, n_rot * bytes_per_launch / 1e6)},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(gpu_launches),
            "clocks": clocks, "total_inst_cycles_timed": float(stats[0].item()), "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
