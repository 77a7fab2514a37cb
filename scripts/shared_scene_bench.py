"""One obstacle list for the whole batch (vfk_buffers.obst_shared) against the same list replicated to every instance.

    python scripts/shared_scene_bench.py [--rounds 3] [--out DIR]

Prints one JSON line (and writes it to DIR/shared_scene_bench.json when --out is given).  Every shape runs both modes on the
same starts, goals and scene, alternating them --rounds times in this one process:
  step   the headline shape (1 M FP32 LWR instances, 32 obstacles) at K = 1 and K = 100, 2 M FP32 instances x 256 obstacles,
         FP64 65,536 x 32 (config 2), 512 k FP32 17-joint DH chains x 64 obstacles (config 5): time per launch (CUDA events
         over a window of launches), instance-cycles/s, the HBM bytes each instance needs per launch -- s (3N + 13) shared,
         s (3N + 13 + 4 Mp) replicated -- with the floor they set at 7.7 TB/s and its share of the measured time, and whether
         q and qdot after one launch from the same state are bit-identical.  Batches under 256 MB (shared mode) are copied
         enough times that the launches of either mode rotate over more than the 126 MB L2.
  solve  the reach workload of scripts/solve_bench.py (65,536 LWR instances, goals at the tool frames of other random
         postures, 1e-3 m / 1e-2 rad, K = 1000) in one scene of 32 obstacles, both precisions: time per call, reached
         fraction and whether cycles and q are bit-identical.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM = 7.7e12                 # B/s, one B200 (data sheet)
L2_ROTATE = 256 << 20


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (out.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def chain_and_params(name):
    from vfclik_b200 import workloads
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
    from vfclik_b200.engine import Params
    if name == "lwr":
        cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
        return chain_from_config(cfg), Params.from_config(cfg)
    return workloads.dual_arm_torso_chain(17), Params()


class Pair:
    """One batch (q, goal, qdot per instance) in `copies` copies, each with the scene both as one shared list and replicated."""

    def __init__(self, eng, n, M, seed, copies=1, reach=False):
        import torch
        from vfclik_b200 import workloads
        self.eng, self.n, self.M = eng, n, M
        scene = workloads.random_batch(eng.chain, 1, M, seed + 1)["obst"][:, 0]          # as workloads.shared_scene_batch
        dev = "cuda:%d" % eng.device
        self.scene = torch.tensor(scene, dtype=eng.torch_dtype, device=dev)
        self.copies = []
        for c in range(copies):
            rep = eng.alloc(M, n, width=4)
            step = max(2, min(M, (1 << 26) // n) & ~1)                                     # whole pairs per packed slice
            for m0 in range(0, M, step):
                m1 = min(M, m0 + step)
                dense = self.scene[m0:m1, None, :].expand(m1 - m0, n, 4).contiguous()
                blk = eng.alloc(m1 - m0, n, width=4)
                eng.pack(dense, blk, m1 - m0, 4, n)
                rep[:, m0:m0 + blk.shape[1]] = blk
                del dense, blk
            db = workloads.random_batch_device(eng, n, 2, seed=seed + 7 * c)
            if reach:
                other = workloads.random_batch_device(eng, n, 2, seed=seed + 1000)
                other._ensure("pose")
                eng.step(dict(q=other.t["q"], goal=other.t["goal"], obst=other.t["obst"], pose=other.t["pose"]), n, 2, 1)
                db.t["goal"][:, 0:12] = other.t["pose"][:, 0:12]
                db.t["goal"][:, 12] = 0.05
                del other
            b = dict(q=db.t["q"], goal=db.t["goal"], qdot=db.t["qdot"])
            self.copies.append(dict(b=b, q0=db.t["q"].clone(), rep=dict(b, obst=rep), shared=dict(b, obst=self.scene, obst_shared=True),
                                    cycles=eng.alloc(1, n, dtype=torch.int32)))
        torch.cuda.synchronize()

    def reset(self):
        for c in self.copies:
            c["b"]["q"].copy_(c["q0"])


def timed(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3          # us


def step_shape(label, precision, chain_name, n, M, K, launches, rounds):
    import torch
    from vfclik_b200.engine import Engine
    chain, params = chain_and_params(chain_name)
    eng = Engine(chain, precision=precision, params=params)
    s = precision // 8
    N = chain.n_joints
    per_shared, per_rep = s * (3 * N + 13), s * (3 * N + 13 + 4 * ((M + 1) & ~1))
    copies = max(1, math.ceil(L2_ROTATE / (n * per_shared)))          # enough for the smaller of the two working sets
    p = Pair(eng, n, M, seed=3, copies=copies)
    # outputs: one launch of each mode from the same state
    c0 = p.copies[0]
    got = {}
    for mode in ("shared", "rep"):
        p.reset()
        eng.step(c0[mode], n, M, K)
        got[mode] = (c0["b"]["q"].clone(), c0["b"]["qdot"].clone())
    same = all(torch.equal(a, b) for a, b in zip(got["shared"], got["rep"]))
    times = {"shared": [], "rep": []}
    for _ in range(rounds):
        for mode in ("shared", "rep"):
            p.reset()

            def window():
                for i in range(launches):
                    eng.step(p.copies[i % copies][mode], n, M, K)
            window()                                    # warm-up and steady clocks
            times[mode].append(timed(window) / launches)
    eng.close()
    del p
    torch.cuda.empty_cache()
    res = dict(shape=label, precision=precision, n=n, N=N, M=M, K=K, copies_rotated=copies, launches_per_window=launches,
               q_qdot_bit_identical=bool(same))
    for mode, per in (("shared", per_shared), ("rep", per_rep)):
        t = float(np.median(times[mode]))
        floor = n * per / HBM * 1e6
        res[mode] = dict(us_per_launch=t, us_all=times[mode], instance_cycles_per_s=n * K / (t * 1e-6), bytes_per_instance=per,
                         hbm_floor_us=floor, of_hbm_roofline=floor / t)
    res["speedup"] = res["rep"]["us_per_launch"] / res["shared"]["us_per_launch"]
    return res


def solve_shape(precision, n=1 << 16, M=32, K=1000, rounds=2, tol_t=1e-3, tol_r=1e-2):
    import torch
    from vfclik_b200.engine import Engine
    chain, params = chain_and_params("lwr")
    eng = Engine(chain, precision=precision, params=params)
    p = Pair(eng, n, M, seed=5, reach=True)
    c0 = p.copies[0]
    dist = eng.alloc(2, n)
    out, times = {}, {"shared": [], "rep": []}
    for r in range(rounds + 1):                       # the first round warms up
        for mode in ("shared", "rep"):
            p.reset()
            bufs = {k: v for k, v in c0[mode].items() if k != "qdot"}
            t = timed(lambda: eng.solve(bufs, n, M, K, tol_t, tol_r, c0["cycles"], dist))
            if r:
                times[mode].append(t)
            out[mode] = (c0["cycles"].clone(), c0["b"]["q"].clone(), dist.clone())
    same = all(torch.equal(a, b) for a, b in zip(out["shared"], out["rep"]))
    cyc = out["shared"][0].cpu().numpy().reshape(-1)[:n]
    eng.close()
    res = dict(shape="reach, one scene", precision=precision, n=n, M=M, K=K, tol_trans=tol_t, tol_rot=tol_r,
               reached_fraction=float((cyc >= 0).mean()), cycles_q_dist_bit_identical=bool(same))
    for mode in ("shared", "rep"):
        t = float(np.median(times[mode]))
        res[mode] = dict(us_per_call=t, us_all=times[mode])
    res["speedup"] = res["rep"]["us_per_call"] / res["shared"]["us_per_call"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("shared_scene_bench needs a CUDA device")
    name, power = card()
    r = args.rounds
    res = dict(gpu=name, power_limit=power, step=[
        step_shape("headline", 32, "lwr", 1 << 20, 32, 1, 200, r),
        step_shape("headline", 32, "lwr", 1 << 20, 32, 100, 10, r),
        step_shape("config 4 shard", 32, "lwr", 2 << 20, 256, 1, 50, r),
        step_shape("config 2", 64, "lwr", 1 << 16, 32, 1, 400, r),
        step_shape("config 5", 32, "dh17", 1 << 19, 64, 1, 100, r),
    ], solve=[solve_shape(32), solve_shape(64)])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "shared_scene_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
