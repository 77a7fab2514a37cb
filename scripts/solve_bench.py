"""vfk_solve on one GPU: what the stop rule costs when nothing stops, and what it saves on a reach workload.

    python scripts/solve_bench.py [--reps 5] [--out DIR]

Prints one JSON line (and writes it to DIR/solve_bench.json when --out is given):
  overhead  the headline shape (1 M FP32 LWR instances, 32 obstacles) and FP64 config 2 (65,536 instances, 32 obstacles):
            vfk_solve with both tolerances 0 (never met) at K = 100, alternated with vfk_step(K = 100) on the same batch
            from the same q; time per call of each (median over --reps) and whether the final q is bit-identical.
  reach     goals = the tool frames of random reachable postures, random starts, obstacles as config 2, tol 1e-3 m /
            1e-2 rad, K = 1000, both precisions: reached fraction, percentiles of the reported cycles, time per call,
            useful instance-cycles per second (sum over instances of the cycles each one needed, K for those that never
            arrived, over the call's time) and vfk_step(K = 1000) on the same batch as the fixed-budget comparison.
Times are CUDA-event intervals around single calls.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (out.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def timed(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3          # us


def setup(precision, n, M, seed, reach=False):
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
    from vfclik_b200.engine import Engine, Params
    cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
    chain = chain_from_config(cfg)
    eng = Engine(chain, precision=precision, params=Params.from_config(cfg))
    db = workloads.random_batch_device(eng, n, M, seed=seed)
    if reach:
        # the goal of every instance is the tool frame of another random posture: reachable, and (obstacles aside) on a path
        # the field can follow
        other = workloads.random_batch_device(eng, n, 2, seed=seed + 1)
        other._ensure("pose")
        # the tool frame of the other posture: pose is written before the cycle integrates
        eng.step(dict(q=other.t["q"], goal=other.t["goal"], obst=other.t["obst"], pose=other.t["pose"]), n, 2, 1)
        db.t["goal"][:, 0:12] = other.t["pose"][:, 0:12]
        db.t["goal"][:, 12] = 0.05
        del other
    db._ensure("cycles")
    db._ensure("solve_dist")
    torch.cuda.synchronize()
    return eng, db


def overhead(precision, n, M, reps, K=100):
    import torch
    eng, db = setup(precision, n, M, seed=1)
    q0 = db.t["q"].clone()
    step_bufs = db.bufs
    solve_bufs = {k: v for k, v in step_bufs.items() if k != "qdot"}

    def solve():
        eng.solve(solve_bufs, n, M, K, 0.0, 0.0, db.t["cycles"], None)

    def step():
        eng.step(step_bufs, n, M, K)

    for fn in (solve, step):                # warm-up (module load, launch plans)
        db.t["q"].copy_(q0)
        fn()
    ts, tp = [], []
    for _ in range(reps):
        db.t["q"].copy_(q0)
        ts.append(timed(solve))
        qs = db.t["q"].clone()
        db.t["q"].copy_(q0)
        tp.append(timed(step))
    same = bool(torch.equal(qs, db.t["q"]))
    cyc_ok = bool((db.download("cycles")[0] == -1).all())
    eng.close()
    s, p = float(np.median(ts)), float(np.median(tp))
    return dict(n=n, M=M, precision=precision, K=K, solve_us=s, step_us=p, solve_over_step=s / p, q_bit_identical=same,
                all_cycles_minus_one=cyc_ok, solve_us_all=ts, step_us_all=tp)


def reach(precision, n, M, reps, K=1000, tol_t=1e-3, tol_r=1e-2):
    eng, db = setup(precision, n, M, seed=5, reach=True)
    q0 = db.t["q"].clone()
    step_bufs = db.bufs
    solve_bufs = {k: v for k, v in step_bufs.items() if k != "qdot"}

    def solve():
        eng.solve(solve_bufs, n, M, K, tol_t, tol_r, db.t["cycles"], db.t["solve_dist"])

    def step():
        eng.step(step_bufs, n, M, K)

    ts, tp = [], []
    for _ in range(reps + 1):               # the first pair warms up
        db.t["q"].copy_(q0)
        ts.append(timed(solve))
        cyc = db.download("cycles")[0]
        db.t["q"].copy_(q0)
        tp.append(timed(step))
    ts, tp = ts[1:], tp[1:]
    eng.close()
    s, p = float(np.median(ts)), float(np.median(tp))
    got = cyc >= 0
    useful = float(np.where(got, cyc, K).sum())
    pct = {str(x): (float(np.percentile(cyc[got], x)) if got.any() else None) for x in (10, 50, 90, 99)}
    return dict(n=n, M=M, precision=precision, K=K, tol_trans=tol_t, tol_rot=tol_r, reached_fraction=float(got.mean()),
                cycles_percentiles_of_reached=pct, solve_us=s, step_us=p, useful_instance_cycles_per_s=useful / (s * 1e-6),
                step_instance_cycles_per_s=n * K / (p * 1e-6), solve_us_all=ts, step_us_all=tp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("solve_bench needs a CUDA device")
    name, power = card()
    res = dict(gpu=name, power_limit=power,
               overhead=[overhead(32, 1 << 20, 32, args.reps), overhead(64, 1 << 16, 32, args.reps)],
               reach=[reach(32, 1 << 16, 32, max(2, args.reps // 2)), reach(64, 1 << 16, 32, max(2, args.reps // 2))])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "solve_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
