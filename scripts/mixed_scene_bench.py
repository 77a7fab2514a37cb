"""A mixed scene (vfk_buffers.obst_shared = 2: own obstacles per instance plus one shared workcell) against the same scene as
one per-instance list [own ; shared] (workloads.concat_scene), which is what a caller had to build before.

    python scripts/mixed_scene_bench.py [--rounds 3] [--out DIR]

Prints one JSON line (and writes it to DIR/mixed_scene_bench.json when --out is given).  Every shape runs both arms on the same
starts, goals and scene, alternating them --rounds times in this one process:
  step   1 M FP32 LWR instances x (8 own + 256 shared) at K = 1 and K = 100, FP64 65,536 x (8 + 32), 512 k FP32 17-joint DH
         chains x (16 + 64): time per launch (CUDA events over a window of launches), instance-cycles/s, the HBM bytes each
         instance needs per launch -- s (3N + 13 + 4 Mip) mixed, s (3N + 13 + 4 (Mi + Ms) p) concatenated -- with the floor
         they set at 7.7 TB/s and its share of the measured time, and whether q and qdot after one launch from the same state
         are bit-identical (every own count here is a multiple of 8).  Batches under 256 MB (mixed arm) are copied enough
         times that the launches of either arm rotate over more than the 126 MB L2.
  solve  the reach workload of scripts/solve_bench.py (65,536 LWR instances, goals at the tool frames of other random
         postures, 1e-3 m / 1e-2 rad, K = 1000) with 8 own + 32 shared obstacles, both precisions: time per call, reached
         fraction and whether cycles, q and distance are bit-identical.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from shared_scene_bench import HBM, L2_ROTATE, card, chain_and_params, timed   # noqa: E402


class MixedPair:
    """One batch (q, goal, own obstacles, qdot per instance) in `copies` copies, each as a mixed scene and concatenated."""

    def __init__(self, eng, n, Mi, Ms, seed, copies=1, reach=False):
        import torch
        from vfclik_b200 import workloads
        self.eng, self.n, self.Mi, self.Ms = eng, n, Mi, Ms
        assert Mi % 2 == 0, "the blocked concatenation below keeps obstacle pairs whole"
        scene = workloads.random_batch(eng.chain, 1, Ms, seed + 1)["obst"][:, 0]
        dev = "cuda:%d" % eng.device
        self.scene = torch.tensor(scene, dtype=eng.torch_dtype, device=dev)
        rep = eng.alloc(Ms, n, width=4)                                                   # the shared list, replicated
        step = max(2, min(Ms, (1 << 26) // n) & ~1)
        for m0 in range(0, Ms, step):
            m1 = min(Ms, m0 + step)
            dense = self.scene[m0:m1, None, :].expand(m1 - m0, n, 4).contiguous()
            blk = eng.alloc(m1 - m0, n, width=4)
            eng.pack(dense, blk, m1 - m0, 4, n)
            rep[:, m0:m0 + blk.shape[1]] = blk
            del dense, blk
        self.copies = []
        for c in range(copies):
            db = workloads.random_batch_device(eng, n, Mi, seed=seed + 7 * c)
            if reach:
                other = workloads.random_batch_device(eng, n, 2, seed=seed + 1000)
                other._ensure("pose")
                eng.step(dict(q=other.t["q"], goal=other.t["goal"], obst=other.t["obst"], pose=other.t["pose"]), n, 2, 1)
                db.t["goal"][:, 0:12] = other.t["pose"][:, 0:12]
                db.t["goal"][:, 12] = 0.05
                del other
            b = dict(q=db.t["q"], goal=db.t["goal"], qdot=db.t["qdot"])
            own = db.t["obst"]
            cat = torch.cat([own, rep], dim=1).contiguous()      # blocked [own ; shared]: pair rows of an even own count stay whole
            self.copies.append(dict(b=b, q0=db.t["q"].clone(), mixed=dict(b, obst=own, obst_shared=2, shared_obst=self.scene),
                                    concat=dict(b, obst=cat), cycles=eng.alloc(1, n, dtype=torch.int32)))
        del rep
        torch.cuda.synchronize()

    def m(self, arm):
        return self.Mi if arm == "mixed" else self.Mi + self.Ms

    def reset(self):
        for c in self.copies:
            c["b"]["q"].copy_(c["q0"])


def step_shape(label, precision, chain_name, n, Mi, Ms, K, launches, rounds):
    import torch
    from vfclik_b200.engine import Engine
    chain, params = chain_and_params(chain_name)
    eng = Engine(chain, precision=precision, params=params)
    s = precision // 8
    N = chain.n_joints
    per_mixed, per_cat = s * (3 * N + 13 + 4 * ((Mi + 1) & ~1)), s * (3 * N + 13 + 4 * ((Mi + Ms + 1) & ~1))
    copies = max(1, math.ceil(L2_ROTATE / (n * per_mixed)))
    p = MixedPair(eng, n, Mi, Ms, seed=3, copies=copies)
    c0 = p.copies[0]
    got = {}
    for arm in ("mixed", "concat"):
        p.reset()
        eng.step(c0[arm], n, p.m(arm), K)
        got[arm] = (c0["b"]["q"].clone(), c0["b"]["qdot"].clone())
    same = all(torch.equal(a, b) for a, b in zip(got["mixed"], got["concat"]))
    times = {"mixed": [], "concat": []}
    for _ in range(rounds):
        for arm in ("mixed", "concat"):
            p.reset()

            def window():
                for i in range(launches):
                    eng.step(p.copies[i % copies][arm], n, p.m(arm), K)
            window()                                    # warm-up and steady clocks
            times[arm].append(timed(window) / launches)
    eng.close()
    del p
    torch.cuda.empty_cache()
    res = dict(shape=label, precision=precision, n=n, N=N, Mi=Mi, Ms=Ms, K=K, copies_rotated=copies, launches_per_window=launches,
               q_qdot_bit_identical=bool(same))
    for arm, per in (("mixed", per_mixed), ("concat", per_cat)):
        t = float(np.median(times[arm]))
        floor = n * per / HBM * 1e6
        res[arm] = dict(us_per_launch=t, us_all=times[arm], instance_cycles_per_s=n * K / (t * 1e-6), bytes_per_instance=per,
                        hbm_floor_us=floor, of_hbm_roofline=floor / t)
    res["speedup"] = res["concat"]["us_per_launch"] / res["mixed"]["us_per_launch"]
    return res


def solve_shape(precision, n=1 << 16, Mi=8, Ms=32, K=1000, rounds=2, tol_t=1e-3, tol_r=1e-2):
    import torch
    from vfclik_b200.engine import Engine
    chain, params = chain_and_params("lwr")
    eng = Engine(chain, precision=precision, params=params)
    p = MixedPair(eng, n, Mi, Ms, seed=5, reach=True)
    c0 = p.copies[0]
    dist = eng.alloc(2, n)
    out, times = {}, {"mixed": [], "concat": []}
    for r in range(rounds + 1):                       # the first round warms up
        for arm in ("mixed", "concat"):
            p.reset()
            bufs = {k: v for k, v in c0[arm].items() if k != "qdot"}
            t = timed(lambda: eng.solve(bufs, n, p.m(arm), K, tol_t, tol_r, c0["cycles"], dist))
            if r:
                times[arm].append(t)
            out[arm] = (c0["cycles"].clone(), c0["b"]["q"].clone(), dist.clone())
    same = all(torch.equal(a, b) for a, b in zip(out["mixed"], out["concat"]))
    cyc = out["mixed"][0].cpu().numpy().reshape(-1)[:n]
    eng.close()
    res = dict(shape="reach, mixed scene", precision=precision, n=n, Mi=Mi, Ms=Ms, K=K, tol_trans=tol_t, tol_rot=tol_r,
               reached_fraction=float((cyc >= 0).mean()), cycles_q_dist_bit_identical=bool(same))
    for arm in ("mixed", "concat"):
        t = float(np.median(times[arm]))
        res[arm] = dict(us_per_call=t, us_all=times[arm])
    res["speedup"] = res["concat"]["us_per_call"] / res["mixed"]["us_per_call"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mixed_scene_bench needs a CUDA device")
    name, power = card()
    r = args.rounds
    res = dict(gpu=name, power_limit=power, step=[
        step_shape("headline + workcell", 32, "lwr", 1 << 20, 8, 256, 1, 100, r),
        step_shape("headline + workcell", 32, "lwr", 1 << 20, 8, 256, 100, 5, r),
        step_shape("config 2", 64, "lwr", 1 << 16, 8, 32, 1, 400, r),
        step_shape("config 5", 32, "dh17", 1 << 19, 16, 64, 1, 100, r),
    ], solve=[solve_shape(32), solve_shape(64)])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "mixed_scene_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
