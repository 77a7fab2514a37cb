"""Small invocations of every kernel shape added in round 2, for `compute-sanitizer --tool memcheck`."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from vfclik_b200 import workloads
from vfclik_b200.config import PACKAGE_CONFIG_DIR, chain_from_config, config_filename, load_config
from vfclik_b200.engine import DeviceBatch, Engine, Params
cfg = load_config(config_filename(PACKAGE_CONFIG_DIR + "/lwr/", "lwr", "right"))
lwr = chain_from_config(cfg)

def run(chain, precision, n, m, k=2, outputs=("qdot",), params=None, extra=None):
    dt = np.float32 if precision == 32 else np.float64
    e = Engine(chain, precision=precision, params=params or Params())
    w = workloads.random_batch(chain, n, m, seed=5, dtype=dt)
    db = DeviceBatch(e, n, m, outputs=outputs, inputs=tuple((extra or {}).keys()))
    db.upload("q", w["q"]); db.upload("goal", w["goal"])
    if m:
        db.upload("obst", w["obst"])
        assert np.array_equal(db.download("obst"), w["obst"])
    for name, arr in (extra or {}).items():
        db.upload(name, arr.astype(dt))
    db.step(k)
    out = db.download("qdot")
    assert np.all(np.isfinite(out))
    e.close()
    return out

full = ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "twist", "flags")
for precision in (32, 64):
    run(lwr, precision, 70, 33)                                             # lean, odd obstacle count (padding slot), ragged tile
    run(lwr, precision, 70, 9, outputs=full)                                # general
    run(workloads.dual_arm_torso_chain(), precision, 100, 20)               # FP32: DhPattern lean (slim path, 3 stages); FP64: lane-split kernel (tensor-map TMA)
    run(workloads.dual_arm_torso_chain(), precision, 40, 20)                # two tiles: two warps of the CTA have no work (they still pass the table barrier)
    run(workloads.torso_arm_chain(8), precision, 64, 5, outputs=full)       # padded chain in the 10-joint instantiation
    run(workloads.torso_arm_chain(3), precision, 64, 5, outputs=full)
run(workloads.torso_arm_chain(10), 64, 64, 4, outputs=full, params=Params(ns_mode=2, ns_control=(0.3, -0.2, 0.1, 0.2)),
    extra={"ns_lastvec": np.zeros((40, 64))})                               # control nullspace, 4 basis vectors
run(lwr, 64, 64, 4, outputs=full, params=Params(ns_mode=1, ns_lambda=0.0))  # undamped projector through the Householder basis
run(lwr, 64, 64, 4, outputs=full, params=Params(ik_mode=1))                 # truncated IK (one-sided Jacobi)
run(lwr, 64, 64, 0, outputs=full, params=Params(mixer_w=(0, 0, 1.0, 0, 0, 0)),
    extra={"jp_ref": np.zeros((7, 64)), "jp_lo": -np.ones((7, 64)), "jp_hi": np.ones((7, 64))})
print("sanitize_small: all shapes ran")
