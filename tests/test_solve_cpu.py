"""CPU tests of vfk_solve: the obstacle ring's cursor arithmetic on early exit (tests/ring_model.cpp driving
vfclik_b200/csrc/vfk_ring.cuh) and the oracle's ``solve`` against its own ``step``."""
import os
import subprocess

import numpy as np
import pytest

import solve_oracle
from helpers import near_goal, oracle_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The oracle's batched numpy / LAPACK calls round a row differently (by ~1e-17) when other rows of the batch hold other
# values, and a frozen instance does; so its solve matches its step to rounding, not to the bit.  The GPU kernel has no such
# coupling and is held to the bit (tests/test_gpu_solve.py).
ORACLE_ATOL = 1e-12


def test_ring_cursor_model(tmp_path):
    """Random ring shapes (chunks 1-9, 1-3 stages, K 1-5, strides, unit counts) and random exits: at cycle 0, at the last
    cycle, never, anywhere in a streaming unit, and with fewer than S uses left.  Every copy is waited exactly once, no wait
    finds an empty slot or an older phase, and the producer is exactly S uses ahead at every unit's start."""
    exe = tmp_path / "ring_model"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "vfclik_b200", "csrc"),
                           os.path.join(ROOT, "tests", "ring_model.cpp"), "-o", str(exe)])
    res = subprocess.run([str(exe), "30000"], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip() == "ok 30000", res.stdout + res.stderr


def _batch(lwr, n=96, M=8, seed=3, **kw):
    chain, cfg = lwr
    w, meta = near_goal(chain, n, M, seed, **kw)
    from vfclik_b200.engine import Params
    prm = oracle_params(Params.from_config(cfg))
    q = w["q"].T.astype(np.float64)
    goal = w["goal"].T.astype(np.float64)
    obst = w["obst"].transpose(1, 0, 2).astype(np.float64)
    return chain, prm, q, goal, obst, meta


def test_oracle_solve_equals_step_at_each_instance_cycle(lwr):
    from oracle import batch
    chain, prm, q, goal, obst, _ = _batch(lwr)
    K = 40
    res = solve_oracle.solve(chain, prm, q, goal, obst, K, 0.02, 0.2)
    cyc = res["cycles"]
    assert (cyc == 0).any() and ((cyc > 0) & (cyc < K)).any() and (cyc == -1).any(), np.bincount(cyc + 1)
    for c in np.unique(cyc):
        idx = np.nonzero(cyc == c)[0]
        k = K if c == -1 else int(c)
        ref = q if k == 0 else batch.step(chain, prm, q, goal, obst, k_cycles=k)["q"]
        np.testing.assert_allclose(res["q"][idx], ref[idx], rtol=0, atol=ORACLE_ATOL)
    d, a = solve_oracle.goal_distance(chain, prm, res["q"], goal)
    np.testing.assert_array_equal(res["dist"], np.stack([d, a], axis=1))
    reached = cyc >= 0
    assert np.all(d[reached] < 0.02) and np.all(a[reached] < 0.2)


def test_oracle_solve_at_the_goal_stops_at_cycle_zero(lwr):
    """Goals at 1e-7 m / 1e-7 rad from the tool frame, tolerances above that: nothing moves."""
    chain, prm, q, goal, obst, meta = _batch(lwr, n=400)
    at = (meta["d"] == 1e-7) & (meta["theta"] == 1e-7)
    assert at.sum() >= 2
    res = solve_oracle.solve(chain, prm, q[at], goal[at], obst[at], 5, 1e-6, 1e-6)
    assert np.all(res["cycles"] == 0)
    np.testing.assert_array_equal(res["q"], q[at])


def test_oracle_solve_zero_tolerance_never_stops(lwr):
    from oracle import batch
    chain, prm, q, goal, obst, _ = _batch(lwr, n=64)
    for tt, tr in ((0.0, 1.0), (1.0, 0.0)):
        res = solve_oracle.solve(chain, prm, q, goal, obst, 3, tt, tr)
        assert np.all(res["cycles"] == -1)
        np.testing.assert_array_equal(res["q"], batch.step(chain, prm, q, goal, obst, k_cycles=3)["q"])


def test_oracle_solve_tol_rot_pi_ignores_orientation(lwr):
    chain, prm, q, goal, obst, meta = _batch(lwr, n=400)
    far_rot = meta["theta"] > 1.0                       # position close, orientation far
    res = solve_oracle.solve(chain, prm, q, goal, obst, 1, 1e-3, np.pi)
    d0, _ = solve_oracle.goal_distance(chain, prm, q, goal)
    np.testing.assert_array_equal(res["cycles"] == 0, d0 < 1e-3)
    assert np.any((res["cycles"] == 0) & far_rot)
    strict = solve_oracle.solve(chain, prm, q, goal, obst, 1, 1e-3, 1.0)
    assert not np.any((strict["cycles"] == 0) & far_rot)


@pytest.mark.parametrize("mode", ["jp_limits", "control"])
def test_oracle_solve_freezes_carried_state(lwr, mode):
    """jp_ref (with per-instance limits) and the control-mode lastvec keep the value of the instance's last cycle."""
    import dataclasses
    from oracle import batch
    chain, prm, q, goal, obst, _ = _batch(lwr, n=96)
    I, N = q.shape
    kw = {}
    if mode == "jp_limits":
        kw = dict(jp_ref=np.full((I, N), 2.5), jp_limits=(np.tile(chain.q_lo, (I, 1)) * 0.5, np.tile(chain.q_hi, (I, 1)) * 0.5))
    else:
        prm = dataclasses.replace(prm, ns_mode=2, ns_control=(0.3, 0.0, 0.0, 0.0))
    K = 30
    res = solve_oracle.solve(chain, prm, q, goal, obst, K, 0.02, 0.2, **kw)
    cyc = res["cycles"]
    key = "jp_ref" if mode == "jp_limits" else "lastvec"
    for c in np.unique(cyc):
        idx = np.nonzero(cyc == c)[0]
        k = K if c == -1 else int(c)
        if k == 0:
            continue
        ref = batch.step(chain, prm, q, goal, obst, k_cycles=k, **kw)
        np.testing.assert_allclose(res["q"][idx], ref["q"][idx], rtol=0, atol=ORACLE_ATOL)
        np.testing.assert_allclose(res[key][idx], ref[key][idx], rtol=0, atol=ORACLE_ATOL)
