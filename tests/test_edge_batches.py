"""The batch constructors of tests/helpers.py that put goals and obstacles next to the tool, and postures next to kinematic
singularities (CPU only): through the oracle's FK the requested distances and angles come out as asked, every combination
is drawn, FP32 batches stay clear of the repeller-weight saturation, and singular postures have the chain's known rank."""
import numpy as np
import pytest

import helpers
from helpers import near_goal, near_obstacles, near_singular, tool_frame


def _chains(lwr):
    from vfclik_b200 import workloads
    return {"lwr": (lwr[0], None), "dh17": (workloads.dual_arm_torso_chain(17), None),
            "tool10": (workloads.torso_arm_chain(10), (0, -1, 0, 1, 0, 0, 0, 0, 1, 0.03, -0.02, 0.15))}


@pytest.mark.parametrize("which", ["lwr", "dh17", "tool10"])
@pytest.mark.parametrize("rot_slowdown", [0.09, 0.5, 0.0])
def test_near_goal_distances_and_angles(lwr, which, rot_slowdown):
    from oracle import batch
    chain, tool = _chains(lwr)[which]
    n = 800
    w, meta = near_goal(chain, n, 4, seed=5, rot_slowdown=rot_slowdown, tool=tool)
    R, p = tool_frame(chain, w["q"], tool)
    goal = w["goal"].T
    assert np.max(np.abs(np.linalg.norm(goal[:, 9:12] - p, axis=1) - meta["d"])) <= 1e-12
    _, angle = batch.rot_axis_angle(goal[:, 0:9].reshape(n, 3, 3) @ np.transpose(R, (0, 2, 1)))
    assert np.max(np.abs(angle - meta["theta"])) <= 1e-12
    assert np.array_equal(goal[:, 12], meta["slowdown"])
    # every (slowdown, distance, angle) combination is drawn
    combos = {(s, d, t) for s in helpers.SLOWDOWNS for d in helpers.goal_distances(s) for t in helpers.goal_angles(rot_slowdown)}
    assert set(zip(meta["slowdown"], meta["d"], meta["theta"])) == combos
    # the states the slowdowns act on are there: S0 < 1 and S1 < 1 together
    if rot_slowdown > 0:
        assert np.any((meta["d"] < meta["slowdown"]) & (meta["theta"] < rot_slowdown) & (meta["d"] <= 1e-4))


@pytest.mark.parametrize("which", ["lwr", "dh17", "tool10"])
@pytest.mark.parametrize("ext", [True, False])
def test_near_obstacles_distances(lwr, which, ext):
    chain, tool = _chains(lwr)[which]
    n, M = 600, 19
    w, meta = near_obstacles(chain, n, M, seed=6, obst_ext=ext, safe=1e-3, order=20.0, n_near=3, tool=tool)
    _, pt = tool_frame(chain, w["q"], tool)
    cols = np.arange(n)
    for k in range(3):
        o = w["obst"][meta["slot"][k], cols]
        assert np.max(np.abs(np.linalg.norm(o[:, 0:3] - pt, axis=1) - meta["d"][k])) <= 1e-12
    assert np.all(meta["slot"][0] != meta["slot"][1]) and np.all(meta["slot"][1] != meta["slot"][2])
    if ext:
        assert set(np.unique(w["obst_ext"][:, :, 0])) == set(helpers.OBST_SAFES)
        assert set(np.unique(w["obst_ext"][:, :, 1])) == set(helpers.OBST_ORDERS)
        safe = w["obst_ext"][meta["slot"][0], cols, 0]
        d = meta["d"][0]
        assert np.any(d < safe) and np.any((d > safe) & (safe > 0))        # inside and outside the safe distance
    else:
        assert np.any(meta["d"] < 1e-3)


@pytest.mark.parametrize("ext,safe,order", [(True, 1e-3, 20.0), (False, 1e-3, 20.0), (False, 0.0, 7.5), (False, 0.05, 2.0)])
def test_near_obstacles_fp32_weights_stay_below_saturation(lwr, ext, safe, order):
    n, M = 600, 17
    w, meta = near_obstacles(lwr[0], n, M, seed=7, dtype=np.float32, obst_ext=ext, safe=safe, order=order, n_near=2)
    assert w["obst"].dtype == np.float32
    _, pt = tool_frame(lwr[0], w["q"])
    cols = np.arange(n)
    for k in range(2):
        o = w["obst"][meta["slot"][k], cols].astype(np.float64)
        d = np.linalg.norm(o[:, 0:3] - pt, axis=1)
        sf, od = (w["obst_ext"][meta["slot"][k], cols, 0], w["obst_ext"][meta["slot"][k], cols, 1]) if ext else (safe, order)
        wgt = (o[:, 3] / np.maximum(d, sf)) ** od / d
        assert np.all(wgt <= 1.5 * helpers.FP32_WEIGHT_LIMIT)
        if ext:
            assert np.any(wgt > 1e10)                              # still steep: the bound lowers orders only where needed


def _singular_cases():
    return [("lwr", "home"), ("lwr", "elbow"), ("tool10", "home"), ("dh17", "home"), ("generic17", "home")]


@pytest.mark.parametrize("which,kind", _singular_cases())
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_near_singular_levels_rank_and_limits(lwr, which, kind, dtype):
    """near_singular: every level is drawn; at delta = 0 the oracle's Jacobian has the chain's known rank (numpy's pinv cutoff,
    1e-15 sigma_max); sigma_min / sigma_max grows linearly with delta (all these singularities are first order: within a
    factor of the median over the batch at every level); q stays inside the limits and in the requested dtype; elbow moves
    q[3] only."""
    from vfclik_b200 import workloads
    chain = {"lwr": lambda: lwr[0], "tool10": lambda: workloads.torso_arm_chain(10),
             "dh17": lambda: workloads.dual_arm_torso_chain(17),
             "generic17": lambda: workloads.dual_arm_torso_chain(17, dh=False)}[which]()
    rank0 = {("lwr", "home"): 3, ("lwr", "elbow"): 5, ("tool10", "home"): 4, ("dh17", "home"): 5, ("generic17", "home"): 4}
    n = 1200
    w, meta = near_singular(chain, n, 4, seed=8, dtype=dtype, kind=kind)
    q = w["q"]
    assert q.dtype == dtype and q.shape == (len(chain.q_lo), n)
    assert np.all(q >= chain.q_lo[:, None]) and np.all(q <= chain.q_hi[:, None])
    assert set(meta["delta"]) == set(helpers.SINGULAR_LEVELS)
    counts = np.array([np.count_nonzero(meta["delta"] == d) for d in helpers.SINGULAR_LEVELS])
    assert counts.max() - counts.min() <= 1
    sigma = meta["sigma"]
    assert np.array_equal(sigma, helpers.singular_values(chain, q))
    rel = sigma / sigma[:, :1]
    at0 = meta["delta"] == 0
    assert np.all(np.count_nonzero(rel[at0] > 1e-15, axis=1) == rank0[(which, kind)])
    assert np.all(np.isinf(meta["cond"][at0]) | (meta["cond"][at0] > 1e15))
    if kind == "home":
        assert np.all(q[:, at0] == 0)
    else:
        ref = workloads.random_batch(chain, n, 4, seed=8, dtype=dtype)["q"]
        assert np.all(q[3, at0] == 0)
        assert np.array_equal(np.delete(q, 3, axis=0), np.delete(ref, 3, axis=0))
        assert np.array_equal(np.abs(q[3]).astype(np.float64), meta["delta"].astype(dtype).astype(np.float64))
    # first order: sigma_min / sigma_max / delta stays within a factor of its median, at every level from 1e-12 to 1e-1
    smin = rel[:, -1]
    med = {}
    for d in helpers.SINGULAR_LEVELS[1:]:
        at = meta["delta"] == d
        med[d] = np.median(smin[at] / d)
        assert np.all(smin[at] > 0)
        assert np.quantile(smin[at] / d, 0.05) > med[d] / 100
        assert np.all(smin[at] / d < 30 * med[d])
    ratios = np.array(list(med.values()))
    assert ratios.max() / ratios.min() < 10
