"""Reference for vfk_solve (test infrastructure): ``oracle.batch.step`` run one cycle at a time until each instance's tool
reaches its goal.  Kept beside the tests that use it; it only calls the oracle's published functions."""
import numpy as np

from oracle import batch


def goal_distance(chain, prm: batch.Params, q, goal):
    """Distance monitor of ``scripts/monitor_distance:148-219`` for the tool frame at q [I, N]: ``(|p_goal - p_tool|,
    angle of R_goal R_tool^T in [0, pi])`` in metres and radians, each [I]."""
    I = q.shape[0]
    tool = np.asarray(prm.tool, dtype=np.float64)
    R, p, _ = batch.fk_jac(chain, q)
    Rt = R @ tool[:9].reshape(3, 3)
    pt = p + R @ tool[9:12]
    goal = np.asarray(goal, dtype=np.float64)
    d = np.linalg.norm(goal[:, 9:12] - pt, axis=1)
    _, angle = batch.rot_axis_angle(goal[:, 0:9].reshape(I, 3, 3) @ np.transpose(Rt, (0, 2, 1)))
    return d, angle


def solve(chain, prm: batch.Params, q, goal, obst, max_cycles: int, tol_trans: float, tol_rot: float, **step_kw):
    """Each instance's control loop until its tool reaches the goal (``vfk_solve``, include/vfk.h): the batched
    ``HandleArm.gotoFrame(frame, wait, goal_precision)`` (``src/handlers.py:346-387``), which polls the distance monitor
    until both distances are below ``goal_precision`` (strict, ``:123``).  ``tol_rot >= pi`` ignores the orientation.

    ``step`` one cycle at a time; before every cycle, and once after the last, the rule is checked at the current q, and an
    instance that meets it is frozen: no further integration, and the state ``step`` carries (``jp_ref`` with
    ``jp_limits``, ``lastvec``) keeps its value.  Returns ``q``, ``cycles`` [I] (the first c in 0..max_cycles with the rule
    at q_c, or -1), ``dist`` [I, 2] (``goal_distance`` at the returned q), and ``jp_ref`` / ``lastvec`` where ``step``
    returns them."""
    q = np.array(q, dtype=np.float64, copy=True)
    I, N = q.shape
    jp_ref = step_kw.pop("jp_ref", None)
    lastvec = step_kw.pop("lastvec", None)
    if jp_ref is not None:
        jp_ref = np.array(jp_ref, dtype=np.float64, copy=True)
    if lastvec is None and prm.ns_mode == 2:
        lastvec = np.zeros((I, max(1, batch.ns_ctrl_vectors(N)) * N))
    elif lastvec is not None:
        lastvec = np.array(lastvec, dtype=np.float64, copy=True)
    cycles = np.full(I, -1, dtype=np.int32)
    done = np.zeros(I, dtype=bool)
    for c in range(max_cycles + 1):
        d, angle = goal_distance(chain, prm, q, goal)
        hit = ~done & (d < tol_trans) & ((angle < tol_rot) | (tol_rot >= np.pi))
        cycles[hit] = c
        done |= hit
        if c == max_cycles or done.all():
            break
        out = batch.step(chain, prm, q, goal, obst, jp_ref=jp_ref, lastvec=lastvec, k_cycles=1, **step_kw)
        run = ~done
        q[run] = out["q"][run]
        if jp_ref is not None and "jp_ref" in out:
            jp_ref[run] = out["jp_ref"][run]
        if lastvec is not None and "lastvec" in out:
            lastvec[run] = out["lastvec"][run]
    res = dict(q=q, cycles=cycles, dist=np.stack([d, angle], axis=1))
    if jp_ref is not None and step_kw.get("jp_limits") is not None:
        res["jp_ref"] = jp_ref
    if lastvec is not None:
        res["lastvec"] = lastvec
    return res
