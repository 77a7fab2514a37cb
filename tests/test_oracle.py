"""CPU tests of the oracle itself: self-consistency and the reference golden vectors."""
import io
import os
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import batch, refshape
from vfclik_b200 import workloads


def test_fk_jacobian_finite_differences(lwr):
    chain, _ = lwr
    rng = np.random.default_rng(0)
    q = rng.uniform(chain.q_lo, chain.q_hi, size=(64, 7))
    R, p, J = batch.fk_jac(chain, q)
    eps = 1e-6
    for j in range(7):
        qp, qm = q.copy(), q.copy()
        qp[:, j] += eps
        qm[:, j] -= eps
        Rp, pp, _ = batch.fk_jac(chain, qp)
        Rm, pm, _ = batch.fk_jac(chain, qm)
        assert np.allclose((pp - pm) / (2 * eps), J[:, 0:3, j], atol=1e-8)
        dR = ((Rp - Rm) / (2 * eps)) @ np.transpose(R, (0, 2, 1))
        w = np.stack([dR[:, 2, 1], dR[:, 0, 2], dR[:, 1, 0]], axis=1)
        assert np.allclose(w, J[:, 3:6, j], atol=1e-8)
    # rotations stay orthonormal, home pose is the stretched arm: 0.31+0.40+0.39+0.078
    assert np.allclose(R @ np.transpose(R, (0, 2, 1)), np.eye(3), atol=1e-12)
    assert np.allclose(batch.fk_jac(chain, np.zeros((1, 7)))[1] - chain.base[9:12] + [0, 0, 0.31], [[0, 0, 1.178]])


def test_fk_all_joint_types_finite_differences():
    """RotX/RotY/Trans* joints (the kernel canonicalises them to Z joints on the host)."""
    from vfclik_b200 import kdl
    from vfclik_b200.config import chain_from_segments
    segs = [kdl.Segment(kdl.Joint(t), kdl.Frame(kdl.Rotation.RotX(0.3 * (i + 1)) * kdl.Rotation.RotZ(0.2 * i),
                                                 kdl.Vector(0.1 * i, 0.05, 0.2)))
            for i, t in enumerate([kdl.Joint.RotX, kdl.Joint.TransY, kdl.Joint.RotY, kdl.Joint.RotZ,
                                   kdl.Joint.TransX, kdl.Joint.TransZ])]
    chain = chain_from_segments(segs, [[-1, 1]] * 6)
    rng = np.random.default_rng(1)
    q = rng.uniform(-1, 1, size=(16, 6))
    R, p, J = batch.fk_jac(chain, q)
    eps = 1e-6
    for j in range(6):
        qp, qm = q.copy(), q.copy()
        qp[:, j] += eps
        qm[:, j] -= eps
        assert np.allclose((batch.fk_jac(chain, qp)[1] - batch.fk_jac(chain, qm)[1]) / (2 * eps), J[:, 0:3, j], atol=1e-8)


def test_dls_closed_form_equals_svd_form(lwr):
    chain, _ = lwr
    rng = np.random.default_rng(2)
    q = rng.uniform(chain.q_lo, chain.q_hi, size=(256, 7))
    _, _, J = batch.fk_jac(chain, q)
    tw = rng.normal(size=(256, 6))
    prm = batch.Params(ik_lambda=0.05, w_task=(1, 2, 1, 0.5, 1, 1), w_joint=(1, 1, 0.5, 1, 2, 1, 1))
    qd = batch.ikv_dls(prm, J, tw, 7)
    wt, wj = np.asarray(prm.w_task), np.asarray(prm.w_joint)
    for i in range(256):
        Jw = np.diag(wt) @ J[i] @ np.diag(wj)
        U, s, Vt = np.linalg.svd(Jw, full_matrices=False)
        ref = wj * (Vt.T @ np.diag(s / (s * s + prm.ik_lambda ** 2)) @ U.T @ (wt * tw[i]))
        assert np.allclose(qd[i], ref, rtol=1e-9, atol=1e-12)


def test_projector_identities(lwr):
    chain, _ = lwr
    rng = np.random.default_rng(3)
    q = rng.uniform(0.5 * chain.q_lo, 0.5 * chain.q_hi, size=(64, 7))
    _, _, J = batch.fk_jac(chain, q)
    x = rng.normal(size=(64, 7))
    prm = batch.Params(ns_lambda=0.0)
    Bx = batch.ns_project(prm, J, x)
    assert np.allclose(np.einsum("ikn,in->ik", J, Bx), 0, atol=1e-9)          # J B x = 0
    assert np.allclose(batch.ns_project(prm, J, Bx), Bx, atol=1e-9)           # idempotent
    u = batch.ns_basis_1d(prm, J, np.zeros((64, 7)))
    assert np.allclose(np.einsum("in,in->i", u, x)[:, None] * u, Bx, atol=1e-9)   # B = u u^T (1-D nullspace)


def test_rot_axis_angle_round_trip():
    rng = np.random.default_rng(4)
    axis = rng.normal(size=(500, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    ang = np.concatenate([rng.uniform(0, np.pi, 480), np.pi - rng.uniform(0, 1e-6, 10), rng.uniform(0, 1e-7, 10)])
    K = np.zeros((500, 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 0] = -axis[:, 2], axis[:, 1], axis[:, 2]
    K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -axis[:, 0], -axis[:, 1], axis[:, 0]
    R = np.eye(3) + np.sin(ang)[:, None, None] * K + (1 - np.cos(ang))[:, None, None] * (K @ K)
    a2, g2 = batch.rot_axis_angle(R)
    assert np.allclose(g2, ang, atol=1e-7)
    big = ang > 1e-3
    assert np.allclose((a2 * g2[:, None])[big], (axis * ang[:, None])[big], atol=1e-6) or \
        np.allclose(np.abs(np.einsum("in,in->i", a2[big], axis[big])), 1, atol=1e-9)


@pytest.mark.parametrize("ns_mode", [0, 1, 2])
def test_batch_equals_reference_shaped_loop(lwr, ns_mode):
    """oracle.batch (vectorised) and oracle.refshape (reference-shaped scalar loop) agree."""
    chain, cfg = lwr
    I, M = 24, 5
    K = 4 if ns_mode != 2 else 1     # mode 2: LAPACK's first-cycle sign is arbitrary, so trajectories may mirror
    w = workloads.random_batch(chain, I, M, seed=10 + ns_mode)
    q = w["q"].T
    goal = w["goal"].T
    obst = w["obst"].transpose(1, 0, 2)
    # mode 2 (reference control interface) is the reference's algorithm only with the undamped pinv
    prm = batch.Params(ns_mode=ns_mode, ns_lambda=0.0 if ns_mode == 2 else 0.1,
                       jp_ref=tuple(cfg.initial_joint_pos), ns_control=(0.4, 0, 0, 0),
                       mixer_w=(1.0, 1.0, 0.25, 0, 0, 0), tool=(0, -1, 0, 1, 0, 0, 0, 0, 1, 0.02, -0.01, 0.12))
    out = batch.step(chain, prm, q, goal, obst, k_cycles=K)
    for i in range(I):
        g = goal[i]
        g17 = [g[0], g[1], g[2], g[9], g[3], g[4], g[5], g[10], g[6], g[7], g[8], g[11], 0, 0, 0, 1, g[12]]
        loop = refshape.ControlLoop(chain, prm, q[i], g17, obstacles=obst[i])
        loop.run(K)
        keys = ["qdot_vf", "qdot_jp", "qdot"] if ns_mode != 2 else ["qdot_vf", "qdot_jp"]
        for k in keys + (["qdot_ns"] if ns_mode == 1 else []):
            assert np.allclose(loop.last[k], out[k][i], rtol=1e-9, atol=1e-12), (i, k)
        if ns_mode == 2:
            # LAPACK's first-cycle sign is arbitrary: compare up to one global sign per instance
            a, b = np.asarray(loop.last["qdot_ns"]), out["qdot_ns"][i]
            assert np.allclose(a, b, rtol=1e-8, atol=1e-11) or np.allclose(a, -b, rtol=1e-8, atol=1e-11)
        else:
            assert np.allclose(loop.q, out["q"][i], rtol=1e-10, atol=1e-12)
            assert loop.last["flags"] == out["flags"][i]
        T = np.asarray(loop.last["pose"]).reshape(4, 4)
        assert np.allclose(np.concatenate([T[:3, :3].reshape(9), T[:3, 3]]), out["pose"][i], atol=1e-12)


def test_config1_runs_and_converges(lwr):
    """BASELINE config 1: single LWR, goal of old/system_start.sh.old:346, 3 obstacles, 1000 cycles."""
    chain, cfg = lwr
    w = workloads.config1(chain, cfg)
    prm = batch.Params(jp_ref=tuple(cfg.initial_joint_pos), speed_scale=cfg.speedScale, dt=cfg.rate)
    out = batch.step(chain, prm, w["q"].T, w["goal"].T, w["obst"].transpose(1, 0, 2), k_cycles=1000)
    assert np.all(np.isfinite(out["q"]))
    d0 = np.linalg.norm(batch.fk_jac(chain, w["q"].T)[1][0] - w["goal"][9:12, 0])
    d1 = np.linalg.norm(out["pose"][0, 9:12] - w["goal"][9:12, 0])
    assert d1 < 0.02 < d0            # reached the goal's slow-down ball
    assert np.all(out["q"] >= chain.q_lo - 1e-9) and np.all(out["q"] <= chain.q_hi + 1e-9)


# ------------------------------------------------------------------ golden vectors (real reference code)

def test_golden_command_mixer(golden):
    """refshape.CommandMixer reproduces the real src/command_mixer.py on a scripted port sequence."""
    ev, wev, short = golden["mixer_events"], golden["mixer_wevents"], golden["mixer_short"]
    steps, n_ports, n = ev.shape
    now = [1000.0]
    ports = [refshape.Port() for _ in range(n_ports)]
    wport = refshape.Port()
    mixer = refshape.CommandMixer(ports, wport, n, 2.0, [1.0, 1.0, 0.0, 0.0, 0.0, 0.0], clock=lambda: now[0])
    for s in range(steps):
        now[0] += float(golden["mixer_dts"][s])
        for p in range(n_ports):
            if not np.isnan(ev[s, p, 0]):
                ports[p].write_list(ev[s, p])
            elif short[s, p]:
                ports[p].write_list([0.0] * (n - 2))
        wv = wev[s][~np.isnan(wev[s])]
        if wv.size:
            wport.write_list(wv)
        with redirect_stdout(io.StringIO()):
            out = mixer.read()
        assert np.array_equal(np.asarray(out), golden["mixer_out"][s]), s       # bit-exact: same op order
        assert np.array_equal(np.asarray(mixer.weights), golden["mixer_weights_after"][s])
    with redirect_stdout(io.StringIO()):
        m2 = refshape.CommandMixer([refshape.Port(), refshape.Port()], None, 3, 1.0, [1.0])
    assert np.array_equal(np.asarray(m2.weights), golden["mixer_bad_init_weights"])


def test_golden_nullspace(golden, lwr):
    """refshape.Nullspace and oracle.batch reproduce the real scripts/nullspace functions."""
    chain, _ = lwr
    q, J = golden["ns_q"], golden["ns_J"]
    assert np.allclose(batch.fk_jac(chain, q)[2], J, atol=1e-14)       # fixture J is this oracle's J
    ns = refshape.Nullspace(7, ns_lambda=0.0)
    control = list(golden["ns_control"])
    limits = [[float(a), float(b)] for a, b in zip(chain.q_lo, chain.q_hi)]
    prm0 = batch.Params(ns_lambda=0.0)
    lastvec = np.zeros((1, 7))
    for s in range(q.shape[0]):
        B = ns.restrict(np.eye(6), J[s])
        assert np.allclose(B, golden["ns_B"][s], atol=1e-10)
        qd = ns.move_in_nullspace(np.eye(6), J[s], control)
        assert np.allclose(qd, golden["ns_qdot"][s], atol=1e-10)
        scaled = [v * (25.0 if s % 3 == 2 else 1.0) for v in golden["ns_qdot"][s]]
        out, hit = refshape.Nullspace.check_limits(list(q[s]), scaled, limits)
        assert np.allclose(out, golden["ns_limited"][s], atol=1e-12) and hit == bool(golden["ns_hit"][s])
        # batch oracle: projector columns and the 1-D basis (up to the LAPACK first-cycle sign)
        Bb = np.stack([batch.ns_project(prm0, J[s:s + 1], np.eye(7)[j:j + 1])[0] for j in range(7)], axis=1)
        assert np.allclose(Bb, golden["ns_B"][s], atol=1e-9)
        u = batch.ns_basis_1d(prm0, J[s:s + 1], lastvec)
        lastvec = u
        g = golden["ns_basis"][s]
        assert np.allclose(u[0], g, atol=1e-8) or np.allclose(u[0], -g, atol=1e-8)
    assert np.any(golden["ns_hit"]) and not np.all(golden["ns_hit"])
    assert int(golden["ns_rank"]) == 6
    # sign continuity: the batch basis never flips between consecutive cycles, like the reference's
    Jr = golden["ns_Jrand"]
    for k in range(Jr.shape[0]):
        Bb = np.stack([batch.ns_project(prm0, Jr[k:k + 1], np.eye(7)[j:j + 1])[0] for j in range(7)], axis=1)
        assert np.allclose(Bb, golden["ns_Brand"][k], atol=1e-9)


@pytest.mark.parametrize("n", [10, 8])
def test_golden_nullspace_wide(golden, n):
    """k = N - 6 > 1 (the reference's iCub shape, 10 joints -> 4 vectors; 8 joints -> 2): the oracle's basis against the
    executed ``scripts/nullspace`` functions.  The basis of a degenerate singular subspace is LAPACK's free choice, so the
    comparison is through what IS determined: the projector ``sum u u^T``, the span, the number of vectors, orthonormality,
    sign continuity, and the length of the motion for the same four control floats."""
    tag = "ns%d_" % n
    J, B, Uref, qd_ref = golden[tag + "J"], golden[tag + "B"], golden[tag + "basis"], golden[tag + "qdot"]
    control = golden[tag + "control"]
    steps, k = J.shape[0], n - 6
    assert Uref.shape == (steps, k, n) and batch.ns_ctrl_vectors(n) == min(4, k)
    chain = workloads.torso_arm_chain(n)
    assert np.allclose(batch.fk_jac(chain, golden[tag + "q"])[2], J, atol=1e-14)
    prm0 = batch.Params(ns_lambda=0.0)
    U = batch.ns_basis(J)                                                   # [steps, k, n]
    for s in range(steps):
        # the executed reference: projector and its own basis agree, and the basis is orthonormal
        assert np.allclose(Uref[s].T @ Uref[s], B[s], atol=1e-10)
        Q = np.linalg.qr(J[s].T, mode="complete")[0]
        assert np.allclose(U[s], Q[:, 6:].T, atol=1e-12)                    # LAPACK's own Householder QR
        assert np.allclose(U[s] @ U[s].T, np.eye(k), atol=1e-12)
        assert np.allclose(U[s].T @ U[s], B[s], atol=1e-9)                  # same projector
        assert np.allclose(U[s] @ B[s], U[s], atol=1e-9)                    # same span
        assert np.linalg.matrix_rank(np.vstack([U[s], Uref[s]]), tol=1e-8) == k
        Bb = np.stack([batch.ns_project(prm0, J[s:s + 1], np.eye(n)[j:j + 1])[0] for j in range(n)], axis=1)
        assert np.allclose(Bb, B[s], atol=1e-10)
    # control motion: sum of min(4, k) orthonormal vectors -> |qdot| = |control[:kk]|, inside null(J); sign-continuous
    kk = min(4, k)
    last = np.zeros((1, kk * n))
    prev = None
    for s in range(steps):
        qd, last = batch.ns_control_motion(J[s:s + 1], last, control[None, :])
        assert np.allclose(np.linalg.norm(qd), np.linalg.norm(control[:kk]), rtol=1e-12)
        assert np.allclose(np.linalg.norm(qd_ref[s]), np.linalg.norm(control[:kk]), rtol=1e-10)
        assert np.allclose(J[s] @ qd[0], 0, atol=1e-12) and np.allclose(J[s] @ qd_ref[s], 0, atol=1e-10)
        assert np.allclose(B[s] @ qd[0], qd[0], atol=1e-9)
        u = last.reshape(kk, n)
        if prev is not None:
            assert np.all(np.einsum("kn,kn->k", u, prev) >= 0.0)
        prev = u


def test_ns_basis_small_and_padded_chains():
    """N <= 6: empty nullspace, zero motion.  Zero Jacobian columns (how the kernel pads a short chain into a larger
    instantiation) leave the leading vectors of the basis untouched."""
    rng = np.random.default_rng(12)
    for n in (3, 6):
        J = rng.normal(size=(5, 6, n))
        assert batch.ns_basis(J).shape == (5, 0, n)
        qd, _ = batch.ns_control_motion(J, np.zeros((5, n)), np.ones((5, 4)))
        assert np.all(qd == 0)
    J = rng.normal(size=(5, 6, 8))
    Jp = np.concatenate([J, np.zeros((5, 6, 2))], axis=2)
    assert np.allclose(batch.ns_basis(Jp, 2)[:, :, :8], batch.ns_basis(J), atol=1e-14)
    assert np.all(batch.ns_basis(Jp, 2)[:, :, 8:] == 0)


def test_ik_mode_kdl_wdls_form(lwr):
    """ORACLE_CHOICES 'velocity IK vs KDL': away from singularities the truncated form is the plain weighted pseudo-inverse
    and differs from north_star's uniformly damped form by O(lambda^2 / sigma^2); with lambda = 0 the two coincide."""
    chain, _ = lwr
    rng = np.random.default_rng(13)
    q = rng.uniform(0.5 * chain.q_lo, 0.5 * chain.q_hi, size=(64, 7))
    _, _, J = batch.fk_jac(chain, q)
    tw = rng.normal(size=(64, 6))
    a = batch.ikv_dls(batch.Params(ik_lambda=0.0), J, tw, 7)
    b = batch.ikv_dls(batch.Params(ik_lambda=0.1, ik_mode=1), J, tw, 7)
    assert np.allclose(a, b, rtol=1e-7, atol=1e-9)
    assert np.allclose(np.einsum("ikn,in->ik", J, b), tw, atol=1e-8)          # exact task-space tracking
    c = batch.ikv_dls(batch.Params(ik_lambda=0.1), J, tw, 7)
    assert not np.allclose(c, b, rtol=1e-3)


@pytest.mark.skipif(not os.path.isdir(os.environ.get("VFCLIK_REFERENCE", "")),
                    reason="needs the original vfclik sources: set VFCLIK_REFERENCE to a checkout of them")
def test_golden_is_reproducible_from_reference(golden):
    """Regenerating from the real reference gives the committed vectors (guards a stale fixture)."""
    from oracle import gen_golden
    rng = np.random.default_rng(20261018)
    data = gen_golden.gen_mixer(rng)
    data.update(gen_golden.gen_nullspace(rng))
    data.update(gen_golden.gen_bridge(rng))
    data.update(gen_golden.gen_feeder())
    data.update(gen_golden.gen_jp(rng))
    data.update(gen_golden.gen_vf(rng))
    data.update(gen_golden.gen_bridge_loop(rng))
    data.update(gen_golden.gen_dmonitor(rng))
    data.update(gen_golden.gen_nullspace_loop(rng))
    data.update(gen_golden.gen_handlers())
    data.update(gen_golden.gen_nullspace_wide())
    data.update(gen_golden.gen_bridge_readpos())
    for k, v in data.items():
        if np.asarray(v).dtype.kind in "US":
            assert [str(x) for x in v] == [str(x) for x in golden[k]], k
            continue
        assert np.allclose(np.asarray(v, dtype=np.float64), np.asarray(golden[k], dtype=np.float64), equal_nan=True,
                           atol=1e-12), k


def test_operation_count_is_frozen_and_counts_the_oracle(lwr):
    """SURVEY.md 8(d): the FLOP constants bench.py computes the K-fused roofline from are an exact count of the oracle's
    cycle -- the counting implementation must reproduce oracle.batch.step, and its counts must equal the frozen table."""
    from oracle import opcount
    chain, _ = lwr
    prm = batch.Params()
    rng = np.random.default_rng(5)
    w = workloads.random_batch(chain, 4, 32, seed=11)
    for i in range(4):
        q, goal, obst = w["q"][:, i], w["goal"][:, i], w["obst"][:, i, :]
        out, _ = opcount.cycle(chain, prm, q, goal, obst)
        ref = batch.step(chain, prm, q[None, :], goal[None, :], obst[None, :, :])
        assert np.allclose(out["qdot"], ref["qdot"][0], rtol=1e-10, atol=1e-13)
        assert np.allclose(out["q"], ref["q"][0], rtol=1e-12, atol=1e-13)
    for (n, m), (flops, trans) in workloads.ALGORITHMIC_OPS.items():
        ch = chain if n == 7 else workloads.dual_arm_torso_chain()
        c = opcount.count(ch, m, samples=3)
        assert (c.flops, c.transcendentals) == (flops, trans), ((n, m), c.flops, c.transcendentals)
    assert workloads.algorithmic_flops(7, 64) == workloads.ALGORITHMIC_OPS[(7, 32)][0] + 20 * 32


def test_powercube_bridge_restatement_matches_batch(lwr):
    """Row f4: the statement-for-statement Powercube set_vel of the reference-shaped loop (scripts/bridge:288-305)
    equals the vectorised oracle, including the doubled leading ratio when the shoulder limit is not hit."""
    import dataclasses
    chain, cfg = lwr
    prm = dataclasses.replace(batch.Params(), speed_scale=0.41, max_vel=0.3, bridge_kind=1, shoulder_vel=(0.05, -0.08))
    w = workloads.random_batch(chain, 12, 3, seed=23)
    seen = set()
    for i in range(12):
        q, goal, obst = w["q"][:, i], w["goal"][:, i], w["obst"][:, i, :]
        ref = batch.step(chain, prm, q[None], goal[None], obst[None])
        g = goal
        g17 = [g[0], g[1], g[2], g[9], g[3], g[4], g[5], g[10], g[6], g[7], g[8], g[11], 0, 0, 0, 1, g[12]]
        loop = refshape.ControlLoop(chain, prm, q, g17, obstacles=obst)
        with redirect_stdout(io.StringIO()):
            qd = loop.cycle()
        assert np.allclose(qd, ref["qdot"][0], rtol=1e-9, atol=1e-12)
        assert np.allclose(loop.last["cmd"], ref["qdot"][0], rtol=1e-9, atol=1e-12)
        lead = np.max(np.abs(ref["qdot_mix"][0]))
        first = ref["qdot_mix"][0, 0] * min(1.0, prm.max_vel / lead)
        seen.add("shoulder" if (first > 0.05 or first < -0.08) else ("double" if lead > prm.max_vel else "none"))
    assert {"shoulder", "double"} <= seen


def test_golden_bridge_backends_joint_limits_and_weight_matrix(golden, capsys):
    """Vectors produced by executing the reference's own `set_vel` of the three bridge back-ends, `set_torso_cjoints`,
    `joint_p_controller.check_limits` and `vf.get_weight_matrix` (oracle/gen_golden.py:gen_bridge) against the oracle's
    restatement and the host modules' parsers."""
    import dataclasses
    import types
    g = golden
    qdot, q, qc = g["br_qdot"], g["br_q"], g["br_qcmded"]
    max_vel, sh_pos, sh_neg = [float(v) for v in g["br_cfg"]]
    base = dataclasses.replace(batch.Params(), max_vel=max_vel, shoulder_vel=(sh_pos, sh_neg))
    for direct in (0, 1):
        _, cmd, _ = batch.bridge_set_vel(base, qdot, q, qc, bool(direct))
        assert np.allclose(cmd, g["br_lwr_cmd_direct%d" % direct], rtol=1e-14, atol=1e-15)
    for kind, key in ((1, "br_powercube_cmd"), (2, "br_icub_cmd")):
        qd, cmd, _ = batch.bridge_set_vel(dataclasses.replace(base, bridge_kind=kind), qdot, q, qc, False)
        assert np.allclose(cmd, g[key], rtol=1e-14, atol=1e-15) and np.array_equal(cmd, qd)
    # the vectors exercise every branch: no clamp, leading clamp only (applied twice by the Powercube code), shoulder clamp
    lead = np.max(np.abs(qdot), axis=1)
    first = qdot[:, 0] * np.minimum(1.0, max_vel / lead)
    assert np.any(lead <= max_vel) and np.any((lead > max_vel) & (first <= sh_pos) & (first >= sh_neg))
    assert np.any(first > sh_pos) and np.any(first < sh_neg)
    # joint_p_controller.check_limits through the module's own clamp (posture-dependent limits)
    from vfclik_b200.joint_p_controller import JointPControllerModule
    sent = []
    jp = object.__new__(JointPControllerModule)
    jp.nJoints = 7
    jp.rt = types.SimpleNamespace(config=types.SimpleNamespace(updateJntLimits=lambda cur: [[-0.5 - abs(cur[0]), 0.4 + abs(cur[1])]] * 7),
                                  set_jp_ref=lambda r: sent.append(list(r)))
    for k in range(g["jp_ref"].shape[0]):
        jp.ref = list(g["jp_ref"][k])
        jp._ref_sent = None
        jp._apply_position_dependent_limits(list(q[k]))
        assert np.array_equal(jp._ref_sent, g["jp_ref_clamped"][k])
    capsys.readouterr()
    # vf.get_weight_matrix: diagonal of the reference's matrix; wrong sizes ignored
    from vfclik_b200 import ports as yarp
    from vfclik_b200.vf import get_weight_matrix
    for tag, w, mat, n in (("t", g["vf_wt"], g["vf_wt_matrix"], 6), ("j", g["vf_wj"], g["vf_wj_matrix"], 7)):
        b = yarp.Bottle.from_list([tag] + [float(v) for v in w])
        got = get_weight_matrix(b, n)
        assert np.array_equal(np.diag(got), mat)
        assert get_weight_matrix(yarp.Bottle.from_list([tag] + [float(v) for v in w[:3]]), n) is None
    assert "Wrong size" in capsys.readouterr().out


def test_golden_joint_p_controller_loop(golden, lwr):
    """The reference-shaped loop's joint-controller stage against the reference's own loop (scripts/joint_p_controller:96-146)
    run on a scripted sequence with the LWR's static limits: clamp, P law and the signed at-goal compare."""
    chain, cfg = lwr
    g = golden
    kp, delta = [float(v) for v in g["jp_kp_delta"]]
    assert np.allclose(g["jp_static_limits"], np.stack([chain.q_lo, chain.q_hi], axis=1))
    prm = batch.Params(jp_kp=kp, jp_delta=delta, jp_ref=tuple(cfg.initial_joint_pos))
    steps = {int(k): g["jp_ref_msgs"][i] for i, k in enumerate(g["jp_ref_steps"])}
    loop = refshape.ControlLoop(chain, prm, g["jp_q"][0], cfg.initial_vf_pose[2])
    for k in range(g["jp_q"].shape[0]):
        if k in steps:
            loop.ref = [float(v) for v in steps[k]]
        loop.q = [float(v) for v in g["jp_q"][k]]
        with redirect_stdout(io.StringIO()):
            loop.cycle()
        assert np.allclose(loop.last["qdot_jp"], g["jp_out_static"][k], rtol=1e-13, atol=1e-15), k
        assert bool(loop.last["flags"] & batch.FLAG_AT_GOAL) == bool(g["jp_at_goal_static"][k]), k
        # the vectorised oracle on the same step (any goal: the joint controller does not look at it)
        goal = np.array([[1, 0, 0, 0, 1, 0, 0, 0, 1, 0.5, 0.0, 0.8, 0.05]], dtype=np.float64)
        ref_b = batch.step(chain, prm, g["jp_q"][k][None], goal, None, jp_ref=np.asarray(steps[max(s for s in steps if s <= k)])[None])
        assert np.allclose(ref_b["qdot_jp"][0], g["jp_out_static"][k], rtol=1e-13, atol=1e-15), k


def test_golden_distance_monitor_loop(golden):
    """oracle/monitor.py (the restatement the vfk_monitor kernel is tested against) versus what the reference's own
    monitor_distance loop body (scripts/monitor_distance:107-221, with its orientLength) wrote for a scripted approach:
    distances to every object each cycle, and the 20-sample majority state messages -- including the reference sending the
    xyz state under the "rot" tag."""
    import json
    from oracle import monitor
    from oracle.refshape import listToKdlFrame
    g = golden
    dm = monitor.DistanceMonitor()
    objects = {}
    last_x = last_r = "on goal"
    n_msgs = 0
    for k in range(g["dm_script"].shape[0]):
        ev = json.loads(str(g["dm_script"][k]))
        want = json.loads(str(g["dm_out"][k]))
        def apply(m):
            if m[0] == "add":
                objects[m[1]] = m[2]
            else:
                objects.pop(m[1], None)
        pending = list(ev.get("objects", []))
        if pending:                        # the loop takes ONE /objectsIn message per iteration; the pose is consumed by the first
            apply(pending.pop(0))
        frame = listToKdlFrame(ev["pose"])
        msgs = []
        rows = []
        for oid in sorted(objects):
            goal = listToKdlFrame(objects[oid])
            if oid == 0:
                dx, do, mx, mr = dm.update(frame, goal, ev["track_error"])
                if mx is not None and mx != last_x:
                    last_x = mx
                    msgs.append(["xyz", mx])
                if mr is not None and mr != last_r:
                    last_r = mr
                    msgs.append(["rot", mx])                  # sic: scripts/monitor_distance:215 sends the xyz state
            else:
                d = frame.p - goal.p
                dx, do = float(np.sqrt(d @ d)), monitor.orientLength(goal, frame)
            rows.append([float(oid), dx, do])
        assert len(want["distOut"]) == 1
        assert np.allclose(rows, want["distOut"][0], rtol=1e-12, atol=1e-12), k
        assert msgs == want["tracking_state"], (k, msgs, want["tracking_state"])
        n_msgs += len(msgs)
        for m in pending:
            apply(m)
    assert n_msgs >= 6
