"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle.

Tolerances (BASELINE.json north_star): joint velocities within 1e-9 relative in the FP64
mode and 1e-4 in the FP32 mode; "relative" = per-instance max-norm error over
max(|qdot_ref|_inf, 1e-3 rad/s) (tests/helpers.py:rel_err).  K-cycle trajectories:
1e-9 rad (FP64, K=50) and 2e-3 rad (FP32, K=50).
"""
import dataclasses

import numpy as np
import pytest

from helpers import FP32_RTOL, FP64_RTOL, check, oracle_parallel, oracle_params, rel_err, run_gpu, run_oracle, to_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng(lwr, built_lib):
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr
    engines = {}

    def get(precision, chain_=None):
        key = (precision, id(chain_))
        if key not in engines:
            engines[key] = Engine(chain_ or chain, precision=precision, params=Params.from_config(cfg) if chain_ is None else Params())
        return engines[key]
    yield get
    for e in engines.values():
        e.close()


@pytest.mark.parametrize("n", [1, 127, 4096])
def test_fp64_cycle_matches_oracle(eng, lwr, n):
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(64)
    w = workloads.random_batch(chain, n, 32, seed=0)
    out = run_gpu(e, w, 32)
    ref = run_oracle(chain, e.params, w, 32)
    check(out, ref, FP64_RTOL, pose_atol=1e-12)
    assert np.array_equal(out["flags"], ref["flags"])
    assert np.max(np.abs(out["q"] - ref["q"])) < 1e-12


def test_fp64_config2_65536_instances(eng, lwr):
    """BASELINE config 2: 65,536 LWR instances, FP64, K = 1, per-cycle qdot vs the oracle."""
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(64)
    w = workloads.random_batch(chain, 65536, 32, seed=0)
    out = run_gpu(e, w, 32)
    ref = run_oracle(chain, e.params, w, 32)
    check(out, ref, FP64_RTOL, pose_atol=1e-12)
    assert np.array_equal(out["flags"], ref["flags"])


@pytest.mark.parametrize("n", [1, 1000, 65536])
def test_fp32_cycle_matches_oracle(eng, lwr, n):
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(32)
    w = workloads.random_batch(chain, n, 32, seed=1, dtype=np.float32)
    out = run_gpu(e, w, 32)
    ref = run_oracle(chain, e.params, w, 32)
    check(out, ref, FP32_RTOL, pose_atol=5e-6)
    # flags may differ only where a comparison sits within FP32 rounding of its threshold
    assert np.mean(out["flags"] != ref["flags"]) < 1e-3


@pytest.mark.parametrize("precision,traj_tol", [(64, 1e-9), (32, 2e-3)])
def test_k_cycle_trajectory(eng, lwr, precision, traj_tol):
    """K fused cycles == K oracle cycles: final q within the stated joint-space tolerance (1e-9 rad FP64, 2e-3 rad FP32 after
    50 cycles).  The cycle has two discontinuities -- the all-or-nothing nullspace limit check and the velocity clamp -- so in
    FP32 an instance within rounding of a threshold may take the other branch in some cycle.  Those instances are identified
    by comparing the per-cycle flags; the tolerance is asserted as a MAX over every instance whose flags agree in all 50
    cycles, every outlier must be one of the flag-mismatch instances, and those must stay rare."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    from oracle import batch
    chain, _ = lwr
    e = eng(precision)
    n, M, K = 2048, 8, 50
    w = workloads.random_batch(chain, n, M, seed=2, dtype=np.float32 if precision == 32 else np.float64)
    out = run_gpu(e, w, M, k=K)
    # cycle by cycle on both sides, flags recorded
    db = DeviceBatch(e, n, M, outputs=("qdot", "flags"))
    db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
    q_o, goal_o, obst_o = to_oracle(w, M)
    prm = oracle_params(e.params)
    mismatch = np.zeros(n, dtype=bool)
    for _ in range(K):
        db.step(1)
        o = batch.step(chain, prm, q_o, goal_o, obst_o)
        q_o = o["q"]
        mismatch |= db.download("flags")[0] != o["flags"]
    q_gpu = db.download("q").T
    assert np.array_equal(q_gpu, out["q"])                  # K launches of 1 cycle == 1 launch of K cycles (bit-exact)
    err = np.max(np.abs(q_gpu - q_o), axis=1)
    if precision == 64:
        assert not mismatch.any() and err.max() <= traj_tol
    else:
        assert err[~mismatch].max() <= traj_tol, float(err[~mismatch].max())
        assert np.all(mismatch[err > traj_tol])             # every outlier took a different branch somewhere
        assert mismatch.mean() < 0.02, float(mismatch.mean())


@pytest.mark.parametrize("ns_mode", [0, 1, 2])
def test_nullspace_modes_fp64(eng, lwr, ns_mode):
    """Off / damped projector / the reference's control interface, each at the FP64 tolerance.  Mode 2 is undamped like the
    reference (scripts/nullspace:75-107): the Householder basis of null(J) keeps it at cond(J) * eps, well inside 1e-9."""
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(64)
    old = e.params
    try:
        e.set_params(ns_mode=ns_mode, ns_lambda=0.0 if ns_mode == 2 else 0.05, ns_control=(0.3, 0, 0, 0),
                     mixer_w=(1.0, 1.0, 0.5, 0, 0, 0))
        w = workloads.random_batch(chain, 3000, 4, seed=3)
        extra = {"ns_lastvec": np.zeros((7, 3000))} if ns_mode == 2 else None
        out = run_gpu(e, w, 4, k=3, extra=extra)
        ref = run_oracle(chain, e.params, w, 4, k=3)
        check(out, ref, FP64_RTOL)
        if ns_mode == 2:
            assert np.max(np.abs(out["lastvec"] - ref["lastvec"])) < 1e-9
            assert np.allclose(np.linalg.norm(out["lastvec"], axis=1), 1.0, atol=1e-12)
    finally:
        e.set_params(old)


def test_ik_mode_truncated_fp64(lwr, built_lib):
    """VFK_IK_TRUNCATED: the KDL-wdls-style velocity IK (plain weighted pseudo-inverse above ik_eps, damped below; see
    ORACLE_CHOICES 'velocity IK vs KDL') through the kernel's one-sided Jacobi SVD against the oracle's numpy SVD, unit and
    non-unit weights, at the FP64 tolerance; FP32 refuses it."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params, VfkError
    chain, cfg = lwr
    e = Engine(chain, precision=64, params=Params.from_config(cfg, ik_mode=1, ik_eps=1e-5))
    try:
        for kw in ({}, {"w_task": (1, 1, 1, 0.5, 0.5, 0.5), "w_joint": (1, 0.8, 1, 1.2, 1, 1, 0.5)}):
            e.set_params(**kw)
            w = workloads.random_batch(chain, 2500, 6, seed=51)
            out = run_gpu(e, w, 6, outputs=("qdot_vf", "qdot", "twist", "pose"))
            ref = run_oracle(chain, e.params, w, 6)
            check(out, ref, FP64_RTOL, keys=("qdot_vf", "qdot"))
            # away from singularities the task twist is tracked exactly -- what distinguishes it from the damped form
            from oracle import batch
            J = batch.fk_jac(chain, w["q"].T)[2]
            sig = np.linalg.svd(J, compute_uv=False)
            if not kw:
                ok = sig[:, -1] > 1e-3
                assert np.allclose(np.einsum("ikn,in->ik", J, out["qdot_vf"])[ok], ref["twist"][ok], atol=1e-9)
    finally:
        e.close()
    e32 = Engine(chain, precision=32, params=Params.from_config(cfg))
    try:
        with pytest.raises(VfkError):
            e32.set_params(ik_mode=1)
    finally:
        e32.close()


def test_undamped_projector_is_the_references_restrict(eng, lwr):
    """ns_lambda = 0 in projector mode: B x = (I - pinv(J) J) x of scripts/nullspace:75-79 (numpy SVD pinv in the oracle,
    Q diag(0, 1) Q^T x on the GPU) at the FP64 tolerance, and in the FP32 mode at its own."""
    from vfclik_b200 import workloads
    chain, _ = lwr
    for precision, tol, dt in ((64, FP64_RTOL, np.float64), (32, FP32_RTOL, np.float32)):
        e = eng(precision)
        old = e.params
        try:
            e.set_params(ns_mode=1, ns_lambda=0.0)
            w = workloads.random_batch(chain, 3000, 4, seed=13, dtype=dt)
            rng = np.random.default_rng(14)
            x = rng.normal(scale=0.2, size=(7, 3000)).astype(dt)
            out = run_gpu(e, w, 4, extra={"ns_in": x})
            ref = run_oracle(chain, e.params, w, 4, ns_in=x.T.astype(np.float64))
            if precision == 64:
                check(out, ref, tol, keys=("qdot_ns", "qdot"))
            else:
                # undamped: the FP32 Jacobian's rounding (6e-8) is amplified by cond(J), with nothing to bound it
                from oracle import batch
                cond = np.linalg.cond(batch.fk_jac(chain, w["q"].T.astype(np.float64))[2])
                err = rel_err(out["qdot_ns"].astype(np.float64), ref["qdot_ns"])
                assert np.all(err <= np.maximum(tol, 2e-6 * cond)), float(np.max(err / np.maximum(tol, 2e-6 * cond)))
                assert np.quantile(err, 0.99) <= tol
        finally:
            e.set_params(old)


@pytest.mark.parametrize("n_joints", [10, 8, 17])
def test_control_nullspace_wide_chains(built_lib, n_joints):
    """k = N - 6 > 1: the four control floats mix min(4, k) basis vectors, each sign-continuous over the fused cycles
    (scripts/nullspace:91-117 with nJoints = 10, the reference's iCub shape)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params, ns_ctrl_vectors
    chain = workloads.torso_arm_chain(n_joints)
    kk = ns_ctrl_vectors(n_joints)
    n = 1200
    e = Engine(chain, precision=64, params=Params(ns_mode=2, ns_control=(0.3, -0.2, 0.25, 0.1), mixer_w=(1.0, 1.0, 0, 0, 0, 0)))
    try:
        w = workloads.random_batch(chain, n, 4, seed=21)
        rng = np.random.default_rng(22)
        ctrl = rng.uniform(-0.4, 0.4, size=(4, n))
        out = run_gpu(e, w, 4, k=4, outputs=("qdot_vf", "qdot_ns", "qdot", "flags"),
                      extra={"ns_lastvec": np.zeros((kk * n_joints, n)), "ns_in": ctrl})
        ref = run_oracle(chain, e.params, w, 4, k=4, ns_in=ctrl.T)
        check(out, ref, FP64_RTOL, keys=("qdot_vf", "qdot_ns", "qdot"))
        assert np.array_equal(out["flags"], ref["flags"])
        assert np.max(np.abs(out["lastvec"] - ref["lastvec"])) < 1e-9
        u = out["lastvec"].reshape(n, kk, n_joints)
        assert np.allclose(np.einsum("ikn,iln->ikl", u, u), np.eye(kk)[None], atol=1e-12)
    finally:
        e.close()


def test_control_nullspace_against_the_executed_reference_n10(built_lib, golden):
    """The GPU's control-mode motion on the recorded 10-joint trajectory against what the reference's own functions
    produced (tests/golden ns10_*): inside the same nullspace (projector B), same length for the same four control floats
    (LAPACK's rotation of the basis inside the degenerate subspace is the only freedom)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    chain = workloads.torso_arm_chain(10)
    q, B, qd_ref, control = golden["ns10_q"], golden["ns10_B"], golden["ns10_qdot"], golden["ns10_control"]
    steps = q.shape[0]
    e = Engine(chain, precision=64, params=Params(ns_mode=2, ns_control=tuple(control), mixer_w=(0, 1.0, 0, 0, 0, 0),
                                                  integrate=0, max_vel=100.0, ns_gain=1.0, ns_lookahead=0.0))
    try:
        db = DeviceBatch(e, steps, 0, outputs=("qdot_ns",), inputs=("ns_lastvec",))
        db.upload("q", q.T)
        goal = np.zeros((13, steps)); goal[0] = goal[4] = goal[8] = 1.0
        db.upload("goal", goal)
        db.step(1)
        got = db.download("qdot_ns").T
        for s in range(steps):
            assert np.allclose(B[s] @ got[s], got[s], rtol=0, atol=1e-9)              # in the reference's nullspace
            assert np.allclose(np.linalg.norm(got[s]), np.linalg.norm(qd_ref[s]), rtol=1e-9)
    finally:
        e.close()


@pytest.mark.parametrize("m,k,n", [(64, 1, 4128), (9, 3, 1000), (32, 2, 4160), (32, 1, 4128), (3, 4, 37), (20, 2, 4100),
                                   (8, 1, 999)])
def test_lane_split_shape(built_lib, monkeypatch, m, k, n):
    """Two lanes per instance (vfk_split.cuh; the lean call shape of the FP64 17-joint chain, where it measured 25 % faster and
    is the default): against the oracle at the FP64 tolerance, and against the one-thread-per-instance kernel (VFK_NO_SPLIT=1).
    Partial tiles, a single obstacle chunk and resident rings, remainder chunks, K > 1.  Batches with M >= 16 obstacles have
    n > 4096 instances, where the cooperative shape does not take them."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain = workloads.dual_arm_torso_chain(17)                              # DH form: what the split kernel takes
    e = Engine(chain, precision=64, params=Params())
    try:
        w = workloads.random_batch(chain, n, m, seed=57 + m, dtype=np.float64)
        out = run_gpu(e, w, m, k=k, outputs=("qdot",))
        monkeypatch.setenv("VFK_NO_SPLIT", "1")
        solo = run_gpu(e, w, m, k=k, outputs=("qdot",))
        monkeypatch.delenv("VFK_NO_SPLIT")
        dflt = run_gpu(e, w, m, k=k, outputs=("qdot",))
        assert np.array_equal(dflt["qdot"], out["qdot"])                      # the default choice is the split kernel again
        ref = run_oracle(chain, e.params, w, m, k=k)
        assert np.max(rel_err(out["qdot"], ref["qdot"])) <= FP64_RTOL
        assert np.max(rel_err(solo["qdot"], ref["qdot"])) <= FP64_RTOL
        qtol = 1e-11
        assert np.abs(out["q"] - ref["q"]).max() <= qtol and np.abs(out["q"] - solo["q"]).max() <= qtol
        assert np.all(np.isfinite(out["qdot"]))
        assert not np.array_equal(out["qdot"], solo["qdot"])                       # two different kernels really ran
    finally:
        e.close()


@pytest.mark.parametrize("n_joints", [1, 3, 5, 8, 9, 12, 14, 16])
def test_any_joint_count(built_lib, n_joints):
    """Chains whose joint count has no instantiation of its own run padded in the next larger generic one
    (config.nJoints is free in the reference, scripts/vf:143): every output of every controller, both precisions."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain = workloads.torso_arm_chain(n_joints)
    n = 700
    for precision, tol, dt in ((64, FP64_RTOL, np.float64), (32, FP32_RTOL, np.float32)):
        e = Engine(chain, precision=precision, params=Params(mixer_w=(1.0, 1.0, 0.5, 0, 0, 0), jp_ref=tuple([0.1] * n_joints)))
        try:
            w = workloads.random_batch(chain, n, 5, seed=30 + n_joints, dtype=dt)
            out = run_gpu(e, w, 5, k=2)
            ref = run_oracle(chain, e.params, w, 5, k=2)
            check(out, ref, tol, pose_atol=1e-11 if precision == 64 else 1e-5)
            if precision == 64:
                assert np.array_equal(out["flags"], ref["flags"])
                assert np.max(np.abs(out["q"] - ref["q"])) < 1e-11
            # the lean shape (q / qdot only) takes the same padded route
            lean = run_gpu(e, w, 5, k=2, outputs=("qdot",))
            assert np.array_equal(lean["qdot"], out["qdot"]) or rel_err(lean["qdot"].astype(np.float64), ref["qdot"]).max() <= tol
        finally:
            e.close()


def test_per_instance_inputs_weights_tool_and_ext_ports(eng, lwr):
    """jp_ref / qdot0 / q_cmded / extra mixer ports per instance; non-identity IK weights and tool frame."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    chain, _ = lwr
    e = eng(64)
    old = e.params
    try:
        e.set_params(w_task=(1, 1, 1, 0.5, 0.5, 0.5), w_joint=(1, 0.8, 1, 1.2, 1, 1, 0.5), ns_lambda=0.07,
                     tool=(0, -1, 0, 1, 0, 0, 0, 0, 1, 0.03, -0.02, 0.15), mixer_w=(0.9, 0.8, 0.7, 0.6, 0.5, 0.4))
        n, M = 2500, 6
        rng = np.random.default_rng(5)
        w = workloads.random_batch(chain, n, M, seed=4, obst_ext=True)
        w["obst_ext"][:, :, 1] = rng.uniform(2, 25, size=(M, n))         # per-obstacle decay order
        w["obst_ext"][:, :, 0] = rng.uniform(5e-4, 5e-3, size=(M, n))    # per-obstacle safe distance
        jp_ref = rng.uniform(-3.2, 3.2, size=(7, n))          # some beyond the limits -> clamped
        qd0 = rng.normal(size=(7, n))
        q_cmded = w["q"] + rng.normal(scale=0.01, size=(7, n))
        ext = [rng.normal(scale=0.1, size=(7, n)) for _ in range(3)]
        db = DeviceBatch(e, n, M, obst_ext=True, outputs=("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "flags"))
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
        db.upload("obst_ext", w["obst_ext"])
        db.upload("jp_ref", jp_ref); db.upload("ns_in", qd0); db.upload("q_cmded", q_cmded)
        for k in range(3):
            db.ext_cmd[k] = db.to_blocked(ext[k])
        db.step(1)
        out = {k: db.download(k).T for k in ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd")}
        ref = run_oracle(chain, e.params, w, M, jp_ref=jp_ref.T, ns_in=qd0.T, q_cmded=q_cmded.T,
                         ext_cmd=tuple(x.T for x in ext))
        check(out, ref, FP64_RTOL)
        assert np.array_equal(db.download("flags")[0], ref["flags"])
    finally:
        e.set_params(old)


def test_edge_cases(eng, lwr):
    """No obstacles; zero-radius padding obstacles; goal frame already reached."""
    from oracle import batch
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(64)
    w = workloads.random_batch(chain, 300, 4, seed=6)
    out0 = run_gpu(e, dict(w), 0)
    ref0 = run_oracle(chain, e.params, w, 0)
    check(out0, ref0, FP64_RTOL)
    wz = {k: v.copy() for k, v in w.items()}
    wz["obst"][:, :, 3] = 0.0                                     # radius 0 = inactive
    outz = run_gpu(e, wz, 4)
    assert np.array_equal(outz["qdot"], out0["qdot"])
    # instance 0: goal frame == current tool frame (dist ~ 0, angle ~ 0).  (An obstacle exactly on the tool
    # position is a singular point of the field -- d = 0 -- and is covered by the pose-driven field query in
    # test_field_eval_and_mix, where both sides see bit-identical positions.)
    R, p, _ = batch.fk_jac(chain, w["q"].T)
    w["goal"][0:9, 0] = R[0].reshape(9)
    w["goal"][9:12, 0] = p[0]
    out = run_gpu(e, w, 4)
    ref = run_oracle(chain, e.params, w, 4)
    assert np.all(np.isfinite(out["qdot"]))
    check(out, ref, FP64_RTOL)
    assert np.max(np.abs(out["qdot_vf"][0])) < 1e-6


@pytest.mark.parametrize("dh", [True, False])
def test_17_dof_chain(eng, built_lib, dh):
    """BASELINE config 5 shape: 3-DOF torso + 14 arm joints as one serial chain (6x17 Jacobian): in DH form (the kernels'
    DhPattern) and with a mixed-axis torso (RotX joint -> general tip -> GenericPattern)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine
    chain = workloads.dual_arm_torso_chain(dh=dh)
    for precision, tol, dt in ((64, FP64_RTOL, np.float64), (32, FP32_RTOL, np.float32)):
        e = Engine(chain, precision=precision)
        assert e.chain_pattern == ("dh" if dh else "generic")
        try:
            w = workloads.random_batch(chain, 1500, 8, seed=7, dtype=dt)
            out = run_gpu(e, w, 8, outputs=("qdot_vf", "qdot_ns", "qdot", "pose"))
            ref = run_oracle(chain, e.params, w, 8)
            check(out, ref, tol, keys=("qdot_vf", "qdot_ns", "qdot"), pose_atol=1e-11 if precision == 64 else 1e-5)
        finally:
            e.close()


def test_all_joint_types(built_lib):
    """RotX/RotY/Trans* joints are canonicalised to Z joints on the host; results match the oracle's direct form."""
    from vfclik_b200 import kdl
    from vfclik_b200.config import chain_from_segments
    from vfclik_b200.engine import Engine
    types = [kdl.Joint.RotX, kdl.Joint.TransY, kdl.Joint.RotY, kdl.Joint.RotZ, kdl.Joint.TransX, kdl.Joint.RotX,
             kdl.Joint.TransZ]
    segs = [kdl.Segment(kdl.Joint(t), kdl.Frame(kdl.Rotation.RotX(0.3 * (i + 1)) * kdl.Rotation.RotZ(0.2 * i),
                                                 kdl.Vector(0.1, 0.05 * i, 0.2))) for i, t in enumerate(types)]
    chain = chain_from_segments(segs, [[-1.0, 1.0]] * 7)
    from vfclik_b200 import workloads
    e = Engine(chain, precision=64)
    try:
        w = workloads.random_batch(chain, 500, 3, seed=8, shoulder=(0.3, 0.2, 0.8), box=0.6)
        out = run_gpu(e, w, 3, outputs=("qdot_vf", "qdot_ns", "qdot", "pose"))
        ref = run_oracle(chain, e.params, w, 3)
        check(out, ref, FP64_RTOL, keys=("qdot_vf", "qdot_ns", "qdot"), pose_atol=1e-12)
    finally:
        e.close()


@pytest.mark.parametrize("precision, rtol, pose_atol", [(64, FP64_RTOL, 1e-12), (32, FP32_RTOL, 2e-6)])
def test_joint_angles_beyond_one_turn(lwr, built_lib, precision, rtol, pose_atol):
    """Continuous joints: angles of several turns (limits +-4 pi) go through the kernels' own sin / cos (reduction to the
    nearest of 128 table angles in the FP32 mode's wide chain, quadrant reduction in the FP64 mode) and still match the
    oracle's libm."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr
    wide = dataclasses.replace(chain, q_lo=np.full(7, -4 * np.pi), q_hi=np.full(7, 4 * np.pi))
    e = Engine(wide, precision=precision, params=Params.from_config(cfg))
    try:
        w = workloads.random_batch(wide, 4096, 8, seed=21, dtype=np.float64 if precision == 64 else np.float32)
        assert np.abs(w["q"]).max() > 3 * np.pi
        out = run_gpu(e, w, 8, outputs=("qdot_vf", "qdot_ns", "qdot", "pose"))
        ref = run_oracle(wide, e.params, w, 8)
        check(out, ref, rtol, keys=("qdot_vf", "qdot_ns", "qdot"), pose_atol=pose_atol)
        lean = run_gpu(e, w, 8, outputs=("qdot",))          # the lean instantiation (q / qdot only) takes the same chain
        check(lean, ref, rtol, keys=("qdot",))
    finally:
        e.close()


@pytest.mark.parametrize("n", [40, 3000])
def test_long_chain_fp32_table_sincos(built_lib, n):
    """The FP32 mode takes the sin / cos of its FP64 kinematic chain from the 128-entry shared-memory table (vfk_math.cuh:
    sincos_table); here on the 17-joint chain: joint angles of several turns in both directions still match the oracle's
    libm, in the lean and in the general instantiation; n = 40 leaves two warps of the only CTA without a tile (they must
    still pass the table's barrier); K fused cycles stay bit-identical to K single-cycle launches (every instantiation
    uses the table)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch, Engine
    chain = workloads.dual_arm_torso_chain()
    wide = dataclasses.replace(chain, q_lo=np.full(17, -4 * np.pi), q_hi=np.full(17, 4 * np.pi))
    e = Engine(wide, precision=32)
    try:
        w = workloads.random_batch(wide, n, 20, seed=33, dtype=np.float32)
        assert np.abs(w["q"]).max() > 3 * np.pi and w["q"].min() < -3 * np.pi
        out = run_gpu(e, w, 20, outputs=("qdot_vf", "qdot_ns", "qdot", "pose"))
        ref = run_oracle(wide, e.params, w, 20)
        check(out, ref, FP32_RTOL, keys=("qdot_vf", "qdot_ns", "qdot"), pose_atol=1e-5)
        lean = run_gpu(e, w, 20, outputs=("qdot",))
        check(lean, ref, FP32_RTOL, keys=("qdot",))
        db = DeviceBatch(e, n, 20, outputs=("qdot",))
        db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
        db.upload("q", w["q"])
        for _ in range(4):
            db.step(1)
        q_loop, qd_loop = db.download("q"), db.download("qdot")
        db.upload("q", w["q"])
        db.step(4)
        assert np.array_equal(db.download("q"), q_loop) and np.array_equal(db.download("qdot"), qd_loop)
    finally:
        e.close()


def test_host_session_matches_device_path(eng, lwr):
    """The host-buffer C-ABI session (numpy in / numpy out) gives the same numbers as the device path."""
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(64)
    n, M = 1111, 5
    w = workloads.random_batch(chain, n, M, seed=9)
    ref = run_oracle(chain, e.params, w, M, k=2)
    s = e.session(n, M)
    try:
        s.set_goal(w["goal"]); s.set_obstacles(w["obst"])
        s.enable("qdot_vf", "pose")
        qd = np.empty((7, n)); qo = np.empty((7, n)); fl = np.empty(n, dtype=np.int32)
        assert s.cycle(q_in=w["q"], k_cycles=2, qdot_out=qd, q_out=qo, flags_out=fl) == 4   # pack q, cycle kernel, unpack qdot, unpack q
        assert rel_err(qd.T, ref["qdot"]).max() <= FP64_RTOL
        assert np.max(np.abs(qo.T - ref["q"])) < 1e-12 and np.array_equal(fl, ref["flags"])
        assert rel_err(s.read("qdot_vf").T, ref["qdot_vf"]).max() <= FP64_RTOL
        assert np.max(np.abs(s.read("pose").T - ref["pose"])) < 1e-12
        # second call continues from the resident state (no q upload)
        ref2 = run_oracle(chain, e.params, dict(w, q=ref["q"].T), M, k=1)
        s.cycle(k_cycles=1, qdot_out=qd)
        assert rel_err(qd.T, ref2["qdot"]).max() <= 1e-8
    finally:
        s.close()


def test_field_eval_and_mix(eng, lwr):
    """/pose_in -> /vector_out query (scripts/vf:469-503) and the stand-alone mixer sum (src/command_mixer.py:78-82)."""
    from oracle import batch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    chain, _ = lwr
    e = eng(64)
    n, M = 700, 6
    w = workloads.random_batch(chain, n, M, seed=11)
    q, goal, obst = to_oracle(w, M)
    R, p, _ = batch.fk_jac(chain, q)
    obst[5, 0, 0:3] = p[5]                      # an obstacle centred exactly on the query position (d = 0)
    w["obst"][0, 5, 0:3] = p[5]
    goal[6, 9:12] = p[6]                        # a goal position exactly on the query position
    w["goal"][9:12, 6] = p[6]
    v, om = batch.field_eval(oracle_params(e.params), R, p, goal, obst)
    db = DeviceBatch(e, n, M, outputs=())
    db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
    pose = db.upload("pose", np.concatenate([R.reshape(n, 9), p], axis=1).T)
    tw = db._ensure("twist")
    assert e.field_eval(pose, db.t["goal"], db.t["obst"], tw, n, M) == 1
    got = db.download("twist").T
    assert np.allclose(got, np.concatenate([v, om], axis=1), rtol=1e-9, atol=1e-12)
    # mixer
    rng = np.random.default_rng(12)
    cmds = [rng.normal(size=(7, n)) for _ in range(6)]
    cmds[4][3, 17] = np.nan
    wts = [1.0, 1.0, 0.3, 0.0, 0.25, -0.5]
    dev = [db.to_blocked(c) for c in cmds]
    dev[3] = None                                            # an unconnected port
    out = db._ensure("mix_out")
    flags = db._ensure("flags")
    e.mix(dev, wts, out, 7, n, nan_flags=flags)
    want = np.zeros((7, n))
    for c, wt, d in zip(cmds, wts, dev):
        if d is not None:
            want = want + c * wt
    got = db.download("mix_out")
    ok = ~np.isnan(want)
    assert np.allclose(got[ok], want[ok], rtol=1e-12, atol=1e-14) and np.isnan(got[3, 17])
    fl = db.download("flags")[0]
    assert fl[17] == 4 and fl.sum() == 4


def test_invalid_arguments_return_errors(eng, lwr):
    from vfclik_b200._lib import VfkError
    from vfclik_b200.engine import DeviceBatch
    e = eng(32)
    db = DeviceBatch(e, 64, 2)
    with pytest.raises(VfkError):
        e.step(db.bufs, 64, -1)
    with pytest.raises(VfkError):
        e.step(db.bufs, 64, 2, k_cycles=0)
    with pytest.raises(VfkError):
        e.step({"q": db.t["q"]}, 64, 0)             # goal missing
    with pytest.raises(VfkError):
        e.step(dict(db.bufs, goal=db.t["goal"].data_ptr() + 4), 64, 2)     # misaligned base pointer
    with pytest.raises(VfkError):
        e.set_params(ns_mode=7)
    with pytest.raises(VfkError):
        e.set_params(ik_lambda=0.0)                 # outside the FP32 domain
    e.set_params(ns_lambda=0.0)                     # the undamped projector goes through the Householder basis: no pivots to lose
    e.set_params(ns_lambda=0.1, ns_mode=1)


def test_pack_unpack_round_trip(eng, lwr):
    """Dense SoA <-> tile-blocked conversion kernels: exact, for ragged n and every element width."""
    from vfclik_b200.engine import DeviceBatch
    e = eng(32)
    rng = np.random.default_rng(13)
    for n in (1, 31, 32, 33, 1000):
        db = DeviceBatch(e, n, 3, obst_ext=True, outputs=("qdot",))
        a = rng.normal(size=(7, n)).astype(np.float32)
        o = rng.normal(size=(3, n, 4)).astype(np.float32)
        x = rng.normal(size=(3, n, 2)).astype(np.float32)
        db.upload("q", a); db.upload("obst", o); db.upload("obst_ext", x)
        assert np.array_equal(db.download("q"), a)
        assert np.array_equal(db.download("obst"), o)
        assert np.array_equal(db.download("obst_ext"), x)
        # the documented index formula: element (c, i) at ((i // 32) * C + c) * 32 + i % 32
        flat = db.t["q"].reshape(-1).cpu().numpy()
        i = n - 1
        assert flat[((i // 32) * 7 + 3) * 32 + i % 32] == a[3, i]
        # obstacles, FP32: pair p = m // 2 of a tile is two planes of 32 x float4, {x0, x1, y0, y1} and {z0, z1, r0, r1}
        # (slot s = m % 2); 3 obstacles are padded to 2 pairs with a zero-radius slot
        oflat = db.t["obst"].reshape(-1).cpu().numpy()
        for m, c in ((2, 1), (1, 0), (0, 3), (1, 2)):
            pair, slot = m // 2, m % 2
            at = (((i // 32) * 2 + pair) * 2 + c // 2) * 128 + (i % 32) * 4 + (c % 2) * 2 + slot
            assert oflat[at] == o[m, i, c]
        assert np.all(oflat.reshape(-1, 2, 2, 32, 2, 2)[:, 1, :, :, :, 1] == 0)          # the padding slot of pair 1
        assert np.array_equal(db.obstacles_of(np.arange(n)), o)


@pytest.mark.parametrize("precision,m,k", [(64, 64, 3), (64, 100, 1), (32, 100, 2), (32, 256, 1), (64, 3, 1), (32, 9, 4)])
def test_obstacle_ring_shapes(eng, lwr, precision, m, k):
    """Streaming ring (more chunks than stages), ragged last chunk, K > 1 re-streaming, resident small lists."""
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(precision)
    n = 1500
    w = workloads.random_batch(chain, n, m, seed=30 + m, dtype=np.float32 if precision == 32 else np.float64)
    out = run_gpu(e, w, m, k=k, outputs=("qdot_vf", "qdot"))
    ref = run_oracle(chain, e.params, w, m, k=k)
    tol = FP64_RTOL if precision == 64 else FP32_RTOL * (1 if k == 1 else 3)
    check(out, ref, tol, keys=("qdot_vf", "qdot"))


def test_config4_and_config5_shapes_fp32(eng, built_lib):
    """BASELINE configs[3] (256 obstacles, repulsor-sum dominated) and configs[4] (17-DOF, 64 obstacles) at test size."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine
    chain = workloads.dual_arm_torso_chain()
    e = Engine(chain, precision=32)
    try:
        w = workloads.random_batch(chain, 4096, 64, seed=41, dtype=np.float32)
        out = run_gpu(e, w, 64, outputs=("qdot_vf", "qdot_ns", "qdot"))
        ref = run_oracle(chain, e.params, w, 64)
        check(out, ref, FP32_RTOL, keys=("qdot_vf", "qdot_ns", "qdot"))
    finally:
        e.close()


def test_host_session_chunk_pipeline(eng, lwr):
    """Large sessions split the call into tile-aligned chunks on several streams (H2D / kernel / D2H overlap);
    results must be identical to the single-launch device path, including a ragged last chunk."""
    import torch
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(32)
    n, M = 200_003, 4
    w = workloads.random_batch(chain, n, M, seed=51, dtype=np.float32)
    dev = run_gpu(e, w, M, k=2, outputs=("qdot", "flags"))
    s = e.session(n, M)
    try:
        s.set_goal(w["goal"]); s.set_obstacles(w["obst"])
        q_pin = torch.from_numpy(w["q"]).pin_memory()
        qd = torch.empty((7, n), dtype=torch.float32).pin_memory()
        qo = np.empty((7, n), dtype=np.float32)                      # pageable output goes through the staging copy
        fl = np.empty(n, dtype=np.int32)
        launches = s.cycle(q_in=q_pin.numpy(), k_cycles=2, qdot_out=qd.numpy(), q_out=qo, flags_out=fl)
        assert launches == 3 * 4                                      # 3 chunks x (pack q, cycle, unpack qdot, unpack q)
        assert np.array_equal(qd.numpy().T, dev["qdot"]) and np.array_equal(qo.T, dev["q"]) and np.array_equal(fl, dev["flags"])
        # same buffers again: the second call captures the pipeline into a CUDA graph, later calls replay it
        for _ in range(3):
            qd.zero_(); qo[:] = 0; fl[:] = -1
            assert s.cycle(q_in=q_pin.numpy(), k_cycles=2, qdot_out=qd.numpy(), q_out=qo, flags_out=fl) == 12
            assert np.array_equal(qd.numpy().T, dev["qdot"]) and np.array_equal(qo.T, dev["q"]) and np.array_equal(fl, dev["flags"])
        # a parameter change invalidates the captured graph (the constants are baked into the kernel nodes)
        old = e.params
        e.set_params(speed_scale=0.1)
        s.cycle(q_in=q_pin.numpy(), k_cycles=2, qdot_out=qd.numpy())
        s.cycle(q_in=q_pin.numpy(), k_cycles=2, qdot_out=qd.numpy())
        slow = qd.numpy().copy()
        e.set_params(old)
        assert not np.array_equal(slow.T, dev["qdot"])
        s.cycle(q_in=q_pin.numpy(), k_cycles=2, qdot_out=qd.numpy())
        assert np.array_equal(qd.numpy().T, dev["qdot"])
    finally:
        s.close()


@pytest.mark.parametrize("precision", [64, 32])
def test_auxiliary_fields_types_4_and_5(eng, lwr, precision):
    """Hemisphere repellers (vfl type 4) and funnel attractors (type 5) as per-instance auxiliary field records."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    chain, _ = lwr
    e = eng(precision)
    n, M = 3000, 3
    dt = np.float32 if precision == 32 else np.float64
    rng = np.random.default_rng(71)
    w = workloads.random_batch(chain, n, M, seed=70, dtype=dt)
    aux = np.zeros((3, 12, n), dtype=dt)
    aux[0, 0] = 4; aux[0, 1] = -50                                              # table below the workspace
    aux[0, 2:5] = w["goal"][9:12] + rng.uniform(-0.3, 0.3, size=(3, n)); aux[0, 5:8] = rng.normal(size=(3, n))
    aux[0, 8] = rng.uniform(0.01, 0.1, size=n); aux[0, 9] = rng.uniform(2, 6, size=n)
    aux[1, 0] = 5; aux[1, 1] = 30                                               # funnel at the goal
    aux[1, 2:5] = w["goal"][9:12]; aux[1, 5:8] = rng.normal(size=(3, n))
    aux[1, 8] = rng.uniform(0.2, 0.8, size=n); aux[1, 9] = 10; aux[1, 10] = rng.uniform(0.1, 0.5, size=n); aux[1, 11] = 2
    aux[2, 0] = np.where(rng.random(n) < 0.5, 0, 4); aux[2, 1] = -50            # half of the third slots are empty
    aux[2, 2:5] = rng.uniform(-0.5, 0.5, size=(3, n)); aux[2, 5:8] = rng.normal(size=(3, n)); aux[2, 8] = 0.05; aux[2, 9] = 3
    db = DeviceBatch(e, n, M, outputs=("qdot_vf", "qdot", "twist"))
    db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
    db.set_aux(aux)
    assert db.step(1) == 1
    ref = run_oracle(chain, e.params, w, M, aux=aux.transpose(2, 0, 1).astype(np.float64))
    tol = FP64_RTOL if precision == 64 else FP32_RTOL
    for k in ("qdot_vf", "qdot"):
        err = rel_err(db.download(k).T.astype(np.float64), ref[k])
        assert err.max() <= tol, (k, float(err.max()))
    assert np.max(np.abs(db.download("twist").T - ref["twist"])) <= (1e-12 if precision == 64 else 2e-6)
    # and the fields change the answer
    ref0 = run_oracle(chain, e.params, w, M)
    assert np.max(np.abs(ref0["qdot_vf"] - ref["qdot_vf"])) > 1e-3


def test_full_size_config3_properties_and_sampled_oracle(lwr, built_lib):
    """BASELINE configs[2] at full size (1,048,576 instances, 32 obstacles, FP32, nullspace on): the oracle on ALL
    instances (1e-4), flags on a sample, plus size-independent properties on the whole batch -- permutation equivariance,
    an empty obstacle slot changes nothing, K launches == one launch of K cycles, output finiteness and the clamp bound."""
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    chain, cfg = lwr
    e = Engine(chain, precision=32, params=Params.from_config(cfg))
    try:
        n, M = 1 << 20, 32
        w = workloads.random_batch(chain, n, M, seed=1, dtype=np.float32)
        db = DeviceBatch(e, n, M, outputs=("qdot",))
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
        q_before = db.t["q"].clone()
        assert db.step(1) == 1
        qd = db.download("qdot")                                   # [7, n]
        q1 = db.download("q")
        assert np.all(np.isfinite(qd)) and np.max(np.abs(qd)) <= cfg.max_vel * (1 + 1e-6)
        assert np.allclose(q1, w["q"] + np.float32(cfg.rate) * qd, rtol=0, atol=5e-7)      # explicit Euler (fma vs mul+add: 1 ulp at |q| ~ 3)
        # oracle parity on EVERY instance (the vectorised oracle fanned over the host cores), flags on a sample
        ref = oracle_parallel(chain, e.params, w, M, keys=("qdot", "flags"))
        err = rel_err(qd.T.astype(np.float64), ref["qdot"])
        assert err.max() <= FP32_RTOL, (float(err.max()), int(np.argmax(err)))
        rng = np.random.default_rng(5)
        idx = np.sort(rng.choice(n, size=16384, replace=False))
        sub = dict(q=w["q"][:, idx], goal=w["goal"][:, idx], obst=np.ascontiguousarray(w["obst"][:, idx]))
        gen = run_gpu(e, sub, M, outputs=("qdot", "flags"))          # the general instantiation writes the flags
        fl_ref = ref["flags"][idx]
        differ = gen["flags"] != fl_ref
        assert differ.mean() < 1e-3, float(differ.mean())
        assert rel_err(gen["qdot"].astype(np.float64), ref["qdot"][idx]).max() <= FP32_RTOL
        # permutation equivariance (bit-exact): instance order carries no information
        perm = rng.permutation(n)
        dbp = DeviceBatch(e, n, M, outputs=("qdot",))
        dbp.upload("q", w["q"][:, perm]); dbp.upload("goal", w["goal"][:, perm])
        dbp.upload("obst", np.ascontiguousarray(w["obst"][:, perm]))
        dbp.step(1)
        assert np.array_equal(dbp.download("qdot"), qd[:, perm])
        del dbp
        # an extra empty slot (radius 0) is a no-op (bit-exact), and 33 obstacles exercise the ragged last chunk
        obst33 = np.concatenate([w["obst"], np.zeros((1, n, 4), dtype=np.float32)], axis=0)
        obst33[32, :, 0:3] = 0.5
        db33 = DeviceBatch(e, n, M + 1, outputs=("qdot",))
        db33.upload("q", w["q"]); db33.upload("goal", w["goal"]); db33.upload("obst", obst33)
        db33.step(1)
        assert np.array_equal(db33.download("qdot"), qd)
        del db33, obst33
        # K fused cycles == K single-cycle launches (state round-trips HBM bit-exactly)
        db.t["q"].copy_(q_before)
        for _ in range(5):
            db.step(1)
        q_loop, qd_loop = db.download("q"), db.download("qdot")
        db.t["q"].copy_(q_before)
        db.step(5)
        assert np.array_equal(db.download("q"), q_loop) and np.array_equal(db.download("qdot"), qd_loop)
        torch.cuda.synchronize()
    finally:
        e.close()


@pytest.mark.parametrize("precision", [64, 32])
def test_powercube_and_icub_bridge_backends(lwr, built_lib, precision):
    """SURVEY.md 8 row f4: Powercube_Bridge.set_vel's shoulder clamp (scripts/bridge:288-305, incl. the reference's
    double application of the leading ratio) and the iCub / Powercube command form, fused in the cycle kernel."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import BRIDGE_ICUB, BRIDGE_POWERCUBE, Engine, Params
    chain, cfg = lwr
    dt = np.float32 if precision == 32 else np.float64
    w = workloads.random_batch(chain, 3000, 8, seed=17, dtype=dt)
    # fast enough that all three cases occur: no clamp, leading clamp only, shoulder clamp
    base = dataclasses.replace(Params.from_config(cfg), speed_scale=0.41, max_vel=0.3)
    for kind, shoulder in ((BRIDGE_POWERCUBE, (0.05, -0.08)), (BRIDGE_ICUB, (0.0, 0.0))):
        prm = dataclasses.replace(base, bridge_kind=kind, shoulder_vel=shoulder)
        e = Engine(chain, precision=precision, params=prm)
        try:
            out = run_gpu(e, w, 8)
            ref = run_oracle(chain, prm, w, 8)
            check(out, ref, FP64_RTOL if precision == 64 else FP32_RTOL)
            assert np.allclose(out["cmd"], out["qdot"])               # both back-ends command qdot_lim itself
            if kind == BRIDGE_POWERCUBE:
                sh = ref["qdot"][:, 0]
                assert np.all(sh <= shoulder[0] * (1 + 1e-12)) and np.all(sh >= shoulder[1] * (1 + 1e-12))
                lwr_like = run_oracle(chain, dataclasses.replace(prm, bridge_kind=0), w, 8)
                changed = np.any(np.abs(lwr_like["qdot"] - ref["qdot"]) > 1e-12, axis=1)
                assert 0.05 < changed.mean() < 1.0                    # the second clamp really acted on part of the batch
        finally:
            e.close()
    # invalid Powercube limits are refused
    with pytest.raises(Exception):
        Engine(chain, precision=64, params=dataclasses.replace(base, bridge_kind=BRIDGE_POWERCUBE, shoulder_vel=(0.0, 0.0)))


@pytest.mark.parametrize("precision", [32, 64])
def test_host_session_direct_host_io(eng, lwr, precision, monkeypatch):
    """Page-locked caller buffers + a tile-aligned batch: vfk_session_cycle runs ONE kernel that reads q from host memory
    (TMA bulk copies of the dense rows) and writes qdot back itself.  Results are bit-identical to the device path and to
    the chunked copy pipeline (VFK_SESSION_DIRECT=0); pageable buffers and ragged batches fall back to the pipeline."""
    import torch
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(precision)
    dt, tdt = (np.float32, torch.float32) if precision == 32 else (np.float64, torch.float64)
    n, M = 70_016, 12                                               # 2188 tiles: not a multiple of the warp count
    w = workloads.random_batch(chain, n, M, seed=77, dtype=dt)
    dev = run_gpu(e, w, M, k=3, outputs=("qdot", "flags"))
    s = e.session(n, M)
    try:
        s.set_goal(w["goal"]); s.set_obstacles(w["obst"])
        q_pin = torch.from_numpy(w["q"]).pin_memory()
        qd = torch.zeros((7, n), dtype=tdt).pin_memory()
        qo = torch.zeros((7, n), dtype=tdt).pin_memory()
        fl = torch.zeros(n, dtype=torch.int32).pin_memory()
        assert s.cycle(q_in=q_pin.numpy(), k_cycles=3, qdot_out=qd.numpy()) == 1                       # the cycle kernel only
        assert np.array_equal(qd.numpy().T, dev["qdot"])
        qd.zero_()
        assert s.cycle(q_in=q_pin.numpy(), k_cycles=3, qdot_out=qd.numpy(), q_out=qo.numpy(), flags_out=fl.numpy()) == 2
        assert np.array_equal(qd.numpy().T, dev["qdot"]) and np.array_equal(qo.numpy().T, dev["q"])
        assert np.array_equal(fl.numpy(), dev["flags"])
        assert np.array_equal(q_pin.numpy(), w["q"])                                                 # the caller's q is read-only
        # pageable output -> copy pipeline, same numbers
        qd_page = np.zeros((7, n), dtype=dt)
        assert s.cycle(q_in=q_pin.numpy(), k_cycles=3, qdot_out=qd_page) > 1
        assert np.array_equal(qd_page.T, dev["qdot"])
        monkeypatch.setenv("VFK_SESSION_DIRECT", "0")
        qd.zero_()
        assert s.cycle(q_in=q_pin.numpy(), k_cycles=3, qdot_out=qd.numpy()) > 1
        assert np.array_equal(qd.numpy().T, dev["qdot"])
    finally:
        s.close()


@pytest.mark.parametrize("precision", [32, 64])
def test_direct_host_io_keeps_the_sessions_device_state_current(lwr, built_lib, precision):
    """integrate = 0 (ControlRuntime's default: the plant is elsewhere) through the direct path: the kernel reads q from the
    caller's buffer, so the session's own q / qdot must still follow -- q_out, read("q"), read("qdot") and a later cycle
    WITHOUT q_in all see the state of the last call, exactly as through the copy pipeline."""
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr
    dt, tdt = (np.float32, torch.float32) if precision == 32 else (np.float64, torch.float64)
    n, M = 4096, 5
    e = Engine(chain, precision=precision, params=Params.from_config(cfg, integrate=0))
    try:
        wa = workloads.random_batch(chain, n, M, seed=91, dtype=dt)
        wb = workloads.random_batch(chain, n, M, seed=92, dtype=dt)
        results = {}
        for mode in ("direct", "pipeline"):
            s = e.session(n, M)
            s.set_goal(wa["goal"]); s.set_obstacles(wa["obst"]); s.set_q(wa["q"])
            if mode == "direct":
                q_in = torch.from_numpy(wb["q"]).pin_memory().numpy()
                qd = torch.zeros((7, n), dtype=tdt).pin_memory().numpy()
                qo = torch.zeros((7, n), dtype=tdt).pin_memory().numpy()
                assert s.cycle(q_in=q_in, qdot_out=qd, q_out=qo) == 2            # cycle kernel + the un-blocking of q_out
            else:
                q_in, qd, qo = wb["q"].copy(), np.zeros((7, n), dtype=dt), np.zeros((7, n), dtype=dt)
                assert s.cycle(q_in=q_in, qdot_out=qd, q_out=qo) > 2
            assert np.array_equal(qo, wb["q"])                                   # integrate = 0: q_out is the q that came in
            assert np.array_equal(s.read("q"), wb["q"]) and np.array_equal(s.read("qdot"), qd)
            again = np.zeros((7, n), dtype=dt)
            s.cycle(qdot_out=again)                                              # no q_in: continues from the session's q
            assert np.array_equal(again, qd)
            results[mode] = qd.copy()
            s.close()
        assert np.array_equal(results["direct"], results["pipeline"])
    finally:
        e.close()


def test_batched_posture_dependent_joint_limits(lwr, built_lib, golden):
    """Row a12 at batch > 1: ``config.updateJntLimits(q)`` evaluated per instance and handed to the kernel as ``jp_lo`` /
    ``jp_hi``; the clamped reference persists in ``jp_ref`` like the loop variable of scripts/joint_p_controller:121.
    Instance 0 replays the trajectory recorded from the reference's own loop with posture-dependent limits
    (tests/golden jp_out_dynamic / jp_at_goal_dynamic), the other instances run their own postures against the oracle."""
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    from oracle import batch
    chain, cfg = lwr
    g = golden
    q_gold, steps = g["jp_q"], g["jp_q"].shape[0]
    kp, delta = g["jp_kp_delta"]
    n = 96
    rng = np.random.default_rng(61)
    e = Engine(chain, precision=64, params=Params.from_config(cfg, jp_kp=float(kp), jp_delta=float(delta), integrate=0,
                                                              mixer_w=(0, 0, 1.0, 0, 0, 0)))
    prm = oracle_params(e.params)
    try:
        db = DeviceBatch(e, n, 0, outputs=("qdot_jp", "flags"), inputs=("jp_ref", "jp_lo", "jp_hi"))
        goal = np.zeros((13, n)); goal[0] = goal[4] = goal[8] = 1.0
        db.upload("goal", goal)
        ref = np.tile(np.asarray(cfg.initial_joint_pos, dtype=np.float64)[:, None], (1, n))          # [7, n]
        db.upload("jp_ref", ref)
        ref_o = ref.T.copy()
        msgs = {int(k): m for k, m in zip(g["jp_ref_steps"], g["jp_ref_msgs"])}
        for k in range(steps):
            q = rng.uniform(-1.0, 1.0, size=(n, 7))
            q[0] = q_gold[k]
            if k in msgs:                                            # a new reference arrives (instance 0: the recorded one)
                ref_o = rng.uniform(-3.0, 3.0, size=(n, 7))
                ref_o[0] = msgs[k]
                db.upload("jp_ref", ref_o.T)
            lo = np.tile((-0.5 - np.abs(q[:, 0]))[:, None], (1, 7))   # the golden record's hook, per instance
            hi = np.tile((0.4 + np.abs(q[:, 1]))[:, None], (1, 7))
            db.upload("q", q.T); db.upload("jp_lo", lo.T); db.upload("jp_hi", hi.T)
            assert db.step(1) == 1
            got = db.download("qdot_jp").T
            flags = db.download("flags")[0]
            o = batch.step(chain, prm, q, goal.T, None, jp_ref=ref_o, jp_limits=(lo, hi))
            ref_o = o["jp_ref"]
            assert np.allclose(got, o["qdot_jp"], rtol=1e-13, atol=1e-15)
            assert np.array_equal(flags & 1, o["flags"] & 1)
            assert np.allclose(db.download("jp_ref").T, ref_o, rtol=0, atol=0)          # the clamp persisted on the device
            assert np.allclose(got[0], g["jp_out_dynamic"][k], rtol=1e-12, atol=1e-14), k
            assert int(flags[0] & 1) == int(g["jp_at_goal_dynamic"][k]), k
    finally:
        e.close()


@pytest.mark.parametrize("which", ["config4", "config5"])
def test_full_size_config4_and_config5_shards(lwr, built_lib, which):
    """BASELINE configs[3] / [4] at their per-GPU shard size on 8 GPUs (2,097,152 LWR instances x 256 obstacles;
    524,288 17-DOF instances x 64 obstacles), drawn on the device like bench.py does: finiteness and the clamp bound on
    the whole shard, the explicit-Euler relation, and the oracle on a random sample of 2048 instances (FP32, 1e-4)."""
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain_lwr, cfg = lwr
    if which == "config4":
        chain, n, M, params = chain_lwr, 1 << 21, 256, Params.from_config(cfg)
    else:
        chain, n, M, params = workloads.dual_arm_torso_chain(), 1 << 19, 64, Params()
    N = chain.n_joints
    e = Engine(chain, precision=32, params=params)
    try:
        db = workloads.random_batch_device(e, n, M, seed=9)
        q0 = db.download("q")                                           # dense [N, n]
        goal = db.download("goal")
        rng = np.random.default_rng(3)
        idx = np.sort(rng.choice(n, size=2048, replace=False))
        obst = db.obstacles_of(idx)                                     # [M, 2048, 4]
        assert db.step(1) == 1
        qd = db.download("qdot")
        q1 = db.download("q")
        assert np.all(np.isfinite(qd)) and np.max(np.abs(qd)) <= params.max_vel * (1 + 1e-6)
        assert np.allclose(q1, q0 + np.float32(params.dt) * qd, rtol=0, atol=5e-7)
        sub = dict(q=q0[:, idx], goal=goal[:, idx], obst=obst)
        ref = run_oracle(chain, e.params, sub, M)
        err = rel_err(qd[:, idx].T.astype(np.float64), ref["qdot"])
        assert err.max() <= FP32_RTOL, float(err.max())
        gen = run_gpu(e, sub, M, outputs=("qdot", "flags"))          # flags come from the general instantiation
        assert (gen["flags"] != ref["flags"]).mean() < 2e-3
        assert rel_err(gen["qdot"].astype(np.float64), ref["qdot"]).max() <= FP32_RTOL
        assert qd.shape == (N, n)
    finally:
        e.close()


def test_fp32_obstacle_almost_at_the_tool_saturates_instead_of_overflowing(eng, lwr):
    """(radius / d)^20 / d exceeds the FP32 range once d < radius / 75.  The FP32 mode saturates that weight (the field is
    normalised afterwards, so only the direction matters) and must agree with the FP64 oracle, not return NaN."""
    from oracle import batch
    from vfclik_b200 import workloads
    chain, _ = lwr
    e = eng(32)
    n, M = 256, 8
    w = workloads.random_batch(chain, n, M, seed=61, dtype=np.float32)
    _, p_tool, _ = batch.fk_jac(chain, w["q"].T.astype(np.float64))              # identity tool: flange = tool position
    rng = np.random.default_rng(2)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    dist = np.where(np.arange(n) % 2 == 0, 2e-4, 9e-4)[:, None]                  # both far inside radius / 75 = 1.3e-3
    w["obst"][3, :, 0:3] = (p_tool + dist * u).astype(np.float32)
    w["obst"][3, :, 3] = 0.1
    out = run_gpu(e, w, M, outputs=("qdot_vf", "qdot"))
    assert np.all(np.isfinite(out["qdot"])) and np.all(np.isfinite(out["qdot_vf"]))
    ref = run_oracle(chain, e.params, w, M)
    # the FP32 obstacle coordinates quantise d itself (ulp 6e-8 at ~1 m on a 2e-4 m offset): the direction agrees to ~1e-3
    err = rel_err(out["qdot_vf"].astype(np.float64), ref["qdot_vf"])
    assert np.quantile(err, 0.95) < 5e-3 and err.max() < 5e-2, (float(np.quantile(err, 0.95)), float(err.max()))


@pytest.mark.parametrize("precision", [32, 64])
def test_outputs_stay_inside_their_buffers(eng, lwr, precision):
    """Guard bands (compute-sanitizer is not available on the pool): every output of the cycle kernel, of the general and
    the lean instantiation, sits inside a larger tensor filled with a sentinel; after ragged launches (n not a multiple
    of 32, 13 obstacles, K = 2) the bands are untouched.  Same for the session's page-locked host buffers in the direct
    host I/O path and in the copy pipeline."""
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch
    chain, _ = lwr
    e = eng(precision)
    dt, tdt = (np.float32, torch.float32) if precision == 32 else (np.float64, torch.float64)
    SENT = -777.25
    for n, outputs in ((1000 - 7, ("qdot",)), (1000 - 7, ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "twist", "flags"))):
        M = 13
        w = workloads.random_batch(chain, n, M, seed=91, dtype=dt)
        db = DeviceBatch(e, n, M, outputs=outputs)
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
        guarded = {}
        for name in outputs + ("q",):
            t = db.t[name]
            pad = 4096 // t.element_size()
            big = torch.full((t.numel() + 2 * pad,), SENT if t.dtype.is_floating_point else -777, dtype=t.dtype, device=t.device)
            big[pad:pad + t.numel()] = t.reshape(-1)
            db.t[name] = big[pad:pad + t.numel()].view(t.shape)
            guarded[name] = (big, pad, t.numel())
        assert db.step(2) == 1
        torch.cuda.synchronize()
        for name, (big, pad, cnt) in guarded.items():
            sent = SENT if big.dtype.is_floating_point else -777
            assert bool((big[:pad] == sent).all()) and bool((big[pad + cnt:] == sent).all()), name
        ref = run_oracle(chain, e.params, w, M, k=2)
        assert rel_err(db.download("qdot").T.astype(np.float64), ref["qdot"]).max() <= (FP32_RTOL if precision == 32 else FP64_RTOL)
    # host side: direct host I/O (n multiple of 32) and the copy pipeline (ragged n), pinned buffers with bands
    for n in (4096, 4096 - 5):
        M = 13
        w = workloads.random_batch(chain, n, M, seed=92, dtype=dt)
        s = e.session(n, M)
        try:
            s.set_goal(w["goal"]); s.set_obstacles(w["obst"])
            pad = 1024
            q_big = torch.full((7 * n + 2 * pad,), SENT, dtype=tdt).pin_memory()
            qd_big = torch.full((7 * n + 2 * pad,), SENT, dtype=tdt).pin_memory()
            q_big[pad:pad + 7 * n] = torch.from_numpy(np.ascontiguousarray(w["q"])).reshape(-1)
            q_view = q_big[pad:pad + 7 * n].view(7, n).numpy()
            qd_view = qd_big[pad:pad + 7 * n].view(7, n).numpy()
            s.cycle(q_in=q_view, k_cycles=2, qdot_out=qd_view)
            assert bool((qd_big[:pad] == SENT).all()) and bool((qd_big[pad + 7 * n:] == SENT).all())
            assert bool((q_big[:pad] == SENT).all()) and bool((q_big[pad + 7 * n:] == SENT).all())
            assert np.array_equal(q_view, w["q"])
            ref = run_oracle(chain, e.params, w, M, k=2)
            assert rel_err(qd_view.T.astype(np.float64), ref["qdot"]).max() <= (FP32_RTOL if precision == 32 else FP64_RTOL)
        finally:
            s.close()


@pytest.mark.parametrize("precision", [32, 64])
def test_round2_shapes_stay_inside_their_buffers(lwr, built_lib, precision):
    """Guard bands (compute-sanitizer is closed on the pool) around everything the round-2 shapes write: the nullspace
    state of a 10-joint chain (4 basis vectors), the joint-controller reference written back under per-instance limits, q and
    qdot of a padded 8-joint chain and of the 17-joint DH chain (FP32: the DH-pattern kernel, FP64: the lane-split kernel),
    and the obstacle array packed from an odd obstacle count -- ragged batches, K = 2."""
    import torch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    dt = np.float32 if precision == 32 else np.float64
    SENT = -777.25

    def guard(db, names):
        held = {}
        for name in names:
            t = db.t[name]
            pad = 4096 // t.element_size()
            big = torch.full((t.numel() + 2 * pad,), SENT, dtype=t.dtype, device=t.device)
            big[pad:pad + t.numel()] = t.reshape(-1)
            db.t[name] = big[pad:pad + t.numel()].view(t.shape)
            held[name] = (big, pad, t.numel())
        return held

    def intact(held):
        torch.cuda.synchronize()
        for name, (big, pad, cnt) in held.items():
            assert bool((big[:pad] == SENT).all()) and bool((big[pad + cnt:] == SENT).all()), name

    cases = [
        (workloads.torso_arm_chain(10), Params(ns_mode=2, ns_control=(0.3, -0.2, 0.1, 0.2)), ("qdot", "qdot_ns"), ("ns_lastvec",)),
        (lwr[0], Params(mixer_w=(1.0, 1.0, 0.5, 0, 0, 0)), ("qdot", "qdot_jp"), ("jp_ref", "jp_lo", "jp_hi")),
        (workloads.torso_arm_chain(8), Params(), ("qdot", "qdot_vf", "flags"), ()),
        (workloads.dual_arm_torso_chain(), Params(), ("qdot",), ()),
    ]
    for chain, prm, outputs, inputs in cases:
        n, M = 1000 - 7, 13
        e = Engine(chain, precision=precision, params=prm)
        try:
            w = workloads.random_batch(chain, n, M, seed=93, dtype=dt)
            db = DeviceBatch(e, n, M, outputs=outputs, inputs=inputs)
            held = guard(db, ("obst",))
            db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
            intact(held)                                                        # packing 13 obstacles into 7 pairs
            assert np.array_equal(db.download("obst"), w["obst"])
            if "jp_lo" in inputs:
                db.upload("jp_ref", np.full((chain.n_joints, n), 2.5, dtype=dt))
                db.upload("jp_lo", np.full((chain.n_joints, n), -0.3, dtype=dt)); db.upload("jp_hi", np.full((chain.n_joints, n), 0.4, dtype=dt))
            held.update(guard(db, tuple(x for x in outputs + inputs + ("q",) if db.t[x].dtype.is_floating_point)))
            assert db.step(2) == 1
            intact(held)
            assert np.all(np.isfinite(db.download("qdot")))
            if "jp_lo" in inputs:
                assert np.all(db.download("jp_ref") == dt(0.4))                 # the clamp was stored back, inside its buffer
        finally:
            e.close()


def test_bench_dump_outputs_are_the_last_timed_launch(lwr, built_lib, tmp_path):
    """`bench.py --dump-outputs` writes q and qdot of the last timed step.  At 4096 instances the launches rotate over more
    copies of the seeded batch than warm-up and timed steps together, so the last one advanced its copy once: the dump is
    one cycle of the engine on that batch, bit for bit."""
    import json
    import os
    import subprocess
    import sys
    from vfclik_b200 import workloads
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, m = 4096, 32
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--instances", str(n), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3
    chain, cfg = lwr
    e = Engine(chain, precision=32, params=Params.from_config(cfg))
    try:
        w = workloads.random_batch(chain, n, m, seed=1, dtype=np.float32)
        db = DeviceBatch(e, n, m, outputs=("qdot",))
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"])
        assert db.step(1) == 1
        for name in ("q", "qdot"):
            got = np.load(tmp_path / (name + ".npy"))
            assert got.dtype == np.float32 and np.array_equal(got, db.download(name)), name
    finally:
        e.close()
