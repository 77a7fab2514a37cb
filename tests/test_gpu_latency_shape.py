"""The cooperative latency shape (FP64, n <= 4096 instances, M >= 16 obstacles: 8 lanes share an instance's repulsor sum,
vfk_kernels.cuh G = 8) against the oracle and against the one-thread kernel (VFK_NO_COOP=1); and the field's regimes next
to the goal and next to obstacles -- where a controller converges -- through every kernel shape, in both precisions.

Tolerances are the suite's (test_gpu_parity.py): joint velocities 1e-9 relative in FP64 and 1e-4 in FP32, twist rows 1e-12
(FP64) and 2e-6 (FP32) absolute.  The cooperative and the one-thread FP64 kernels differ only in the order of the repulsor
sum, so they must agree to 1e-11.
"""
import dataclasses

import numpy as np
import pytest

from helpers import (FP32_RTOL, FP64_RTOL, near_goal, near_obstacles, oracle_params, rel_err, run_gpu, run_oracle,
                     to_oracle)

pytestmark = pytest.mark.gpu

COOP_RTOL = 1e-11
# FP32 at a converged state: the field forms the rotation error from the tool rotation rounded to FP32 (6e-8), which below
# rot_slowdown becomes up to speed_scale / rot_slowdown * 6e-8 ~ 1.3e-7 rad/s of angular velocity.  Where the joint velocity
# has converged to ~0 that is more than 1e-4 of rel_err's 1e-3 floor (measured 1.004e-4), so FP32 joint velocities are
# held to DESIGN.md section 2's absolute floor of 5e-7 rad/s there: rel_err with a floor of 5e-3.
FP32_FLOOR = 5e-3
ALL = ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "pose", "twist", "flags")
QDOT_KEYS = ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd")


def edge_batch(chain, n, M, seed, dtype=np.float64, ext=True, safe=1e-3, order=20.0, rot_slowdown=0.09, tool=None):
    """Goals next to the tool (near_goal) for every instance, obstacles next to the tool (near_obstacles) for the odd ones;
    the even ones keep random_batch's obstacles, so the converged attractor is not drowned by a close repeller there."""
    w, _ = near_obstacles(chain, n, M, seed, dtype=dtype, obst_ext=ext, safe=safe, order=order, tool=tool)
    wg, _ = near_goal(chain, n, M, seed, rot_slowdown=rot_slowdown, dtype=dtype, tool=tool)
    assert np.array_equal(w["q"], wg["q"])
    w["goal"] = wg["goal"]
    w["obst"][:, 0::2] = wg["obst"][:, 0::2]
    return w


def coop_and_solo(monkeypatch, e, w, M, k, outputs=ALL, **kw):
    monkeypatch.delenv("VFK_NO_COOP", raising=False)
    coop = run_gpu(e, w, M, k=k, outputs=outputs, **kw)
    monkeypatch.setenv("VFK_NO_COOP", "1")
    solo = run_gpu(e, w, M, k=k, outputs=outputs, **kw)
    monkeypatch.delenv("VFK_NO_COOP")
    return coop, solo


def check_all(coop, solo, ref, keys=QDOT_KEYS, rtol=FP64_RTOL):
    """Every output of the cooperative run against the oracle and against the one-thread run."""
    for key in keys:
        e_ref = rel_err(coop[key].astype(np.float64), ref[key])
        assert e_ref.max() <= rtol, (key, "oracle", float(e_ref.max()), int(np.argmax(e_ref)))
        e_solo = rel_err(coop[key], solo[key])
        assert e_solo.max() <= COOP_RTOL, (key, "one-thread", float(e_solo.max()), int(np.argmax(e_solo)))
    if "pose" in coop:
        assert np.max(np.abs(coop["pose"] - ref["pose"])) <= 1e-12
        assert np.max(np.abs(coop["pose"] - solo["pose"])) <= 1e-14
    if "twist" in coop:
        assert np.max(np.abs(coop["twist"] - ref["twist"])) <= 1e-12
        assert np.max(np.abs(coop["twist"] - solo["twist"])) <= 1e-13
    if "flags" in coop:
        assert np.array_equal(coop["flags"], ref["flags"]) and np.array_equal(coop["flags"], solo["flags"])
    assert np.max(np.abs(coop["q"] - ref["q"])) <= 1e-11 and np.max(np.abs(coop["q"] - solo["q"])) <= 1e-13


@pytest.fixture(scope="module")
def lwr_cfg(lwr, built_lib):
    return lwr


# ------------------------------------------------------------------------------------------------ a. which kernel runs
def test_coop_runs_at_4096_instances_and_16_obstacles(lwr_cfg, monkeypatch):
    """FP64, n = 4096, M = 16 takes the cooperative kernel: its answer differs somewhere from VFK_NO_COOP=1 (a different
    summation order, so a different kernel ran), and both agree with the oracle.  Obstacles next to the tool make the
    repulsor sum large enough that the two orders round differently."""
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    e = Engine(chain, precision=64, params=Params.from_config(cfg))
    try:
        w, _ = near_obstacles(chain, 4096, 16, seed=101, obst_ext=False, n_near=4)
        coop, solo = coop_and_solo(monkeypatch, e, w, 16, 1, outputs=("qdot_vf", "qdot", "flags"))
        assert not np.array_equal(coop["qdot_vf"], solo["qdot_vf"])
        ref = run_oracle(chain, e.params, w, 16)
        check_all(coop, solo, ref, keys=("qdot_vf", "qdot"))
    finally:
        e.close()


@pytest.mark.parametrize("precision,n,M", [(64, 4097, 16), (64, 4096, 15), (32, 64, 32)])
def test_outside_the_coop_switch_nothing_changes(lwr_cfg, monkeypatch, precision, n, M):
    """One instance too many, one obstacle too few, or FP32 (no cooperative instantiation): VFK_NO_COOP=1 changes no bit."""
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    dt = np.float64 if precision == 64 else np.float32
    e = Engine(chain, precision=precision, params=Params.from_config(cfg))
    try:
        w, _ = near_obstacles(chain, n, M, seed=102, dtype=dt, obst_ext=False, n_near=4)
        for outputs in (("qdot",), ALL):
            dflt, solo = coop_and_solo(monkeypatch, e, w, M, 2, outputs=outputs)
            for key in outputs + ("q",):
                assert np.array_equal(dflt[key], solo[key]), key
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ b. parity matrix
NMK = [(1, 16, 1), (3, 17, 3), (4, 24, 1), (5, 23, 3), (33, 100, 1), (127, 17, 3), (4093, 23, 1)]


def _lwr_feature(chain, cfg, feature, n, M, K, seed):
    """(params, batch, GPU keyword arguments, oracle keyword arguments) of one LWR feature set."""
    from vfclik_b200.engine import BRIDGE_POWERCUBE, Params
    rng = np.random.default_rng(seed)
    tool = (0, -1, 0, 1, 0, 0, 0, 0, 1, 0.03, -0.02, 0.15) if feature == "weights_tool_jp_aux" else None
    w = edge_batch(chain, n, M, seed, tool=tool)
    gpu, orc = {}, {}
    if feature == "weights_tool_jp_aux":
        prm = Params.from_config(cfg, w_task=(1, 1, 1, 0.5, 0.5, 0.5), w_joint=(1, 0.8, 1, 1.2, 1, 1, 0.5), ns_lambda=0.07,
                                 tool=tool, mixer_w=(0.9, 0.8, 0.7, 0, 0, 0))
        jp_ref = rng.uniform(-3.2, 3.2, size=(7, n))
        lo = -0.5 - rng.uniform(0, 1.5, size=(7, n))
        hi = 0.4 + rng.uniform(0, 1.5, size=(7, n))
        aux = np.zeros((2, 12, n))
        aux[0, 0] = 4; aux[0, 1] = -50                                       # hemisphere repeller below the goal
        aux[0, 2:5] = w["goal"][9:12] + rng.uniform(-0.3, 0.3, size=(3, n)); aux[0, 5:8] = rng.normal(size=(3, n))
        aux[0, 8] = rng.uniform(0.01, 0.1, size=n); aux[0, 9] = rng.uniform(2, 6, size=n)
        aux[1, 0] = 5; aux[1, 1] = 30                                        # funnel at the goal
        aux[1, 2:5] = w["goal"][9:12]; aux[1, 5:8] = rng.normal(size=(3, n))
        aux[1, 8] = rng.uniform(0.2, 0.8, size=n); aux[1, 9] = 10; aux[1, 10] = rng.uniform(0.1, 0.5, size=n); aux[1, 11] = 2
        gpu = dict(extra={"jp_ref": jp_ref, "jp_lo": lo, "jp_hi": hi}, aux=aux)
        orc = dict(jp_ref=jp_ref.T, jp_limits=(lo.T, hi.T), aux=aux.transpose(2, 0, 1))
    elif feature == "ports_truncated_ik":
        prm = Params.from_config(cfg, ik_mode=1, ik_eps=1e-5, mixer_w=(0.9, 0.8, 0.7, 0.6, 0.5, 0.4))
        x = rng.normal(scale=0.2, size=(7, n))
        q_cmded = w["q"] + rng.normal(scale=0.01, size=(7, n))
        ports = [rng.normal(scale=0.1, size=(7, n)) for _ in range(3)]
        gpu = dict(extra={"ns_in": x, "q_cmded": q_cmded}, ext_cmd=ports)
        orc = dict(ns_in=x.T, q_cmded=q_cmded.T, ext_cmd=tuple(p.T for p in ports))
    else:
        prm = dataclasses.replace(Params.from_config(cfg), speed_scale=0.41, max_vel=0.3, bridge_kind=BRIDGE_POWERCUBE,
                                  shoulder_vel=(0.05, -0.08))
    return prm, w, gpu, orc


@pytest.mark.parametrize("feature", ["weights_tool_jp_aux", "ports_truncated_ik", "powercube"])
@pytest.mark.parametrize("n,M,K", NMK)
def test_coop_lwr_features(lwr_cfg, monkeypatch, feature, n, M, K):
    """The 7-joint LWR through the cooperative kernel with per-obstacle {safe, order} rows next to the tool and goals next to
    it: non-identity IK weights and tool frame with per-instance joint-controller reference and limits (the clamped reference
    written back) and auxiliary fields; nullspace input, commanded q, three extra mixer ports and the truncated IK; the
    Powercube back-end.  n covers partial 4-instance groups, a partial warp and a ragged last tile; M = 16 keeps both chunks
    resident, 17 streams with a one-obstacle last chunk and a padding slot, 23 leaves 7 in the last chunk."""
    from vfclik_b200.engine import Engine
    chain, cfg = lwr_cfg
    prm, w, gpu, orc = _lwr_feature(chain, cfg, feature, n, M, K, seed=200 + n + M)
    e = Engine(chain, precision=64, params=prm)
    try:
        coop, solo = coop_and_solo(monkeypatch, e, w, M, K, **gpu)
        ref = run_oracle(chain, prm, w, M, k=K, **orc)
        check_all(coop, solo, ref)
        if "jp_ref" in ref:
            assert np.array_equal(coop["jp_ref"], ref["jp_ref"]) and np.array_equal(coop["jp_ref"], solo["jp_ref"])
    finally:
        e.close()


@pytest.mark.parametrize("ns_mode", [0, 1, 2])
@pytest.mark.parametrize("n,M,K", [(5, 17, 3), (127, 16, 1), (4093, 24, 3)])
def test_coop_nullspace_modes(lwr_cfg, monkeypatch, ns_mode, n, M, K):
    """Nullspace off, the undamped projector (ns_lambda = 0: the Householder path), and the control interface (state in
    ns_lastvec) through the cooperative kernel."""
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    prm = Params.from_config(cfg, ns_mode=ns_mode, ns_lambda=0.0, ns_control=(0.3, 0, 0, 0), mixer_w=(1.0, 1.0, 0.5, 0, 0, 0))
    e = Engine(chain, precision=64, params=prm)
    try:
        w = edge_batch(chain, n, M, seed=300 + n)
        extra = {"ns_lastvec": np.zeros((7, n))} if ns_mode == 2 else None
        coop, solo = coop_and_solo(monkeypatch, e, w, M, K, extra=extra)
        ref = run_oracle(chain, prm, w, M, k=K)
        check_all(coop, solo, ref)
        if ns_mode == 2:
            assert np.max(np.abs(coop["lastvec"] - ref["lastvec"])) < 1e-9
            assert np.max(np.abs(coop["lastvec"] - solo["lastvec"])) < 1e-11
    finally:
        e.close()


@pytest.mark.parametrize("n,M", [(33, 17), (4093, 23)])
def test_coop_control_nullspace_10_joints(built_lib, monkeypatch, n, M):
    """Generic 10-joint chain, control-mode nullspace (k = 4 basis vectors), K = 4 fused cycles: the per-group ns_lastvec
    writes against the oracle and orthonormal."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain = workloads.torso_arm_chain(10)
    prm = Params(ns_mode=2, ns_control=(0.3, -0.2, 0.25, 0.1), mixer_w=(1.0, 1.0, 0, 0, 0, 0))
    e = Engine(chain, precision=64, params=prm)
    try:
        w = edge_batch(chain, n, M, seed=400 + n)
        ctrl = np.random.default_rng(401).uniform(-0.4, 0.4, size=(4, n))
        coop, solo = coop_and_solo(monkeypatch, e, w, M, 4, outputs=("qdot_vf", "qdot_ns", "qdot", "flags"),
                                   extra={"ns_lastvec": np.zeros((40, n)), "ns_in": ctrl})
        ref = run_oracle(chain, prm, w, M, k=4, ns_in=ctrl.T)
        check_all(coop, solo, ref, keys=("qdot_vf", "qdot_ns", "qdot"))
        assert np.max(np.abs(coop["lastvec"] - ref["lastvec"])) < 1e-9
        u = coop["lastvec"].reshape(n, 4, 10)
        assert np.allclose(np.einsum("ikn,iln->ikl", u, u), np.eye(4)[None], atol=1e-12)
    finally:
        e.close()


@pytest.mark.parametrize("chain_name", ["dh10", "dh17", "generic17"])
@pytest.mark.parametrize("ext", [False, True])
@pytest.mark.parametrize("n,M,K", [(3, 16, 1), (127, 17, 3), (4093, 24, 1)])
def test_coop_long_chains(built_lib, monkeypatch, chain_name, ext, n, M, K):
    """The DH-pattern 10- and 17-joint chains and the generic 17-joint chain through the cooperative kernel, default parameters,
    with uniform and with per-obstacle {safe, order}."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine
    chain = {"dh10": lambda: workloads.dual_arm_torso_chain(10), "dh17": workloads.dual_arm_torso_chain,
             "generic17": lambda: workloads.dual_arm_torso_chain(dh=False)}[chain_name]()
    e = Engine(chain, precision=64)
    assert e.chain_pattern == ("generic" if chain_name == "generic17" else "dh")
    try:
        w = edge_batch(chain, n, M, seed=500 + n + M, ext=ext)
        coop, solo = coop_and_solo(monkeypatch, e, w, M, K)
        check_all(coop, solo, run_oracle(chain, e.params, w, M, k=K))
    finally:
        e.close()


@pytest.mark.parametrize("n_joints", [3, 8, 12])
@pytest.mark.parametrize("n,M,K", [(4, 17, 2), (4093, 23, 2)])
def test_coop_padded_chains(built_lib, monkeypatch, n_joints, n, M, K):
    """Joint counts without an instantiation of their own run padded in the next larger generic kernel, cooperative shape too:
    every output, the flags and q (what test_any_joint_count checks in the one-thread shape)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain = workloads.torso_arm_chain(n_joints)
    prm = Params(mixer_w=(1.0, 1.0, 0.5, 0, 0, 0), jp_ref=tuple([0.1] * n_joints))
    e = Engine(chain, precision=64, params=prm)
    try:
        w = edge_batch(chain, n, M, seed=600 + n_joints, ext=False)
        coop, solo = coop_and_solo(monkeypatch, e, w, M, K)
        check_all(coop, solo, run_oracle(chain, prm, w, M, k=K))
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ c. invariants
def test_coop_k_fused_equals_single_launches(lwr_cfg):
    """K = 4 fused cycles in the cooperative kernel are bit-identical to 4 single-cycle launches."""
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    chain, cfg = lwr_cfg
    e = Engine(chain, precision=64, params=Params.from_config(cfg, mixer_w=(1.0, 1.0, 0.5, 0, 0, 0)))
    try:
        n, M = 127, 17
        w = edge_batch(chain, n, M, seed=700)
        db = DeviceBatch(e, n, M, obst_ext=True, outputs=("qdot_vf", "qdot", "twist", "flags"))
        db.upload("goal", w["goal"]); db.upload("obst", w["obst"]); db.upload("obst_ext", w["obst_ext"])
        db.upload("q", w["q"])
        for _ in range(4):
            db.step(1)
        loop = {k: db.download(k) for k in ("q", "qdot_vf", "qdot", "twist", "flags")}
        db.upload("q", w["q"])
        db.step(4)
        for k, v in loop.items():
            assert np.array_equal(db.download(k), v), k
    finally:
        e.close()


@pytest.mark.parametrize("n", [37, 4093])
def test_coop_outputs_stay_inside_their_buffers(lwr_cfg, n):
    """Guard bands around every output of the cooperative kernel and around the state it writes in place (ns_lastvec, the
    clamped jp_ref): ragged batches, 19 obstacles with {safe, order} rows, K = 2."""
    import torch
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    chain, cfg = lwr_cfg
    SENT = -777.25
    M = 19
    e = Engine(chain, precision=64, params=Params.from_config(cfg, ns_mode=2, ns_control=(0.3, 0, 0, 0),
                                                              mixer_w=(1.0, 1.0, 0.5, 0, 0, 0)))
    try:
        w = edge_batch(chain, n, M, seed=800 + n)
        db = DeviceBatch(e, n, M, obst_ext=True, outputs=ALL, inputs=("jp_ref", "jp_lo", "jp_hi", "ns_lastvec"))
        db.upload("q", w["q"]); db.upload("goal", w["goal"]); db.upload("obst", w["obst"]); db.upload("obst_ext", w["obst_ext"])
        db.upload("jp_ref", np.full((7, n), 2.5)); db.upload("jp_lo", np.full((7, n), -0.3)); db.upload("jp_hi", np.full((7, n), 0.4))
        guarded = {}
        for name in ALL + ("q", "jp_ref", "ns_lastvec"):
            t = db.t[name]
            pad = 4096 // t.element_size()
            sent = SENT if t.dtype.is_floating_point else -777
            big = torch.full((t.numel() + 2 * pad,), sent, dtype=t.dtype, device=t.device)
            big[pad:pad + t.numel()] = t.reshape(-1)
            db.t[name] = big[pad:pad + t.numel()].view(t.shape)
            guarded[name] = (big, pad, t.numel(), sent)
        assert db.step(2) == 1
        torch.cuda.synchronize()
        for name, (big, pad, cnt, sent) in guarded.items():
            assert bool((big[:pad] == sent).all()) and bool((big[pad + cnt:] == sent).all()), name
        assert np.all(db.download("jp_ref") == 0.4)
        ref = run_oracle(chain, e.params, w, M, k=2, jp_ref=np.full((n, 7), 2.5), jp_limits=(np.full((n, 7), -0.3), np.full((n, 7), 0.4)))
        assert rel_err(db.download("qdot").T, ref["qdot"]).max() <= FP64_RTOL
    finally:
        e.close()


@pytest.mark.parametrize("n,M", [(1, 16), (4096, 24)])
def test_coop_session_paths(lwr_cfg, n, M):
    """The host-buffer session in the cooperative shape: one robot with 16 obstacle slots and {safe, order} rows through the
    copy pipeline (what ControlRuntime runs), and 4096 instances with page-locked buffers (direct host I/O: the kernel reads
    q from host memory).  Both bit-identical to the device path."""
    import torch
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    e = Engine(chain, precision=64, params=Params.from_config(cfg))
    try:
        w = edge_batch(chain, n, M, seed=900 + n)
        dev = run_gpu(e, w, M, k=2, outputs=("qdot", "flags"))
        s = e.session(n, M, obst_ext=True)
        try:
            s.set_goal(w["goal"]); s.set_obstacles(w["obst"], w["obst_ext"])
            if n >= 1024:
                q_in = torch.from_numpy(w["q"]).pin_memory().numpy()
                qd = torch.zeros((7, n), dtype=torch.float64).pin_memory().numpy()
                assert s.cycle(q_in=q_in, k_cycles=2, qdot_out=qd) == 1                # direct host I/O: the cycle kernel only
            else:
                qd = np.zeros((7, n))
                assert s.cycle(q_in=w["q"], k_cycles=2, qdot_out=qd) > 1               # copy pipeline
            assert np.array_equal(qd.T, dev["qdot"])
            qo, fl = np.zeros((7, n)), np.zeros(n, dtype=np.int32)
            s.cycle(q_in=w["q"], k_cycles=2, qdot_out=qd, q_out=qo, flags_out=fl)
            assert np.array_equal(qd.T, dev["qdot"]) and np.array_equal(qo.T, dev["q"]) and np.array_equal(fl, dev["flags"])
        finally:
            s.close()
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 2. field regimes
UNIFORM = [(order, safe) for order in (2.0, 5.0, 20.0, 3.0, 7.5) for safe in (0.0, 1e-3, 0.05)]
SHAPES = [(64, "lean"), (64, "general"), (64, "ext"), (64, "coop"), (64, "split17"),
          (32, "lean"), (32, "general"), (32, "ext"), (32, "split17"), (32, "split10")]


@pytest.mark.parametrize("rot_slowdown", [0.09, 0.5, 0.0])
@pytest.mark.parametrize("precision,shape", SHAPES)
def test_field_regimes(lwr_cfg, monkeypatch, precision, shape, rot_slowdown):
    """Goals within 1e-7 m / 1e-7 rad of the tool up to far away, translational slowdowns on and off, obstacles inside and
    outside their safe distance, through every kernel shape: the lean and the general one-thread instantiations, the
    per-obstacle {safe, order} path (FP32: the scalar MUFU repeller), the cooperative shape (FP64, M >= 16) and the lane
    split (the FP64 17-joint chain).  "split17" / "split10" are the 17- and 10-joint DH chains in the lean call shape; in
    FP32 they run the one-thread DhPattern kernel, which took them over when the FP32 split shape was removed.  Uniform
    decay orders 2 / 5 / 20 (FP64 multiplication chains), 3 (square-and-multiply) and 7.5 (pow), safe distances 0 / 1e-3 /
    0.05; rot_slowdown 0.09 (FP32: the small-angle asin series), 0.5 (atan2) and 0 (off)."""
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    dt = np.float64 if precision == 64 else np.float32
    tol = FP64_RTOL if precision == 64 else FP32_RTOL
    tw_tol = 1e-12 if precision == 64 else 2e-6
    n, M = (700, 17) if shape == "coop" else (700, 13)
    outputs = ("qdot",) if shape in ("lean", "split17", "split10") else ("qdot_vf", "qdot", "twist")
    prm = Params.from_config(cfg, rot_slowdown=rot_slowdown)
    if shape.startswith("split"):
        chain = workloads.dual_arm_torso_chain(17 if shape == "split17" else 10)
        prm = Params(rot_slowdown=rot_slowdown)
    elif shape != "coop":
        monkeypatch.setenv("VFK_NO_COOP", "1")
    e = Engine(chain, precision=precision, params=prm)
    try:
        for order, safe in ([(20.0, 1e-3)] if shape in ("ext",) else UNIFORM):
            e.set_params(obst_order=order, obst_safe=safe)
            w = edge_batch(chain, n, M, seed=1000 + int(10 * order) + int(1e3 * safe), dtype=dt, ext=shape == "ext",
                           safe=safe, order=order, rot_slowdown=rot_slowdown)
            out = run_gpu(e, w, M, outputs=outputs)
            ref = run_oracle(chain, e.params, w, M)
            for key in outputs:
                if key == "twist":
                    err = np.abs(out[key] - ref[key]).max()
                    assert err <= tw_tol, (order, safe, key, float(err))
                else:
                    err = rel_err(out[key].astype(np.float64), ref[key], floor=1e-3 if precision == 64 else FP32_FLOOR)
                    assert err.max() <= tol, (order, safe, key, float(err.max()), int(np.argmax(err)))
            assert np.all(np.isfinite(out["qdot"]))
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 3. rot_slowdown = 0
@pytest.mark.parametrize("precision,shape", [(64, "general"), (64, "coop"), (32, "general")])
def test_goal_orientation_reached_exactly(lwr_cfg, monkeypatch, precision, shape):
    """A goal whose orientation is the tool's own, bit for bit (a caller that keeps the current orientation sets the goal
    rotation from the pose): R_goal R_tool^T is then exactly symmetric, the rotation error exactly 0, and the rotational
    slowdown factor min(1, 0 / rot_slowdown) is 0 * inf with the slowdown off (rot_slowdown = 0).  The cycle must treat
    that as the oracle does (factor 1, no rotation to do): no NaN flag, finite joint velocities, zero angular twist, and
    the same joint velocities as with rot_slowdown = 0.09."""
    from vfclik_b200.engine import Engine, Params
    chain, cfg = lwr_cfg
    dt = np.float64 if precision == 64 else np.float32
    if shape == "general":
        monkeypatch.setenv("VFK_NO_COOP", "1")
    e = Engine(chain, precision=precision, params=Params.from_config(cfg))
    try:
        n, M = 200, 16
        w = edge_batch(chain, n, M, seed=1100, dtype=dt)
        first = run_gpu(e, w, M, outputs=("qdot", "pose", "flags"))
        w["goal"][0:9] = first["pose"].T[0:9]                         # the tool's rotation as output by the kernel
        outs = {}
        for rs in (0.0, 0.09):
            e.set_params(rot_slowdown=rs)
            out = run_gpu(e, w, M, outputs=("qdot_vf", "qdot", "twist", "flags"))
            assert not np.any(out["flags"] & 4), (rs, int(np.count_nonzero(out["flags"] & 4)))
            assert np.all(np.isfinite(out["qdot"])) and np.all(np.isfinite(out["qdot_vf"]))
            assert np.all(out["twist"][:, 3:6] == 0)
            outs[rs] = out
        assert np.array_equal(outs[0.0]["qdot"], outs[0.09]["qdot"]) and np.array_equal(outs[0.0]["twist"], outs[0.09]["twist"])
        # rot_slowdown = 0.09 against the oracle, whose own rotation error is the rounding of the kernel's pose (FP32: 6e-8)
        ref = run_oracle(chain, e.params, w, M)
        tol, floor = (FP64_RTOL, 1e-3) if precision == 64 else (FP32_RTOL, FP32_FLOOR)
        for key in ("qdot_vf", "qdot"):
            assert rel_err(outs[0.09][key].astype(np.float64), ref[key], floor=floor).max() <= tol, key
    finally:
        e.close()


@pytest.mark.parametrize("precision", [64, 32])
def test_field_query_at_the_goal_orientation(lwr_cfg, precision):
    """The same through Engine.field_eval, in both precisions: the query pose's rotation is the goal's own, so the rotation
    error is exactly 0; obstacles with {safe, order} rows next to the query position."""
    from oracle import batch
    from vfclik_b200.engine import DeviceBatch, Engine, Params
    chain, cfg = lwr_cfg
    dt = np.float64 if precision == 64 else np.float32
    e = Engine(chain, precision=precision, params=Params.from_config(cfg))
    try:
        n, M = 300, 6
        w = edge_batch(chain, n, M, seed=1200, dtype=dt)
        q, goal, obst = to_oracle(w, M)
        _, p, _ = batch.fk_jac(chain, q)
        pose = np.concatenate([w["goal"][0:9], p.T.astype(dt)], axis=0)
        got = {}
        for rs in (0.0, 0.09):
            e.set_params(rot_slowdown=rs)
            db = DeviceBatch(e, n, M, obst_ext=True, outputs=())
            db.upload("goal", w["goal"]); db.upload("obst", w["obst"]); db.upload("obst_ext", w["obst_ext"])
            pz = db.upload("pose", pose)
            assert e.field_eval(pz, db.t["goal"], db.t["obst"], db._ensure("twist"), n, M, obst_ext=db.t["obst_ext"]) == 1
            got[rs] = db.download("twist").T
            assert np.all(np.isfinite(got[rs])) and np.all(got[rs][:, 3:6] == 0)
        assert np.array_equal(got[0.0], got[0.09])
        v, _ = batch.field_eval(oracle_params(e.params), goal[:, 0:9].reshape(n, 3, 3), pose[9:12].T.astype(np.float64), goal, obst)
        assert np.allclose(got[0.09][:, 0:3], v, rtol=0, atol=1e-12 if precision == 64 else 2e-6)
    finally:
        e.close()
