"""The velocity IK and the nullspace at and near kinematic singularities, against the oracle.

Batches come from helpers.near_singular: the home posture q = 0 of every chain (rank 3 to 5) and the LWR's straight elbow
(rank 5), each moved by delta in {0, 1e-12, 1e-9, 1e-6, 1e-3, 1e-1}.  Random postures almost never come this close: there
the Cholesky of J J^T + lambda^2 I meets zero pivots, the Jacobi SVD zero singular values and the Householder QR exact
zeros.

Tolerances.  Where damping bounds the problem (the default lambda = 0.1, the truncated IK's damped branch) or where an
exact zero singular value is cut (the undamped projector at delta = 0), the suite's flat bounds hold: 1e-9 relative in
FP64, 1e-4 in FP32.  Elsewhere two correct FP64 implementations agree only to about eps64 * cond, so the bound is
max(1e-9, C * eps64 * cond), cond being the condition number that governs the problem:
- DLS with small lambda: cond(A) = (s_max^2 + lambda^2) / (s_min^2 + lambda^2), C = C_DLS.  The spread between
  numpy.linalg.solve (LU) and scipy.linalg.cho_solve (Cholesky) on these batches reaches 1.3 eps64 * cond(A).
- undamped projector, control basis, truncated IK: cond = s_max / s_kept, s_kept the smallest singular value the method
  keeps, C = C_SVD.  The spread between numpy's pinv (LAPACK gesdd) and one through LAPACK gesvd on these batches
  reaches 133 eps64 * cond (rel_err's 1e-3 floor counts an error against a projection of 1e-3 of x's size).
"""
import dataclasses

import numpy as np
import pytest

from helpers import FP32_RTOL, FP64_RTOL, near_singular, rel_err, run_gpu, run_oracle

pytestmark = pytest.mark.gpu

EPS64 = np.finfo(np.float64).eps
C_DLS = 16.0             # 12x the measured LU / Cholesky spread
C_SVD = 1000.0           # 7.5x the measured gesdd / gesvd spread
FLAG_NS_LIMIT, FLAG_NAN, FLAG_CLAMPED = 2, 4, 8
KINDS = [("lwr", "home"), ("lwr", "elbow"), ("torso10", "home"), ("dh17", "home"), ("generic17", "home")]


def _chain(lwr, name):
    from vfclik_b200 import workloads
    return {"lwr": lambda: lwr[0], "torso10": lambda: workloads.torso_arm_chain(10),
            "dh17": lambda: workloads.dual_arm_torso_chain(17),
            "generic17": lambda: workloads.dual_arm_torso_chain(17, dh=False)}[name]()


def _params(lwr, name, **over):
    from vfclik_b200.engine import Params
    return Params.from_config(lwr[1], **over) if name == "lwr" else Params(**over)


def _run(monkeypatch, e, w, M, shape, k=1, **kw):
    """One launch in the given shape: "lean" (qdot only), "general" (every output), both with VFK_NO_COOP=1; "coop" (FP64,
    n <= 4096, M >= 16); "split" (the FP64 17-joint lane split / the FP32 DhPattern kernel: lean call, M < 16)."""
    if shape in ("lean", "general"):
        monkeypatch.setenv("VFK_NO_COOP", "1")
    else:
        monkeypatch.delenv("VFK_NO_COOP", raising=False)
    outputs = ("qdot",) if shape in ("lean", "split") else ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd", "flags")
    try:
        return run_gpu(e, w, M, k=k, outputs=outputs, **kw)
    finally:
        monkeypatch.delenv("VFK_NO_COOP", raising=False)


def _sub(w, idx):
    return {k: (v[:, idx] if k != "obst" else v[:, idx, :]) for k, v in w.items()}


# ------------------------------------------------------------------------------------------------ a. DLS, lambda = 0.1
DLS_SHAPES = [(64, "lean"), (64, "general"), (64, "coop"), (64, "split"), (32, "lean"), (32, "general"), (32, "split")]


@pytest.mark.parametrize("precision,shape", DLS_SHAPES)
@pytest.mark.parametrize("chain_name,kind", KINDS)
def test_dls_default_lambda(lwr, built_lib, monkeypatch, precision, shape, chain_name, kind):
    """The default damping (lambda = 0.1) at every level including the exact singularity: the suite's flat bounds, since
    cond(J J^T + lambda^2 I) <= (s_max^2 + 0.01) / 0.01.  FP64 flags equal, FP32 flags as rare as in the random batches.
    The general shape passes a random ns_in: at q = 0 with symmetric limits the built-in limit gradient is 0."""
    from vfclik_b200.engine import Engine
    if shape == "split":
        if chain_name != "dh17":
            pytest.skip("the lane split / DhPattern shape is the 17-joint DH chain's")
    chain = _chain(lwr, chain_name)
    dt = np.float64 if precision == 64 else np.float32
    n, M = (1200, 16) if shape == "coop" else (1200, 8)
    w, meta = near_singular(chain, n, M, seed=10 + len(chain.q_lo), dtype=dt, kind=kind)
    e = Engine(chain, precision=precision, params=_params(lwr, chain_name))
    try:
        kw, okw = {}, {}
        if shape == "general":
            x = np.random.default_rng(11).normal(scale=0.2, size=(len(chain.q_lo), n)).astype(dt)
            kw, okw = dict(extra={"ns_in": x}), dict(ns_in=x.T.astype(np.float64))
        out = _run(monkeypatch, e, w, M, shape, **kw)
        ref = run_oracle(chain, e.params, w, M, **okw)
        tol = FP64_RTOL if precision == 64 else FP32_RTOL
        for key in [k for k in ("qdot_vf", "qdot_ns", "qdot_jp", "qdot", "cmd") if k in out]:
            err = rel_err(out[key].astype(np.float64), ref[key])
            assert err.max() <= tol, (key, float(err.max()), float(meta["delta"][np.argmax(err)]))
        assert np.all(np.isfinite(out["qdot"]))
        if "flags" in out:
            if precision == 64:
                assert np.array_equal(out["flags"], ref["flags"])
            else:
                assert np.mean(out["flags"] != ref["flags"]) < 1e-3
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ b. DLS, small lambda
def _dls_contract(out, prm, q0, K=None, q=None):
    """What the pivot floor guarantees where the oracle cannot follow: finite values, no NaN flag, the clamp holds and is
    flagged, and K integrated cycles move q at most K dt max_vel."""
    for key in ("qdot", "cmd", "q"):
        assert np.all(np.isfinite(out[key])), key
    assert not np.any(out["flags"] & FLAG_NAN)
    assert np.all(np.max(np.abs(out["qdot"]), axis=1) <= prm.max_vel * (1 + 1e-12))
    mix = sum(out[k] * wgt for k, wgt in zip(("qdot_vf", "qdot_ns", "qdot_jp"), prm.mixer_w))
    over = np.max(np.abs(mix), axis=1) > prm.max_vel * (1 + 1e-9)
    assert np.all(out["flags"][over] & FLAG_CLAMPED)
    if K is not None:
        assert np.all(np.abs(q - q0) <= K * prm.dt * prm.max_vel * (1 + 1e-12) + 1e-15)


@pytest.mark.parametrize("ik_lambda", [1e-2, 1e-4, 0.0])
@pytest.mark.parametrize("shape", ["general", "coop"])
@pytest.mark.parametrize("chain_name,kind", KINDS)
def test_dls_small_lambda_fp64(lwr, built_lib, monkeypatch, ik_lambda, shape, chain_name, kind):
    """FP64 DLS with lambda down to 0 (the reference's undamped pinv; FP32 refuses it).  Where eps64 cond(A) <= 1e-4 the
    oracle's solve is meaningful: rel_err <= max(1e-9, C_DLS eps64 cond(A)).  Elsewhere (A singular or nearly) the contract
    of the pivot floor: finite, no NaN flag, |qdot| <= max_vel with the clamp flagged, and after 5 integrated cycles
    |dq| <= 5 dt max_vel."""
    from vfclik_b200.engine import Engine
    chain = _chain(lwr, chain_name)
    n, M = 1200, 16
    w, meta = near_singular(chain, n, M, seed=20 + len(chain.q_lo), kind=kind)
    prm = _params(lwr, chain_name, ik_lambda=ik_lambda)
    e = Engine(chain, precision=64, params=prm)
    try:
        out = _run(monkeypatch, e, w, M, shape)
        s2 = meta["sigma"] ** 2 + ik_lambda ** 2
        with np.errstate(divide="ignore"):
            condA = s2[:, 0] / s2[:, -1]
        ok = EPS64 * condA <= 1e-4
        assert ok.sum() >= n // 4                            # lambda = 0: the levels 1e-3 and 1e-1, a third of the batch
        idx = np.flatnonzero(ok)
        ref = run_oracle(chain, prm, _sub(w, idx), M)
        tol = np.maximum(FP64_RTOL, C_DLS * EPS64 * condA[idx])
        for key in ("qdot_vf", "qdot", "cmd"):
            err = rel_err(out[key][idx], ref[key])
            assert np.all(err <= tol), (key, float(np.max(err / tol)), float(meta["delta"][idx][np.argmax(err / tol)]))
        assert np.array_equal(out["flags"][idx], ref["flags"])
        _dls_contract(out, prm, w["q"].T)
        K = 5
        outk = _run(monkeypatch, e, w, M, shape, k=K)
        _dls_contract(outk, prm, w["q"].T, K=K, q=outk["q"])
    finally:
        e.close()


@pytest.mark.parametrize("shape", ["general", "coop"])
def test_undamped_dls_at_lwr_home_is_the_minimum_norm_solution(lwr, built_lib, monkeypatch, shape):
    """At the LWR's q = 0, J has exactly zero rows; at lambda = 0 the floored pivots decouple them, and qdot_vf must be the
    minimum-norm pinv(J) t (numpy, 1e-9) -- provided the kernel's FK gives those zeros exactly (it does: the test fails
    otherwise, as a 1e-17 entry against a floored pivot of 1e-28 trace would be amplified far past 1e-9)."""
    from oracle import batch
    from vfclik_b200.engine import Engine
    chain = lwr[0]
    n, M = 600, 16
    w, meta = near_singular(chain, n, M, seed=30, kind="home", levels=(0.0,))
    J = batch.fk_jac(chain, w["q"].T)[2]
    zero_rows = np.all(J == 0.0, axis=2)
    assert np.all(zero_rows.sum(axis=1) == 3)
    prm = _params(lwr, "lwr", ik_lambda=0.0, max_vel=1e6)
    e = Engine(chain, precision=64, params=prm)
    try:
        out = _run(monkeypatch, e, w, M, shape)
        # the task twist t of the IK, through the oracle at lambda = 0.1 (its solve rejects the singular A of lambda = 0)
        ref = run_oracle(chain, dataclasses.replace(prm, ik_lambda=0.1), w, M)
        tool = np.asarray(prm.tool, dtype=np.float64)
        R, p, _ = batch.fk_jac(chain, w["q"].T)
        dp = -(R @ tool[9:12])
        v, om = ref["twist"][:, 0:3], ref["twist"][:, 3:6]
        t = np.concatenate([v + np.cross(om, dp), om], axis=1)
        mn = np.einsum("ink,ik->in", np.linalg.pinv(J), t)
        err = rel_err(out["qdot_vf"], mn)
        assert err.max() <= FP64_RTOL, (float(err.max()), int(np.argmax(err)))
        assert not np.any(out["flags"] & FLAG_NAN)
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ c. truncated IK
@pytest.mark.parametrize("ik_eps", [1e-5, 1e-3, 1e-1])
@pytest.mark.parametrize("ik_lambda", [0.1, 1e-3])
@pytest.mark.parametrize("weights", ["unit", "weighted"])
@pytest.mark.parametrize("shape", ["general", "coop"])
@pytest.mark.parametrize("kind", ["home", "elbow"])
def test_truncated_ik_across_eps(lwr, built_lib, monkeypatch, ik_eps, ik_lambda, weights, shape, kind):
    """VFK_IK_TRUNCATED (FP64) on the LWR: 40 % of the batch near the singularity, the rest random postures, so that at least 20 %
    of the instances take the damped branch (a singular value of Jw below ik_eps) and at least 20 % take only the plain
    one.  Instances with a singular value within 1e-8 of ik_eps (either branch is right) are left out, at most 1 %.
    Tolerance max(1e-9, C_SVD eps64 s_max / s_kept), s_kept the smallest singular value >= ik_eps; at delta = 0 the flat
    1e-9."""
    from oracle import batch
    from vfclik_b200 import workloads
    from vfclik_b200.engine import Engine
    chain = lwr[0]
    n, M = 1200, 16
    seed = 40 + int(-np.log10(ik_eps))
    w, meta = near_singular(chain, n, M, seed=seed, kind=kind)
    h = 2 * n // 5
    w["q"][:, h:] = workloads.random_batch(chain, n, M, seed)["q"][:, h:]
    delta = np.where(np.arange(n) < h, meta["delta"], np.nan)
    over = dict(ik_mode=1, ik_eps=ik_eps, ik_lambda=ik_lambda)
    if weights == "weighted":
        over.update(w_task=(1, 1, 1, 0.5, 0.5, 0.5), w_joint=(1, 0.8, 1, 1.2, 1, 1, 0.5))
    prm = _params(lwr, "lwr", **over)
    wt = np.asarray(prm.w_task, dtype=np.float64)
    wj = np.ones(7) if prm.w_joint is None else np.asarray(prm.w_joint, dtype=np.float64)
    J = batch.fk_jac(chain, w["q"].T)[2]
    sg = np.linalg.svd(wt[None, :, None] * J * wj[None, None, :], compute_uv=False)
    damped = np.any(sg < ik_eps, axis=1)
    assert damped.mean() >= 0.2 and (~damped).mean() >= 0.2, (damped.mean(), ik_eps)
    edge = np.any(np.abs(sg / ik_eps - 1) < 1e-8, axis=1)
    assert edge.mean() <= 0.01
    e = Engine(chain, precision=64, params=prm)
    try:
        out = _run(monkeypatch, e, w, M, shape)
        ref = run_oracle(chain, prm, w, M)
        kept = np.where(sg >= ik_eps, sg, np.inf).min(axis=1)
        tol = np.maximum(FP64_RTOL, C_SVD * EPS64 * sg[:, 0] / np.where(np.isinf(kept), sg[:, 0], kept))
        tol[delta == 0] = FP64_RTOL
        for key in ("qdot_vf", "qdot"):
            err = rel_err(out[key], ref[key])[~edge]
            assert np.all(err <= tol[~edge]), (key, float(np.max(err / tol[~edge])), float(delta[~edge][np.argmax(err / tol[~edge])]))
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ d. undamped projector
def _kept_cond(sigma, cut):
    """s_max / (smallest singular value above cut * s_max): the condition number of the part of J a projector keeps."""
    kept = np.where(sigma > cut * sigma[:, :1], sigma, np.inf).min(axis=1)
    return sigma[:, 0] / kept


@pytest.mark.parametrize("precision,shape", [(64, "general"), (64, "coop"), (32, "general")])
@pytest.mark.parametrize("chain_name,kind", KINDS)
def test_undamped_projector_near_singular(lwr, built_lib, monkeypatch, precision, shape, chain_name, kind):
    """ns_mode = 1, ns_lambda = 0 with a random ns_in: I - pinv(J) J (numpy's pinv in the oracle).
    - delta = 0: flat 1e-9 (FP64) / 1e-4 (FP32).  The gap between the kept singular values and the exact zeros makes that
      projector well-conditioned; a projector that is not rank-revealing misses rank(J) - 6 dimensions of null(J) here.
    - near: FP64 max(1e-9, C_SVD eps64 cond), cond over the singular values above pinv's cutoff.  FP32 (J rounded to float)
      max(1e-4, 2e-6 cond(J)) as for random postures, where s_min > 1e-5 s_max; between that and 0 the FP32 cutoff
      (1e-6 s_max) may cut a direction the FP64 oracle keeps, and only the contract below is asserted.
    - every level: J qdot_ns stays at rounding of |J| |x| (1e-12 in FP64, 1e-6 in FP32), and the projector does not expand."""
    from oracle import batch
    from vfclik_b200.engine import Engine
    chain = _chain(lwr, chain_name)
    N = len(chain.q_lo)
    dt = np.float64 if precision == 64 else np.float32
    n, M = 1200, 16
    w, meta = near_singular(chain, n, M, seed=50 + N, dtype=dt, kind=kind)
    x = np.random.default_rng(51).normal(scale=0.2, size=(N, n)).astype(dt)
    prm = _params(lwr, chain_name, ns_mode=1, ns_lambda=0.0, ns_gain=1.0, mixer_w=(1.0, 1.0, 0, 0, 0, 0))
    e = Engine(chain, precision=precision, params=prm)
    try:
        out = _run(monkeypatch, e, w, M, shape, extra={"ns_in": x})
        ref = run_oracle(chain, prm, w, M, ns_in=x.T.astype(np.float64))
        live = (out["flags"] & FLAG_NS_LIMIT) == 0
        assert live.mean() > 0.5
        at0 = meta["delta"] == 0
        err = rel_err(out["qdot_ns"].astype(np.float64), ref["qdot_ns"])
        if precision == 64:
            tol = np.maximum(FP64_RTOL, C_SVD * EPS64 * _kept_cond(meta["sigma"], 1e-15))
            tol[at0] = FP64_RTOL
            check = np.ones(n, dtype=bool)
        else:
            tol = np.maximum(FP32_RTOL, 2e-6 * meta["cond"])
            tol[at0] = FP32_RTOL
            check = at0 | (meta["sigma"][:, -1] > 1e-5 * meta["sigma"][:, 0])
        bad = check & (err > tol)
        assert not bad.any(), (int(bad.sum()), float(np.max(err[check] / tol[check])),
                               sorted(set(meta["delta"][bad].tolist())), float(err[at0].max()))
        # the contract at every level, on the instances whose projection the limit check let through
        J = batch.fk_jac(chain, w["q"].T.astype(np.float64))[2]
        raw = out["qdot_ns"].astype(np.float64)[live]
        xl = x.T.astype(np.float64)[live]
        nJ = np.linalg.norm(J[live], ord=2, axis=(1, 2))
        res = np.linalg.norm(np.einsum("ikn,in->ik", J[live], raw), axis=1)
        assert np.all(res <= (1e-12 if precision == 64 else 1e-6) * nJ * np.linalg.norm(xl, axis=1))
        assert np.all(np.linalg.norm(raw, axis=1) <= np.linalg.norm(xl, axis=1) * (1 + (1e-14 if precision == 64 else 1e-6)))
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ e. control interface
@pytest.mark.parametrize("shape", ["general", "coop"])
@pytest.mark.parametrize("chain_name,kind", [("lwr", "home"), ("lwr", "elbow"), ("torso10", "home"), ("dh17", "home"),
                                             ("generic17", "home")])
def test_control_basis_near_singular(lwr, built_lib, monkeypatch, shape, chain_name, kind):
    """ns_mode = 2 (FP64): the Householder basis of null(J).  Near the singularity, lastvec against the oracle at
    max(1e-9, C_SVD eps64 cond(J)).  At delta = 0 the reference would find rank-deficiency's extra vectors and the oracle
    assumes full rank, so there the contract, with integrate = 0 (the posture stays put): unit vectors, mutually
    orthogonal, |J u| <= 1e-12 |J|, and the same vectors after 1 and after 3 cycles."""
    from oracle import batch
    from vfclik_b200.engine import Engine, ns_ctrl_vectors
    chain = _chain(lwr, chain_name)
    N = len(chain.q_lo)
    kk = ns_ctrl_vectors(N)
    n, M = 1200, 16
    w, meta = near_singular(chain, n, M, seed=60 + N, kind=kind)
    ctrl = np.random.default_rng(61).uniform(-0.4, 0.4, size=(4, n))
    prm = _params(lwr, chain_name, ns_mode=2, mixer_w=(1.0, 1.0, 0, 0, 0, 0), integrate=0)
    e = Engine(chain, precision=64, params=prm)
    try:
        outs = {}
        for K in (1, 3):
            outs[K] = _run(monkeypatch, e, w, M, shape, k=K, extra={"ns_lastvec": np.zeros((kk * N, n)), "ns_in": ctrl})
        at0 = meta["delta"] == 0
        near = ~at0
        idx = np.flatnonzero(near)
        ref = run_oracle(chain, prm, _sub(w, idx), M, k=1, ns_in=ctrl.T[idx])
        tol = np.maximum(1e-9, C_SVD * EPS64 * meta["cond"][idx])
        err = np.max(np.abs(outs[1]["lastvec"][idx] - ref["lastvec"]), axis=1)
        assert np.all(err <= tol), (float(np.max(err / tol)), float(meta["delta"][idx][np.argmax(err / tol)]))
        err = rel_err(outs[1]["qdot_ns"][idx], ref["qdot_ns"])
        assert np.all(err <= tol), ("qdot_ns", float(np.max(err / tol)))
        # delta = 0: the contract
        J = batch.fk_jac(chain, w["q"].T)[2][at0]
        u = outs[1]["lastvec"][at0].reshape(-1, kk, N)
        assert np.all(np.isfinite(u))
        assert np.allclose(np.einsum("ikn,iln->ikl", u, u), np.eye(kk)[None], rtol=0, atol=1e-12)
        nJ = np.linalg.norm(J, ord=2, axis=(1, 2))
        assert np.all(np.linalg.norm(np.einsum("irn,ikn->ikr", J, u), axis=2) <= 1e-12 * nJ[:, None])
        assert np.array_equal(outs[3]["lastvec"][at0], outs[1]["lastvec"][at0])
        assert np.array_equal(outs[3]["q"], w["q"].T)
    finally:
        e.close()
