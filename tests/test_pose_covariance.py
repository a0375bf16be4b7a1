"""Per-pair 6x6 pose covariance (dvo_pose_covariance) and its propagation along the key-frame chain (dvo_run_sequences_cov).

CPU: the dvo_cov_info layout, and a Monte-Carlo check of the propagation rule and the tangent convention
(psi = (rho, omega), T <- T exp(psi)) with the oracle's SE(3) exp / log.
GPU: parity with a covariance built from the oracle's per-point outputs, launch-size independence, device == host
output, no side effects on solver state, degenerate slots, and the sequence loop.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import rgbd_odometry_b200 as dvo


def skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]], np.float64)


def adjoint(R, t):
    """Ad(T) for tangent (rho, omega): [[R, [t]x R], [0, R]]."""
    A = np.zeros((6, 6))
    A[:3, :3] = R; A[:3, 3:] = skew(t) @ R; A[3:, 3:] = R
    return A


def adjoint_inv(R, t):
    return adjoint(R.T, -R.T @ t)


def propagate(rel, kind, rel_cov):
    """numpy reference of the global covariance: Sigma_g(i) = Ad(Tr^-1) Sigma_key Ad(Tr^-1)^T + Sigma_rel(i), Sigma_key <- Sigma_g(i) where
    kind[i] != 0.  rel (nseq, nframes, 12), kind (nseq, nframes), rel_cov (nseq, nframes, 6, 6)."""
    out = np.empty_like(rel_cov)
    for s in range(rel.shape[0]):
        key = np.zeros((6, 6))
        for i in range(rel.shape[1]):
            A = adjoint_inv(rel[s, i, :9].reshape(3, 3), rel[s, i, 9:])
            out[s, i] = A @ key @ A.T + rel_cov[s, i]
            if kind[s, i] != 0:
                key = out[s, i]
    return out


# ------------------------------------------------------------------------------------------------ CPU
def test_cov_info_layout_matches_header():
    assert C.sizeof(dvo.CovInfo) == 32
    assert (dvo.CovInfo.status.offset, dvo.CovInfo.level.offset, dvo.CovInfo.nvis.offset) == (0, 4, 8)
    assert (dvo.CovInfo.sigma2.offset, dvo.CovInfo.logdet.offset) == (16, 24)


def _random_spd(rng, scale):
    A = rng.standard_normal((6, 6))
    return scale * (A @ A.T + 0.5 * np.eye(6))


def test_propagation_rule_and_convention_monte_carlo():
    """T_k exp(dk) T_r exp(dr) mapped back with log(T_g^-1 sample): its sample covariance is Ad(Tr^-1) Sk Ad(Tr^-1)^T + Sr."""
    rng = np.random.default_rng(7)
    Rk, tk = O.se3_exp(np.array([0.3, -0.2, 0.5, 0.2, -0.4, 0.3]))
    Rr, tr = O.se3_exp(np.array([0.4, -0.3, 0.5, 0.3, 0.5, -0.4]))
    Sk, Sr = _random_spd(rng, 1e-6), _random_spd(rng, 1e-6)
    Rg, tg = Rk @ Rr, Rk @ tr + tk
    n = 20000
    dk = rng.multivariate_normal(np.zeros(6), Sk, n)
    dr = rng.multivariate_normal(np.zeros(6), Sr, n)
    samples = np.empty((n, 6))
    for i in range(n):
        Ek, ek = O.se3_exp(dk[i]); Er, er = O.se3_exp(dr[i])
        R1, t1 = Rk @ Ek, Rk @ ek + tk                       # T_k exp(dk)
        R2, t2 = R1 @ Rr, R1 @ tr + t1                       # .. T_r
        R3, t3 = R2 @ Er, R2 @ er + t2                       # .. exp(dr)
        samples[i] = O.se3_log(Rg.T @ R3, Rg.T @ (t3 - tg))  # log(T_g^-1 sample)
    got = np.cov(samples.T)
    A = adjoint_inv(Rr, tr)
    want = A @ Sk @ A.T + Sr
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < 0.05
    # the other orders are measurably wrong: the rule pins the convention
    for wrong in (Sk + Sr, adjoint(Rr, tr) @ Sk @ adjoint(Rr, tr).T + Sr):
        assert np.linalg.norm(got - wrong) / np.linalg.norm(want) > 0.1


# ------------------------------------------------------------------------------------------------ GPU
K320 = (262.5, 262.5, 159.5, 119.5)


def oracle_cov(ref_gray, ref_depth, now_gray, level, R, T, K, weight, huber_k=1.345, residual=O.RES_DT_FLOOR):
    """H_o, sigma2_o, nvis from the oracle's per-point EXACT-Jacobian outputs at (R, T)."""
    ref = O.preprocess_level(ref_gray, ref_depth, level)
    now = O.preprocess_level(now_gray, None, level)
    X, Y, Z, _, _ = O.select_points(ref["edge"], ref["depth"], level, K)
    o = O.evaluate(X, Y, Z, now["dtn"], now["gx"], now["gy"], level, R, T, K=K, jac=O.JAC_EXACT, weight=weight, huber_k=huber_k,
                   per_point=True, residual=residual)
    iu = np.triu_indices(6)
    H = np.zeros((6, 6)); H[iu] = o["H"][iu]; H = H + np.triu(H, 1).T       # the accumulated upper triangle, mirrored
    s2 = float(np.sum(o["w"].astype(np.float64) * o["eps"].astype(np.float64) ** 2)) / (o["nvis"] - 6)
    return H, s2, o["nvis"]


def check_against_oracle(cov, inf, H, s2, nvis, level):
    assert inf.status == 0 and inf.level == level and inf.nvis == nvis
    assert abs(inf.sigma2 - s2) <= 1e-10 * s2
    assert np.abs(cov @ H / s2 - np.eye(6)).max() < 1e-6
    assert np.array_equal(cov, cov.T)
    assert abs(inf.logdet - (6 * np.log(s2) - np.linalg.slogdet(H)[1])) < 1e-8


@pytest.fixture(scope="module")
def small_batch():
    W, H, L, n = 320, 240, 4, 8
    d = O.synth_batch(4100, n, W, H, K320)
    al = dvo.BatchAligner(W, H, L, max_batch=n, intrinsics=K320)
    al.set_frames(dvo.FRAME_REF, d["ref_gray"], d["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, d["now_gray"], None)
    al.build_pyramids(n)
    al.prepare(n)
    yield al, d, n
    al.close()


CASES = [  # (solver, weight, residual, iters, level)
    (dvo.GN, dvo.W_REF_CAUCHY, dvo.RES_DT_FLOOR, (10, 10, 10, 10), -1),
    (dvo.GN, dvo.W_HUBER, dvo.RES_DT_FLOOR, (10, 10, 10, 10), -1),
    (dvo.SUBGRAD_REF, dvo.W_REF_CAUCHY, dvo.RES_DT_FLOOR, (30, 30, 30, 30), -1),
    (dvo.GN, dvo.W_REF_CAUCHY, dvo.RES_DT_INTERP, (8, 8, 8, 8), -1),
    (dvo.GN, dvo.W_REF_CAUCHY, dvo.RES_DT_FLOOR, (10, 10, 10, 10), 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("solver,weight,residual,iters,level", CASES)
def test_covariance_matches_oracle_320x240(small_batch, solver, weight, residual, iters, level):
    al, d, n = small_batch
    prm = dvo.solver_params(solver=solver, weight=weight, residual=residual, iters=iters)
    al.set_initial_pose(n, None)
    al.run(n, prm)
    poses, _ = al.get_poses(n)
    cov, info = al.pose_covariance(n, prm, level=level)
    lv = 0 if level < 0 else level
    for i in (0, 3, 7):
        R, T = poses[i, :9].reshape(3, 3), poses[i, 9:]
        H, s2, nvis = oracle_cov(d["ref_gray"][i], d["ref_depth"][i], d["now_gray"][i], lv, R, T, K320, weight, residual=residual)
        check_against_oracle(cov[i], info[i], H, s2, nvis, lv)


NFULL = 160            # > 148 SMs: the 256-thread solver shape of the 1024-pair benchmark


@pytest.fixture(scope="module")
def full_load():
    d = O.synth_batch(5000, NFULL)
    al = dvo.BatchAligner(640, 480, 4, max_batch=NFULL)
    al.set_frames(dvo.FRAME_REF, d["ref_gray"], d["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, d["now_gray"], None)
    al.build_pyramids(NFULL)
    al.prepare(NFULL)
    yield al, d
    al.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver,weight,iters", [(dvo.GN, dvo.W_REF_CAUCHY, (10, 10, 10, 10)), (dvo.GN, dvo.W_HUBER, (10, 10, 10, 10)),
                                                 (dvo.SUBGRAD_REF, dvo.W_REF_CAUCHY, (50, 50, 50, 50))])
def test_covariance_matches_oracle_full_load_640x480(full_load, solver, weight, iters):
    al, d = full_load
    prm = dvo.solver_params(solver=solver, weight=weight, iters=iters)
    al.set_initial_pose(NFULL, None)
    al.run(NFULL, prm)
    poses, _ = al.get_poses(NFULL)
    cov, info = al.pose_covariance(NFULL, prm)
    assert all(info[i].status == 0 for i in range(NFULL))
    for i in (0, 80, 159):
        R, T = poses[i, :9].reshape(3, 3), poses[i, 9:]
        H, s2, nvis = oracle_cov(d["ref_gray"][i], d["ref_depth"][i], d["now_gray"][i], 0, R, T, O.K640, weight)
        check_against_oracle(cov[i], info[i], H, s2, nvis, 0)


@pytest.mark.gpu
def test_covariance_does_not_depend_on_launch_size_and_device_equals_host(full_load):
    import torch
    al, d = full_load
    prm = dvo.solver_params(solver=dvo.GN, iters=(10, 10, 10, 10))
    al.set_initial_pose(NFULL, None)
    al.run(NFULL, prm)
    want, winfo = al.pose_covariance(NFULL, prm)
    got5, _ = al.pose_covariance(5, prm, first=33)
    assert np.array_equal(got5, want[33:38])
    got1, _ = al.pose_covariance(1, prm, first=159)
    assert np.array_equal(got1, want[159:160])
    dcov = torch.empty((NFULL, 36), dtype=torch.float64, device="cuda")
    dinfo = torch.empty((NFULL * C.sizeof(dvo.CovInfo),), dtype=torch.uint8, device="cuda")
    al.pose_covariance_device(NFULL, prm, dcov.data_ptr(), info_ptr=dinfo.data_ptr())
    al.synchronize()
    assert np.array_equal(dcov.cpu().numpy().view(np.uint64), want.reshape(NFULL, 36).view(np.uint64))
    ginfo = (dvo.CovInfo * NFULL).from_buffer_copy(dinfo.cpu().numpy().tobytes())
    for g, w in zip(ginfo, winfo):                                    # field by field: the struct's padding is not written
        assert (g.status, g.level, g.nvis) == (w.status, w.level, w.nvis)
        assert np.array_equal(np.array([g.sigma2, g.logdet]).view(np.uint64), np.array([w.sigma2, w.logdet]).view(np.uint64))
    al.pose_covariance_device(NFULL, prm, dcov.data_ptr())            # info may be NULL
    al.synchronize()
    assert np.array_equal(dcov.cpu().numpy().view(np.uint64), want.reshape(NFULL, 36).view(np.uint64))


@pytest.mark.gpu
def test_covariance_has_no_side_effects(small_batch):
    al, d, n = small_batch
    prm = dvo.solver_params(solver=dvo.GN, iters=(10, 10, 10, 10))
    al.set_initial_pose(n, None)
    al.run(n, prm)
    p0, i0 = al.get_poses(n)
    al.pose_covariance(n, prm)
    p1, i1 = al.get_poses(n)
    assert np.array_equal(p0.view(np.uint64), p1.view(np.uint64)) and bytes(i0) == bytes(i1)
    al.run(n, prm)                                                   # a later solve is unaffected too
    p2, i2 = al.get_poses(n)
    assert np.array_equal(p0.view(np.uint64), p2.view(np.uint64)) and bytes(i0) == bytes(i2)


@pytest.mark.gpu
def test_degenerate_slots_give_nan_and_status(small_batch):
    """slot 1: blank now frame (no now edges) -> bit0; slot 3: pose moved so that no point reprojects -> bit1.  The good slots of the
    same launch equal their covariance computed alone."""
    _, d, _ = small_batch
    W, H, L, n = 320, 240, 4, 4
    now = d["now_gray"][:n].copy()
    now[1] = 0
    al = dvo.BatchAligner(W, H, L, max_batch=n, intrinsics=K320)
    al.set_frames(dvo.FRAME_REF, d["ref_gray"][:n], d["ref_depth"][:n])
    al.set_frames(dvo.FRAME_NOW, now, None)
    al.build_pyramids(n); al.prepare(n)
    prm = dvo.solver_params(solver=dvo.GN, iters=(10, 10, 10, 10))
    al.set_initial_pose(n, None)
    al.run(n, prm)
    far = np.concatenate([np.eye(3).reshape(9), [50.0, 0.0, 0.0]])
    al.set_initial_pose(1, far, first=3)
    al.run(1, dvo.solver_params(solver=dvo.GN, iters=(0, 0, 0, 0)), first=3)   # no iterations: the pose stays where it was put
    cov, info = al.pose_covariance(n, prm)
    assert info[1].status == 1 and info[3].status == 2 and info[3].nvis < 7
    for i in (1, 3):
        assert np.isnan(cov[i]).all() and np.isnan(info[i].sigma2) and np.isnan(info[i].logdet)
    for i in (0, 2):
        assert info[i].status == 0 and np.isfinite(cov[i]).all()
        alone, ainfo = al.pose_covariance(1, prm, first=i)
        assert np.array_equal(alone[0], cov[i]) and ainfo[0].sigma2 == info[i].sigma2
    al.close()


def reference_of(kind_s, t):
    return max(k for k in range(t) if kind_s[k] != 0)


def check_sequence(al, gray, depth, nseq, nframes, prm, pol, K, L, frames):
    want = al.run_sequences_mem(gray, depth, nseq, nframes, prm, pol)
    rel, kind, reason, glob, rel_cov, glob_cov = al.run_sequences_cov(gray, depth, nseq, nframes, prm, pol)
    for a, b in zip(want, (rel, kind, reason, glob)):
        assert np.array_equal(a, b)
    assert not rel_cov[:, 0].any()
    finest = [l for l in range(L) if prm.iters[l] > 0][0]
    for s in range(nseq):
        for t in frames:
            r = reference_of(kind[s], t)
            R, T = rel[s, t, :9].reshape(3, 3), rel[s, t, 9:]
            H, s2, nvis = oracle_cov(gray[s, r], depth[s, r], gray[s, t], finest, R, T, K, dvo.W_REF_CAUCHY)
            cov = rel_cov[s, t]
            assert np.abs(cov @ H / s2 - np.eye(6)).max() < 1e-6, (s, t, r)
    prop = propagate(rel, kind, rel_cov)
    assert np.all(np.abs(glob_cov - prop) <= 1e-12 * np.abs(prop).max(axis=(2, 3), keepdims=True))
    return kind


@pytest.mark.gpu
def test_sequence_covariances_320x240():
    W, H, L, K = 320, 240, 3, K320
    nseq, nframes = 4, 8
    seqs = [O.synth_sequence(90 + s, nframes, W, H, K, max_angle_deg=0.4, max_trans_m=0.008) for s in range(nseq)]
    gray = np.stack([s[0] for s in seqs]); depth = np.stack([s[1] for s in seqs])
    prm = dvo.solver_params(iters=(8, 8, 8))
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K)
    kind = check_sequence(al, gray, depth, nseq, nframes, prm, dvo.keyframe_policy(keyframe_every=3), K, L, (1, 3, 4, 7))
    assert list(np.nonzero(kind[0] == 2)[0]) == [2, 4, 6]            # frames 3, 5, 7 were re-solved after a switch
    gated = dvo.keyframe_policy(keyframe_every=0, use_quality_gates=True, laplacian_thresh=9.5, visible_ratio_thresh=0.95)
    check_sequence(al, gray, depth, nseq, nframes, prm, gated, K, L, (1, 2, 5, 7))
    al.close()


@pytest.mark.gpu
def test_sequence_covariances_1280x720_5_levels():
    W, H, L, K = 1280, 720, 5, O.K1280
    nseq, nframes = 2, 7
    seqs = [O.synth_sequence(170 + s, nframes, W, H, K, max_angle_deg=0.4, max_trans_m=0.008) for s in range(nseq)]
    gray = np.stack([s[0] for s in seqs]); depth = np.stack([s[1] for s in seqs])
    prm = dvo.solver_params(iters=(50, 50, 50, 50, 50))
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K)
    kind = check_sequence(al, gray, depth, nseq, nframes, prm, dvo.keyframe_policy(), K, L, (1, 5, 6))
    assert list(np.nonzero(kind[0] == 2)[0]) == [4]                  # frame 5 was re-solved after a switch
    al.close()


@pytest.mark.gpu
def test_pose_covariance_rejects_bad_arguments(small_batch):
    al, _, n = small_batch
    prm = dvo.solver_params(solver=dvo.GN, iters=(10, 10, 10, 10))
    with pytest.raises(dvo.DvoError):
        al.pose_covariance(n + 1, prm)
    with pytest.raises(dvo.DvoError):
        al.pose_covariance(n, prm, level=4)
    with pytest.raises(dvo.DvoError, match="no level has iterations"):
        al.pose_covariance(n, dvo.solver_params(iters=(0, 0, 0, 0)))
