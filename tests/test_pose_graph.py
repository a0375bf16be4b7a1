"""Windowed pose-graph optimisation (dvo_pose_graph_optimize): the CPU oracle (LM over a sequential banded Cholesky) against
scipy / numpy on small graphs, and the device (one CTA per graph, block cyclic reduction) against the oracle, against the
covariance convention of dvo_run_sequences_cov, for bit-reproducibility and for its error reporting."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_lib as O
import pgo_oracle_lib as PG
import rgbd_odometry_b200 as dvo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRM = dict(max_iterations=100, lambda0=1e-4, rel_tol=1e-10)


# ---------------------------------------------------------------- graph construction
def compose(A, B):
    R = A[:9].reshape(3, 3) @ B[:9].reshape(3, 3)
    return np.concatenate([R.reshape(9), A[9:] + A[:9].reshape(3, 3) @ B[9:]])


def inverse(A):
    Rt = A[:9].reshape(3, 3).T
    return np.concatenate([Rt.reshape(9), -Rt @ A[9:]])


def exp12(psi):
    R, t = O.se3_exp(np.asarray(psi, np.float64))
    return np.concatenate([np.asarray(R).reshape(9), np.asarray(t).reshape(3)])


def random_spd(rng, sigma):
    A = rng.normal(size=(6, 6))
    S = A @ A.T / 6 + 0.2 * np.eye(6)
    d = np.diag(sigma)
    return d @ S @ d


def edge_list(N, lag, backward=True):
    """every (t - j, t), and with backward every (t, t - j) of lag j <= 2 plus a duplicate of each lag-1 edge"""
    e = [(t - j, t) for j in range(1, lag + 1) for t in range(j, N)]
    if backward:
        e += [(t, t - j) for j in range(1, min(lag, 2) + 1) for t in range(j, N)]
        e += [(t - 1, t) for t in range(1, N)]
    return e


def make_graphs(seed, G, N, lag, noise=3e-3, init=2e-2, nan_edges=0.05, backward=True):
    """G graphs over the same edge list: seeded random-walk ground truth, measurements perturbed by noise drawn from each edge's
    random SPD covariance, a perturbed initial guess (node 0 exact), and a fraction of NaN covariances off the lag-1 chain."""
    rng = np.random.default_rng(seed)
    edges = edge_list(N, lag, backward)
    E = len(edges)
    ref = np.array([[a for a, _ in edges]] * G, np.int32)
    now = np.array([[b for _, b in edges]] * G, np.int32)
    meas = np.empty((G, E, 12)); cov = np.empty((G, E, 6, 6)); gt = np.empty((G, N, 12)); x0 = np.empty((G, N, 12))
    sig = np.array([noise] * 3 + [noise / 2] * 3)
    for g in range(G):
        gt[g, 0] = exp12(rng.normal(0, 0.3, 6))
        for i in range(1, N):
            gt[g, i] = compose(gt[g, i - 1], exp12(np.concatenate([rng.normal(0, 0.05, 3), rng.normal(0, 0.03, 3)])))
        for e, (a, b) in enumerate(edges):
            S = random_spd(rng, sig)
            n = np.linalg.cholesky(S) @ rng.normal(size=6)
            meas[g, e] = compose(compose(inverse(gt[g, a]), gt[g, b]), exp12(n))
            cov[g, e] = S
            if abs(a - b) > 1 and rng.random() < nan_edges:
                cov[g, e, rng.integers(6), rng.integers(6)] = np.nan
        x0[g, 0] = gt[g, 0]
        for i in range(1, N):
            x0[g, i] = compose(gt[g, i], exp12(rng.normal(0, init, 6)))
    return ref, now, meas, cov, x0, gt


def pose_err(A, B):
    """max rotation angle (rad) and translation distance (m) between two stacks of 12-double poses"""
    A = A.reshape(-1, 12); B = B.reshape(-1, 12)
    ang = [np.linalg.norm(O.se3_log(a[:9].reshape(3, 3).T @ b[:9].reshape(3, 3), np.zeros(3))[3:]) for a, b in zip(A, B)]
    return max(ang), np.abs(A[:, 9:] - B[:, 9:]).max()


# ---------------------------------------------------------------- CPU: interface and oracle
def test_struct_layouts_match_header():
    assert C.sizeof(dvo.PgoParams) == 24 and dvo.PgoParams.lambda0.offset == 8 and dvo.PgoParams.rel_tol.offset == 16
    assert C.sizeof(dvo.PgoInfo) == 32 and dvo.PgoInfo.edges_used.offset == 12 and dvo.PgoInfo.cost_initial.offset == 16
    assert dvo.PgoInfo.cost_final.offset == 24
    hdr = open(os.path.join(ROOT, "include", "dvo_b200.h")).read()
    assert int(re.search(r"#define DVO_PGO_MAX_LAG (\d+)", hdr).group(1)) == dvo.PGO_MAX_LAG == 8
    body = re.search(r"typedef struct dvo_pgo_info \{(.*?)\} dvo_pgo_info;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    assert re.findall(r"\b(status|iterations|accepted|edges_used|cost_initial|cost_final)\b", body) == [f for f, _ in dvo.PgoInfo._fields_]


def whitened(ref, now, meas, cov, x0):
    """residual function of the tangent offsets xi (node i >= 1: G_i = x0_i exp(xi_i)), whitened by chol(Omega)"""
    N = x0.shape[0]
    Ls = []
    for S in cov:
        Om = np.linalg.inv(S)
        Ls.append(np.linalg.cholesky(Om).T)                      # r^T Omega r = |L^T r|^2

    def fun(xi):
        X = x0.copy()
        for i in range(1, N):
            X[i] = compose(x0[i], exp12(xi[6 * (i - 1):6 * i]))
        r = PG.pgo_system(ref, now, meas, cov, X, 8)["r"]
        return np.concatenate([L @ ri for L, ri in zip(Ls, r)])
    return fun


@pytest.mark.parametrize("N,lag,seed", [(2, 1, 1), (5, 2, 2), (7, 4, 3), (12, 3, 4), (12, 8, 5)])
def test_oracle_reaches_the_least_squares_minimum(N, lag, seed):
    """Noise 1e-3 keeps the first-order inverse Jacobian's offset of the fixed point (|r|^3 / 12) far below 1e-8."""
    from scipy.optimize import least_squares
    ref, now, meas, cov, x0, _ = make_graphs(seed, 1, N, lag, noise=1e-3, nan_edges=0.0)
    X, info, _ = PG.pose_graph(ref, now, meas, cov, x0, lag, **PRM)
    assert info["status"][0] == 0 and info["cost_final"][0] <= info["cost_initial"][0]
    fun = whitened(ref[0], now[0], meas[0], cov[0], x0[0])
    sol = least_squares(fun, np.zeros(6 * (N - 1)), method="lm", jac="3-point", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    Xs = x0[0].copy()
    for i in range(1, N):
        Xs[i] = compose(x0[0][i], exp12(sol.x[6 * (i - 1):6 * i]))
    ang, tr = pose_err(X[0], Xs)
    assert ang < 1e-8 and tr < 1e-8, (ang, tr)
    assert abs(info["cost_final"][0] - 0.5 * np.sum(sol.fun ** 2)) <= 1e-8 * info["cost_final"][0]


@pytest.mark.parametrize("N,lag,lam", [(5, 1, 0.0), (9, 2, 1e-3), (12, 4, 1.0), (12, 8, 1e-4)])
def test_oracle_linear_step_matches_dense_solve(N, lag, lam):
    ref, now, meas, cov, x0, _ = make_graphs(10 + N, 1, N, lag)
    s = PG.pgo_system(ref[0], now[0], meas[0], cov[0], x0[0], lag, lam)
    H = s["H"]
    assert np.allclose(H, H.T, rtol=0, atol=1e-12 * np.abs(H).max())
    Hd = H + lam * np.diag(np.diag(H))
    want = np.linalg.solve(Hd, -s["g"])
    assert np.abs(s["delta"] - want).max() <= 1e-10 * np.abs(want).max()
    valid = s["valid"]
    assert valid.sum() < len(valid) or lag <= 2 or N < 5          # the generator's NaN covariances drop out
    Om = [np.linalg.inv(S) for S in cov[0]]
    F = sum(0.5 * r @ W @ r for r, W, v in zip(s["r"], Om, valid) if v)
    assert abs(s["F"] - F) <= 1e-12 * F


@pytest.mark.parametrize("N,lag", [(6, 2), (11, 4), (12, 8)])
def test_oracle_marginals_are_inverse_hessian_blocks(N, lag):
    ref, now, meas, cov, x0, _ = make_graphs(20 + N, 1, N, lag)
    X, info, nc = PG.pose_graph(ref, now, meas, cov, x0, lag, marginals=True, **PRM)
    assert info["status"][0] == 0
    Hi = np.linalg.inv(PG.pgo_system(ref[0], now[0], meas[0], cov[0], X[0], lag)["H"])
    assert not nc[0, 0].any()
    for i in range(1, N):
        blk = Hi[6 * (i - 1):6 * i, 6 * (i - 1):6 * i]
        assert np.abs(nc[0, i] - blk).max() <= 1e-10 * np.abs(blk).max()


def test_oracle_reports_bad_and_disconnected_graphs():
    ref, now, meas, cov, x0, _ = make_graphs(30, 3, 6, 2, nan_edges=0.0)
    ref[0, 0] = 9                                                  # out of range
    cov[1, :, 0, 0] = np.nan                                       # no usable edge
    X, info, nc = PG.pose_graph(ref, now, meas, cov, x0, 2, marginals=True, **PRM)
    assert list(info["status"]) == [1, 2, 0]
    assert np.array_equal(X[:2], x0[:2]) and np.isnan(nc[:2]).all() and not np.isnan(nc[2]).any()


# ---------------------------------------------------------------- GPU
def device_run(al, ref, now, meas, cov, x0, lag, marginals=True, device=False, **kw):
    p = dict(PRM); p.update(kw)
    if not device:
        return al.optimize_pose_graph(ref, now, meas, cov, x0, lag, marginals=marginals, **p)
    import torch
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dt)  # noqa: E731
    r = al.optimize_pose_graph(t(ref, torch.int32), t(now, torch.int32), t(meas, torch.float64), t(cov, torch.float64),
                               t(x0, torch.float64), lag, marginals=marginals, device=True, **p)
    al.synchronize()
    out = [r[0].cpu().numpy(), dvo.records(r[1], dvo.PgoInfo)]
    if marginals:
        out.append(r[2].cpu().numpy())
    return tuple(out)


def info_tuple(I):
    return (I.status, I.iterations, I.accepted, I.edges_used, I.cost_initial, I.cost_final)


def check_against_oracle(poses, info, nc, ref, now, meas, cov, x0, lag):
    X, oi, onc = PG.pose_graph(ref, now, meas, cov, x0, lag, marginals=nc is not None, **PRM)
    for g in range(ref.shape[0]):
        assert info[g].status == oi["status"][g] == 0
        assert info[g].edges_used == oi["edges_used"][g]
        assert abs(info[g].cost_initial - oi["cost_initial"][g]) <= 1e-12 * oi["cost_initial"][g]
        assert abs(info[g].cost_final - oi["cost_final"][g]) <= 1e-9 * oi["cost_final"][g], (info[g].cost_final, oi["cost_final"][g])
        assert info[g].cost_final <= info[g].cost_initial
        ang, tr = pose_err(poses[g], X[g])
        assert ang < 1e-9 and tr < 1e-9, (g, ang, tr, info_tuple(info[g]), oi["iterations"][g])
        assert np.array_equal(poses[g, 0], x0[g, 0])
        if nc is not None:
            assert not nc[g, 0].any()
            scale = np.abs(onc[g]).max(axis=(1, 2))
            assert (np.abs(nc[g] - onc[g]).max(axis=(1, 2)) <= 1e-8 * np.maximum(scale, 1e-300)).all()


CASES = [(2, 1), (2, 8), (5, 2), (5, 4), (7, 4), (7, 8), (64, 1), (64, 2), (64, 8), (1024, 4), (1024, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,lag", CASES)
def test_device_matches_oracle(N, lag):
    G = 3 if N < 1024 else 1
    ref, now, meas, cov, x0, _ = make_graphs(100 + N + lag, G, N, lag)
    al = dvo.BatchAligner(64, 64, 1, max_batch=1)
    poses, info, nc = device_run(al, ref, now, meas, cov, x0, lag)
    al.close()
    check_against_oracle(poses, info, nc, ref, now, meas, cov, x0, lag)


def last_key_before(kind_s, t):
    return max(k for k in range(t) if kind_s[k] != 0)


@pytest.mark.gpu
def test_tree_graph_reproduces_the_key_frame_chain():
    """rel_poses / rel_cov of dvo_run_sequences_cov as edges (key frame k -> t): a tree, so the optimum satisfies every edge
    exactly; the poses are global_poses and the marginals global_cov (first-order propagation along the chain)."""
    W, H, L, K = 320, 240, 3, (262.5, 262.5, 159.5, 119.5)
    nseq, F = 2, 16
    seqs = [O.synth_sequence(500 + s, F, W, H, K, max_angle_deg=0.4, max_trans_m=0.008) for s in range(nseq)]
    gray = np.stack([s[0] for s in seqs]); depth = np.stack([s[1] for s in seqs])
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K)
    prm = dvo.solver_params(solver=dvo.GN, iters=(10, 10, 10))
    rel, kind, _, glob, rel_cov, glob_cov = al.run_sequences_cov(gray, depth, nseq, F, prm, dvo.keyframe_policy(keyframe_every=5))
    ref = np.array([[last_key_before(kind[s], t) for t in range(1, F)] for s in range(nseq)], np.int32)
    now = np.array([list(range(1, F))] * nseq, np.int32)
    assert (now - ref).max() <= 5
    meas = rel[:, 1:]; cov = rel_cov[:, 1:]
    rng = np.random.default_rng(7)
    x0 = glob[:, :, :12].copy()
    for s in range(nseq):
        for t in range(1, F):
            x0[s, t] = compose(x0[s, t], exp12(rng.normal(0, 0.01, 6)))
    poses, info, nc = al.optimize_pose_graph(ref, now, meas, cov, x0, 5, marginals=True, **PRM)
    al.close()
    for s in range(nseq):
        assert info[s].status == 0 and info[s].edges_used == F - 1
        ang, tr = pose_err(poses[s], glob[s, :, :12])
        assert ang < 1e-12 and tr < 1e-12, (ang, tr)
        scale = np.abs(glob_cov[s]).max(axis=(1, 2))
        assert not nc[s, 0].any() and not glob_cov[s, 0].any()
        assert (np.abs(nc[s, 1:] - glob_cov[s, 1:]).max(axis=(1, 2)) <= 1e-9 * scale[1:]).all()


def same(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


@pytest.mark.gpu
def test_graph_results_do_not_depend_on_batch_memory_or_run():
    ref, now, meas, cov, x0, _ = make_graphs(300, 300, 24, 3)
    al = dvo.BatchAligner(64, 64, 1, max_batch=1)
    P, I, NC = device_run(al, ref, now, meas, cov, x0, 3)
    P2, I2, NC2 = device_run(al, ref, now, meas, cov, x0, 3)
    Pd, Id, NCd = device_run(al, ref, now, meas, cov, x0, 3, device=True)
    assert same(P, P2) and same(NC, NC2) and bytes(I) == bytes(I2)
    assert same(P, Pd) and same(NC, NCd) and bytes(I) == bytes(Id)
    assert all(i.status == 0 for i in I)
    for g in (0, 137, 299):
        p, i, nc = device_run(al, ref[g:g + 1], now[g:g + 1], meas[g:g + 1], cov[g:g + 1], x0[g:g + 1], 3)
        assert same(p[0], P[g]) and same(nc[0], NC[g]) and bytes(i[0]) == bytes(I[g])
        perm = [5, g, 9] if g not in (5, 9) else [g, 5, 9]           # the same graph at another position
        k = perm.index(g)
        p, i, nc = device_run(al, ref[perm], now[perm], meas[perm], cov[perm], x0[perm], 3, device=True)
        assert same(p[k], P[g]) and same(nc[k], NC[g]) and bytes(i[k]) == bytes(I[g])
    al.close()


@pytest.mark.gpu
def test_errors():
    ref, now, meas, cov, x0, _ = make_graphs(400, 4, 9, 2, nan_edges=0.0)
    al = dvo.BatchAligner(64, 64, 1, max_batch=1)
    for bad in ((9, 1), (-1, 0), (3, 3), (1, 4)):                  # out of range, negative, self, over the lag
        r = ref.copy(); n = now.copy()
        r[2, 5], n[2, 5] = bad
        with pytest.raises(dvo.DvoError, match="-1"):
            al.optimize_pose_graph(r, n, meas, cov, x0, 2)
        p, i, nc = device_run(al, r, n, meas, cov, x0, 2, device=True)
        assert i[2].status & 1 and same(p[2], x0[2]) and np.isnan(nc[2]).all()
        assert all(i[g].status == 0 for g in (0, 1, 3))
    c = cov.copy(); c[1, :, 2, 2] = np.nan                          # every covariance NaN
    r, n = ref.copy(), now.copy()
    c[3, (r[3] == 8) | (n[3] == 8)] = np.nan                        # graph 3: no usable edge reaches node 8
    p, i, nc = al.optimize_pose_graph(r, n, meas, c, x0, 2, marginals=True)
    assert i[1].status == 2 and i[1].edges_used == 0 and same(p[1], x0[1]) and np.isnan(nc[1]).all()
    assert i[3].status == 2 and same(p[3], x0[3])
    assert i[0].status == 0 and i[2].status == 0
    for args in ((ref, now, meas, cov, x0, 9), (ref[:, :0], now[:, :0], meas[:, :0], cov[:, :0], x0[:, :1], 2)):
        with pytest.raises(dvo.DvoError, match="-1"):
            al.optimize_pose_graph(*args)
    prm = dvo.PgoParams(10, 1e-4, 1e-10)
    lib = al.lib
    ref_ = np.ascontiguousarray(ref); now_ = np.ascontiguousarray(now)
    rc = lib.dvo_pose_graph_optimize(al.h, 4, 9, ref.shape[1], 2, ref_.ctypes.data, now_.ctypes.data, meas.ctypes.data, cov.ctypes.data,
                                     None, C.byref(prm), None, None, 0)
    assert rc == -1
    al.close()


@pytest.mark.gpu
def test_end_to_end_on_images():
    """align_pairs over a window of 4 in both directions with covariances, the lag-1 chain through gop_compose as the initial
    guess, then the optimiser.  The trajectory errors are printed, not asserted: whether smoothing reduces drift on this
    synthetic data is not established."""
    W, H, L, F, k = 640, 480, 4, 64, 4
    g, d, Rg, Tg = O.synth_sequence(9100, F, W, H, O.K640)
    al = dvo.BatchAligner(W, H, L, max_batch=F, intrinsics=O.K640)
    al.load_frames(g, d)
    pairs = [(t - j, t) for j in range(1, k + 1) for t in range(j, F)] + [(t, t - j) for j in range(1, k + 1) for t in range(j, F)]
    ri = np.array([a for a, _ in pairs], np.int32); ni = np.array([b for _, b in pairs], np.int32)
    prm = dvo.solver_params(solver=dvo.GN, iters=(10,) * L)
    poses, info, cov, cinfo = al.align_pairs(ri, ni, prm, covariance=True)
    rel = np.tile(np.eye(3).reshape(9).tolist() + [0, 0, 0], (1, F, 1)).astype(np.float64)
    for e, (a, b) in enumerate(pairs):
        if b == a + 1:
            rel[0, b] = poses[e]
    chain = al.gop_compose(np.ones((1, F), np.int32), rel)[:, :, :12]
    P, I, NC = al.optimize_pose_graph(ri[None], ni[None], poses[None], cov[None], chain, k, marginals=True)
    al.close()
    assert I[0].status == 0 and I[0].cost_final <= I[0].cost_initial
    assert I[0].edges_used == sum(c.status == 0 for c in cinfo)
    check_against_oracle(P, I, NC, ri[None], ni[None], poses[None], cov[None], chain, k)
    gt = np.stack([np.concatenate([Rg[i].reshape(9), Tg[i]]) for i in range(F)])
    gt = np.stack([compose(inverse(gt[0]), gt[i]) for i in range(F)])
    ate = lambda X: float(np.sqrt(np.mean(np.sum((X[:, 9:] - gt[:, 9:]) ** 2, axis=1))))  # noqa: E731
    print(f"\nATE (m, RMS translation) over {F} frames: lag-1 chain {ate(chain[0]):.6f}, optimised {ate(P[0]):.6f}; "
          f"{I[0].edges_used} edges, {I[0].iterations} iterations, cost {I[0].cost_initial:.3f} -> {I[0].cost_final:.3f}")
