"""dvo_align_pairs: any (reference, now) pair of frames prepared in one context, addressed by slot index.

Every check is bit for bit against the per-slot path: a context whose slot holds pair (i, j) as its reference / now frames,
run through dvo_build_pyramids + dvo_prepare + dvo_run + dvo_pose_covariance with the same thread shape per pair.
"""
import numpy as np
import pytest

import oracle_lib as O
import rgbd_odometry_b200 as dvo

W, H, L = 640, 480, 4


def window_pairs(n, k):
    """(i, j) for 1 <= |i - j| <= k, both directions."""
    return [(i, j) for i in range(n) for j in range(n) if i != j and abs(i - j) <= k]


def same(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


def same_cov_info(a, b):
    return all((x.status, x.level, x.nvis) == (y.status, y.level, y.nvis) and same([x.sigma2, x.logdet], [y.sigma2, y.logdet])
               for x, y in zip(a, b))


def per_slot(gray, depth, pairs, prm, max_batch, pose0=None):
    """poses, info bytes, cov, cov_info of every pair through the per-slot path, max_batch pairs per pass."""
    al = dvo.BatchAligner(W, H, L, max_batch=max_batch)
    poses, info, cov, cinfo = [], b"", [], []
    for s in range(0, len(pairs), max_batch):
        chunk = pairs[s:s + max_batch]
        n = len(chunk)
        ri = [i for i, _ in chunk]; ni = [j for _, j in chunk]
        al.set_frames(dvo.FRAME_REF, gray[ri], depth[ri])
        al.set_frames(dvo.FRAME_NOW, gray[ni], None)
        al.build_pyramids(n); al.prepare(n)
        al.set_initial_pose(n, None if pose0 is None else pose0[s:s + n])
        al.run(n, prm)
        p, i = al.get_poses(n)
        c, ci = al.pose_covariance(n, prm)
        poses.append(p); info += bytes(i); cov.append(c); cinfo += list(ci)
    al.close()
    return np.concatenate(poses), info, np.concatenate(cov), cinfo


def check_pairs_against_slots(al, gray, depth, pairs, prm, max_batch):
    ri = [i for i, _ in pairs]; ni = [j for _, j in pairs]
    poses, info, cov, cinfo = al.align_pairs(ri, ni, prm, covariance=True)
    wp, wi, wc, wci = per_slot(gray, depth, pairs, prm, max_batch)
    assert all(r.status == 0 for r in info)
    assert same(poses, wp)
    assert bytes(info) == wi
    assert same(cov, wc)
    assert same_cov_info(cinfo, wci)
    return poses, info, cov, cinfo


# ------------------------------------------------------------------------------------------------ shape 512 (max_batch <= SM count)
NF = 12
PAIRS12 = window_pairs(NF, 2)          # 42 pairs


@pytest.fixture(scope="module")
def frames12():
    gray, depth, _, _ = O.synth_sequence(7100, NF, W, H)
    al = dvo.BatchAligner(W, H, L, max_batch=NF)
    al.load_frames(gray, depth)
    yield al, gray, depth
    al.close()


CASES512 = {
    "subgrad_shipped": dict(),
    "gn_exact_huber": dict(solver=dvo.GN, jacobian=dvo.JAC_EXACT, weight=dvo.W_HUBER, iters=(10, 10, 10, 10)),
    "lm_exact_huber": dict(solver=dvo.LM, jacobian=dvo.JAC_EXACT, weight=dvo.W_HUBER, iters=(10, 10, 10, 10)),
    "gn_dt_interp": dict(solver=dvo.GN, residual=dvo.RES_DT_INTERP, iters=(10, 10, 10, 10)),
    "gn_fast": dict(solver=dvo.GN, arithmetic=dvo.ARITH_FAST, iters=(10, 10, 10, 10)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES512))
def test_pairs_equal_per_slot_path_512(frames12, case):
    al, gray, depth = frames12
    check_pairs_against_slots(al, gray, depth, PAIRS12, dvo.solver_params(**CASES512[case]), len(PAIRS12))


# ------------------------------------------------------------------------------------------------ shape 256 (max_batch > SM count)
NF256 = 160
PAIRS160 = window_pairs(NF256, 2)      # 634 pairs > max_batch


@pytest.fixture(scope="module")
def frames160():
    gray, depth, _, _ = O.synth_sequence(7200, NF256, W, H)
    al = dvo.BatchAligner(W, H, L, max_batch=NF256)
    al.load_frames(gray, depth)
    yield al, gray, depth
    al.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(solver=dvo.GN, iters=(10, 10, 10, 10)), dict()], ids=["gn", "subgrad_shipped"])
def test_pairs_equal_per_slot_path_256(frames160, kw):
    al, gray, depth = frames160
    check_pairs_against_slots(al, gray, depth, PAIRS160, dvo.solver_params(**kw), 200)


# ------------------------------------------------------------------------------------------------ order, memory modes, pose0
GN10 = dict(solver=dvo.GN, iters=(10, 10, 10, 10))


@pytest.mark.gpu
def test_result_depends_neither_on_npairs_nor_position(frames12):
    al, _, _ = frames12
    prm = dvo.solver_params(**GN10)
    ri = np.array([i for i, _ in PAIRS12]); ni = np.array([j for _, j in PAIRS12])
    p, i, c, ci = al.align_pairs(ri, ni, prm, covariance=True)
    perm = np.random.default_rng(3).permutation(len(ri))
    pp, ip, cp, cip = al.align_pairs(ri[perm], ni[perm], prm, covariance=True)
    assert same(pp, p[perm]) and same(cp, c[perm])
    assert all(bytes(ip[k]) == bytes(i[perm[k]]) for k in range(len(ri)))
    assert same_cov_info(cip, [ci[q] for q in perm])
    for k in (0, 17, 41):
        p1, i1, c1, ci1 = al.align_pairs(ri[k:k + 1], ni[k:k + 1], prm, covariance=True)
        assert same(p1[0], p[k]) and bytes(i1[0]) == bytes(i[k]) and same(c1[0], c[k]) and same_cov_info(ci1, [ci[k]])


@pytest.fixture(scope="module")
def regular():
    """a context whose slots hold distinct reference / now frames, solved by dvo_run"""
    n = 8
    d = O.synth_batch(7300, n, W, H)
    al = dvo.BatchAligner(W, H, L, max_batch=n)
    al.set_frames(dvo.FRAME_REF, d["ref_gray"], d["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, d["now_gray"], None)
    al.build_pyramids(n); al.prepare(n)
    yield al, n
    al.close()


def pose0_of(n, seed):
    rng = np.random.default_rng(seed)
    out = np.empty((n, 12))
    for k in range(n):
        R, T = O.se3_exp(np.concatenate([rng.normal(0, 0.005, 3), rng.normal(0, 0.004, 3)]))
        out[k, :9], out[k, 9:] = np.asarray(R).reshape(9), T
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("with_pose0", [False, True])
def test_diagonal_pairs_equal_dvo_run_host_and_device(regular, with_pose0):
    import torch
    al, n = regular
    prm = dvo.solver_params(**GN10)
    P0 = pose0_of(n, 5) if with_pose0 else None
    al.set_initial_pose(n, P0)
    al.run(n, prm)
    wp, wi = al.get_poses(n)
    wc, wci = al.pose_covariance(n, prm)
    s = np.arange(n)
    p, i, c, ci = al.align_pairs(s, s, prm, pose0=P0, covariance=True)
    assert same(p, wp) and bytes(i) == bytes(wi) and same(c, wc) and same_cov_info(ci, wci)
    ts = torch.arange(n, dtype=torch.int32, device="cuda")
    tp0 = None if P0 is None else torch.from_numpy(P0).cuda()
    dp, di, dc, dci = al.align_pairs(ts, ts, prm, pose0=tp0, covariance=True, device=True)
    al.synchronize()
    assert same(dp.cpu().numpy(), wp) and bytes(dvo.records(di, dvo.PairInfo)) == bytes(wi)
    assert same(dc.cpu().numpy(), wc) and same_cov_info(dvo.records(dci, dvo.CovInfo), wci)
    if with_pose0:                                           # the initial pose matters: identity gives other poses
        ip, _ = al.align_pairs(s, s, prm)
        assert not same(ip, p)


@pytest.mark.gpu
def test_align_pairs_has_no_side_effects_on_slots(regular):
    al, n = regular
    prm = dvo.solver_params(**GN10)
    al.set_initial_pose(n, None)
    al.run(n, prm)
    p0, i0 = al.get_poses(n)
    e0 = [al.get_energies(s, l) for s in range(n) for l in range(L)]
    c0, ci0 = al.pose_covariance(n, prm)
    al.align_pairs([3, 0, 5, 7, 7], [1, 6, 5, 2, 0], dvo.solver_params(iters=(30, 30, 30, 30)), pose0=pose0_of(5, 9), covariance=True)
    p1, i1 = al.get_poses(n)
    e1 = [al.get_energies(s, l) for s in range(n) for l in range(L)]
    c1, ci1 = al.pose_covariance(n, prm)
    assert same(p0, p1) and bytes(i0) == bytes(i1)
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(e0, e1))
    assert same(c0, c1) and same_cov_info(ci0, ci1)


# ------------------------------------------------------------------------------------------------ errors
@pytest.mark.gpu
def test_host_indices_out_of_range_are_rejected(frames12):
    al, _, _ = frames12
    prm = dvo.solver_params(**GN10)
    for ri, ni in (([0, NF], [1, 2]), ([0, 1], [-1, 2]), ([-5], [0])):
        with pytest.raises(dvo.DvoError, match=r"\(-1\)"):
            al.align_pairs(ri, ni, prm)


@pytest.mark.gpu
def test_device_indices_out_of_range_give_status_bit1_and_nan(frames12):
    import torch
    al, _, _ = frames12
    prm = dvo.solver_params(**GN10)
    ri = [0, -1, 3, 2, 5]; ni = [1, 2, NF, 3, 65536]
    dp, di, dc, dci = al.align_pairs(torch.tensor(ri, dtype=torch.int32, device="cuda"), torch.tensor(ni, dtype=torch.int32, device="cuda"),
                                     prm, covariance=True, device=True)
    al.synchronize()
    p, c = dp.cpu().numpy(), dc.cpu().numpy()
    info, cinfo = dvo.records(di, dvo.PairInfo), dvo.records(dci, dvo.CovInfo)
    for k in (1, 2, 4):
        assert info[k].status == 2 and np.isnan(p[k]).all() and list(info[k].npts) == [0] * 6
        assert cinfo[k].status == 1 and np.isnan(c[k]).all() and np.isnan(cinfo[k].sigma2)
    wp, wi, wc, wci = al.align_pairs([0, 2], [1, 3], prm, covariance=True)
    assert same(p[[0, 3]], wp) and bytes(info[0]) + bytes(info[3]) == bytes(wi)
    assert same(c[[0, 3]], wc) and same_cov_info([cinfo[0], cinfo[3]], wci)


@pytest.mark.gpu
def test_unprepared_slot_gives_status_bit0(frames12):
    _, gray, depth = frames12
    al = dvo.BatchAligner(W, H, L, max_batch=4)
    al.load_frames(gray[:2], depth[:2])
    prm = dvo.solver_params(**GN10)
    p, info, c, cinfo = al.align_pairs([0, 3, 1], [3, 0, 0], prm, covariance=True)
    assert info[0].status == 1 and info[1].status == 1 and info[2].status == 0
    assert same(p[:2], np.tile(np.concatenate([np.eye(3).reshape(9), np.zeros(3)]), (2, 1)))
    assert cinfo[0].status == 1 and cinfo[1].status == 1 and np.isnan(c[:2]).all() and cinfo[2].status == 0
    al.close()
