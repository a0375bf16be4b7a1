"""Entropy-ratio key frames (dvo_run_sequences_entropy): the DVO-SLAM rule (Kerl, Sturm, Cremers, IROS 2013) as a gate of the
device-side key-frame policy.

CPU: the oracle's decision helper on hand-built log-determinants (sign handling, NaN covariances, h_ref >= 0, the
lastRef == t - 1 guard, the order of the reasons), so that the GPU tests rest on a checked oracle.
GPU: a disabled gate is dvo_run_sequences_cov exactly; an enabled gate matches a CPU loop driven by the oracle's solver and
covariance frame by frame; input memory kinds and launch subsets give identical records; a degenerate frame never fires it.
"""
import numpy as np
import pytest

import oracle_lib as O
import rgbd_odometry_b200 as dvo

K320 = (262.5, 262.5, 159.5, 119.5)
H0 = 3.0 * (1.0 + np.log(2.0 * np.pi))     # h(Sigma) = H0 + logdet(Sigma) / 2 for a 6-D Gaussian, nats


def entropy(logdet):
    return H0 + 0.5 * np.float64(logdet)


def keyframe_decision(t, last_ref, quality_reasons, logdet_t, logdet_ref, thr, every):
    """seq_gate_kernel's decision for one sequence at frame t: (switch, reason, alpha).  quality_reasons: the quality gates that
    fired, in the order 2, 3, 4; logdet_t: covariance of frame t's first solve; logdet_ref: final covariance of frame
    last_ref + 1.  Gates in the order quality, entropy, periodic; the last one that fires names the reason."""
    signal, why, alpha = False, 0, np.nan
    for r in quality_reasons:
        signal, why = True, r
    if last_ref != t - 1:
        h_ref = entropy(logdet_ref)
        with np.errstate(divide="ignore", invalid="ignore"):
            alpha = float(entropy(logdet_t) / h_ref)
        if np.isfinite(alpha) and h_ref < 0 and alpha < thr:
            signal, why = True, 6
    if every > 0 and t - last_ref == every:
        signal, why = True, 5
    if signal and last_ref != t - 1:
        return True, why, alpha
    return False, 0, alpha


def oracle_cov(ref_gray, ref_depth, now_gray, level, R, T, K, weight=O.W_REF_CAUCHY, huber_k=1.345, residual=O.RES_DT_FLOOR):
    """H, sigma2, nvis from the oracle's per-point EXACT-Jacobian outputs at (R, T) (as in test_pose_covariance)."""
    ref = O.preprocess_level(ref_gray, ref_depth, level)
    now = O.preprocess_level(now_gray, None, level)
    X, Y, Z, _, _ = O.select_points(ref["edge"], ref["depth"], level, K)
    o = O.evaluate(X, Y, Z, now["dtn"], now["gx"], now["gy"], level, R, T, K=K, jac=O.JAC_EXACT, weight=weight, huber_k=huber_k,
                   per_point=True, residual=residual)
    iu = np.triu_indices(6)
    H = np.zeros((6, 6)); H[iu] = o["H"][iu]; H = H + np.triu(H, 1).T
    s2 = float(np.sum(o["w"].astype(np.float64) * o["eps"].astype(np.float64) ** 2)) / (o["nvis"] - 6) if o["nvis"] > 6 else np.nan
    return H, s2, o["nvis"]


def oracle_logdet(ref_gray, ref_depth, now_gray, level, R, T, K):
    """log det Sigma as dvo_cov_info.logdet; NaN for a degenerate covariance."""
    H, s2, nvis = oracle_cov(ref_gray, ref_depth, now_gray, level, R, T, K)
    sign, ld = np.linalg.slogdet(H)
    if nvis < 7 or sign <= 0:
        return np.nan
    return 6.0 * np.log(s2) - ld


def oracle_sequence_entropy(gray, depth, levels, iters, K, thr, every=0, gates=False, b_thr=3.0, vis_thr=0.8, min_reproj=50):
    """SolveDVO::loop with the quality gates, the entropy gate and the periodic rule, driven by the CPU oracle.  Returns rel,
    kind, reason, glob, alpha and the quality statistics every decision saw."""
    n = gray.shape[0]
    rel = np.zeros((n, 12)); kind = np.zeros(n, np.int32); reason = np.zeros(n, np.int32); alpha = np.full(n, np.nan)
    rel[0, [0, 4, 8]] = 1.0; kind[0] = 1; reason[0] = 1
    ref = 0; last_ref = 0
    finest = [l for l in range(levels) if iters[l] > 0][0]
    final_logdet = np.full(n, np.nan)                   # of the frames that were first against their key frame
    R, T = np.eye(3), np.zeros(3)
    stats = []
    for t in range(1, n):
        o = O.align_pair(gray[ref], depth[ref], gray[t], levels, iters, K, R0=R, T0=T, stats=True)
        stats.append((o["b_cap"], float(o["visible_ratio"][finest]), int(o["npts"][finest])))
        q = []
        if gates:
            if o["b_cap"] > b_thr: q.append(2)
            if o["visible_ratio"][finest] < vis_thr: q.append(3)
            if o["npts"][finest] < min_reproj: q.append(4)
        ld_t = oracle_logdet(gray[ref], depth[ref], gray[t], finest, o["R"], o["T"], K) if last_ref != t - 1 else np.nan
        switch, why, alpha[t] = keyframe_decision(t, last_ref, q, ld_t, final_logdet[last_ref + 1], thr, every)
        if switch:
            last_ref = t - 1; ref = t - 1; kind[t - 1] = 2; reason[t - 1] = why
            o = O.align_pair(gray[ref], depth[ref], gray[t], levels, iters, K, R0=np.eye(3), T0=np.zeros(3))
        R, T = o["R"], o["T"]
        rel[t, :9] = R.reshape(9); rel[t, 9:] = T
        if last_ref == t - 1:
            final_logdet[t] = oracle_logdet(gray[ref], depth[ref], gray[t], finest, R, T, K)
    glob, _, _ = O.gop_replay(kind, np.maximum(reason, 1), rel)
    return rel, kind, reason, glob, alpha, stats


# ------------------------------------------------------------------------------------------------ CPU
LD_REF = -60.0                                   # h_ref = H0 - 30 < 0


def test_decision_sign_handling():
    h_ref = entropy(LD_REF)
    assert h_ref < 0
    sw, why, a = keyframe_decision(5, 2, [], -50.0, LD_REF, 0.9, 0)          # less certain than after the key frame: alpha < 1
    assert sw and why == 6 and a == pytest.approx(entropy(-50.0) / h_ref) and 0 < a < 0.9
    assert not keyframe_decision(5, 2, [], -50.0, LD_REF, a, 0)[0]           # alpha must be strictly below the threshold
    sw, why, a = keyframe_decision(5, 2, [], -62.0, LD_REF, 0.9, 0)          # more certain: alpha > 1
    assert not sw and why == 0 and a > 1
    sw, _, a = keyframe_decision(5, 2, [], 2 * (1.0 - H0), LD_REF, 0.9, 0)   # h_t > 0 > h_ref: alpha < 0 fires
    assert sw and a < 0


def test_decision_nan_covariances_decide_nothing():
    for ld_t, ld_ref in ((np.nan, LD_REF), (-50.0, np.nan), (np.nan, np.nan)):
        sw, why, a = keyframe_decision(5, 2, [], ld_t, ld_ref, 0.9, 0)
        assert not sw and why == 0 and np.isnan(a)
    sw, why, _ = keyframe_decision(5, 2, [3], np.nan, LD_REF, 0.9, 0)         # the other gates still decide
    assert sw and why == 3


def test_decision_silent_when_h_ref_not_negative():
    for ld_ref in (2 * (1.0 - H0), -2 * H0):                                  # h_ref = 1, h_ref = 0
        assert entropy(ld_ref) >= 0
        for ld_t in (-60.0, -2 * H0 + 0.5, 0.0):
            sw, why, a = keyframe_decision(5, 2, [], ld_t, ld_ref, 0.9, 0)
            assert not sw and why == 0
    sw, _, a = keyframe_decision(5, 2, [], -60.0, 2 * (1.0 - H0), 0.9, 0)
    assert np.isfinite(a) and a < 0.9                                          # alpha is reported but does not fire


def test_decision_guard_previous_frame_already_key():
    sw, why, a = keyframe_decision(3, 2, [2, 4], -50.0, LD_REF, 0.9, 1)      # every gate would fire, but frame 2 already is the key frame
    assert not sw and why == 0 and np.isnan(a)
    sw, why, a = keyframe_decision(1, 0, [], -50.0, LD_REF, 0.9, 0)
    assert not sw and np.isnan(a)


def test_decision_reason_order():
    fire, calm = -50.0, -62.0
    assert keyframe_decision(5, 2, [2], calm, LD_REF, 0.9, 0)[:2] == (True, 2)
    assert keyframe_decision(5, 2, [2, 3, 4], calm, LD_REF, 0.9, 0)[:2] == (True, 4)
    assert keyframe_decision(5, 2, [2, 4], fire, LD_REF, 0.9, 0)[:2] == (True, 6)      # entropy after the quality gates
    assert keyframe_decision(5, 2, [3], fire, LD_REF, 0.9, 3)[:2] == (True, 5)         # periodic last
    assert keyframe_decision(5, 2, [], fire, LD_REF, 0.9, 4)[:2] == (True, 6)          # periodic not due
    assert keyframe_decision(5, 2, [], calm, LD_REF, 0.9, 3)[:2] == (True, 5)


# ------------------------------------------------------------------------------------------------ GPU
def rot_angle(Ra, Rb):
    return float(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


def reference_of(kind_s, t):
    return max(k for k in range(t) if kind_s[k] != 0)


def bits(a):
    return None if a is None else np.ascontiguousarray(a).view(np.uint8)


def same_records(a, b):
    return len(a) == len(b) and all((x is None and y is None) or np.array_equal(bits(x), bits(y)) for x, y in zip(a, b))


def make_sequences(seed0, nseq, nframes, W, H, K, max_angle_deg, max_trans_m):
    seqs = [O.synth_sequence(seed0 + s, nframes, W, H, K, max_angle_deg=max_angle_deg, max_trans_m=max_trans_m) for s in range(nseq)]
    return np.stack([s[0] for s in seqs]), np.stack([s[1] for s in seqs])


def check_against_oracle_loop(al, gray, depth, L, iters, K, thr, pol, **gates):
    """Run the GPU loop and the oracle loop; compare everything; return (kind, reason, largest relative alpha difference)."""
    nseq, nframes = gray.shape[:2]
    prm = dvo.solver_params(iters=iters)
    rel, kind, reason, glob, rel_cov, glob_cov, alpha = al.run_sequences_entropy(gray, depth, nseq, nframes, prm, pol, thr)
    finest = [l for l in range(L) if iters[l] > 0][0]
    worst = 0.0
    for s in range(nseq):
        orel, okind, oreason, oglob, oalpha, stats = oracle_sequence_entropy(gray[s], depth[s], L, iters, K, thr, every=pol.keyframe_every,
                                                                             **gates)
        seen = oalpha[np.isfinite(oalpha)]
        assert np.abs(seen - thr).min() > 1e-4, (s, thr, oalpha)            # no decision sits near the threshold
        if gates.get("gates"):
            assert min(abs(b - gates["b_thr"]) for b, _, _ in stats) > 1e-3 and min(abs(v - gates["vis_thr"]) for _, v, _ in stats) > 1e-4
        assert np.array_equal(kind[s], okind), (s, kind[s], okind)
        assert np.array_equal(reason[s], oreason), (s, reason[s], oreason)
        assert np.array_equal(np.isnan(alpha[s]), np.isnan(oalpha)), (s, alpha[s], oalpha)
        fin = np.isfinite(oalpha)
        worst = max(worst, float(np.max(np.abs(alpha[s, fin] - oalpha[fin]) / np.abs(oalpha[fin]))))
        for t in range(nframes):
            assert rot_angle(rel[s, t, :9].reshape(3, 3), orel[t, :9].reshape(3, 3)) < 1e-5 and np.linalg.norm(rel[s, t, 9:] - orel[t, 9:]) < 1e-5
            assert rot_angle(glob[s, t, :9].reshape(3, 3), oglob[t, :9].reshape(3, 3)) < 1e-5 and np.linalg.norm(glob[s, t, 9:12] - oglob[t, 9:12]) < 1e-5
        # NaN exactly at frame 0 and at the frames the gate skipped (t = lastRef + 1 at decision time)
        last_ref, skipped = 0, [0]
        for t in range(1, nframes):
            if last_ref == t - 1:
                skipped.append(t)
            if kind[s, t - 1] == 2:
                last_ref = t - 1
        assert list(np.nonzero(np.isnan(alpha[s]))[0]) == skipped, (s, alpha[s])
        for t in range(1, nframes):                                          # covariance at the GPU's pose, on its final reference
            r = reference_of(kind[s], t)
            R, T = rel[s, t, :9].reshape(3, 3), rel[s, t, 9:]
            H, s2, _ = oracle_cov(gray[s, r], depth[s, r], gray[s, t], finest, R, T, K)
            assert np.abs(rel_cov[s, t] @ H / s2 - np.eye(6)).max() < 1e-6, (s, t, r)
    assert worst < 1e-6, worst
    print(f"largest relative alpha difference GPU vs oracle: {worst:.3e}")
    return kind, reason, worst


@pytest.fixture(scope="module")
def seq320():
    W, H, L = 320, 240, 4
    gray, depth = make_sequences(70, 3, 10, W, H, K320, 0.4, 0.008)
    al = dvo.BatchAligner(W, H, L, max_batch=4, keep_now_depth=True, intrinsics=K320)
    yield al, gray, depth
    al.close()


GATED = dict(keyframe_every=0, use_quality_gates=True, laplacian_thresh=9.5, visible_ratio_thresh=0.95)


@pytest.mark.gpu
@pytest.mark.parametrize("policy", [dict(), dict(keyframe_every=3), GATED], ids=["shipped", "periodic3", "quality_gates"])
def test_disabled_gate_is_run_sequences_cov(seq320, policy):
    al, gray, depth = seq320
    nseq, nframes = gray.shape[:2]
    prm = dvo.solver_params(iters=(8, 8, 8, 8))
    pol = dvo.keyframe_policy(**policy)
    n0 = al.launch_count()
    want = al.run_sequences_cov(gray, depth, nseq, nframes, prm, pol)
    n1 = al.launch_count()
    got = al.run_sequences_entropy(gray, depth, nseq, nframes, prm, pol, 0.0)
    n2 = al.launch_count()
    assert same_records(want, got[:6])
    assert np.isnan(got[6]).all()
    assert n2 - n1 == n1 - n0
    assert same_records(want, al.run_sequences_entropy(gray, depth, nseq, nframes, prm, pol, -1.0)[:6])


# Thresholds: chosen from a run of the oracle loop so that the sequences switch at different frames, and asserted to sit more than 1e-4 away
# from every ratio a decision saw (the GPU and the oracle agree on alpha to about 1e-6, so no decision can flip).
ENT_SEQ = dict(seed0=300, nseq=4, nframes=12, max_angle_deg=0.8, max_trans_m=0.016)
ENT_THR = 0.955


@pytest.mark.gpu
def test_entropy_gate_matches_oracle_loop_320x240():
    W, H, L, iters = 320, 240, 4, (8, 8, 8, 8)
    gray, depth = make_sequences(W=W, H=H, K=K320, **ENT_SEQ)
    al = dvo.BatchAligner(W, H, L, max_batch=4, keep_now_depth=True, intrinsics=K320)
    kind, reason, _ = check_against_oracle_loop(al, gray, depth, L, iters, K320, ENT_THR, dvo.keyframe_policy(keyframe_every=0))
    switches = [tuple(np.nonzero(k == 2)[0]) for k in kind]
    assert set(reason[kind == 2].tolist()) == {6}
    assert any(switches) and len(set(switches)) > 1, switches               # the sequences switch at different frames
    al.close()


@pytest.mark.gpu
def test_entropy_with_periodic_and_quality_gates(seq320):
    """All gates at once: the reasons follow the order 2, 3, 4, 6, 5 of the oracle loop."""
    al, gray, depth = seq320
    pol = dvo.keyframe_policy(keyframe_every=5, use_quality_gates=True, laplacian_thresh=9.5, visible_ratio_thresh=0.95)
    kind, reason, _ = check_against_oracle_loop(al, gray, depth, 4, (8, 8, 8, 8), K320, 0.95, pol, gates=True, b_thr=9.5,
                                                vis_thr=0.95)
    assert {3, 5, 6} <= set(reason[kind == 2].tolist())


@pytest.mark.gpu
def test_entropy_inputs_and_subsets_give_identical_records():
    """Pageable host, pinned host and device-resident inputs give bit-identical records, and so does every sequence run in a
    smaller launch."""
    import torch
    W, H, L = 320, 240, 4
    gray, depth = make_sequences(W=W, H=H, K=K320, **ENT_SEQ)
    nseq, nframes = gray.shape[:2]
    prm = dvo.solver_params(iters=(8, 8, 8, 8))
    pol = dvo.keyframe_policy(keyframe_every=0)
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K320)
    want = al.run_sequences_entropy(gray, depth, nseq, nframes, prm, pol, ENT_THR)
    assert (want[1] == 2).any()
    pg, pd = torch.from_numpy(gray).pin_memory(), torch.from_numpy(depth.view(np.int16)).pin_memory()
    assert same_records(want, al.run_sequences_entropy(pg.data_ptr(), pd.data_ptr(), nseq, nframes, prm, pol, ENT_THR))
    dg, dd = pg.cuda(), pd.cuda()
    torch.cuda.synchronize()
    assert same_records(want, al.run_sequences_entropy(dg.data_ptr(), dd.data_ptr(), nseq, nframes, prm, pol, ENT_THR, device=True))
    for sub in ([1, 2], [3], [0, 2, 3]):
        g, d = np.ascontiguousarray(gray[sub]), np.ascontiguousarray(depth[sub])
        got = al.run_sequences_entropy(g, d, len(sub), nframes, prm, pol, ENT_THR)
        assert same_records([a[sub] for a in want], got), sub
    al.close()


@pytest.mark.gpu
def test_degenerate_frame_never_fires_the_gate():
    """Sequence 1's now frame 5 is blank: no edges at the finest level, a NaN covariance, alpha NaN there and no switch.  The
    other sequences' records equal a run without sequence 1."""
    W, H, L = 320, 240, 4
    gray, depth = make_sequences(W=W, H=H, K=K320, **ENT_SEQ)
    gray[1, 5] = 128
    nseq, nframes = gray.shape[:2]
    prm = dvo.solver_params(iters=(8, 8, 8, 8))
    pol = dvo.keyframe_policy(keyframe_every=0)
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K320)
    rel, kind, reason, glob, rel_cov, glob_cov, alpha = al.run_sequences_entropy(gray, depth, nseq, nframes, prm, pol, ENT_THR)
    assert np.isnan(alpha[1, 5]) and kind[1, 4] == 0 and reason[1, 4] == 0
    assert np.isnan(rel_cov[1, 5]).all()
    others = [0, 2, 3]
    got = al.run_sequences_entropy(np.ascontiguousarray(gray[others]), np.ascontiguousarray(depth[others]), 3, nframes, prm, pol, ENT_THR)
    assert same_records([a[others] for a in (rel, kind, reason, glob, rel_cov, glob_cov, alpha)], got)
    al.close()


ENT_SEQ_1280 = dict(seed0=170, nseq=2, nframes=7, max_angle_deg=0.8, max_trans_m=0.016)
ENT_THR_1280 = 0.99


@pytest.mark.gpu
def test_entropy_gate_matches_oracle_loop_1280x720_5_levels():
    W, H, L, K = 1280, 720, 5, O.K1280
    gray, depth = make_sequences(W=W, H=H, K=K, **ENT_SEQ_1280)
    al = dvo.BatchAligner(W, H, L, max_batch=2, keep_now_depth=True, intrinsics=K)
    kind, reason, _ = check_against_oracle_loop(al, gray, depth, L, (50,) * 5, K, ENT_THR_1280, dvo.keyframe_policy(keyframe_every=0))
    assert set(reason[kind == 2].tolist()) == {6}
    al.close()
