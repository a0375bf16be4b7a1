"""Buffers a context grows on demand: growth is transparent.

Each grow path is called on one context with a small size, then a larger one, then the small one again, so that a buffer is
replaced after it has been used and then reused at less than its capacity.  Every result must equal, bit for bit, the result of
a fresh context of the same configuration that makes only that call.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import rgbd_odometry_b200 as dvo

W, H, L = 320, 240, 3
K = (262.5, 262.5, 159.5, 119.5)
PRM = dvo.solver_params(iters=(8, 8, 8))


def same(a, b):
    """Bit-for-bit equality of numpy arrays (NaN payloads included), and of ctypes record arrays field by field: the padding
    bytes of a record (dvo_cov_info has 4 after nvis) are never written, so they are not compared."""
    if isinstance(a, np.ndarray):
        return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()
    rec = type(a)._type_
    size, fields = C.sizeof(rec), [(getattr(rec, f[0]).offset, getattr(rec, f[0]).size) for f in rec._fields_]
    ra, rb = bytes(a), bytes(b)
    return len(a) == len(b) and all(ra[i * size + o:i * size + o + n] == rb[i * size + o:i * size + o + n]
                                    for i in range(len(a)) for o, n in fields)


def check_same(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert (g is None) == (w is None), k
        if g is not None:
            assert same(g, w), k


@pytest.fixture(scope="module")
def sequences():
    seqs = [O.synth_sequence(300 + s, 8, W, H, K, max_angle_deg=0.4, max_trans_m=0.008) for s in range(4)]
    return np.stack([s[0] for s in seqs]), np.stack([s[1] for s in seqs])


@pytest.mark.gpu
@pytest.mark.parametrize("entropy", [False, True])
def test_sequence_buffers_grow_transparently(sequences, entropy):
    gray, depth = sequences
    pol = dvo.keyframe_policy(keyframe_every=3)

    def run(al, nseq, nframes):
        g = np.ascontiguousarray(gray[:nseq, :nframes]); d = np.ascontiguousarray(depth[:nseq, :nframes])
        if entropy:
            return al.run_sequences_entropy(g, d, nseq, nframes, PRM, pol, 0.95)
        return al.run_sequences_cov(g, d, nseq, nframes, PRM, pol)

    al = dvo.BatchAligner(W, H, L, max_batch=4, keep_now_depth=True, intrinsics=K)
    for nseq, nframes in ((2, 4), (4, 8), (2, 4)):
        got = run(al, nseq, nframes)
        fresh = dvo.BatchAligner(W, H, L, max_batch=4, keep_now_depth=True, intrinsics=K)
        check_same(got, run(fresh, nseq, nframes))
        fresh.close()
    al.close()


NF = 6


@pytest.fixture(scope="module")
def frames():
    gray, depth, _, _ = O.synth_sequence(310, NF, W, H, K)
    return gray, depth


def loaded(frames):
    al = dvo.BatchAligner(W, H, L, max_batch=NF, intrinsics=K)
    al.load_frames(*frames)
    return al


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True])
def test_pair_buffers_grow_transparently(frames, device):
    import torch

    def run(al, k):
        pairs = [(i, j) for i in range(NF) for j in range(NF) if i != j and abs(i - j) <= k]
        ri = [i for i, _ in pairs]; ni = [j for _, j in pairs]
        if device:
            poses, info, cov, cinfo = al.align_pairs(torch.tensor(ri, dtype=torch.int32, device="cuda"),
                                                     torch.tensor(ni, dtype=torch.int32, device="cuda"), PRM, covariance=True, device=True)
            al.synchronize()
            return poses.cpu().numpy(), dvo.records(info, dvo.PairInfo), cov.cpu().numpy(), dvo.records(cinfo, dvo.CovInfo)
        return al.align_pairs(ri, ni, PRM, covariance=True)

    al = loaded(frames)
    for k in (1, 3, 1):                      # 10, 24, 10 pairs
        got = run(al, k)
        fresh = loaded(frames)
        check_same(got, run(fresh, k))
        fresh.close()
    al.close()


@pytest.mark.gpu
def test_covariance_buffer_grows_transparently(frames):
    gray, depth = frames

    def solved():
        al = dvo.BatchAligner(W, H, L, max_batch=NF - 1, intrinsics=K)
        al.set_frames(dvo.FRAME_REF, gray[:-1], depth[:-1])
        al.set_frames(dvo.FRAME_NOW, gray[1:])
        al.build_pyramids(NF - 1); al.prepare(NF - 1); al.run(NF - 1, PRM)
        return al

    al = solved()
    for count in (2, NF - 1, 2):
        got = al.pose_covariance(count, PRM)
        fresh = solved()
        check_same(got, fresh.pose_covariance(count, PRM))
        fresh.close()
    al.close()


@pytest.mark.gpu
def test_raw_staging_grows_transparently():
    d = O.synth_batch(320, 4, W, H, K, bgr=True)
    bgr, dm = d["ref_bgr"], d["ref_depth"].astype(np.float32) / np.float32(1000.0)

    def levels(al, count):
        return [al.get_level_buffer(s, dvo.FRAME_REF, 0, which) for s in range(count) for which in ("gray", "depth")]

    al = dvo.BatchAligner(W, H, L, max_batch=4, intrinsics=K)
    for first, count in ((3, 1), (0, 4), (1, 1)):          # the small calls take other images than the slots they write held
        al.set_frames_raw(dvo.FRAME_REF, bgr[first:first + count], dm[first:first + count])
        fresh = dvo.BatchAligner(W, H, L, max_batch=4, intrinsics=K)
        fresh.set_frames_raw(dvo.FRAME_REF, bgr[first:first + count], dm[first:first + count])
        check_same(levels(al, count), levels(fresh, count))
        fresh.close()
    al.close()
