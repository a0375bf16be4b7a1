"""Device memory comes back when a context closes.

Five cycles of: create a BatchAligner, a PhotoEstimator and an RGBDAligner (320x240), drive every buffer that grows on demand
from a small to a larger size, call every inspection entry point, close.  After each close it prints the free device memory
(torch.cuda.mem_get_info).  From cycle 2 on the figure must not go down; cycle 1 may differ, since the CUDA runtime keeps
module and local-memory reservations once made.  Not a test: the figure covers the whole device, and other processes on a
shared GPU move it.  Needs a CUDA device.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle_lib as O  # noqa: E402
import rgbd_odometry_b200 as dvo  # noqa: E402

W, H = 320, 240
K = (262.5, 262.5, 159.5, 119.5)


def free():
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


def batch_aligner(seq, pair):
    gray, depth = seq
    prm = dvo.solver_params(iters=(8, 8, 8))
    pol = dvo.keyframe_policy(keyframe_every=3)
    al = dvo.BatchAligner(W, H, 3, max_batch=4, keep_now_depth=True, trace_iters=2, intrinsics=K)
    for nseq, nf in ((2, 4), (4, 8)):
        g, d = np.ascontiguousarray(gray[:nseq, :nf]), np.ascontiguousarray(depth[:nseq, :nf])
        al.run_sequences_cov(g, d, nseq, nf, prm, pol)
        rel, kind, *_ = al.run_sequences_entropy(g, d, nseq, nf, prm, pol, 0.95)
    al.gop_compose(kind, rel)
    al.load_frames(gray[0, :4], depth[0, :4])
    for k in (1, 3):
        pairs = [(i, j) for i in range(4) for j in range(4) if i != j and abs(i - j) <= k]
        ri = [i for i, _ in pairs]; ni = [j for _, j in pairs]
        al.align_pairs(ri, ni, prm, covariance=True)
        al.align_pairs(torch.tensor(ri, dtype=torch.int32, device="cuda"), torch.tensor(ni, dtype=torch.int32, device="cuda"), prm,
                       covariance=True, device=True)
    al.synchronize()
    al.set_frames(dvo.FRAME_REF, pair["ref_gray"], pair["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, pair["now_gray"], pair["now_depth"])
    al.build_pyramids(4); al.prepare(4); al.run(4, prm)
    for count in (2, 4):
        al.pose_covariance(count, prm)
    for count in (1, 4):
        al.set_frames_raw(dvo.FRAME_NOW, pair["now_bgr"][:count], pair["now_depth"][:count].astype(np.float32) / np.float32(1000.0))
    al.build_pyramids(4); al.prepare(4); al.run(4, prm)
    for which in ("gray", "depth", "edge", "d2", "dtn", "gx", "gy"):
        al.get_level_buffer(0, dvo.FRAME_NOW, 1, which)
    n = len(al.get_points(0, 1)[0])
    al.eval_normal_equations(0, 1, np.eye(3), np.zeros(3), per_point=True, npts=n)
    al.get_trace(0, 1); al.get_energies(0, 1)
    dvo.undistort(pair["now_bgr"], (K[0], K[1], K[2], K[3]), (0.05, -0.02, 0.001, 0.001, 0.0))
    al.close()


def photo_estimator(pair):
    ph = dvo.PhotoEstimator(W, H, 3, max_batch=4, intrinsics=K)
    ph.set_frames(dvo.FRAME_REF, pair["ref_bgr"], pair["ref_depth"])
    ph.set_frames(dvo.FRAME_NOW, pair["now_bgr"], pair["now_depth"])
    ph.prepare_ref(4)
    ph.set_pose(4, np.tile(np.r_[np.eye(3).ravel(), np.zeros(3)], (4, 1)))
    ph.estimate(4, 1)
    ph.get_poses(4)
    for level in (0, 1):
        for which in ("bgr", "X", "J", "blueVals"):
            ph.get_level(0, dvo.FRAME_REF, level, which)
        ph.eval(0, level, np.eye(3), np.zeros(3), want_canvas=True)
    ph.close()


def rgbd_aligner(pair):
    rg = dvo.RGBDAligner(W, H, 3, max_batch=4, intrinsics=K)
    rg.set_frames(dvo.FRAME_REF, pair["ref_bgr"], pair["ref_depth"])
    rg.set_frames(dvo.FRAME_NOW, pair["now_bgr"], pair["now_depth"])
    rg.compute_jacobians(4)
    rg.set_pose(4, np.tile(np.eye(4), (4, 1, 1)))
    rg.gauss_newton(4, 1)
    rg.get_poses(4)
    rg.get_level(0, dvo.FRAME_REF, 1); rg.get_A(0, 1)
    rg.eval(0, 1, np.eye(4))
    rg.close()


def main():
    seqs = [O.synth_sequence(400 + s, 8, W, H, K, max_angle_deg=0.4, max_trans_m=0.008) for s in range(4)]
    seq = (np.stack([s[0] for s in seqs]), np.stack([s[1] for s in seqs]))
    pair = O.synth_batch(410, 4, W, H, K, bgr=True, now_depth=True)
    torch.cuda.init()
    print(f"{torch.cuda.get_device_name(0)}: free device memory in bytes after each close")
    print(f"{'cycle':>5} {'BatchAligner':>14} {'PhotoEstimator':>15} {'RGBDAligner':>14}")
    for cycle in range(1, 6):
        batch_aligner(seq, pair); a = free()
        photo_estimator(pair); b = free()
        rgbd_aligner(pair); c = free()
        print(f"{cycle:>5} {a:>14} {b:>15} {c:>14}", flush=True)


if __name__ == "__main__":
    main()
