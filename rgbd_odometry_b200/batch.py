"""BatchAligner: Python host-side mirror of the batch C-ABI (one object = one dvo_ctx on one GPU)."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Config, CovInfo, KeyframePolicy, PairInfo, PgoInfo, PgoParams, SolverParams, check

SUBGRAD_REF, GN, LM = 0, 1, 2
JAC_REFERENCE, JAC_EXACT = 0, 1
W_REF_CAUCHY, W_HUBER, W_NONE = 0, 1, 2
ARITH_EXACT, ARITH_FAST = 0, 1
RES_DT_FLOOR, RES_DT_INTERP = 0, 1
FRAME_REF, FRAME_NOW = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
BUF = {"gray": (0, np.uint8), "depth": (1, np.uint16), "edge": (2, np.uint8), "d2": (3, np.int32),
       "dtn": (4, np.float32), "gx": (5, np.float32), "gy": (6, np.float32)}


def solver_params(solver=SUBGRAD_REF, jacobian=JAC_REFERENCE, weight=W_REF_CAUCHY, arithmetic=ARITH_EXACT, huber_k=1.345,
                  lm_lambda0=1e-3, iters=(50, 50, 50, 50), residual=RES_DT_FLOOR):
    p = SolverParams()
    p.solver, p.jacobian, p.weight, p.arithmetic, p.residual = solver, jacobian, weight, arithmetic, residual
    p.huber_k, p.lm_lambda0 = huber_k, lm_lambda0
    for i in range(_lib.MAX_LEVELS):
        p.iters[i] = int(iters[i]) if i < len(iters) else 0
    return p


def keyframe_policy(keyframe_every=5, use_quality_gates=False, laplacian_thresh=3.0, visible_ratio_thresh=0.8, min_reprojections=50):
    """Defaults are the reference's constants (src/SolveDVO.cpp:22-23, :2145, :2156); the gates ship disabled there."""
    return KeyframePolicy(keyframe_every, int(use_quality_gates), laplacian_thresh, visible_ratio_thresh, min_reprojections)


def undistort(img, K, D):
    """cv::undistort of a batch of images (N, H, W[, 3]) u8 or (N, H, W) u16 on the GPU (dvo_undistort, host buffers)."""
    lib = _lib.load()
    img = np.ascontiguousarray(img)
    n, h, w = img.shape[:3]
    typ = 2 if img.dtype == np.uint16 else (1 if img.ndim == 4 and img.shape[3] == 3 else 0)
    out = np.empty_like(img)
    K4 = np.array(K, np.float64); D5 = np.array(D, np.float64)
    check(lib.dvo_undistort(img.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), w, h, typ, n, K4.ctypes.data_as(C.c_void_p),
                            D5.ctypes.data_as(C.c_void_p), MEM_HOST, None), "dvo_undistort")
    return out


def records(raw, cls):
    """ctypes array of `cls` (PairInfo, CovInfo, PgoInfo) from the raw records align_pairs(device=True) returns as a uint8 CUDA tensor."""
    return (cls * raw.shape[0]).from_buffer_copy(raw.cpu().numpy().tobytes())


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


class BatchAligner:
    """Owns a dvo_ctx.  Arrays are numpy (host) unless `device=True`, in which case raw device pointers (ints) are passed."""

    def __init__(self, width=640, height=480, levels=4, max_batch=1, device=0, keep_now_depth=False, trace_iters=0,
                 intrinsics=(525.0, 525.0, 319.5, 239.5)):
        self.lib = _lib.load()
        self.cfg = Config(width, height, levels, max_batch, device, int(keep_now_depth), trace_iters)
        self.h = C.c_void_p()
        check(self.lib.dvo_create(C.byref(self.cfg), C.byref(self.h)), "dvo_create")
        self.levels, self.max_batch, self.width, self.height = levels, max_batch, width, height
        if intrinsics is not None:
            self.set_intrinsics(*intrinsics)

    def close(self):
        if self.h:
            self.lib.dvo_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, stream_ptr):
        check(self.lib.dvo_set_stream(self.h, C.c_void_p(stream_ptr) if stream_ptr else None), "dvo_set_stream")

    def synchronize(self):
        check(self.lib.dvo_synchronize(self.h), "dvo_synchronize")

    def set_intrinsics(self, fx, fy, cx, cy):
        check(self.lib.dvo_set_intrinsics(self.h, fx, fy, cx, cy), "dvo_set_intrinsics")

    def set_frames(self, frame, gray, depth=None, first=0, count=None, device=False):
        if not device:
            gray = np.ascontiguousarray(gray, np.uint8)
            count = gray.shape[0] if count is None else count
            if depth is not None:
                depth = np.ascontiguousarray(depth, np.uint16)
        check(self.lib.dvo_set_frames(self.h, frame, first, count, _ptr(gray), _ptr(depth), MEM_DEVICE if device else MEM_HOST),
              "dvo_set_frames")

    def set_frames_raw(self, frame, bgr, depth_m=None, first=0, count=None, device=False):
        """Raw sensor frames: bgr (n, H, W, 3) u8 and depth_m (n, H, W) f32 metres (dvo_set_frames_raw)."""
        if not device:
            bgr = np.ascontiguousarray(bgr, np.uint8)
            count = bgr.shape[0] if count is None else count
            if depth_m is not None:
                depth_m = np.ascontiguousarray(depth_m, np.float32)
        check(self.lib.dvo_set_frames_raw(self.h, frame, first, count, _ptr(bgr), _ptr(depth_m), MEM_DEVICE if device else MEM_HOST),
              "dvo_set_frames_raw")

    def build_pyramids(self, count, first=0, frames_mask=3):
        check(self.lib.dvo_build_pyramids(self.h, first, count, frames_mask), "dvo_build_pyramids")

    def prepare(self, count, first=0, frames_mask=3):
        check(self.lib.dvo_prepare(self.h, first, count, frames_mask), "dvo_prepare")

    def promote_now_to_ref(self, count, first=0):
        check(self.lib.dvo_promote_now_to_ref(self.h, first, count), "dvo_promote_now_to_ref")

    def set_initial_pose(self, count, poses=None, first=0):
        if poses is not None:
            poses = np.ascontiguousarray(poses, np.float64).reshape(count, 12)
        check(self.lib.dvo_set_initial_pose(self.h, first, count, _ptr(poses), MEM_HOST), "dvo_set_initial_pose")

    def run(self, count, params, first=0):
        check(self.lib.dvo_run(self.h, first, count, C.byref(params)), "dvo_run")

    def process(self, count, params, first=0, poses_out=None):
        """build_pyramids + prepare + run on resident frames; large ranges run as two staggered half batches (dvo_process).
        poses_out: optional raw device pointer (count x 12 doubles) the poses are copied to without joining."""
        check(self.lib.dvo_process(self.h, first, count, C.byref(params), C.c_void_p(poses_out) if poses_out else None), "dvo_process")

    def join(self):
        check(self.lib.dvo_join(self.h), "dvo_join")

    def join_stream(self, stream_ptr):
        check(self.lib.dvo_join_stream(self.h, C.c_void_p(stream_ptr)), "dvo_join_stream")

    def get_poses(self, count, first=0, want_info=True):
        poses = np.empty((count, 12), np.float64)
        info = (PairInfo * count)() if want_info else None
        check(self.lib.dvo_get_poses(self.h, first, count, _ptr(poses), C.cast(info, C.c_void_p) if want_info else None, MEM_HOST),
              "dvo_get_poses")
        return poses, info

    def get_poses_device(self, count, dst_ptr, first=0):
        check(self.lib.dvo_get_poses(self.h, first, count, C.c_void_p(dst_ptr), None, MEM_DEVICE), "dvo_get_poses")

    def align_batch(self, ref_gray, ref_depth, now_gray, params, now_depth=None, want_info=True):
        ref_gray = np.ascontiguousarray(ref_gray, np.uint8)
        ref_depth = np.ascontiguousarray(ref_depth, np.uint16)
        now_gray = np.ascontiguousarray(now_gray, np.uint8)
        n = ref_gray.shape[0]
        poses = np.empty((n, 12), np.float64)
        info = (PairInfo * n)() if want_info else None
        check(self.lib.dvo_align_batch(self.h, n, _ptr(ref_gray), _ptr(ref_depth), _ptr(now_gray), _ptr(now_depth), C.byref(params),
                                       _ptr(poses), C.cast(info, C.c_void_p) if want_info else None), "dvo_align_batch")
        return poses, info

    def run_sequences(self, gray, depth, params, keyframe_every=5):
        """SolveDVO::loop over nseq sequences in lock step.  gray/depth: (nseq, nframes, H, W)."""
        gray = np.ascontiguousarray(gray, np.uint8)
        depth = np.ascontiguousarray(depth, np.uint16)
        nseq, nframes = gray.shape[:2]
        rel = np.empty((nseq, nframes, 12), np.float64)
        kind = np.empty((nseq, nframes), np.int32)
        glob = np.empty((nseq, nframes, 19), np.float64)
        check(self.lib.dvo_run_sequences(self.h, nseq, nframes, _ptr(gray), _ptr(depth), C.byref(params), keyframe_every, _ptr(rel),
                                         _ptr(kind), _ptr(glob)), "dvo_run_sequences")
        return rel, kind, glob

    def run_sequences_gated(self, gray, depth, params, policy):
        """SolveDVO::loop with the key-frame decision (periodic rule and / or the quality gates) taken per sequence on the device."""
        gray = np.ascontiguousarray(gray, np.uint8)
        depth = np.ascontiguousarray(depth, np.uint16)
        nseq, nframes = gray.shape[:2]
        rel = np.empty((nseq, nframes, 12), np.float64)
        kind = np.empty((nseq, nframes), np.int32)
        reason = np.empty((nseq, nframes), np.int32)
        glob = np.empty((nseq, nframes, 19), np.float64)
        check(self.lib.dvo_run_sequences_gated(self.h, nseq, nframes, _ptr(gray), _ptr(depth), C.byref(params), C.byref(policy), _ptr(rel),
                                               _ptr(kind), _ptr(reason), _ptr(glob)), "dvo_run_sequences_gated")
        return rel, kind, reason, glob

    def run_sequences_mem(self, gray, depth, nseq, nframes, params, policy, device=False, want_global=True):
        """dvo_run_sequences_mem: gray / depth are numpy arrays (host; pinned arrays upload asynchronously) or, with device=True,
        raw device pointers to [nseq][nframes][H][W] buffers."""
        rel = np.empty((nseq, nframes, 12), np.float64)
        kind = np.empty((nseq, nframes), np.int32)
        reason = np.empty((nseq, nframes), np.int32)
        glob = np.empty((nseq, nframes, 19), np.float64) if want_global else None
        check(self.lib.dvo_run_sequences_mem(self.h, nseq, nframes, _ptr(gray), _ptr(depth), MEM_DEVICE if device else MEM_HOST,
                                             C.byref(params), C.byref(policy), _ptr(rel), _ptr(kind), _ptr(reason), _ptr(glob)),
              "dvo_run_sequences_mem")
        return rel, kind, reason, glob

    def run_sequences_cov(self, gray, depth, nseq, nframes, params, policy, device=False, want_global=True):
        """dvo_run_sequences_cov: run_sequences_mem's (rel, kind, reason, glob) plus rel_cov (nseq, nframes, 6, 6) -- the covariance of
        each relative pose, zeros at frame 0 -- and global_cov (nseq, nframes, 6, 6) propagated along the key-frame chain (None
        unless want_global).  Tangent (rho, omega), translation first, for T <- T exp(psi)."""
        rel = np.empty((nseq, nframes, 12), np.float64)
        kind = np.empty((nseq, nframes), np.int32)
        reason = np.empty((nseq, nframes), np.int32)
        glob = np.empty((nseq, nframes, 19), np.float64) if want_global else None
        rel_cov = np.empty((nseq, nframes, 6, 6), np.float64)
        glob_cov = np.empty((nseq, nframes, 6, 6), np.float64) if want_global else None
        check(self.lib.dvo_run_sequences_cov(self.h, nseq, nframes, _ptr(gray), _ptr(depth), MEM_DEVICE if device else MEM_HOST,
                                             C.byref(params), C.byref(policy), _ptr(rel), _ptr(kind), _ptr(reason), _ptr(glob),
                                             _ptr(rel_cov), _ptr(glob_cov)), "dvo_run_sequences_cov")
        return rel, kind, reason, glob, rel_cov, glob_cov

    def run_sequences_entropy(self, gray, depth, nseq, nframes, params, policy, entropy_ratio_thresh, device=False, want_global=True):
        """dvo_run_sequences_entropy: run_sequences_cov with the entropy-ratio key-frame rule of DVO-SLAM added to `policy` (reason 6).
        Returns run_sequences_cov's six records plus entropy_ratio (nseq, nframes): the ratio each decision saw, NaN where the gate
        was not evaluated.  entropy_ratio_thresh <= 0 disables the gate (the result is then run_sequences_cov's)."""
        rel = np.empty((nseq, nframes, 12), np.float64)
        kind = np.empty((nseq, nframes), np.int32)
        reason = np.empty((nseq, nframes), np.int32)
        glob = np.empty((nseq, nframes, 19), np.float64) if want_global else None
        rel_cov = np.empty((nseq, nframes, 6, 6), np.float64)
        glob_cov = np.empty((nseq, nframes, 6, 6), np.float64) if want_global else None
        ratio = np.empty((nseq, nframes), np.float64)
        check(self.lib.dvo_run_sequences_entropy(self.h, nseq, nframes, _ptr(gray), _ptr(depth), MEM_DEVICE if device else MEM_HOST,
                                                 C.byref(params), C.byref(policy), float(entropy_ratio_thresh), _ptr(rel), _ptr(kind),
                                                 _ptr(reason), _ptr(glob), _ptr(rel_cov), _ptr(glob_cov), _ptr(ratio)),
              "dvo_run_sequences_entropy")
        return rel, kind, reason, glob, rel_cov, glob_cov, ratio

    def pose_covariance(self, count, params, first=0, level=-1):
        """6x6 covariance of the pose the last solve left in slots [first, first+count), evaluated on the resident frames
        (dvo_pose_covariance): returns (cov (count, 6, 6), info array of CovInfo).  level = -1: finest level with iterations."""
        cov = np.empty((count, 6, 6), np.float64)
        info = (CovInfo * max(count, 1))()
        check(self.lib.dvo_pose_covariance(self.h, first, count, C.byref(params), level, _ptr(cov), C.cast(info, C.c_void_p), MEM_HOST),
              "dvo_pose_covariance")
        return cov, info

    def pose_covariance_device(self, count, params, cov_ptr, first=0, level=-1, info_ptr=None):
        """dvo_pose_covariance into device memory (count x 36 doubles at cov_ptr; optional count dvo_cov_info at info_ptr), asynchronous on
        the context stream."""
        check(self.lib.dvo_pose_covariance(self.h, first, count, C.byref(params), level, C.c_void_p(cov_ptr),
                                           C.c_void_p(info_ptr) if info_ptr else None, MEM_DEVICE), "dvo_pose_covariance")

    def load_frames(self, gray, depth, first=0, device=False, count=None):
        """Load n frames into BOTH roles of slots [first, first+n) -- reference and now get the same images -- then build_pyramids(3)
        and prepare(3), so that every one of these slots can serve as either side of align_pairs.  gray (n, H, W) u8 and depth
        (n, H, W) u16 numpy arrays, or with device=True raw device pointers and `count`."""
        if not device:
            gray = np.ascontiguousarray(gray, np.uint8)
            depth = np.ascontiguousarray(depth, np.uint16)
            count = gray.shape[0]
        for frame in (FRAME_REF, FRAME_NOW):
            self.set_frames(frame, gray, depth, first=first, count=count, device=device)
        self.build_pyramids(count, first=first, frames_mask=3)
        self.prepare(count, first=first, frames_mask=3)

    def align_pairs(self, ref_slots, now_slots, params, pose0=None, covariance=False, device=False):
        """dvo_align_pairs: pair k aligns the reference data of slot ref_slots[k] against the now data of slot now_slots[k], both
        already prepared (see load_frames).  Returns (poses (n, 12), info), plus (cov (n, 6, 6), cov_info) when covariance=True.
        Host (device=False): index sequences and pose0 ((n, 12) or None = identity) on the host; numpy poses / cov and ctypes
        arrays of PairInfo / CovInfo.  device=True: int32 CUDA tensors of indices and a float64 CUDA tensor pose0; the results are
        CUDA tensors -- poses, cov, and the raw info / cov_info records as uint8 (n, record size), see `records` -- written
        asynchronously on the context stream (synchronize() before reading them).  Out-of-range device indices give info status
        bit 1 and NaN poses; on the host they raise."""
        if device:
            import torch
            n = int(ref_slots.shape[0])
            dev = ref_slots.device
            poses = torch.empty((n, 12), dtype=torch.float64, device=dev)
            info = torch.empty((n, C.sizeof(PairInfo)), dtype=torch.uint8, device=dev)
            cov = torch.empty((n, 6, 6), dtype=torch.float64, device=dev) if covariance else None
            cinfo = torch.empty((n, C.sizeof(CovInfo)), dtype=torch.uint8, device=dev) if covariance else None
            ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
            check(self.lib.dvo_align_pairs(self.h, n, ptr(ref_slots), ptr(now_slots), ptr(pose0), C.byref(params), ptr(poses), ptr(info),
                                           ptr(cov), ptr(cinfo), MEM_DEVICE), "dvo_align_pairs")
        else:
            ref_slots = np.ascontiguousarray(ref_slots, np.int32)
            now_slots = np.ascontiguousarray(now_slots, np.int32)
            n = ref_slots.shape[0]
            if now_slots.shape[0] != n:
                raise ValueError("ref_slots and now_slots differ in length")
            if pose0 is not None:
                pose0 = np.ascontiguousarray(pose0, np.float64).reshape(n, 12)
            poses = np.empty((n, 12), np.float64)
            info = (PairInfo * max(n, 1))()
            cov = np.empty((n, 6, 6), np.float64) if covariance else None
            cinfo = (CovInfo * max(n, 1))() if covariance else None
            check(self.lib.dvo_align_pairs(self.h, n, _ptr(ref_slots), _ptr(now_slots), _ptr(pose0), C.byref(params), _ptr(poses),
                                           C.cast(info, C.c_void_p), _ptr(cov), C.cast(cinfo, C.c_void_p) if covariance else None,
                                           MEM_HOST), "dvo_align_pairs")
        return (poses, info, cov, cinfo) if covariance else (poses, info)

    def level_dims(self, level):
        w, h = C.c_int(), C.c_int()
        check(self.lib.dvo_level_dims(self.h, level, C.byref(w), C.byref(h)), "dvo_level_dims")
        return w.value, h.value

    def get_level_buffer(self, slot, frame, level, which):
        code, dt = BUF[which]
        w, h = self.level_dims(level)
        out = np.empty((h, w), dt)
        check(self.lib.dvo_get_level_buffer(self.h, slot, frame, level, code, _ptr(out), out.nbytes), "dvo_get_level_buffer")
        return out

    def get_points(self, slot, level):
        w, h = self.level_dims(level)
        cap = w * h
        X, Y, Z = (np.empty(cap, np.float32) for _ in range(3))
        n = C.c_int()
        check(self.lib.dvo_get_points(self.h, slot, level, _ptr(X), _ptr(Y), _ptr(Z), cap, C.byref(n)), "dvo_get_points")
        return X[: n.value].copy(), Y[: n.value].copy(), Z[: n.value].copy()

    def eval_normal_equations(self, slot, level, R, T, jacobian=JAC_REFERENCE, weight=W_REF_CAUCHY, arithmetic=ARITH_EXACT,
                              huber_k=1.345, per_point=False, npts=None, residual=RES_DT_FLOOR):
        pose = np.concatenate([np.asarray(R, np.float64).reshape(9), np.asarray(T, np.float64).reshape(3)])
        H = np.empty(36, np.float64)
        g = np.empty(6, np.float64)
        sumsq, nvis = C.c_double(), C.c_int()
        pp = {}
        if per_point:
            pp = {"eps": np.zeros(npts, np.float32), "w": np.zeros(npts, np.float32), "u": np.zeros(npts, np.float32),
                  "v": np.zeros(npts, np.float32), "J": np.zeros((npts, 6), np.float32)}
        prm = solver_params(jacobian=jacobian, weight=weight, arithmetic=arithmetic, huber_k=huber_k, residual=residual)
        check(self.lib.dvo_eval_normal_equations_ex(self.h, slot, level, _ptr(pose), C.byref(prm), _ptr(H), _ptr(g),
                                                    C.byref(sumsq), C.byref(nvis), _ptr(pp.get("eps")), _ptr(pp.get("w")),
                                                    _ptr(pp.get("u")), _ptr(pp.get("v")), _ptr(pp.get("J"))), "dvo_eval_normal_equations_ex")
        out = {"H": H.reshape(6, 6), "g": g, "sumsq": sumsq.value, "nvis": nvis.value}
        out.update(pp)
        return out

    def get_trace(self, slot, level):
        n = self.cfg.trace_iters
        tr = np.zeros((n, 56), np.float64)
        check(self.lib.dvo_get_trace(self.h, slot, level, _ptr(tr)), "dvo_get_trace")
        return {"g": tr[:, 0:6], "H": tr[:, 6:42].reshape(n, 6, 6), "energy": tr[:, 42], "nvis": tr[:, 43],
                "R": tr[:, 44:53].reshape(n, 3, 3), "T": tr[:, 53:56]}

    def get_energies(self, slot, level, n=128):
        out = np.zeros(n, np.float32)
        check(self.lib.dvo_get_energies(self.h, slot, level, _ptr(out), n), "dvo_get_energies")
        return out

    def enable_timing(self, on=True):
        check(self.lib.dvo_enable_timing(self.h, int(on)), "dvo_enable_timing")

    def stage_ms(self):
        ms = (C.c_float * len(_lib.STAGES))()
        check(self.lib.dvo_get_stage_ms(self.h, ms), "dvo_get_stage_ms")
        return dict(zip(_lib.STAGES, list(ms)))

    def launch_count(self):
        return int(self.lib.dvo_launch_count(self.h))

    def gop_compose(self, kind, rel):
        kind = np.ascontiguousarray(kind, np.int32)
        nseq, nframes = kind.shape
        rel = np.ascontiguousarray(rel, np.float64).reshape(nseq, nframes, 12)
        out = np.empty((nseq, nframes, 19), np.float64)
        check(self.lib.dvo_gop_compose(self.h, nseq, nframes, _ptr(kind), _ptr(rel), _ptr(out), MEM_HOST), "dvo_gop_compose")
        return out

    def optimize_pose_graph(self, edge_ref, edge_now, meas, cov, poses0, max_lag, max_iterations=100, lambda0=1e-4, rel_tol=1e-10,
                            marginals=False, device=False):
        """dvo_pose_graph_optimize: G graphs of N nodes and E edges each; edge e of graph k constrains G_b = G_a Z with covariance
        cov, a = edge_ref[k, e], b = edge_now[k, e], 1 <= |a - b| <= max_lag <= 8; node 0 stays at its input pose.
        Shapes: edge_ref / edge_now (G, E), meas (G, E, 12), cov (G, E, 6, 6), poses0 (G, N, 12).  Returns (poses, info) or, with
        marginals=True, (poses, info, node_cov (G, N, 6, 6)).  Host (device=False): numpy arrays and a ctypes array of PgoInfo;
        bad edge indices raise.  device=True: int32 / float64 CUDA tensors in, CUDA tensors out (info as raw uint8 records for
        `records(raw, PgoInfo)`), asynchronous on the context stream; bad indices give info status bit 0."""
        prm = PgoParams(int(max_iterations), float(lambda0), float(rel_tol))
        if device:
            import torch
            G, E = int(edge_ref.shape[0]), int(edge_ref.shape[1])
            N = int(poses0.shape[1])
            dev = poses0.device
            poses = poses0.detach().clone().contiguous()
            info = torch.empty((G, C.sizeof(PgoInfo)), dtype=torch.uint8, device=dev)
            ncov = torch.empty((G, N, 6, 6), dtype=torch.float64, device=dev) if marginals else None
            ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
            check(self.lib.dvo_pose_graph_optimize(self.h, G, N, E, int(max_lag), ptr(edge_ref.contiguous()), ptr(edge_now.contiguous()),
                                                   ptr(meas.contiguous()), ptr(cov.contiguous()), ptr(poses), C.byref(prm), ptr(ncov),
                                                   ptr(info), MEM_DEVICE), "dvo_pose_graph_optimize")
        else:
            edge_ref = np.ascontiguousarray(edge_ref, np.int32)
            edge_now = np.ascontiguousarray(edge_now, np.int32)
            G, E = edge_ref.shape
            poses = np.array(poses0, np.float64, order="C", copy=True)
            N = poses.shape[1]
            if edge_now.shape != (G, E) or poses.shape != (G, N, 12):
                raise ValueError("edge_now must be (G, E) like edge_ref and poses0 (G, N, 12)")
            meas = np.ascontiguousarray(meas, np.float64).reshape(G, E, 12)
            cov = np.ascontiguousarray(cov, np.float64).reshape(G, E, 6, 6)
            info = (PgoInfo * max(G, 1))()
            ncov = np.empty((G, N, 6, 6), np.float64) if marginals else None
            check(self.lib.dvo_pose_graph_optimize(self.h, G, N, E, int(max_lag), _ptr(edge_ref), _ptr(edge_now), _ptr(meas), _ptr(cov),
                                                   _ptr(poses), C.byref(prm), _ptr(ncov), C.cast(info, C.c_void_p), MEM_HOST),
                  "dvo_pose_graph_optimize")
        return (poses, info, ncov) if marginals else (poses, info)
