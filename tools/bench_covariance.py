"""Cost of the pose covariance (dvo_pose_covariance, dvo_run_sequences_cov) on seeded synthetic data generated as bench.py does.

  config 2  1024 pairs 640x480x4, GN 10 it/level: a dvo_process step with and without a following dvo_pose_covariance (device
            output), alternated in one run, plus the covariance pass alone on the solved batch;
  config 4  148 sequences x 8 frames of 1280x720, 5 levels, SUBGRAD_REF 50 it/level: dvo_run_sequences_mem against
            dvo_run_sequences_cov (device-resident inputs), alternated;
  entropy   the same config 4 workload: dvo_run_sequences_cov, dvo_run_sequences_entropy with the gate disabled and with a
            threshold at which some sequences switch (the median of the ratios an enabled, never-firing gate reports),
            alternated.

--configs picks the arms (default: 2,4).

CUDA events on the context's stream, warm-up first.  The card name and power limit are read in the same run.  Writes one JSON
file (--out) and prints it.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle_lib as O  # noqa: E402
import rgbd_odometry_b200 as dvo  # noqa: E402


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                 # the query is informational; the timings stand without it
        out["power_limit"] = f"unavailable ({e})"
    return out


def timed(stream, fn, n, finish=None):
    """ms per call of n calls of fn between two events on the launching stream; finish() makes that stream wait for all their work."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(n):
        fn()
    if finish:
        finish()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def config2(args, stream):
    W, H, L, K, B = 640, 480, 4, O.K640, args.pairs
    d = O.synth_batch(0, B, W, H, K, nthreads=os.cpu_count() or 1)
    al = dvo.BatchAligner(W, H, L, max_batch=B, intrinsics=K)
    al.set_stream(stream.cuda_stream)
    prm = dvo.solver_params(solver=dvo.GN, iters=(10,) * L)
    al.set_frames(dvo.FRAME_REF, d["ref_gray"], d["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, d["now_gray"], None)
    poses = torch.empty((B, 12), dtype=torch.float64, device="cuda")
    cov = torch.empty((B, 36), dtype=torch.float64, device="cuda")

    def step():
        al.process(B, prm, poses_out=poses.data_ptr())

    def step_cov():
        al.process(B, prm, poses_out=poses.data_ptr())
        al.pose_covariance_device(B, prm, cov.data_ptr())

    def finish():
        al.join()

    for _ in range(args.warmup):
        step(); step_cov()
    finish()
    plain, withcov = [], []
    for _ in range(args.rounds):                                   # alternated: A, B, A, B, ...
        plain.append(timed(stream, step, args.steps, finish))
        withcov.append(timed(stream, step_cov, args.steps, finish))
    al.synchronize()
    alone = [timed(stream, lambda: al.pose_covariance_device(B, prm, cov.data_ptr()), args.steps) for _ in range(args.rounds)]
    _, info = al.get_poses(B)
    _, cinfo = al.pose_covariance(B, prm)
    npts0 = int(sum(info[i].npts[0] for i in range(B)))
    ms_alone = float(np.median(alone))
    al.close()
    return {"workload": f"{B} synthetic pairs 640x480x4 (seeds 0..{B - 1}), GN 10 it/level, dvo_process on resident frames",
            "step_ms_median": float(np.median(plain)), "step_with_cov_ms_median": float(np.median(withcov)),
            "step_overhead_ms": float(np.median(withcov) - np.median(plain)),
            "step_overhead_frac": float((np.median(withcov) - np.median(plain)) / np.median(plain)),
            "cov_pass_ms_per_launch_median": ms_alone, "cov_pass_ms_per_1024_pairs": ms_alone * 1024 / B,
            "step_ms_rounds": plain, "step_with_cov_ms_rounds": withcov, "cov_pass_ms_rounds": alone,
            "level0_points": npts0, "algorithmic_bytes": 20 * npts0,
            "algorithmic_gbs": 20 * npts0 / (ms_alone * 1e-3) / 1e9,
            "cov_status_nonzero": int(sum(cinfo[i].status != 0 for i in range(B))),
            "note": "the step with the covariance joins dvo_process's internal streams before the covariance launch, so the "
                    "next step's preprocessing no longer overlaps the previous step's second-half solve"}


def config4(args, stream):
    W, H, L, K = 1280, 720, 5, O.K1280
    nseq, nframes = args.sequences, args.seq_frames
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        seqs = list(ex.map(lambda s: O.synth_sequence(700000 + s, nframes, W, H, K, max_angle_deg=0.4, max_trans_m=0.008), range(nseq)))
    gray = torch.from_numpy(np.stack([s[0] for s in seqs])).cuda()
    depth = torch.from_numpy(np.stack([s[1] for s in seqs]).view(np.int16)).cuda()
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K)
    al.set_stream(stream.cuda_stream)
    prm = dvo.solver_params(iters=(50,) * L)
    pol = dvo.keyframe_policy()
    run = lambda: al.run_sequences_mem(gray.data_ptr(), depth.data_ptr(), nseq, nframes, prm, pol, device=True)
    run_cov = lambda: al.run_sequences_cov(gray.data_ptr(), depth.data_ptr(), nseq, nframes, prm, pol, device=True)
    a, b = run(), run_cov()
    same = all(np.array_equal(x, y) for x, y in zip(a, b[:4]))
    plain, withcov = [], []
    for _ in range(args.rounds):
        plain.append(timed(stream, run, 1))
        withcov.append(timed(stream, run_cov, 1))
    al.close()
    fp = nseq * (nframes - 1)
    return {"workload": f"{nseq} synthetic sequences x {nframes} frames 1280x720, 5 levels, SUBGRAD_REF 50 it/level, key frame every 5, "
                        "device-resident inputs", "run_ms_median": float(np.median(plain)), "run_cov_ms_median": float(np.median(withcov)),
            "overhead_ms": float(np.median(withcov) - np.median(plain)),
            "overhead_frac": float((np.median(withcov) - np.median(plain)) / np.median(plain)),
            "frame_pairs_per_s": fp / (np.median(plain) * 1e-3), "frame_pairs_per_s_with_cov": fp / (np.median(withcov) * 1e-3),
            "run_ms_rounds": plain, "run_cov_ms_rounds": withcov, "records_bit_identical": bool(same)}


def entropy(args, stream):
    W, H, L, K = 1280, 720, 5, O.K1280
    nseq, nframes = args.sequences, args.seq_frames
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        seqs = list(ex.map(lambda s: O.synth_sequence(700000 + s, nframes, W, H, K, max_angle_deg=0.4, max_trans_m=0.008), range(nseq)))
    gray = torch.from_numpy(np.stack([s[0] for s in seqs])).cuda()
    depth = torch.from_numpy(np.stack([s[1] for s in seqs]).view(np.int16)).cuda()
    al = dvo.BatchAligner(W, H, L, max_batch=nseq, keep_now_depth=True, intrinsics=K)
    al.set_stream(stream.cuda_stream)
    prm = dvo.solver_params(iters=(50,) * L)
    pol = dvo.keyframe_policy()
    ent = lambda thr: al.run_sequences_entropy(gray.data_ptr(), depth.data_ptr(), nseq, nframes, prm, pol, thr, device=True)
    probe = ent(1e-300)                                              # enabled, never fires: the ratios of the shipped schedule
    thr = float(np.median(probe[6][np.isfinite(probe[6])]))
    run_cov = lambda: al.run_sequences_cov(gray.data_ptr(), depth.data_ptr(), nseq, nframes, prm, pol, device=True)
    run_off = lambda: ent(0.0)
    run_on = lambda: ent(thr)
    a, b, c = run_cov(), run_off(), run_on()
    off_same = all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b[:6])) and bool(np.isnan(b[6]).all())
    kind, reason = c[1], c[2]
    n0 = al.launch_count(); run_cov(); n1 = al.launch_count(); run_off(); n2 = al.launch_count(); run_on(); n3 = al.launch_count()
    t_cov, t_off, t_on = [], [], []
    for _ in range(args.rounds):                                     # alternated: cov, off, on, cov, off, on, ...
        t_cov.append(timed(stream, run_cov, 1))
        t_off.append(timed(stream, run_off, 1))
        t_on.append(timed(stream, run_on, 1))
    al.close()
    med = lambda v: float(np.median(v))
    return {"workload": f"{nseq} synthetic sequences x {nframes} frames 1280x720, 5 levels, SUBGRAD_REF 50 it/level, key frame every 5, "
                        "device-resident inputs", "entropy_ratio_thresh": thr,
            "sequences_switched_by_entropy": int(((kind == 2) & (reason == 6)).any(axis=1).sum()),
            "entropy_switches": int(((kind == 2) & (reason == 6)).sum()), "periodic_switches": int(((kind == 2) & (reason == 5)).sum()),
            "run_cov_ms_median": med(t_cov), "run_entropy_off_ms_median": med(t_off), "run_entropy_on_ms_median": med(t_on),
            "entropy_on_overhead_ms": med(t_on) - med(t_cov), "entropy_on_overhead_frac": (med(t_on) - med(t_cov)) / med(t_cov),
            "launches_cov": n1 - n0, "launches_entropy_off": n2 - n1, "launches_entropy_on": n3 - n2,
            "run_cov_ms_rounds": t_cov, "run_entropy_off_ms_rounds": t_off, "run_entropy_on_ms_rounds": t_on,
            "disabled_records_bit_identical_to_cov": bool(off_same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--sequences", type=int, default=148)
    ap.add_argument("--seq-frames", type=int, default=8)
    ap.add_argument("--configs", default="2,4", help="comma-separated arms: 2, 4, entropy")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_covariance.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_covariance needs a CUDA device")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    t0 = time.time()
    arms = {"2": ("config2", config2), "4": ("config4", config4), "entropy": ("entropy", entropy)}
    res = {"card": card()}
    for a in args.configs.split(","):
        name, fn = arms[a.strip()]
        res[name] = fn(args, stream)
    res["seconds"] = time.time() - t0
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
