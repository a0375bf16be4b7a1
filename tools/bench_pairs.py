"""Windowed odometry on device-resident frames: every frame t >= 1 of one seeded synthetic 640x480 sequence is aligned against
each of its k predecessors (reference t - j, now t, j = 1..k), 4 levels, GN 10 it/level, EXACT arithmetic.

  arm A  the per-slot path: the pairs become resident in batches of max_batch slots by device-to-device dvo_set_frames copies
         (one copy per role and image plane for each run of consecutive frames), and dvo_process prepares and solves each batch;
  arm B  load_frames once (every frame in both roles of its own slot, pyramids, Canny, EDT, texels), then one dvo_align_pairs
         over all pairs, without and with covariance.  B_pairs times the dvo_align_pairs call alone.

The poses of A and B must be bit-identical (same thread shape per pair: both contexts have max_batch > SM count) before any
time is reported.  CUDA events on one stream, warm-up first, arms alternated round by round.  The card name and power limit are
read in the same run.  Writes one JSON file (--out) and prints it.  Needs a CUDA device.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle_lib as O  # noqa: E402
import rgbd_odometry_b200 as dvo  # noqa: E402
from bench_covariance import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--window", type=int, default=4)
    ap.add_argument("--batch", type=int, default=1024, help="max_batch of the per-slot context (arm A)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_pairs.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pairs needs a CUDA device")
    t0 = time.time()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    W, H, L, K, F, k = 640, 480, 4, O.K640, args.frames, args.window
    g, d, _, _ = O.synth_sequence(9000, F, W, H, K)
    gray, depth = torch.from_numpy(g).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
    P0 = W * H
    # pairs ordered by lag: for lag j the reference frames j.. are the run 0..F-1-j and the now frames the run j..F-1
    pairs = [(t - j, t) for j in range(1, k + 1) for t in range(j, F)]
    n = len(pairs)
    ref = torch.tensor([a for a, _ in pairs], dtype=torch.int32, device="cuda")
    now = torch.tensor([b for _, b in pairs], dtype=torch.int32, device="cuda")
    prm = dvo.solver_params(solver=dvo.GN, iters=(10,) * L)

    B = args.batch
    A = dvo.BatchAligner(W, H, L, max_batch=B, intrinsics=K)
    A.set_stream(stream.cuda_stream)
    poses_a = torch.empty((n, 12), dtype=torch.float64, device="cuda")
    batches = []                                             # per batch: (first pair, count, [(slot, ref frame, now frame, length)])
    for s in range(0, n, B):
        m = min(B, n - s)
        runs, q = [], 0
        while q < m:
            r0, n0 = pairs[s + q]
            ln = 1
            while q + ln < m and pairs[s + q + ln] == (r0 + ln, n0 + ln):
                ln += 1
            runs.append((q, r0, n0, ln)); q += ln
        batches.append((s, m, runs))

    def step_a():                                            # pose0 stays the identity dvo_create put there
        for s, m, runs in batches:
            for slot, r0, n0, ln in runs:
                A.set_frames(dvo.FRAME_REF, gray.data_ptr() + r0 * P0, depth.data_ptr() + 2 * r0 * P0, first=slot, count=ln, device=True)
                A.set_frames(dvo.FRAME_NOW, gray.data_ptr() + n0 * P0, None, first=slot, count=ln, device=True)
            A.process(m, prm, poses_out=poses_a.data_ptr() + 8 * 12 * s)
        A.join()

    Bc = dvo.BatchAligner(W, H, L, max_batch=F, intrinsics=K)
    Bc.set_stream(stream.cuda_stream)
    out = {}

    def load_b():
        Bc.load_frames(gray.data_ptr(), depth.data_ptr(), device=True, count=F)

    def pairs_b(cov=False):
        out["r"] = Bc.align_pairs(ref, now, prm, covariance=cov, device=True)

    load_b()
    step_a(); pairs_b(True)
    torch.cuda.synchronize()
    pa, pb = poses_a.cpu().numpy(), out["r"][0].cpu().numpy()
    identical = bool(np.array_equal(pa.view(np.uint64), pb.view(np.uint64)))
    info_b = dvo.records(out["r"][1], dvo.PairInfo)
    cinfo_b = dvo.records(out["r"][3], dvo.CovInfo)
    if not identical:
        raise SystemExit(f"poses of arm A and arm B differ in {int((pa != pb).any(axis=1).sum())} of {n} pairs: no time is reported")

    arms = {"A_per_slot": step_a, "B_load_and_pairs": lambda: (load_b(), pairs_b(False)),
            "B_load_and_pairs_cov": lambda: (load_b(), pairs_b(True)), "B_pairs": lambda: pairs_b(False),
            "B_pairs_cov": lambda: pairs_b(True), "B_load": load_b}
    for _ in range(args.warmup):
        for fn in arms.values():
            fn()
    rounds = {a: [] for a in arms}
    for _ in range(args.rounds):
        for a, fn in arms.items():
            rounds[a].append(timed(stream, fn, args.steps))
    A.close(); Bc.close()
    med = {a: float(np.median(v)) for a, v in rounds.items()}
    res = {"card": card(),
           "workload": f"one synthetic 640x480 sequence of {F} frames (seed 9000), every frame t >= 1 against its {k} predecessors: {n} "
                       f"pairs, 4 levels, GN 10 it/level, EXACT arithmetic, device-resident frames; arm A context max_batch {B}, "
                       f"arm B context max_batch {F} (both 256 threads per pair)",
           "pairs": n, "poses_bit_identical_A_B": identical,
           "pair_status_nonzero": int(sum(r.status != 0 for r in info_b)), "cov_status_nonzero": int(sum(r.status != 0 for r in cinfo_b)),
           "ms_median": med, "ms_rounds": rounds,
           "speedup_A_over_B_load_and_pairs": med["A_per_slot"] / med["B_load_and_pairs"],
           "steps_per_round": args.steps, "rounds": args.rounds, "seconds": time.time() - t0}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
