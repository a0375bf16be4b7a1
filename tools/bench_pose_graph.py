"""Windowed pose-graph optimisation on the device (dvo_pose_graph_optimize), two workloads:

  (a) the bench_pairs workload: one synthetic 640x480 sequence of 1024 frames, every frame t >= 1 against its 4 predecessors (4086
      pairs, GN 10 it/level, 4 levels, covariances), device-resident.  The lag-1 poses chained through dvo_gop_compose are the
      initial guess of one 1024-node graph over all 4086 edges (max_lag 4).  Times the optimiser call alone, without and with
      marginals, next to the dvo_align_pairs call (with covariances) that produced its input, in the same run; reports the
      trajectory error (RMS translation against the renderer's ground truth, frame 0 aligned) of the chain and of the optimum,
      and the agreement of the device result with the CPU oracle.
  (b) synthetic graphs without images: 148 graphs x 64 nodes, lag 4 (forward edges of lag 1..4, backward of lag 1..2, duplicated
      lag-1 edges, 5% NaN covariances), one call, without and with marginals.

CUDA events on one stream, warm-up first, arms alternated round by round; the card name and power limit are read in the same
run.  Writes one JSON file (--out) and prints it.  Needs a CUDA device.
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
import pgo_oracle_lib as PG  # noqa: E402
import rgbd_odometry_b200 as dvo  # noqa: E402
from bench_covariance import card, timed  # noqa: E402
from test_pose_graph import compose, inverse, make_graphs, pose_err  # noqa: E402

PRM = dict(max_iterations=100, lambda0=1e-4, rel_tol=1e-10)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--window", type=int, default=4)
    ap.add_argument("--graphs", type=int, default=148)
    ap.add_argument("--nodes", type=int, default=64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_pose_graph.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pose_graph needs a CUDA device")
    t0 = time.time()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).cuda()  # noqa: E731
    f64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()  # noqa: E731

    # ---- (a) windowed odometry constraints of a 1024-frame sequence
    W, H, L, K, F, k = 640, 480, 4, O.K640, args.frames, args.window
    g, d, Rg, Tg = O.synth_sequence(9000, F, W, H, K)
    gray, depth = torch.from_numpy(g).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
    pairs = [(t - j, t) for j in range(1, k + 1) for t in range(j, F)]
    n = len(pairs)
    ref, now = i32([a for a, _ in pairs]), i32([b for _, b in pairs])
    prm = dvo.solver_params(solver=dvo.GN, iters=(10,) * L)
    al = dvo.BatchAligner(W, H, L, max_batch=F, intrinsics=K)
    al.set_stream(stream.cuda_stream)
    al.load_frames(gray.data_ptr(), depth.data_ptr(), device=True, count=F)
    out = {}

    def pairs_cov():
        out["pairs"] = al.align_pairs(ref, now, prm, covariance=True, device=True)

    pairs_cov()
    al.synchronize()
    poses, _, cov, cinfo = out["pairs"]
    rel = np.tile(np.eye(3).reshape(9).tolist() + [0.0] * 3, (1, F, 1))
    rel[0, 1:] = poses[:F - 1].cpu().numpy()                       # the lag-1 pairs come first: (t - 1, t) for t = 1..F-1
    chain = al.gop_compose(np.ones((1, F), np.int32), rel)[:, :, :12]
    eref, enow, emeas, ecov, x0 = ref[None], now[None], poses[None].contiguous(), cov[None].contiguous(), f64(chain)

    def opt_a(marg):
        out["a"] = al.optimize_pose_graph(eref, enow, emeas, ecov, x0, k, marginals=marg, device=True, **PRM)

    opt_a(True)
    al.synchronize()
    Pa = out["a"][0].cpu().numpy()
    Ia = dvo.records(out["a"][1], dvo.PgoInfo)[0]
    Xo, Io, _ = PG.pose_graph(ref.cpu().numpy()[None], now.cpu().numpy()[None], emeas.cpu().numpy(), ecov.cpu().numpy(), chain, k, **PRM)
    ang, tr = pose_err(Pa[0], Xo[0])
    gt = np.stack([np.concatenate([Rg[i].reshape(9), Tg[i]]) for i in range(F)])
    gt = np.stack([compose(inverse(gt[0]), gt[i]) for i in range(F)])
    ate = lambda X: float(np.sqrt(np.mean(np.sum((X[:, 9:] - gt[:, 9:]) ** 2, axis=1))))  # noqa: E731

    # ---- (b) batched synthetic graphs
    bref, bnow, bmeas, bcov, bx0, bgt = make_graphs(6000, args.graphs, args.nodes, 4)
    tb = [i32(bref), i32(bnow), f64(bmeas), f64(bcov), f64(bx0)]

    def opt_b(marg):
        out["b"] = al.optimize_pose_graph(*tb, 4, marginals=marg, device=True, **PRM)

    opt_b(True)
    al.synchronize()
    Ib = dvo.records(out["b"][1], dvo.PgoInfo)
    Pb = out["b"][0].cpu().numpy()
    Xb, Iob, _ = PG.pose_graph(bref, bnow, bmeas, bcov, bx0, 4, **PRM)
    bang, btr = pose_err(Pb, Xb)

    arms = {"a_align_pairs_cov": pairs_cov, "a_optimize": lambda: opt_a(False), "a_optimize_marginals": lambda: opt_a(True),
            "b_optimize": lambda: opt_b(False), "b_optimize_marginals": lambda: opt_b(True)}
    for _ in range(args.warmup):
        for fn in arms.values():
            fn()
    rounds = {a: [] for a in arms}
    for _ in range(args.rounds):
        for a, fn in arms.items():
            rounds[a].append(timed(stream, fn, args.steps))
    al.close()
    med = {a: float(np.median(v)) for a, v in rounds.items()}
    res = {"card": card(),
           "workload_a": f"one synthetic 640x480 sequence of {F} frames (seed 9000), every frame t >= 1 against its {k} predecessors: {n} "
                         f"pairs with covariances (4 levels, GN 10 it/level); one graph of {F} nodes and {n} edges, max_lag {k}, "
                         f"initial guess the lag-1 chain; LM {PRM}",
           "workload_b": f"{args.graphs} synthetic graphs x {args.nodes} nodes, lag 4, {bref.shape[1]} edges each (make_graphs seed 6000); LM {PRM}",
           "a_info": {"status": Ia.status, "iterations": Ia.iterations, "accepted": Ia.accepted, "edges_used": Ia.edges_used,
                      "cost_initial": Ia.cost_initial, "cost_final": Ia.cost_final},
           "a_oracle": {"iterations": int(Io["iterations"][0]), "cost_final": float(Io["cost_final"][0]),
                        "max_rot_diff_rad": float(ang), "max_trans_diff_m": float(tr)},
           "a_pair_cov_status_nonzero": int(sum(c.status != 0 for c in dvo.records(cinfo, dvo.CovInfo))),
           "a_ate_m": {"lag1_chain": ate(chain[0]), "optimised": ate(Pa[0])},
           "b_status_nonzero": int(sum(i.status != 0 for i in Ib)), "b_iterations_max": int(max(i.iterations for i in Ib)),
           "b_oracle_max_rot_diff_rad": float(bang), "b_oracle_max_trans_diff_m": float(btr),
           "ms_median": med, "ms_rounds": rounds, "steps_per_round": args.steps, "rounds": args.rounds, "seconds": time.time() - t0}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
