"""Quick solve-stage timing at the bench workload (1024 pairs, or the batch size given as the first argument)."""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as O
import rgbd_odometry_b200 as dvo
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
d = O.synth_batch(0, B)
al = dvo.BatchAligner(640, 480, 4, max_batch=B)
al.set_frames(dvo.FRAME_REF, d["ref_gray"], d["ref_depth"]); al.set_frames(dvo.FRAME_NOW, d["now_gray"], None)
al.build_pyramids(B); al.prepare(B); al.synchronize()
def timed(params, reps=3):
    al.run(B, params); al.synchronize()
    al.enable_timing(True)
    for _ in range(reps): al.run(B, params)
    ms = al.stage_ms()["solve"] / reps
    al.enable_timing(False)
    return ms
out = []
for name, solver, it in (("gn10", dvo.GN, 10), ("subgrad50", dvo.SUBGRAD_REF, 50), ("gn10_L3only", dvo.GN, -1)):
    iters = (it,) * 4 if it > 0 else (0, 0, 0, 50)
    out.append(f"{name}={timed(dvo.solver_params(solver=solver, iters=iters)):.3f}ms")
print(B, " ".join(out))
