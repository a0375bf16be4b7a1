"""Every solve_kernel / solve_pairs_kernel instantiation against the CPU oracle, per iteration, at the precision the kernels reach.

The solver ships one template, solve_body<ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE, PAIRS>, instantiated for slots
(solve_kernel) and pairs (solve_pairs_kernel).  TABLE below names every instantiation and a context shape plus solver
parameters that reach it; the CPU test pins the table to the kernels compiled into libdvo_b200.so, so an instantiation added
later without a row fails the suite.

GPU checks (EXACT arithmetic unless a row says FAST):
  - NEED_H = true rows (a context that keeps a trace): at the pose the trace recorded for iteration i -- the pose the kernel
    evaluated, recorded before the step -- the oracle's nvis equals the kernel's, g and the upper triangle of H agree to 1e-12
    relative, the energy to 1e-12 relative.  GN: one oracle step from trace pose i lands on trace pose i + 1.  Every solver:
    the trajectory, best_index, iterations_run and final pose follow the oracle's align_pair.
  - NEED_H = false rows (sub-gradient without a trace, the shipped kernels): the energy of every iteration within 1 float32
    ulp of the oracle's, best_index / iterations_run exact, best_energy / visible_ratio within 1 ulp, the final pose close to the
    oracle's; also for truncated single-level schedules, and against the traced (NEED_H = true) kernel on the same pairs.
  - every row: a pair launch (solve_pairs_kernel) on the diagonal gives the slot launch's pose and info bit for bit.
  - point counts N on the sweeps' boundaries (partial warps, N < THREADS, ring prologue, k * THREADS +- 1), set exactly by
    keeping depth only at the first N reference edge pixels: the checks above plus dvo_pose_covariance (same sweep, WSQ);
    N = 0 gives status bit 0 and leaves the pose as it was.
The tolerances, and the worst cases measured on a B200 that set them, are listed with their constants below.
"""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import rgbd_odometry_b200 as dvo
from rgbd_odometry_b200 import build as dvo_build

K320 = (262.5, 262.5, 159.5, 119.5)
K160 = (131.25, 131.25, 79.5, 59.5)

# ------------------------------------------------------------------------------------------------ the instantiation table
# key = the template arguments (ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE) of solve_kernel / solve_pairs_kernel:
#   ARITH 0 EXACT / 1 FAST; JAC 0 REFERENCE / 1 EXACT; RES 0 DT_FLOOR / 1 DT_INTERP;
#   WMODE 0 = getWeightOf fixed at compile time, -1 = weight mode read at run time (Huber, none, or FAST / DT_INTERP);
#   PIPE = depth of the cp.async ring of the sweep, 0 = register pipeline (accumulate_points).
# shape: 512 = a context with max_batch <= 148 (the SM count), 256 = a larger one (dispatch: c->solve_shape); FAST arithmetic
# and DT_INTERP always take 256.  traced: the context keeps a trace (trace_iters > 0), which makes SUBGRAD need H; traced rows
# run GN, LM and SUBGRAD, untraced rows SUBGRAD (the only solver that runs without H).
W_HUBER, W_NONE = dvo.W_HUBER, dvo.W_NONE
FAST_ = dict(arithmetic=dvo.ARITH_FAST)
EXJ = dict(jacobian=dvo.JAC_EXACT)
INTERP = dict(residual=dvo.RES_DT_INTERP)
TABLE = [
    # (ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE)  shape traced  params
    ((0, 0, True, 512, 0, 0, 4),     512, True,  dict()),                          # GN / LM ship here at <= 148 pairs
    ((0, 0, True, 512, 0, -1, 0),    512, True,  dict(weight=W_HUBER)),
    ((0, 1, True, 512, 0, 0, 0),     512, True,  dict(**EXJ)),
    ((0, 1, True, 512, 0, -1, 0),    512, True,  dict(**EXJ, weight=W_NONE)),
    ((0, 0, False, 512, 0, 0, 2),    512, False, dict()),                          # the shipped sub-gradient kernel, <= 148 pairs
    ((0, 0, False, 512, 0, -1, 0),   512, False, dict(weight=W_NONE)),
    ((0, 1, False, 512, 0, 0, 0),    512, False, dict(**EXJ)),
    ((0, 1, False, 512, 0, -1, 0),   512, False, dict(**EXJ, weight=W_HUBER)),
    ((0, 0, True, 256, 0, 0, 4),     256, True,  dict()),                          # config 2 (GN at 1024 pairs)
    ((0, 0, True, 256, 0, -1, 0),    256, True,  dict(weight=W_NONE)),
    ((0, 1, True, 256, 0, 0, 0),     256, True,  dict(**EXJ)),
    ((0, 1, True, 256, 0, -1, 0),    256, True,  dict(**EXJ, weight=W_HUBER)),
    ((0, 0, False, 256, 0, 0, 2),    256, False, dict()),                          # the shipped sub-gradient kernel, config 4
    ((0, 0, False, 256, 0, -1, 0),   256, False, dict(weight=W_HUBER)),
    ((0, 1, False, 256, 0, 0, 0),    256, False, dict(**EXJ)),
    ((0, 1, False, 256, 0, -1, 0),   256, False, dict(**EXJ, weight=W_NONE)),
    ((1, 0, True, 256, 0, -1, 0),    256, True,  dict(**FAST_)),
    ((1, 1, True, 256, 0, -1, 0),    256, True,  dict(**FAST_, **EXJ, weight=W_HUBER)),
    ((1, 0, False, 256, 0, -1, 0),   256, False, dict(**FAST_)),
    ((1, 1, False, 256, 0, -1, 0),   256, False, dict(**FAST_, **EXJ, weight=W_NONE)),
    ((0, 0, True, 256, 1, -1, 0),    256, True,  dict(**INTERP)),
    ((0, 1, True, 256, 1, -1, 0),    256, True,  dict(**INTERP, **EXJ, weight=W_HUBER)),
    ((0, 0, False, 256, 1, -1, 0),   256, False, dict(**INTERP)),
    ((0, 1, False, 256, 1, -1, 0),   256, False, dict(**INTERP, **EXJ, weight=W_NONE)),
]
TRACED_SOLVERS = {"gn": dvo.GN, "lm": dvo.LM, "subgrad": dvo.SUBGRAD_REF}


def row_id(key):
    a, j, h, t, r, w, p = key
    return f"{'fast' if a else 'exact'}-{'jexact' if j else 'jref'}-{'H' if h else 'noH'}-{t}-{'interp' if r else 'floor'}-w{w}-pipe{p}"


def dispatch(shape, traced, p):
    """The template arguments dispatch_solve / launch_solve_t / launch_solve_inst / launch_solve_w (csrc/solver.cu) choose."""
    need_h = p.solver != dvo.SUBGRAD_REF or traced
    arith = dvo.ARITH_FAST if p.arithmetic == dvo.ARITH_FAST else dvo.ARITH_EXACT
    jac = dvo.JAC_EXACT if p.jacobian == dvo.JAC_EXACT else dvo.JAC_REFERENCE
    if p.residual == dvo.RES_DT_INTERP:
        assert arith == dvo.ARITH_EXACT, "DT_INTERP is built for EXACT arithmetic only"
        threads, res, wmode = 256, 1, -1
    else:
        threads = 512 if (arith == dvo.ARITH_EXACT and shape == 512) else 256
        res = 0
        wmode = 0 if (arith == dvo.ARITH_EXACT and p.weight == dvo.W_REF_CAUCHY) else -1
    pipe = (4 if need_h else 2) if (wmode == 0 and jac == dvo.JAC_REFERENCE) else 0
    return (arith, jac, need_h, threads, res, wmode, pipe)


def row_solvers(traced):
    return list(TRACED_SOLVERS.values()) if traced else [dvo.SUBGRAD_REF]


def test_table_rows_reach_their_instantiation():
    keys = [k for k, _, _, _ in TABLE]
    assert len(set(keys)) == len(keys) == 24
    for key, shape, traced, kw in TABLE:
        for solver in row_solvers(traced):
            assert dispatch(shape, traced, dvo.solver_params(solver=solver, **kw)) == key, (row_id(key), solver)


def compiled_solve_instances():
    """{kernel name: set of template-argument tuples} of the solve kernels in libdvo_b200.so's sm_100a code (cuobjdump of the
    toolkit that built the library, names demangled by its cu++filt)."""
    if not os.path.exists(dvo_build.LIB):
        pytest.fail(f"{dvo_build.LIB} is missing: build it first (python -m rgbd_odometry_b200.build)")
    bindir = os.path.dirname(os.path.realpath(dvo_build._nvcc()))
    tools = [os.path.join(bindir, t) for t in ("cuobjdump", "cu++filt")]
    for t in tools:
        if not os.path.exists(t):
            pytest.fail(f"{t} is missing: the solve-kernel coverage check needs the CUDA toolkit's cuobjdump and cu++filt")
    sym = subprocess.run([tools[0], "-symbols", "-arch", "sm_100a", dvo_build.LIB], capture_output=True, text=True, check=True).stdout
    mangled = sorted({ln.split()[-1] for ln in sym.splitlines() if "STO_ENTRY" in ln and "solve_" in ln})
    names = subprocess.run([tools[1]], input="\n".join(mangled) + "\n", capture_output=True, text=True, check=True).stdout.splitlines()
    out = {"solve_kernel": set(), "solve_pairs_kernel": set()}
    for n in names:
        m = re.search(r"::(solve_kernel|solve_pairs_kernel)<([^>]*)>\(", n)
        if not m:
            continue
        args = [re.sub(r"^\((?:int|bool)\)", "", a.strip()) for a in m.group(2).split(",")]
        vals = [a == "true" or a == "1" if i == 2 else int(a) for i, a in enumerate(args)]
        if args[2] not in ("0", "1", "true", "false"):
            pytest.fail(f"cannot parse the NEED_H argument of {n}")
        out[m.group(1)].add(tuple(vals))
    return out


def test_table_equals_compiled_solve_kernels():
    got = compiled_solve_instances()
    want = {k for k, _, _, _ in TABLE}
    for name, inst in got.items():
        assert inst, f"no {name} instantiation found in {dvo_build.LIB}"
        assert inst == want, (f"{name}: compiled but not in TABLE: {sorted(inst - want)}; in TABLE but not compiled: {sorted(want - inst)}")


# ------------------------------------------------------------------------------------------------ tolerances
# Measured on one B200 (1000 W power limit) over every test in this file (worst case, bound / worst in brackets):
#   per-iteration g / H at the kernel's pose, EXACT   1.3e-14 relative   (SUM_REL 1e-12, 78x)
#   per-iteration g / H, FAST vs the EXACT oracle     3.2e-7 relative    (FAST_REL 1e-5, the spec)
#   energies (trace, dvo_get_energies), best_energy,  0 ulp              (ULP_TOL 1)
#     visible_ratio
#   trajectories and final poses vs the oracle        5.4e-14 rad / m    (POSE_TOL 1e-11, 190x)
#   one GN step from the same pose                    2.8e-14            (STEP_TOL 1e-12, 36x)
#   NEED_H = false vs NEED_H = true kernel poses      1.4e-17            (GROUP_TOL 1e-14, 700x)
#   covariance: |Sigma H / sigma^2 - I| / cond(H)     6.6e-16            (COV_REL 1e-14, 15x); sigma^2 3e-16 relative
SUM_REL = 1e-12
FAST_REL = 1e-5
ULP_TOL = 1
POSE_TOL = 1e-11
STEP_TOL = 1e-12
GROUP_TOL = 1e-14
COV_REL = 1e-14


# ------------------------------------------------------------------------------------------------ helpers
def rot_angle(Ra, Rb):
    """Angle of Ra^T Rb from its skew part: accurate for the tiny angles compared here, where arccos of the trace bottoms out
    at ~2e-8 rad."""
    R = np.asarray(Ra).T @ np.asarray(Rb)
    v = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(v))))


def same(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


def ulps(a, b):
    """float32 ulp distance (non-negative values)."""
    a = np.atleast_1d(np.asarray(a, np.float32)).view(np.int32).astype(np.int64)
    b = np.atleast_1d(np.asarray(b, np.float32)).view(np.int32).astype(np.int64)
    return np.abs(a - b)


def ocfg(solver, kw):
    return O.cfg(solver, kw.get("jacobian", dvo.JAC_REFERENCE), kw.get("weight", dvo.W_REF_CAUCHY), kw.get("huber_k", 1.345),
                 kw.get("lm_lambda0", 1e-3), kw.get("residual", dvo.RES_DT_FLOOR))


class Frames:
    """A batch of pairs, the oracle's per-level data, and lazily created contexts holding them."""

    def __init__(self, d, W, H, L, K, shape):
        self.d, self.W, self.H, self.L, self.K, self.shape = d, W, H, L, K, shape
        self.n = d["ref_gray"].shape[0]
        self.ctx = {}
        self._lv = {}

    def context(self, traced):
        if traced not in self.ctx:
            mb = self.n if self.shape == 512 else 160
            assert (mb <= 148) == (self.shape == 512)
            al = dvo.BatchAligner(self.W, self.H, self.L, max_batch=mb, trace_iters=50 if traced else 0, intrinsics=self.K)
            al.set_frames(dvo.FRAME_REF, self.d["ref_gray"], self.d["ref_depth"])
            al.set_frames(dvo.FRAME_NOW, self.d["now_gray"], None)
            al.build_pyramids(self.n)
            al.prepare(self.n)
            self.ctx[traced] = al
        return self.ctx[traced]

    def level(self, s, l):
        if (s, l) not in self._lv:
            ref = O.preprocess_level(self.d["ref_gray"][s], self.d["ref_depth"][s], l)
            now = O.preprocess_level(self.d["now_gray"][s], None, l)
            X, Y, Z, _, _ = O.select_points(ref["edge"], ref["depth"], l, self.K)
            self._lv[(s, l)] = (X, Y, Z, now["dtn"], now["gx"], now["gy"])
        return self._lv[(s, l)]

    def evaluate(self, s, l, R, T, kw, per_point=False):
        X, Y, Z, dtn, gx, gy = self.level(s, l)
        return O.evaluate(X, Y, Z, dtn, gx, gy, l, R, T, K=self.K, jac=kw.get("jacobian", dvo.JAC_REFERENCE),
                          weight=kw.get("weight", dvo.W_REF_CAUCHY), huber_k=kw.get("huber_k", 1.345), per_point=per_point,
                          residual=kw.get("residual", dvo.RES_DT_FLOOR))

    def oracle(self, s, solver, kw, iters, pose0=None):
        R0, T0 = (None, None) if pose0 is None else (pose0[:9], pose0[9:])
        return O.align_pair(self.d["ref_gray"][s], self.d["ref_depth"][s], self.d["now_gray"][s], self.L, iters, K=self.K,
                            scfg=ocfg(solver, kw), R0=R0, T0=T0, trace=True)

    def close(self):
        for al in self.ctx.values():
            al.close()
        self.ctx = {}


def run(al, n, prm, pose0=None):
    al.set_initial_pose(n, pose0)
    al.run(n, prm)
    return al.get_poses(n)


def check_pair_launch(al, n, prm, poses, info, pose0=None):
    """solve_pairs_kernel on the diagonal (reference and now data of slot s) == the slot launch, bit for bit."""
    s = np.arange(n)
    pp, pi = al.align_pairs(s, s, prm, pose0=pose0)
    assert same(pp, poses), "pair launch pose differs from the slot launch"
    assert bytes(pi) == bytes(info), "pair launch info differs from the slot launch"


def check_sums_at_kernel_pose(F, s, l, tr, n, kw, tag):
    """Trace row i holds the sums the kernel reduced at trace pose i (the pose before the step): the oracle at that pose."""
    fast = kw.get("arithmetic", dvo.ARITH_EXACT) == dvo.ARITH_FAST
    rel = FAST_REL if fast else SUM_REL
    iu = np.triu_indices(6)
    for i in range(n):
        o = F.evaluate(s, l, tr["R"][i], tr["T"][i], kw)
        where = f"{tag} slot {s} L{l} iteration {i}"
        assert tr["nvis"][i] == o["nvis"], f"{where}: nvis {tr['nvis'][i]} vs oracle {o['nvis']}"
        gs, Hs = np.abs(o["g"]).max(), np.abs(o["H"][iu]).max()
        dg, dH = np.abs(tr["g"][i] - o["g"]).max(), np.abs(tr["H"][i][iu] - o["H"][iu]).max()
        assert dg <= rel * gs, f"{where}: g off by {dg:.3g} (scale {gs:.3g})"
        assert dH <= rel * Hs, f"{where}: H off by {dH:.3g} (scale {Hs:.3g})"
        e = np.float32(np.sqrt(o["sumsq"]))
        assert abs(tr["energy"][i] - e) <= SUM_REL * e, f"{where}: energy {tr['energy'][i]!r} vs oracle {e!r}"


def divergence(F, s, l, kw, gR, gT, oR, oT, n, tol):
    """None when the two trajectories agree to tol; otherwise where they first part and which point's texel differs there."""
    dev = np.maximum(np.abs(gR[:n] - oR[:n]).max(axis=(1, 2)), np.abs(gT[:n] - oT[:n]).max(axis=1))
    bad = np.nonzero(dev > tol)[0]
    if not len(bad):
        return None
    i = int(bad[0]); j = max(i - 1, 0)
    a = F.evaluate(s, l, gR[j], gT[j], kw, per_point=True)
    b = F.evaluate(s, l, oR[j], oT[j], kw, per_point=True)
    diff = np.nonzero((np.floor(a["u"]) != np.floor(b["u"])) | (np.floor(a["v"]) != np.floor(b["v"])) | (a["eps"] != b["eps"]))[0]
    msg = f"slot {s} L{l}: trajectories part at iteration {i} (deviation {dev[i]:.3g} > {tol:g})"
    if len(diff):
        k = int(diff[0])
        frac = min(abs(a["u"][k] - np.round(a["u"][k])), abs(a["v"][k] - np.round(a["v"][k])))
        msg += (f"; at iteration {j} {len(diff)} point(s) see another texel, first point {k}: kernel (u, v) = ({a['u'][k]!r}, "
                f"{a['v'][k]!r}), oracle ({b['u'][k]!r}, {b['v'][k]!r}), {frac:.2g} px from an integer")
    else:
        msg += f"; at iteration {j} every point sees the same texel at both poses: not a floor flip"
    return msg


def check_trajectory(F, s, info, gtr, o, iters, kw, tol, traced=True):
    """Trace poses (traced contexts), iterations_run and best_index against the oracle's align_pair."""
    for l in range(F.L):
        if iters[l] <= 0:
            continue
        n = int(info.iterations_run[l])
        if traced:
            m = min(n, int(o["iterations_run"][l]))
            gR, gT = gtr[l]["R"], gtr[l]["T"]
            oR, oT = o["trace"]["R"][l], o["trace"]["T"][l]
            msg = divergence(F, s, l, kw, gR, gT, oR, oT, m, tol)
            assert msg is None, msg
        assert n == o["iterations_run"][l], f"slot {s} L{l}: iterations_run {n} vs oracle {o['iterations_run'][l]}"
        assert info.best_index[l] == o["best_index"][l], f"slot {s} L{l}: best_index {info.best_index[l]} vs {o['best_index'][l]}"


def check_final_pose(pose, o, tol, tag):
    R, T = pose[:9].reshape(3, 3), pose[9:]
    dR, dT = rot_angle(R, o["R"]), float(np.linalg.norm(T - o["T"]))
    assert dR <= tol and dT <= tol, f"{tag}: final pose dR {dR:.3g} dT {dT:.3g} > {tol:g}"


# ------------------------------------------------------------------------------------------------ GPU fixtures
NP = 3


@pytest.fixture(scope="module")
def frames():
    """shape 512: 2 levels of 320x240; shape 256: a 160-slot context of 160x120 frames, the first NP slots in use."""
    out = {512: Frames(O.synth_batch(9100, NP, 320, 240, K320), 320, 240, 2, K320, 512),
           256: Frames(O.synth_batch(9200, NP, 160, 120, K160), 160, 120, 2, K160, 256)}
    yield out
    for F in out.values():
        F.close()


TRACED_ROWS = [(k, sh, kw) for k, sh, tr, kw in TABLE if tr]
UNTRACED_ROWS = [(k, sh, kw) for k, sh, tr, kw in TABLE if not tr]
TRACED_ITERS = {dvo.GN: (20, 20), dvo.LM: (20, 20), dvo.SUBGRAD_REF: (50, 50)}


@pytest.mark.gpu
@pytest.mark.parametrize("solver", list(TRACED_SOLVERS), ids=list(TRACED_SOLVERS))
@pytest.mark.parametrize("key,shape,kw", TRACED_ROWS, ids=[row_id(r[0]) for r in TRACED_ROWS])
def test_traced_rows_per_iteration(frames, key, shape, kw, solver):
    """NEED_H = true: per-iteration nvis / g / H / energy at the kernel's own pose, the GN step, and the whole trajectory.
    Measured on a B200: the trajectories (2 levels x 20 GN / LM or 50 sub-gradient iterations) stay within 5.4e-14 of the
    oracle's, one GN step within 2.8e-14 (see the tolerance table)."""
    F = frames[shape]
    sv = TRACED_SOLVERS[solver]
    iters = TRACED_ITERS[sv]
    prm = dvo.solver_params(solver=sv, iters=iters, **kw)
    al = F.context(True)
    poses, info = run(al, F.n, prm)
    fast = kw.get("arithmetic", dvo.ARITH_EXACT) == dvo.ARITH_FAST
    for s in range(F.n):
        assert info[s].status == 0
        gtr = [al.get_trace(s, l) for l in range(F.L)]
        for l in range(F.L):
            n = int(info[s].iterations_run[l])
            assert 0 < n <= 50
            check_sums_at_kernel_pose(F, s, l, gtr[l], n, kw, row_id(key))
            if sv == dvo.GN and not fast:
                X, Y, Z, dtn, gx, gy = F.level(s, l)
                for i in range(n - 1):
                    r = O.run_iterations(X, Y, Z, dtn, gx, gy, l, 2, R0=gtr[l]["R"][i], T0=gtr[l]["T"][i], K=F.K, scfg=ocfg(sv, kw), trace=True)
                    assert r["iterations_run"] == 2, f"slot {s} L{l} iteration {i}: the oracle stops where the kernel steps on"
                    d = max(np.abs(r["trace"]["R"][1] - gtr[l]["R"][i + 1]).max(), np.abs(r["trace"]["T"][1] - gtr[l]["T"][i + 1]).max())
                    assert d <= STEP_TOL, f"slot {s} L{l}: GN step from trace pose {i} misses trace pose {i + 1} by {d:.3g}"
        o = F.oracle(s, sv, kw, iters)
        if fast:
            check_final_pose(poses[s], o, 1e-5, "fast")
        else:
            check_trajectory(F, s, info[s], gtr, o, iters, kw, POSE_TOL)
            check_final_pose(poses[s], o, POSE_TOL, "traced")
    check_pair_launch(al, F.n, prm, poses, info)


def check_untraced_against_oracle(F, s, pose, info, kw, iters, pose0=None, tag="untraced"):
    """NEED_H = false: energies per iteration within 1 ulp, best_index / iterations_run exact, best_energy / visible_ratio within
    1 ulp, final pose within POSE_TOL of the oracle run from the same pose0."""
    al = F.context(False)
    o = F.oracle(s, dvo.SUBGRAD_REF, kw, iters, pose0)
    check_trajectory(F, s, info, None, o, iters, kw, POSE_TOL, traced=False)
    for l in range(F.L):
        if iters[l] <= 0:
            continue
        n = int(info.iterations_run[l])
        e = al.get_energies(s, l)[:n]
        oe = o["trace"]["energy"][l, :n].astype(np.float32)
        assert (ulps(e, oe) <= ULP_TOL).all(), f"slot {s} L{l}: energies differ by > {ULP_TOL} ulp at iterations {np.nonzero(ulps(e, oe) > ULP_TOL)[0][:5]}"
        assert ulps(info.best_energy[l], o["best_energy"][l]).max() <= ULP_TOL
        assert ulps(info.visible_ratio[l], o["visible_ratio"][l]).max() <= ULP_TOL
    check_final_pose(pose, o, POSE_TOL, tag)


TRUNCATED = [(1, 0), (2, 0), (3, 0), (5, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("key,shape,kw", UNTRACED_ROWS, ids=[row_id(r[0]) for r in UNTRACED_ROWS])
def test_untraced_rows_against_oracle(frames, key, shape, kw):
    """NEED_H = false (the sub-gradient kernels no trace can see): the full schedule and truncated single-level schedules, where a
    wrong g shows in the first steps, against the oracle; a pair launch against the slot launch."""
    F = frames[shape]
    al = F.context(False)
    fast = kw.get("arithmetic", dvo.ARITH_EXACT) == dvo.ARITH_FAST
    for iters in [(50, 50)] + TRUNCATED:
        prm = dvo.solver_params(iters=iters, **kw)
        poses, info = run(al, F.n, prm)
        for s in range(F.n):
            assert info[s].status == 0
            if fast:
                check_final_pose(poses[s], F.oracle(s, dvo.SUBGRAD_REF, kw, iters), 1e-5, "fast")
            else:
                check_untraced_against_oracle(F, s, poses[s], info[s], kw, iters)
        check_pair_launch(al, F.n, prm, poses, info)


@pytest.mark.gpu
@pytest.mark.parametrize("key,shape,kw", UNTRACED_ROWS, ids=[row_id(r[0]) for r in UNTRACED_ROWS])
def test_untraced_kernel_matches_traced_kernel(frames, key, shape, kw):
    """The same sub-gradient run through the NEED_H = true kernel (traced context): only the grouping of g's partial sums differs,
    so the poses agree to GROUP_TOL and the energies to ULP_TOL.  For FAST arithmetic, whose trajectories the EXACT oracle
    cannot pin, this ties the NEED_H = false kernel to the traced one the per-iteration test holds to the spec."""
    F = frames[shape]
    prm = dvo.solver_params(iters=(50, 50), **kw)
    ua, ut = F.context(False), F.context(True)
    a, ai = run(ua, F.n, prm)
    b, bi = run(ut, F.n, prm)
    for s in range(F.n):
        d = np.abs(a[s] - b[s]).max()
        assert d <= GROUP_TOL, f"slot {s}: NEED_H = false vs true kernel poses differ by {d:.3g}"
        assert list(ai[s].iterations_run) == list(bi[s].iterations_run) and list(ai[s].best_index) == list(bi[s].best_index)
        for l in range(F.L):
            n = int(ai[s].iterations_run[l])
            du = ulps(ua.get_energies(s, l)[:n], ut.get_energies(s, l)[:n]).max()
            assert du <= ULP_TOL, f"slot {s} L{l}: energies of the two kernels differ by {du} ulp"


# ------------------------------------------------------------------------------------------------ point counts on the sweep boundaries
NS = [0, 1, 2, 31, 32, 33, 255, 256, 257, 511, 512, 513, 767, 768, 769, 1023, 1024, 1025, 2047, 2048, 2049, 5000]


@pytest.fixture(scope="module")
def nsweep():
    """One pair at 320x240, one level; slot k keeps depth > 100 only at the first NS[k] Canny edge pixels of the reference frame
    in column-major order (the order select_points takes them), so level 0 has exactly NS[k] points."""
    p = O.synth_pair(9300, 320, 240, K320)
    edge = O.canny(p["ref_gray"])
    xs, ys = np.nonzero(edge.T)                          # column-major: x outer, y inner
    assert len(xs) > max(NS)
    n = len(NS)
    depth = np.zeros((n, 240, 320), np.uint16)
    for k, N in enumerate(NS):
        depth[k, ys[:N], xs[:N]] = np.maximum(p["ref_depth"][ys[:N], xs[:N]], 101)
    d = {"ref_gray": np.repeat(p["ref_gray"][None], n, 0), "ref_depth": depth, "now_gray": np.repeat(p["now_gray"][None], n, 0)}
    out = {512: Frames(d, 320, 240, 1, K320, 512), 256: Frames(d, 320, 240, 1, K320, 256)}
    yield out
    for F in out.values():
        F.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [512, 256])
def test_nsweep_point_counts_are_exact(nsweep, shape):
    F = nsweep[shape]
    al = F.context(False)
    for k, N in enumerate(NS):
        assert len(al.get_points(k, 0)[0]) == N
        assert len(F.level(k, 0)[0]) == N


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [512, 256])
@pytest.mark.parametrize("solver", ["gn", "subgrad"])
@pytest.mark.parametrize("kw", [dict(), dict(weight=W_HUBER)], ids=["ring4", "register"])
def test_nsweep_traced_per_iteration(nsweep, shape, solver, kw):
    """The ring sweep (D = 4) and the register pipeline at every N: per-iteration sums at the kernel's pose; for the sub-gradient
    solver also the trajectory.  (GN's few-point normal equations are nearly singular, N < 64 gives condition numbers ~1e12,
    so its trajectory is no test of the sweep; its sums are.)"""
    F = nsweep[shape]
    sv = TRACED_SOLVERS[solver]
    iters = (10,) if sv == dvo.GN else (50,)
    prm = dvo.solver_params(solver=sv, iters=iters, **kw)
    assert dispatch(shape, True, prm)[6] == (4 if not kw else 0)
    al = F.context(True)
    poses, info = run(al, F.n, prm)
    for k, N in enumerate(NS):
        if N == 0:
            assert info[k].status & 1
            continue
        assert info[k].status == 0 and info[k].npts[0] == N
        tr = al.get_trace(k, 0)
        check_sums_at_kernel_pose(F, k, 0, tr, int(info[k].iterations_run[0]), kw, f"N={N}")
        if sv != dvo.GN:
            o = F.oracle(k, sv, kw, iters)
            check_trajectory(F, k, info[k], [tr], o, iters, kw, POSE_TOL)
            check_final_pose(poses[k], o, POSE_TOL, f"N={N}")
    check_pair_launch(al, F.n, prm, poses, info)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [512, 256])
def test_nsweep_shipped_subgradient(nsweep, shape):
    """The shipped sub-gradient kernel (ring D = 2) at every N against the oracle; the pair launch; dvo_pose_covariance at the
    returned poses (cov_kernel, the same sweep accumulating w eps^2 as well) against the oracle's H; N = 0 gives status bit 0."""
    F = nsweep[shape]
    al = F.context(False)
    iters = (50,)
    prm = dvo.solver_params(iters=iters)
    assert dispatch(shape, False, prm)[6] == 2
    poses, info = run(al, F.n, prm)
    for k, N in enumerate(NS):
        if N == 0:
            assert info[k].status & 1 and same(poses[k], np.concatenate([np.eye(3).reshape(9), np.zeros(3)]))
            continue
        assert info[k].status == 0 and info[k].npts[0] == N
        check_untraced_against_oracle(F, k, poses[k], info[k], {}, iters, tag=f"nsweep_N{N}")
    check_pair_launch(al, F.n, prm, poses, info)
    cov, cinfo = al.pose_covariance(F.n, prm)
    iu = np.triu_indices(6)
    for k, N in enumerate(NS):
        ci = cinfo[k]
        if N == 0:
            assert ci.status == 1 and np.isnan(cov[k]).all()
            continue
        R, T = poses[k, :9].reshape(3, 3), poses[k, 9:]
        o = F.evaluate(k, 0, R, T, dict(jacobian=dvo.JAC_EXACT), per_point=True)
        assert ci.nvis == o["nvis"], f"N={N}: covariance nvis {ci.nvis} vs {o['nvis']}"
        if o["nvis"] < 7:
            assert ci.status == 2 and np.isnan(cov[k]).all()
            continue
        H = np.zeros((6, 6)); H[iu] = o["H"][iu]; H = H + np.triu(H, 1).T
        s2 = float(np.sum(o["w"].astype(np.float64) * o["eps"].astype(np.float64) ** 2)) / (o["nvis"] - 6)
        assert ci.status == 0
        assert abs(ci.sigma2 - s2) <= SUM_REL * s2, f"N={N}: sigma2 {ci.sigma2!r} vs {s2!r}"
        err = np.abs(cov[k] @ H / s2 - np.eye(6)).max()
        assert err <= COV_REL * np.linalg.cond(H), f"N={N}: cov H / sigma2 - I = {err:.3g} (cond H {np.linalg.cond(H):.3g})"
    # N = 0 leaves a non-identity initial pose untouched
    P0 = np.tile(np.concatenate([O.se3_exp(np.array([0.002, -0.001, 0.003, 0.001, 0.002, -0.001]))[0].reshape(9), [0.002, -0.001, 0.003]]), (F.n, 1))
    p0, i0 = run(al, F.n, prm, P0)
    assert i0[0].status & 1 and same(p0[0], P0[0])

