"""ctypes binding of the windowed pose-graph oracle (tests/pgo_oracle/pgo_oracle.cpp): the same Levenberg-Marquardt as
dvo_pose_graph_optimize, with a sequential banded Cholesky where the device uses block cyclic reduction.

Test infrastructure: imported only from tests/ and tools/.  The product package never imports this module.  The library is
built with g++ on first use, next to its source, or in the temporary directory when the tree is read-only.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(ROOT, "tests", "pgo_oracle", "pgo_oracle.cpp")
_DEPS = [_SRC, os.path.join(ROOT, "oracle", "dvo_oracle.hpp")]
_FLAGS = ["-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-std=c++17", "-fPIC", "-shared"]
_lib = None


def build(force=False):
    out_dir = os.path.dirname(_SRC)
    if not os.access(out_dir, os.W_OK):
        out_dir = os.path.join(tempfile.gettempdir(), f"dvo_pgo_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libdvo_pgo_oracle.so")
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in _DEPS):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call(["g++"] + _FLAGS + ["-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def pose_graph(edge_ref, edge_now, meas, cov, poses0, max_lag, max_iterations=100, lambda0=1e-4, rel_tol=1e-10, marginals=False):
    """pgo::optimize for G graphs: returns (poses (G, N, 12), info dict of arrays, node_cov (G, N, 6, 6) or None)."""
    a = np.ascontiguousarray(edge_ref, np.int32); b = np.ascontiguousarray(edge_now, np.int32)
    G, E = a.shape
    X = np.array(poses0, np.float64, order="C", copy=True)
    N = X.shape[1]
    Z = np.ascontiguousarray(meas, np.float64).reshape(G, E, 12)
    S = np.ascontiguousarray(cov, np.float64).reshape(G, E, 6, 6)
    nc = np.empty((G, N, 6, 6), np.float64) if marginals else None
    info = np.empty((G, 6), np.float64)
    lib().orc_pose_graph(G, N, E, int(max_lag), _p(a, C.c_int32), _p(b, C.c_int32), _p(Z, C.c_double), _p(S, C.c_double),
                         _p(X, C.c_double), int(max_iterations), C.c_double(lambda0), C.c_double(rel_tol), _p(nc, C.c_double),
                         _p(info, C.c_double))
    keys = ("status", "iterations", "accepted", "edges_used", "cost_initial", "cost_final")
    out = {k: info[:, i].astype(np.int64) if i < 4 else info[:, i].copy() for i, k in enumerate(keys)}
    return X, out, nc


def pgo_system(edge_ref, edge_now, meas, cov, poses, max_lag, lam=0.0):
    """One graph at `poses`: dict with r (E, 6), valid (E,), dense H (n, n), g (n,), F, and delta of (H + lam diag H) delta = -g
    through the oracle's banded factor (None if that is not positive definite)."""
    a = np.ascontiguousarray(edge_ref, np.int32); b = np.ascontiguousarray(edge_now, np.int32)
    E = a.shape[0]
    X = np.ascontiguousarray(poses, np.float64)
    N = X.shape[0]
    n = 6 * (N - 1)
    Z = np.ascontiguousarray(meas, np.float64).reshape(E, 12)
    S = np.ascontiguousarray(cov, np.float64).reshape(E, 6, 6)
    r = np.empty((E, 6)); valid = np.empty(E, np.int32); H = np.empty((n, n)); g = np.empty(n); d = np.empty(n); F = C.c_double()
    rc = lib().orc_pgo_system(N, E, int(max_lag), _p(a, C.c_int32), _p(b, C.c_int32), _p(Z, C.c_double), _p(S, C.c_double),
                              _p(X, C.c_double), C.c_double(lam), _p(r, C.c_double), _p(valid, C.c_int32), _p(H, C.c_double),
                              _p(g, C.c_double), C.byref(F), _p(d, C.c_double))
    return {"r": r, "valid": valid.astype(bool), "H": H, "g": g, "F": F.value, "delta": d if rc == 0 else None}
