"""The edge path has one texel source (packed 8-byte Morton texels) and reads no environment variables.

Environment variables used to select the float4 texel path (DVO_TEXEL_MODE), the EDT band shape (DVO_EDT_BAND), the solver's
threads per pair (DVO_SOLVE_SHAPE), the Canny warps per level (DVO_CANNY_WARPS) and the upload chunk of dvo_align_batch
(DVO_E2E_CHUNK).  DVO_SOLVE_SHAPE regroups the fp64 partial sums, so it made a pair's pose depend on the caller's environment.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rgbd_odometry_b200", "csrc")

OLD_KNOBS = {"DVO_TEXEL_MODE": "0", "DVO_SOLVE_SHAPE": "256", "DVO_EDT_BAND": "-1", "DVO_CANNY_WARPS": "4,4,4,4", "DVO_E2E_CHUNK": "7"}


def test_library_reads_no_environment():
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    assert sources, CSRC
    hits = []
    for f in sources:
        with open(os.path.join(CSRC, f)) as fh:
            hits += [f"{f}:{no}: {line.strip()}" for no, line in enumerate(fh, 1) if re.search(r"\bgetenv\b", line)]
    assert not hits, "\n".join(hits)


# One seeded dvo_align_batch in a fresh process (the library used to read the variables in dvo_create / on first use):
# poses and the raw dvo_pair_info records go to an .npz.
_ALIGN = r"""
import sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import oracle_lib as O
import rgbd_odometry_b200 as dvo
W, H, L, n, out = int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), sys.argv[6]
K = O.K640 if W == 640 else O.K1280
d = O.synth_batch(900 + W, n, W, H, K)
al = dvo.BatchAligner(W, H, L, max_batch=n, intrinsics=K)
poses, info = al.align_batch(d["ref_gray"], d["ref_depth"], d["now_gray"], dvo.solver_params(iters=(50,) * L))
al.close()
np.savez(out, poses=poses, info=np.frombuffer(bytes(info), np.uint8))
"""


def _align_in_subprocess(tmp_path, tag, W, H, L, n, extra_env):
    env = {k: v for k, v in os.environ.items() if k not in OLD_KNOBS and k != "DVO_L2_FETCH"}
    env.update(extra_env)
    out = str(tmp_path / f"{tag}.npz")
    flags = ["-s"] if sys.flags.no_user_site else []
    subprocess.run([sys.executable, *flags, "-c", _ALIGN, ROOT, str(W), str(H), str(L), str(n), out], env=env, check=True, timeout=600)
    r = np.load(out)
    return r["poses"], r["info"]


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,L,n", [(640, 480, 4, 32), (1280, 720, 5, 8)])
def test_old_environment_knobs_change_nothing(tmp_path, W, H, L, n):
    # n <= SM count: the context's solver shape is 512 threads per pair, which DVO_SOLVE_SHAPE=256 used to override.
    # 1280x720 takes the unfused EDT rows + pack kernels; 640x480 the fused band kernel.
    poses, info = _align_in_subprocess(tmp_path, "plain", W, H, L, n, {})
    poses_k, info_k = _align_in_subprocess(tmp_path, "knobs", W, H, L, n, OLD_KNOBS)
    assert poses.shape == (n, 12) and np.isfinite(poses).all()
    assert np.array_equal(poses.view(np.uint64), poses_k.view(np.uint64))
    assert np.array_equal(info, info_k)
