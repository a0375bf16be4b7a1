"""B200-native direct RGB-D alignment (the SolveDVO / EPoseEstimator / PyramidalStorage / GOP hot path of
mpkuse/rgbd_odometry).  The product is libdvo_b200.so (hand-written sm_100a CUDA behind the C-ABI in
include/dvo_b200.h); this package is the thin Python host binding used by tests and bench.py."""
from ._lib import Config, PairInfo, SolverParams, PhotoConfig, PhotoInfo, DvoError, load, SYMBOLS, STAGES  # noqa: F401
from .photo import PhotoEstimator  # noqa: F401
from .rgbd import RGBDAligner, rgbd_params  # noqa: F401
from ._lib import RgbdConfig, RgbdParams, RgbdInfo  # noqa: F401
from .batch import BatchAligner, solver_params, keyframe_policy, undistort, records  # noqa: F401
from ._lib import KeyframePolicy, CovInfo, PgoParams, PgoInfo, PGO_MAX_LAG  # noqa: F401
from .batch import (SUBGRAD_REF, GN, LM, JAC_REFERENCE, JAC_EXACT, W_REF_CAUCHY, W_HUBER, W_NONE, ARITH_EXACT,  # noqa: F401
                    ARITH_FAST, FRAME_REF, FRAME_NOW, RES_DT_FLOOR, RES_DT_INTERP)
