/* dvo_b200.h -- C-ABI of the B200-native direct-alignment hot path (libdvo_b200.so).
 *
 * This is the drop-in boundary for the hot path of mpkuse/rgbd_odometry: plain pointers and sizes only, no
 * torch / Eigen / OpenCV types.  The reference has no FFI of its own -- its interface is the C++ class API of
 * SolveDVO / EPoseEstimator / PyramidalStorageStruct / GOP (include/SolveDVO.h:148-360,
 * include/EPoseEstimator.h:33-106, include/PyramidalStorage.h:37-78, include/GOP.h:67-95).  Each entry point
 * below cites the reference member(s) it replaces; rgbd_odometry_b200/host/ re-creates those classes on top of
 * this ABI, and INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - images are row-major, tightly packed; gray is u8, depth is u16 millimetres, BGR is u8 HWC;
 *   - a context owns device memory for `max_batch` independent frame pairs ("slots"); every call that takes
 *     (first, count) addresses slots [first, first+count);
 *   - rotation matrices are row-major double[9]; a pose record is R[9] followed by T[3] (12 doubles) with the
 *     reference's convention  p_now = R^T (P_ref - T)   (src/SolveDVO.cpp:330);
 *   - `mem` arguments: DVO_MEM_HOST (pageable or pinned host memory) or DVO_MEM_DEVICE (device pointers);
 *   - every function returns 0 on success, <0 on error (see dvo_last_error()); work is enqueued on the
 *     context's CUDA stream and is asynchronous unless the call returns data to host memory.
 *   - There is NO CPU fallback: every entry point fails with DVO_ERR_CUDA when no CUDA device is usable.
 */
#ifndef DVO_B200_H_
#define DVO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVO_MAX_LEVELS 6

/* DVO_ERR_NOMEM: an allocation failed, in whichever entry point made it (context creation, buffers grown on demand, per-call
 * temporaries).  For device memory dvo_last_error() reads "cudaMalloc(<n> bytes) failed: ...".  Earlier versions returned
 * DVO_ERR_CUDA for some of these failures. */
enum { DVO_OK = 0, DVO_ERR_ARG = -1, DVO_ERR_CUDA = -2, DVO_ERR_STATE = -3, DVO_ERR_NOMEM = -4 };
enum { DVO_MEM_HOST = 0, DVO_MEM_DEVICE = 1 };
enum { DVO_FRAME_REF = 0, DVO_FRAME_NOW = 1 };

/* solver (runIterations, src/SolveDVO.cpp:619-1017).  SUBGRAD_REF is the shipped projected sub-gradient
 * method; GN / LM solve the 6x6 normal equations the same kernels accumulate (north_star extension). */
enum { DVO_SOLVER_SUBGRAD_REF = 0, DVO_SOLVER_GN = 1, DVO_SOLVER_LM = 2 };
/* Jacobian: REFERENCE = computeJacobianOfNowFrame as written (normalised coordinates, src/SolveDVO.cpp:383-406);
 * EXACT = analytic derivative of the residual wrt the right-multiplicative pose update. */
enum { DVO_JAC_REFERENCE = 0, DVO_JAC_EXACT = 1 };
/* weights: REF_CAUCHY = getWeightOf (src/SolveDVO.cpp:1047-1053); HUBER; NONE. */
enum { DVO_WEIGHT_REF_CAUCHY = 0, DVO_WEIGHT_HUBER = 1, DVO_WEIGHT_NONE = 2 };
/* per-point fp32 arithmetic: EXACT reproduces the oracle's IEEE operation order bit for bit (no FMA
 * contraction, IEEE division); FAST lets the compiler contract and uses approximate reciprocals. */
enum { DVO_ARITH_EXACT = 0, DVO_ARITH_FAST = 1 };
/* residual: DT_FLOOR = eps = DT(floor v, floor u), the shipped build (src/SolveDVO.cpp:446); DT_INTERP = the
 * reference's compiled-out __INTERPOLATE_DISTANCE_TRANSFORM variant (:443-444, SolveDVO::interpolate :1285-1308):
 * "squared-bilinear" lookup, weights from getWeightOf of the interpolated value.  EXACT arithmetic only. */
enum { DVO_RESIDUAL_DT_FLOOR = 0, DVO_RESIDUAL_DT_INTERP = 1 };
/* pyramid flavour: NEAREST = camTopic2PublisherPyD (src/camTopic2PublisherPyD.cpp:338-348);
 * AREA = EPoseEstimator (src/EPoseEstimator.cpp:251-253, 284-286). */
enum { DVO_PYR_NEAREST = 0, DVO_PYR_AREA = 1 };

/* which = selector for dvo_get_level_buffer */
enum {
    DVO_BUF_GRAY = 0,   /* u8   [h][w]   pyramid level of the gray image                                  */
    DVO_BUF_DEPTH = 1,  /* u16  [h][w]   pyramid level of depth (mm, zeros replaced by 1, SolveDVO.cpp:512) */
    DVO_BUF_EDGE = 2,   /* u8   [h][w]   Canny edge map, 0 / 255                                          */
    DVO_BUF_D2 = 3,     /* i32  [h][w]   exact squared Euclidean distance to the nearest edge pixel       */
    DVO_BUF_DTN = 4,    /* f32  [h][w]   normalised distance transform (0..255)                           */
    DVO_BUF_GX = 5,     /* f32  [h][w]   d(DTn)/dx, central difference * 0.5                              */
    DVO_BUF_GY = 6      /* f32  [h][w]   d(DTn)/dy                                                        */
};

typedef struct dvo_ctx dvo_ctx;

typedef struct dvo_config {
    int width, height;      /* level-0 resolution                                              */
    int levels;             /* pyramid levels, 1..DVO_MAX_LEVELS (reference ships 4)            */
    int max_batch;          /* frame pairs resident on the device per launch                    */
    int device;             /* CUDA device ordinal                                              */
    int keep_now_depth;     /* 1: store the now frame's depth pyramid too (needed only so a now frame can
                               later become the reference, SolveDVO::setPrevFrameAsRefFrame :561-584)   */
    int trace_iters;        /* >0: keep a per-iteration trace (g, H, energy, pose) of this many iterations
                               per level for parity tests; 0 in production                              */
} dvo_config;

typedef struct dvo_solver_params {
    int solver;             /* DVO_SOLVER_*   */
    int jacobian;           /* DVO_JAC_*      */
    int weight;             /* DVO_WEIGHT_*   */
    int arithmetic;         /* DVO_ARITH_*    */
    float huber_k;
    double lm_lambda0;
    int iters[DVO_MAX_LEVELS];  /* iterationsConfig (src/SolveDVO.cpp:30-33); 0 skips the level */
    int residual;           /* DVO_RESIDUAL_* (0 = the shipped build)                             */
} dvo_solver_params;

/* per pair result record (what runIterations returns besides the pose, src/SolveDVO.cpp:997-1005, plus the
 * quiet-path residual statistic of processResidueHistogram :1398-1483) */
typedef struct dvo_pair_info {
    int status;                          /* 0 ok; bit0: a level had no reference points or no now edges;
                                            bit1: slot index out of range (dvo_align_pairs with device indices) */
    int npts[DVO_MAX_LEVELS];            /* selected reference edge points per level                      */
    int best_index[DVO_MAX_LEVELS];      /* bestEnergyIndex per level                                     */
    int iterations_run[DVO_MAX_LEVELS];  /* iterations actually executed per level                        */
    float best_energy[DVO_MAX_LEVELS];   /* ||eps||_2 of the best iterate                                 */
    float visible_ratio[DVO_MAX_LEVELS]; /* finalVisibleRatio                                             */
    float laplacian_b;                   /* mean(eps_best) at the finest executed level                   */
} dvo_pair_info;

const char* dvo_last_error(void);
int dvo_device_count(void);

/* lifetime: replaces the SolveDVO / EPoseEstimator constructors' state (src/SolveDVO.cpp:5-70) */
int dvo_create(const dvo_config* cfg, dvo_ctx** out);
int dvo_destroy(dvo_ctx* ctx);
/* run on a caller-owned CUDA stream (cudaStream_t as void*); NULL restores the context's own stream */
int dvo_set_stream(dvo_ctx* ctx, void* cuda_stream);
int dvo_synchronize(dvo_ctx* ctx);

/* SolveDVO::setCameraMatrix (src/SolveDVO.cpp:88-126): intrinsics of level 0 */
int dvo_set_intrinsics(dvo_ctx* ctx, float fx, float fy, float cx, float cy);

/* frame ingest: SolveDVO::imageArrivedCallBack + setRcvdFrameAsRefFrame / setRcvdFrameAsNowFrame
 * (src/SolveDVO.cpp:490-614).  Full-resolution images; the pyramid is built by dvo_build_pyramids.
 * depth may be NULL for the now frame (the edge solver never reads it, SURVEY A.7). */
int dvo_set_frames(dvo_ctx* ctx, int frame, int first, int count, const uint8_t* gray, const uint16_t* depth, int mem);
/* The same ingest from the RAW sensor frames the pyramid publisher receives (src/camTopic2PublisherPyD.cpp:65-80, :338-348):
 * bgr = u8 HWC (cv_bridge "bgr8"), depth_m = f32 metres (32FC1).  One fused kernel applies depth16 = saturate_u16(cvRound(
 * 1000.0f * depth)), 0 -> 1 (:75-78) and framemono = cvtColor(BGR2GRAY) (:347; OpenCV 4 fixed point, (B*3735 + G*19235 +
 * R*9798 + 2^14) >> 15) straight into the level-0 regions; the publisher's per-level gray equals the NEAREST level of this
 * full-resolution gray because BGR2GRAY is per pixel.  depth_m may be NULL where dvo_set_frames allows depth == NULL. */
int dvo_set_frames_raw(dvo_ctx* ctx, int frame, int first, int count, const uint8_t* bgr, const float* depth_m, int mem);
/* SolveDVO::setPrevFrameAsRefFrame (src/SolveDVO.cpp:561-584): the PREVIOUS now frame of every slot (p_now_*, kept on the
 * device by dvo_set_frames(NOW) when keep_now_depth = 1) becomes its reference frame's level 0; follow with
 * dvo_build_pyramids(.., 1) and dvo_prepare(.., 1) as the reference does. */
int dvo_promote_now_to_ref(dvo_ctx* ctx, int first, int count);

/* pyramid construction (src/camTopic2PublisherPyD.cpp:338-348): levels 1.. from level 0, both frames */
int dvo_build_pyramids(dvo_ctx* ctx, int first, int count, int frames_mask /* bit0 ref, bit1 now */);

/* computeDistTransfrmOfRef/Now + preProcessRefFrame (src/SolveDVO.cpp:1679-1799, 269-303):
 * Canny, exact EDT, normalise, gradient for the now frame; Canny + edge-point back-projection for the
 * reference frame. */
int dvo_prepare(dvo_ctx* ctx, int first, int count, int frames_mask);

/* initial pose per slot (cR_64, cT_64 of src/SolveDVO.cpp:1931-1932); NULL = identity */
int dvo_set_initial_pose(dvo_ctx* ctx, int first, int count, const double* R9T3, int mem);

/* the coarse-to-fine solve (src/SolveDVO.cpp:2097-2104 calling runIterations :619-1017) */
int dvo_run(dvo_ctx* ctx, int first, int count, const dvo_solver_params* params);

/* read back poses (12 doubles per slot) and optional info records */
int dvo_get_poses(dvo_ctx* ctx, int first, int count, double* R9T3, dvo_pair_info* info, int mem);

/* One call for a whole batch with host buffers: upload, pyramids, prepare, run, download (the end-to-end path
 * SolveDVO::loop executes per frame, src/SolveDVO.cpp:2017-2104).  count may exceed max_batch; the batch is
 * processed in chunks.  now_depth may be NULL. */
/* Whole hot path on frames ALREADY RESIDENT in slots [first, first+count): dvo_build_pyramids(3) + dvo_prepare(3) +
 * dvo_run.  Large ranges are processed as two half batches on two internal streams, staggered so that one half's
 * solve (DRAM-transaction bound, a third of the issue slots used) overlaps the other half's Canny / EDT (issue bound);
 * across back-to-back calls the second half's solve overlaps the next call's first preprocessing.  The call returns
 * without joining: every other entry point joins first, dvo_join does it explicitly (device-side wait, no host block).
 * Results are bit-identical to the staged calls.
 * d_poses (optional, DEVICE memory, count x 12 doubles): every half copies its poses there on its own stream, so a
 * caller that only needs the poses on the device never has to join between back-to-back calls. */
int dvo_process(dvo_ctx* ctx, int first, int count, const dvo_solver_params* params, double* d_poses);
int dvo_join(dvo_ctx* ctx);
/* make another CUDA stream (e.g. the one a collective runs on) wait for the work dvo_process left in flight */
int dvo_join_stream(dvo_ctx* ctx, void* cuda_stream);

int dvo_align_batch(dvo_ctx* ctx, int count, const uint8_t* ref_gray, const uint16_t* ref_depth,
                    const uint8_t* now_gray, const uint16_t* now_depth, const dvo_solver_params* params,
                    double* R9T3, dvo_pair_info* info);

/* SolveDVO::loop (src/SolveDVO.cpp:1896-2373) for nseq independent sequences in lock step (slot = sequence).
 * gray / depth: [nseq][nframes][H][W] host buffers.  rel_poses [nseq][nframes][12] (relative to the current key frame),
 * kind [nseq][nframes] (1 key frame, 0 ordinary, 2 ordinary promoted by updateMostRecentToKeyFrame), global_poses
 * [nseq][nframes][19] (may be NULL) as dvo_gop_compose writes them.  Needs keep_now_depth = 1. */
int dvo_run_sequences(dvo_ctx* ctx, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, const dvo_solver_params* params,
                      int keyframe_every, double* rel_poses, int* kind, double* global_poses);

/* Key-frame policy of SolveDVO::loop (src/SolveDVO.cpp:2117-2160): after a frame is solved against the current
 * reference, the residual statistic b = mean(eps_best) (processResidueHistogram :1398-1483), the visible ratio and the
 * number of reprojected points of the finest level decide whether the PREVIOUS frame becomes the new reference (pose
 * reset, re-solve; :2192-2233).  The reference ships with the three quality gates commented out (:2129-2151) and only
 * the periodic rule (:2155-2160); use_quality_gates = 1 evaluates them as designed, in source order, OR-ed with the
 * periodic rule.  Reasons as the reference numbers them: 2 laplacian b, 3 visible ratio, 4 too few points, 5 periodic.
 * Reason 6 (not the reference's) is the entropy ratio of dvo_run_sequences_entropy.  The gates are evaluated in the order
 * 2, 3, 4, 6, 5, and the last one that fires names the reason. */
typedef struct dvo_keyframe_policy {
    int keyframe_every;           /* 5 (:2156); <= 0 disables the periodic rule                 */
    int use_quality_gates;        /* 0 = as shipped                                             */
    float laplacian_thresh;       /* laplacianThreshExitCond = 3.0 (:23)                        */
    float visible_ratio_thresh;   /* ratio_of_visible_pts_thresh = 0.8 (:22)                    */
    int min_reprojections;        /* 50 (:2145)                                                 */
} dvo_keyframe_policy;
/* dvo_run_sequences with the decision taken per sequence ON THE DEVICE from the solver's own outputs: the gate kernel
 * writes a per-slot switch mask and the promote / pyramid / edge / solve kernels of the switch pass skip the other
 * slots, so no pose or statistic crosses PCIe between frames.  reason [nseq][nframes] receives the reference's reason
 * code at the frames that were promoted to key frames (0 elsewhere; frame 0 is a key frame with reason 1, :2016). */
int dvo_run_sequences_gated(dvo_ctx* ctx, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth,
                            const dvo_solver_params* params, const dvo_keyframe_policy* policy, double* rel_poses, int* kind,
                            int* reason, double* global_poses);

/* Both loops above with the INPUT sequences in host (DVO_MEM_HOST; pinned memory makes the uploads asynchronous) or device
 * memory (DVO_MEM_DEVICE).  Host inputs are pipelined: frame t+1 of every sequence is uploaded on a copy stream (one strided
 * 2-D copy per image plane) while frame t is solved.  Outputs are host buffers as above; reason / global_poses may be NULL. */
int dvo_run_sequences_mem(dvo_ctx* ctx, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem,
                          const dvo_solver_params* params, const dvo_keyframe_policy* policy, double* rel_poses, int* kind,
                          int* reason, double* global_poses);

/* ---- pose covariance ----
 * For a slot whose frames were prepared and solved, the Gauss-Newton covariance of its returned pose (R, T), evaluated at
 * pyramid level `level` on the frames resident in the slot:
 *   H      = sum_i w_i J_i^T J_i over the points visible at (R, T), J = the EXACT Jacobian (DVO_JAC_EXACT) in EXACT arithmetic,
 *            fp64 accumulation as the solver's; weight function, huber_k and residual come from `params` (solver, jacobian
 *            and arithmetic are ignored: the REFERENCE Jacobian is not the derivative of the residual);
 *   sigma2 = sum_i double(w_i) double(eps_i)^2 / (nvis - 6);
 *   Sigma  = sigma2 H^-1 from a Cholesky factor of H (no damping term is added);
 *   logdet = log det Sigma = 6 log sigma2 - log det H (for entropy-style criteria).
 * Tangent convention: Sigma is the covariance of psi = (rho, omega), translation first, for the right-multiplicative update
 * the solver applies, T <- T exp(psi) (cT += cR t(psi), cR <- cR R(psi)).  It describes the local curvature of the robust
 * cost; nothing here claims it is calibrated against the true error.
 * A slot whose level has no reference points or no now edges, fewer than 7 visible points, or an H that is not positive
 * definite gets 36 NaNs (not zeros, which would claim certainty) and a status bit. */
typedef struct dvo_cov_info {
    int status;      /* 0 ok; bit0 no reference points / no now edges at the level; bit1 nvis < 7; bit2 H not positive definite */
    int level;       /* level evaluated */
    int nvis;        /* visible reference points at the pose */
    double sigma2;   /* sum w eps^2 / (nvis - 6); NaN when status != 0 */
    double logdet;   /* log det of the covariance; NaN when status != 0 */
} dvo_cov_info;

/* 6x6 covariance (row-major, 36 doubles per slot) of the pose the last dvo_run / dvo_process left in each slot, evaluated on
 * the frames resident in the slots.  level = -1: the finest level with params->iters[l] > 0.  mem = DVO_MEM_HOST: host
 * buffers, returns when they are filled; DVO_MEM_DEVICE: device buffers, asynchronous on the context stream (info may be NULL).
 * One kernel launch for the whole range; the result of a slot does not depend on `count`, and no solver state is written.
 * After dvo_align_batch with count > max_batch only the last chunk's frames and poses are resident. */
int dvo_pose_covariance(dvo_ctx* ctx, int first, int count, const dvo_solver_params* params, int level,
                        double* cov36, dvo_cov_info* info, int mem);

/* Align npairs (reference, now) pairs of frames that are already prepared in this context. Pair k solves the REFERENCE-frame
 * data of slot ref_slot[k] (edge points, npts) against the NOW-frame data of slot now_slot[k] (texels, d2, max d2, edge counts).
 * Both slots must lie in [0, max_batch). A frame serves in both roles once it has been loaded into both roles of a slot
 * (dvo_set_frames REF and NOW with the same images) and built and prepared with frames_mask = 3. npairs may exceed max_batch.
 * pose0: npairs x 12 initial poses (NULL = identity). poses: npairs x 12. info: optional. cov36 / cov_info: optional, the
 * dvo_pose_covariance of each pair at its returned pose (level -1 rule as there). mem applies to every array argument.
 * The slots' own pose, info, energies and trace are not touched.
 *   - One solve launch over all pairs with the kernel configuration dvo_run would choose for these params on this context
 *     (same thread count per pair), so a pair's pose and info equal what dvo_run gives for a slot holding the same two frames,
 *     and do not depend on npairs or on the pair's position in the list.  DT_INTERP with FAST arithmetic is rejected, as there.
 *   - No energies or trace are recorded for pairs: dvo_get_energies / dvo_get_trace keep describing the last dvo_run.
 *   - DVO_MEM_HOST: indices outside [0, max_batch) return DVO_ERR_ARG; the call returns when the outputs are filled.
 *     DVO_MEM_DEVICE: indices are checked on the device; such a pair gets dvo_pair_info.status bit 1, 12 NaNs as its pose and a
 *     NaN covariance with dvo_cov_info.status bit 0; the call is asynchronous on the context stream.
 *   - A slot that was never prepared has no points or edges: status bit 0, as in dvo_run. */
int dvo_align_pairs(dvo_ctx* ctx, int npairs, const int* ref_slot, const int* now_slot, const double* pose0,
                    const dvo_solver_params* params, double* poses, dvo_pair_info* info,
                    double* cov36, dvo_cov_info* cov_info, int mem);

/* dvo_run_sequences_mem plus per-frame covariances: rel_cov [nseq][nframes][36] of rel_poses (frame 0: zeros, it anchors
 * the chain), global_cov [nseq][nframes][36] (may be NULL) of global_poses, first-order propagated along the key-frame chain:
 *   Sigma_g(i) = Ad(Tr^-1) Sigma_key Ad(Tr^-1)^T + Sigma_rel(i),   Ad(R, t) = [[R, [t]x R], [0, R]],  Tr = rel_poses[i],
 * Sigma_key = 0 at the start and Sigma_g(i) after every frame with kind[i] != 0.  The key-frame and relative estimates are
 * treated as independent.  rel_cov[t] is evaluated at the finest level with iterations, against the reference frame t was
 * finally solved against.  The poses, kinds, reasons and global poses equal those of dvo_run_sequences_mem bit for bit. */
int dvo_run_sequences_cov(dvo_ctx* ctx, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem,
                          const dvo_solver_params* params, const dvo_keyframe_policy* policy, double* rel_poses, int* kind,
                          int* reason, double* global_poses, double* rel_cov, double* global_cov);

/* dvo_run_sequences_cov plus the entropy-ratio key-frame rule of DVO-SLAM (Kerl, Sturm, Cremers, IROS 2013), decided per
 * sequence on the device.
 *   h(Sigma) = 3 (1 + ln 2 pi) + logdet(Sigma) / 2   (nats; logdet as dvo_cov_info.logdet)
 *   h_ref    = h of the final covariance of frame lastRef + 1, the first frame solved against the current key frame
 *              (NaN when that covariance is degenerate)
 *   alpha_t  = h(Sigma_t) / h_ref, Sigma_t the covariance of frame t's first solve against the current key frame (finest level
 *              with iterations; weight, huber_k and residual from params), evaluated where a switch is allowed (lastRef != t - 1).
 * The gate fires (reason 6) iff alpha_t is finite, h_ref < 0 and alpha_t < entropy_ratio_thresh: with h_ref < 0, alpha < 1
 * means "less certain than right after the key frame"; with h_ref >= 0 the ratio has no meaning and the gate stays silent.
 * It combines with the policy's quality gates and periodic rule (order above).  entropy_ratio [nseq][nframes] receives the
 * alpha each decision saw (for a switched frame: against the outgoing key frame), NaN where the gate was not evaluated
 * (frame 0, frames t = lastRef + 1) or a covariance was degenerate.  entropy_ratio_thresh <= 0 disables the gate: the call
 * is then dvo_run_sequences_cov exactly, and entropy_ratio is all NaN.  NaN is rejected.  reason, global_poses, rel_cov,
 * global_cov and entropy_ratio may be NULL (the covariances are computed in any case). */
int dvo_run_sequences_entropy(dvo_ctx* ctx, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem,
                              const dvo_solver_params* params, const dvo_keyframe_policy* policy, double entropy_ratio_thresh,
                              double* rel_poses, int* kind, int* reason, double* global_poses, double* rel_cov,
                              double* global_cov, double* entropy_ratio);

/* ---- windowed pose-graph optimisation (the back end DVO-SLAM puts behind this front end; Kerl, Sturm, Cremers, IROS 2013) ----
 * ngraphs independent graphs of the same shape: nnodes nodes and nedges edges each.  Node i has a global pose G_i (12-double
 * record; composition as dvo_gop_compose: G_a G_b = (R_a R_b, T_a + R_a T_b)); node 0 is held at its input pose (the gauge).
 * Edge e = (a, b, Z, Sigma): Z the relative pose of the pair (reference a, now b) as dvo_align_pairs returns it (noise-free:
 * G_b = G_a Z), Sigma its 6x6 covariance as cov36 (tangent (rho, omega), T <- T exp(psi)), information Omega = Sigma^-1.
 *   r_e = log(Z^-1 G_a^-1 G_b) (se3 log, (rho, omega)),  F = 1/2 sum_e r_e^T Omega_e r_e,
 *   right perturbations G <- G exp(d):  dr/dd_b = Jinv(r),  dr/dd_a = -Jinv(r) Ad(G_b^-1 G_a),
 *   Jinv(r) = I + 1/2 ad(r), ad(rho, omega) = [[omega x, rho x], [0, omega x]], Ad(R, t) = [[R, [t]x R], [0, R]] (first-order
 *   inverse Jacobian: it changes the path of the iteration; at a zero-residual optimum it changes nothing).
 * Every edge needs 1 <= |a - b| <= max_lag <= DVO_PGO_MAX_LAG: windowed odometry, forward and backward pairs; loop closures
 * are out of scope.  An edge whose Sigma has a non-finite entry or is not positive definite (its lower triangle is factored)
 * is skipped, so pairs dvo_align_pairs flagged (NaN covariance) drop out on their own.
 * Levenberg-Marquardt with Marquardt damping H + lambda diag(H): an iteration is one damped solve and one cost evaluation; a
 * step is accepted iff the cost decreases (then lambda /= 10, else lambda *= 10).  The loop stops after max_iterations, after
 * an accepted step whose relative decrease (F - F') / F is below rel_tol, or when lambda exceeds DVO_PGO_LAMBDA_MAX.
 * node_cov36 (optional): the 6x6 diagonal blocks of H^-1 with lambda = 0 at the returned poses, same tangent and convention as
 * global_cov of dvo_run_sequences_cov; node 0 gets zeros (it anchors the graph).
 * mem = DVO_MEM_HOST: a bad edge index returns DVO_ERR_ARG before anything is launched; returns when the outputs are filled.
 * DVO_MEM_DEVICE: the device checks the indices (status bit 0); asynchronous on the context stream.  A graph with status bit
 * 0 or 1 keeps its input poses and gets NaN marginals.  Reads no frame data: works on any context.  One kernel launch; a
 * graph's results are bit-identical whatever ngraphs, its position in the batch and mem. */
#define DVO_PGO_MAX_LAG 8
#define DVO_PGO_LAMBDA_MAX 1e16
typedef struct dvo_pgo_params {
    int max_iterations;   /* damped solves, accepted or not (e.g. 100)          */
    double lambda0;       /* initial Marquardt damping (e.g. 1e-4), > 0           */
    double rel_tol;       /* stop after an accepted step with (F - F') / F < rel_tol (e.g. 1e-10) */
} dvo_pgo_params;
typedef struct dvo_pgo_info {
    int status;       /* bit0 an edge index is out of range, a == b or |a-b| > max_lag (device indices); bit1 a node is not
                         connected to node 0 through valid edges; bit2 H not positive definite at the returned poses (marginals NaN) */
    int iterations, accepted, edges_used;
    double cost_initial, cost_final;   /* F at the input and at the returned poses; NaN when status bit 0 or 1 is set */
} dvo_pgo_info;
int dvo_pose_graph_optimize(dvo_ctx* ctx, int ngraphs, int nnodes, int nedges, int max_lag,
                            const int* edge_ref, const int* edge_now,     /* [ngraphs][nedges]       */
                            const double* meas12, const double* cov36,    /* [ngraphs][nedges][12/36] */
                            double* poses12,                              /* [ngraphs][nnodes][12], in: initial, out: optimised */
                            const dvo_pgo_params* prm, double* node_cov36 /* optional [ngraphs][nnodes][36] */,
                            dvo_pgo_info* info /* optional [ngraphs] */, int mem);

/* ---- inspection (parity tests; not on the hot path) ---- */
int dvo_level_dims(dvo_ctx* ctx, int level, int* w, int* h);
int dvo_get_level_buffer(dvo_ctx* ctx, int slot, int frame, int level, int which, void* host_dst, size_t bytes);
/* reference edge points of one slot/level in enumeration order (SpaceCordList _3d, src/SolveDVO.cpp:287-289) */
int dvo_get_points(dvo_ctx* ctx, int slot, int level, float* X, float* Y, float* Z, int capacity, int* n);
/* one evaluation of the normal equations at a given pose: H = J^T W J (row-major 6x6), g = J^T W eps,
 * sumsq = sum eps^2, nvis; optional per-point outputs (capacity = npts): eps, w, reprojection u, v, J (N x 6) */
int dvo_eval_normal_equations(dvo_ctx* ctx, int slot, int level, const double* R9T3, int jacobian, int weight,
                              int arithmetic, float huber_k, double* H36, double* g6, double* sumsq, int* nvis,
                              float* eps, float* w, float* u, float* v, float* J);
/* same, with every evaluation option taken from a dvo_solver_params (jacobian, weight, arithmetic, huber_k, residual) */
int dvo_eval_normal_equations_ex(dvo_ctx* ctx, int slot, int level, const double* R9T3, const dvo_solver_params* prm,
                                 double* H36, double* g6, double* sumsq, int* nvis,
                                 float* eps, float* w, float* u, float* v, float* J);
/* per-iteration trace of the last dvo_run (needs cfg.trace_iters > 0): for level `level`, `trace_iters` records of
 * 56 doubles: g[6], H[36], energy, nvis, R[9], T[3] (zero where not executed) */
int dvo_get_trace(dvo_ctx* ctx, int slot, int level, double* trace);

/* energyAtEachIteration of runIterations (src/SolveDVO.cpp:634, :690): ||eps|| of the first min(capacity, 128) iterations the last
 * dvo_run executed at `level` for `slot`; entries beyond info.iterations_run[level] are stale.  Always recorded (one float per
 * iteration), independent of cfg.trace_iters. */
int dvo_get_energies(dvo_ctx* ctx, int slot, int level, float* energies, int capacity);

/* per-stage device time of the most recent calls, CUDA events on the context stream (ms); enable first */
enum { DVO_STAGE_H2D = 0, DVO_STAGE_PYRAMID, DVO_STAGE_CANNY, DVO_STAGE_EDT_ROWS, DVO_STAGE_NORMGRAD, DVO_STAGE_SOLVE,
       DVO_STAGE_D2H, DVO_STAGE_COUNT };
int dvo_enable_timing(dvo_ctx* ctx, int on);
int dvo_get_stage_ms(dvo_ctx* ctx, float* ms /* DVO_STAGE_COUNT */);
/* number of kernel launches issued by this context since creation */
long long dvo_launch_count(dvo_ctx* ctx);

/* ---- GOP<double> (src/GOP.cpp:138-196): batched composition on the device ----
 * For `nseq` independent sequences of `nframes` relative poses each (12 doubles, relative to the sequence's last
 * key frame) and kind[] (0 ordinary, 1 key frame, 2 ordinary then updateMostRecentToKeyFrame), write global poses
 * out[nseq][nframes][19] = R[9], T[3], px py pz qx qy qz qw. */
int dvo_gop_compose(dvo_ctx* ctx, int nseq, int nframes, const int* kind, const double* rel, double* out, int mem);

/* ================================================================================================================
 * EPoseEstimator / PyramidalStorageStruct (dense photometric estimator, src/EPoseEstimator.cpp, src/PyramidalStorage.cpp)
 * A separate context: BGR u8 (HWC) + depth u16 frames, INTER_AREA pyramids of up to 5 levels (the reference always
 * builds levels 0..4, :88), reference-frame Jacobian.  `compat` = 1 reproduces the reference bug for bug (SURVEY.md
 * Appendix C quirks: duplicated Jacobian column => singular A, row index paired with cx, unscaled fx, residual flattened
 * row-major against column-major J rows, holes count as residuals): it yields the reference's A = J^T J and b = J^T eps
 * entry for entry and takes no step.  `compat` = 0 is the corrected formulation with optional Huber weights
 * (huber_k > 0, intensity units) and LM damping (lambda0 > 0; 0 = Gauss-Newton).
 * ================================================================================================================ */
typedef struct dvo_photo_ctx dvo_photo_ctx;

typedef struct dvo_photo_config {
    int width, height;   /* level-0 resolution; must be divisible by 2^(levels-1) */
    int levels;          /* 1..5 */
    int max_batch;
    int device;
} dvo_photo_config;

typedef struct dvo_photo_info {
    int status;          /* 0 ok; 1 normal equations not positive definite; 2 compat mode (singular A, no step taken) */
    int iters_run;
    int nreproj;         /* nReprojected of the last warp (src/EPoseEstimator.cpp:168) */
    double sumsq_first, sumsq_last;   /* sum eps^2 at the first / last evaluation */
    double visible;      /* nReprojected / (rows*cols) as a real fraction (the reference's integer division gives 0 or 1) */
    double A[36];        /* normal matrix of the last accepted linearisation (compat: J^T J of the level) */
    double b[6];         /* J^T (W) eps of the last accepted linearisation */
} dvo_photo_info;

/* which = selector for dvo_photo_get_level: the members of PyramidalStorageStruct (include/PyramidalStorage.h:63-77) */
enum {
    DVO_PHOTO_BGR = 0,        /* u8  [rows][cols][3]  im_r_color / im_color */
    DVO_PHOTO_GRAY = 1,       /* u8  [rows][cols]     im_r / im             */
    DVO_PHOTO_DEPTH = 2,      /* u16 [rows][cols]     dim_r / dim           */
    DVO_PHOTO_X = 3, DVO_PHOTO_Y = 4, DVO_PHOTO_Z = 5,   /* f64 [rows][cols], metres (evaluate3d :439-477) */
    DVO_PHOTO_J = 6,          /* f64 [rows*cols][6], row k = column-major pixel k (evaluateJacobian :398-415) */
    DVO_PHOTO_GRAYVALS = 7, DVO_PHOTO_REDVALS = 8, DVO_PHOTO_GREENVALS = 9, DVO_PHOTO_BLUEVALS = 10   /* f64 [rows][cols] */
};

int dvo_photo_create(const dvo_photo_config* cfg, dvo_photo_ctx** out);     /* EPoseEstimator::EPoseEstimator */
int dvo_photo_destroy(dvo_photo_ctx* ctx);
int dvo_photo_set_stream(dvo_photo_ctx* ctx, void* cuda_stream);
int dvo_photo_synchronize(dvo_photo_ctx* ctx);
long long dvo_photo_launch_count(dvo_photo_ctx* ctx);
/* EPoseEstimator::setCameraMatrix (src/EPoseEstimator.cpp:35-59): double intrinsics of level 0 */
int dvo_photo_set_intrinsics(dvo_photo_ctx* ctx, double fx, double fy, double cx, double cy);
/* setRefFrame / setNowFrame (:68-126): copy, BGR2GRAY at full resolution, INTER_AREA pyramids (setRefPyramidalImages :266-290,
 * setPyramidalImages :216-260).  depth may be NULL for the now frame. */
int dvo_photo_set_frames(dvo_photo_ctx* ctx, int frame, int first, int count, const uint8_t* bgr, const uint16_t* depth, int mem);
/* evaluateJacobian + evaluate3d for every level and A = J^T J (:88-102, :229, :320-477) */
int dvo_photo_prepare_ref(dvo_photo_ctx* ctx, int first, int count, int compat);
/* initial (R, T) of estimate(); NULL = identity.  12 doubles per slot, host memory. */
int dvo_photo_set_pose(dvo_photo_ctx* ctx, int first, int count, const double* R9T3);
/* setPyramidalImages(level) + estimate(R, T) (:135-209): `iters` iterations (the reference hard-codes 3) */
int dvo_photo_estimate(dvo_photo_ctx* ctx, int first, int count, int level, int iters, int compat, double huber_k, double lambda0);
int dvo_photo_get_poses(dvo_photo_ctx* ctx, int first, int count, double* R9T3, dvo_photo_info* info);
/* PyramidalStorageStruct::getLevel (src/PyramidalStorage.cpp:71-102): any stored member of one slot / level, host copy */
int dvo_photo_get_level(dvo_photo_ctx* ctx, int slot, int frame, int level, int which, void* host_dst, size_t bytes, int compat);
int dvo_photo_get_A(dvo_photo_ctx* ctx, int slot, int level, double* A36);
/* PyramidalStorageStruct::addLevel with the caller's own images (src/PyramidalStorage.cpp:38-65): overwrite one stored level image
 * (which = DVO_PHOTO_GRAY / DVO_PHOTO_DEPTH at any level, DVO_PHOTO_BGR at level 0; host source, exact size).  X / Y / Z / J / *Vals
 * are functions of these and are re-evaluated by the kernels; call dvo_photo_prepare_ref afterwards to refresh A = J^T J. */
int dvo_photo_put_level(dvo_photo_ctx* ctx, int slot, int frame, int level, int which, const void* host_src, size_t bytes);
/* one evaluation of estimate()'s loop body at a given pose (inspection): warped canvas (f64 [rows][cols], may be NULL),
 * b = J^T (W) eps, A, sum eps^2, nReprojected, residual count */
int dvo_photo_eval(dvo_photo_ctx* ctx, int slot, int level, const double* R9T3, int compat, double huber_k, double* b6, double* A36,
                   double* sumsq, int* nreproj, int* nused, double* canvas);

/* ---- device-resident storage blobs: what PyramidalStorageStruct (src/PyramidalStorage.cpp:38-102) keeps per level when a
 * caller pushes its own eleven arrays -- a device allocation with host upload / download instead of a host deep copy ---- */
typedef struct dvo_blob dvo_blob;
int dvo_blob_create(size_t bytes, int device, dvo_blob** out);
int dvo_blob_upload(dvo_blob* blob, const void* host_src, size_t bytes);
int dvo_blob_download(dvo_blob* blob, void* host_dst, size_t bytes);
void* dvo_blob_device_ptr(dvo_blob* blob);
size_t dvo_blob_bytes(dvo_blob* blob);
int dvo_blob_destroy(dvo_blob* blob);

/* ---- undistortion front-end of the publisher (src/camTopic2PublisherPyD.cpp:86-117: cv::undistort of the BGR frame and of
 * the 16-bit depth frame before the pyramid is built).  `count` images of `type`, tightly packed; K4 = fx, fy, cx, cy;
 * D5 = k1, k2, p1, p2, k3 (sensor_msgs/CameraInfo.D, :55-61).  Bilinear, BORDER_CONSTANT 0, bit-exact against
 * cv2.undistort 4.13.  mem = DVO_MEM_DEVICE: both pointers are device memory and the call is asynchronous on
 * `cuda_stream`; DVO_MEM_HOST: staged through temporary device buffers, synchronous. ---- */
enum { DVO_IMG_U8C1 = 0, DVO_IMG_U8C3 = 1, DVO_IMG_U16C1 = 2 };
int dvo_undistort(const void* src, void* dst, int width, int height, int type, int count, const double* K4, const double* D5, int mem,
                  void* cuda_stream);

/* ================================================================================================================
 * RGBDOdometry (src/RGBDOdometry.cpp, include/RGBDOdometry.h:96-131): the semi-dense photometric Gauss-Newton --
 * reference-frame Jacobian at pixels whose forward x-gradient is >= const_gradientThreshold, A = J^T J per level,
 * three iterations of { eps, b = -J^T eps, psi = A.colPivHouseholderQr().solve(b), T <- T exp(psi)^-1 } with the
 * ||eps|| < 200 early exit.  Batched like the other paths: slot = one (reference, now) pair.  Poses are row-major
 * 4x4 affine transforms (TransformRep, include/RGBDOdometry.h:33).  Quirks of the reference are kept (SURVEY F1).
 * ================================================================================================================ */
#define DVO_RGBD_MAX_LEVELS 5
typedef struct dvo_rgbd_ctx dvo_rgbd_ctx;

typedef struct dvo_rgbd_config {
    int width, height;   /* level-0 resolution */
    int levels;          /* 2..5; the reference builds 4 (src/RGBDOdometry.cpp:343) */
    int max_batch;
    int device;
} dvo_rgbd_config;

typedef struct dvo_rgbd_params {
    int iterations;          /* 3   (src/RGBDOdometry.cpp:541) */
    int gradient_threshold;  /* 5   const_gradientThreshold   (:32) */
    int min_points;          /* 100 const_minimumRequiredPts  (:34, assert :497) -> status bit 0 */
    int max_points;          /* 50000 const_maxJacobianSize   (:33, assert :463) -> status bit 1 */
    double eps_norm_exit;    /* 200.0 (:556) */
} dvo_rgbd_params;

typedef struct dvo_rgbd_info {
    int status;                                  /* bit0: too few selected points at a level that ran; bit1: too many */
    int npts[DVO_RGBD_MAX_LEVELS];               /* selected pixels (rows of J) */
    int iters_run[DVO_RGBD_MAX_LEVELS];          /* epsilon evaluations of the last gaussNewtonIterations at the level */
    int updates[DVO_RGBD_MAX_LEVELS];            /* pose updates applied */
    int nvis_last[DVO_RGBD_MAX_LEVELS];          /* selected pixels that reprojected inside the now image */
    double eps_norm_first[DVO_RGBD_MAX_LEVELS];  /* ||eps|| at the first / last evaluation */
    double eps_norm_last[DVO_RGBD_MAX_LEVELS];
} dvo_rgbd_info;

int dvo_rgbd_create(const dvo_rgbd_config* cfg, dvo_rgbd_ctx** out);        /* RGBDOdometry::RGBDOdometry */
int dvo_rgbd_destroy(dvo_rgbd_ctx* ctx);
int dvo_rgbd_set_stream(dvo_rgbd_ctx* ctx, void* cuda_stream);
int dvo_rgbd_synchronize(dvo_rgbd_ctx* ctx);
long long dvo_rgbd_launch_count(dvo_rgbd_ctx* ctx);
/* setCameraMatrix (:38-60): the same K is used at every level (the reference never rescales it) */
int dvo_rgbd_set_intrinsics(dvo_rgbd_ctx* ctx, double fx, double fy, double cx, double cy);
/* setRefFrame (frame 0) / setNowFrame (frame 1) (:330-390): BGR2GRAY at full resolution, INTER_NEAREST pyramids */
int dvo_rgbd_set_frames(dvo_rgbd_ctx* ctx, int frame, int first, int count, const uint8_t* bgr, const uint16_t* depth, int mem);
/* computeJacobianAllLevels (:393-415): A = J^T J and the selection count for levels 1..levels-1 of the reference frame */
int dvo_rgbd_compute_jacobians(dvo_rgbd_ctx* ctx, int first, int count, int gradient_threshold);
/* T of the next gaussNewtonIterations; NULL = identity.  16 doubles per slot (row-major 4x4), host memory. */
int dvo_rgbd_set_pose(dvo_rgbd_ctx* ctx, int first, int count, const double* T16);
/* gaussNewtonIterations(level, T) (:514-597); level 0 is rejected like the reference's assert (:518) */
int dvo_rgbd_gauss_newton(dvo_rgbd_ctx* ctx, int first, int count, int level, const dvo_rgbd_params* prm);
int dvo_rgbd_get_poses(dvo_rgbd_ctx* ctx, int first, int count, double* T16, dvo_rgbd_info* info);
/* inspection */
int dvo_rgbd_level_dims(dvo_rgbd_ctx* ctx, int level, int* rows, int* cols);
int dvo_rgbd_get_level(dvo_rgbd_ctx* ctx, int slot, int frame, int level, uint8_t* gray, uint16_t* depth);
int dvo_rgbd_get_A(dvo_rgbd_ctx* ctx, int slot, int level, double* A36, int* npts);
/* computeJacobian (:407-505) + computeEpsilon (:602-700) of one slot / level at pose T, in the reference's enumeration
 * order (column outer, row inner): ij = (row, col), J (n x 6), eps, uv = floor(outu, outv) or (-1, -1) when unseen */
int dvo_rgbd_eval(dvo_rgbd_ctx* ctx, int slot, int level, const double* T16, int gradient_threshold, int capacity, int* n, int* ij,
                  double* J, double* eps, int* uv, double* b6, double* sumsq, int* nvis);

#ifdef __cplusplus
}
#endif
#endif /* DVO_B200_H_ */
