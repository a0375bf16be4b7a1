// common.cuh -- context layout, geometry helpers and arithmetic policies shared by the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <memory>

#include "../../include/dvo_b200.h"

#define DVO_EDT_INF_1D 16384             // "no edge pixel in this column" (larger than any image dimension)
#define DVO_EDT_INF (1 << 28)            // DVO_EDT_INF_1D squared: d2 of an image without edges

// Pyramid geometry.  Every per-level device array uses the same layout: level-major, then slot, then the
// level's row-major pixels:   element(l, b, i) = base[ off[l] + b * P[l] + i ],  off[l] = Bmax * sum_{k<l} P[k].
struct PyrGeom {
    int L, Bmax;
    int w[DVO_MAX_LEVELS], h[DVO_MAX_LEVELS], P[DVO_MAX_LEVELS];
    long long off[DVO_MAX_LEVELS];
    long long total;
    // packed distance texels (see "packed texel" below): 4x4-pixel tiles, tw[l] tiles per tile row, Pt[l] texels per image
    // (padded to whole tiles), same level-major / slot / texel layout:  element(l, b, i) = base[ offt[l] + b * Pt[l] + i ]
    int tw[DVO_MAX_LEVELS], Pt[DVO_MAX_LEVELS];
    long long offt[DVO_MAX_LEVELS];
    long long total_t;
};
__host__ __device__ inline long long lvl_at(const PyrGeom& g, int l, int b) { return g.off[l] + (long long)b * g.P[l]; }
__host__ __device__ inline long long tex_at(const PyrGeom& g, int l, int b) { return g.offt[l] + (long long)b * g.Pt[l]; }

// ---- packed texel -------------------------------------------------------------------------------------------------
// Everything the solver reads of the now frame at a reprojection -- DTn, its central-difference gradient and
// getWeightOf(DTn) -- is a function of the exact integer d2 at the pixel and at its four stencil neighbours
// (src/SolveDVO.cpp:1774, 1063-1098, 1047-1053).  Those five integers fit 8 bytes (16-byte float texels before):
//   word 0: bits 0..15  d2(y, x)            bits 16..25  d2(y, x-1) - d2(y, x)   (signed 10 bit)    bit 31  escape
//   word 1: bits 0..9   d2(y, x+1) - centre bits 10..19  d2(y-1, x) - centre     bits 20..29  d2(y+1, x) - centre
// (|sqrt d2(p) - sqrt d2(q)| <= 1 for neighbours, so |delta| <= 2 d + 1: ten bits cover every distance below 255 pixels;
// the pack kernel range-checks every field and sets the escape bit otherwise -- the solver then reads the five values
// from the 32-bit d2 image.)  On the first / last column (row) the REFLECT_101 taps coincide and the gradient is exactly
// 0: both deltas are stored as 0.  Texels are stored in 4x4-pixel tiles in Morton order, so a 32-byte sector is a 2x2
// block and a 128-byte line a 4x4 block: an edge contour crossing the block touches one line whatever its direction
// (row-major 16-byte texels: one line per 8x1 pixels).
#define DVO_TEX_ESCAPE 0x80000000u
__host__ __device__ inline int tex_index(int x, int y, int tw) {
    return (((y >> 2) * tw + (x >> 2)) << 4) | ((y & 2) << 2) | ((x & 2) << 1) | ((y & 1) << 1) | (x & 1);
}

struct Intr { float fx, fy, cx, cy; };

// One trace record per executed iteration: g[6], H[36], energy, nvis, R[9], T[3].
#define DVO_TRACE_DOUBLES 56
// energyAtEachIteration (src/SolveDVO.cpp:634): the first DVO_ENERGY_ITERS energies of every level of the last solve are always kept
#define DVO_ENERGY_ITERS 128

void dvo_set_error(const char* fmt, ...);

// Owner of one device allocation (host code only).  reserve() grows and never shrinks: a larger request frees the old
// block first, then allocates (contents are not kept); on failure the buffer is left empty, so the next call retries.
template <typename T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;            // capacity in elements
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { cudaFree(p); }
    int reserve(size_t count) {
        if (count <= n) return DVO_OK;
        cudaFree(p); p = nullptr; n = 0;
        const cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; dvo_set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e)); return DVO_ERR_NOMEM; }
        n = count;
        return DVO_OK;
    }
    T* get() const { return p; }
    operator T*() const { return p; }
};

struct dvo_ctx {
    dvo_config cfg;
    PyrGeom geom;
    Intr K;
    bool haveK;
    cudaStream_t own_stream, stream, copy_stream;
    cudaEvent_t ev_chunk[16], ev_entry;
    cudaStream_t aux[2];            // internal streams of dvo_process (two half batches, staggered)
    cudaEvent_t ev_fork, ev_pre[2], ev_aux_done[2];
    bool aux_pending;               // work is in flight on aux[] that the context stream has not joined yet
    int proc_first, proc_count;     // slot range of the dvo_process call that left that work in flight
    // sequence mode (run_sequences_core): staging for the pipelined uploads and the device record of a run, kept across calls
    // (cudaMalloc / cudaFree of ~0.8 GB per call made the end-to-end sequence rate vary 8x between runs)
    DevBuf<uint8_t> seq_stage_g[2]; DevBuf<uint16_t> seq_stage_d[2];
    cudaEvent_t seq_ev_ready[2], seq_ev_free[2];
    DevBuf<double> seq_rel; DevBuf<int> seq_kind, seq_reason; DevBuf<double> seq_glob;
    DevBuf<double> seq_cov, seq_gcov;   // per-frame relative / global covariances (dvo_run_sequences_cov)
    DevBuf<dvo_cov_info> seq_cov_info;  // per-frame dvo_cov_info of seq_cov; written by the entropy key-frame gate only
    DevBuf<double> seq_ent;             // per-frame entropy ratio the gate saw (dvo_run_sequences_entropy)
    // device results of dvo_pose_covariance / dvo_align_pairs with host outputs, grown on demand
    DevBuf<double> cov_buf; DevBuf<dvo_cov_info> cov_info_buf;
    // dvo_align_pairs: per-pair slot indices, initial / returned poses, info records and launch order, grown on demand
    DevBuf<int> pair_ref, pair_now, pair_order; DevBuf<double> pair_pose0, pair_pose; DevBuf<dvo_pair_info> pair_info;
    int sm_count;
    int solve_shape;         // threads per pair in solve_kernel: 512 when max_batch <= sm_count (one pair per SM at most), else 256
    size_t smem_optin;

    DevBuf<uint8_t> gray[2];     // [frame] gray pyramid
    DevBuf<uint16_t> depth[2];   // [frame] depth pyramid (now: only if keep_now_depth)
    DevBuf<uint8_t> prev_gray;   // level-0 copy of the previous now frame (p_now_framemono, src/SolveDVO.cpp:594-600); keep_now_depth only
    DevBuf<uint16_t> prev_depth; // p_now_depth
    std::unique_ptr<unsigned char[]> now_valid;    // host: slot has received a now frame
    std::unique_ptr<unsigned char[]> prev_valid;   // host: slot has a previous now frame
    DevBuf<uint8_t> edge[2];     // [frame] Canny edge maps 0/255
    DevBuf<uint16_t> gcol;       // now: EDT phase-1 column distances
    DevBuf<int32_t> d2;          // now: exact squared distance
    DevBuf<uint2> tex8;          // now: packed 8-byte texels
    DevBuf<float> ptsX, ptsY, ptsZ;   // ref: back-projected edge points (row-major pixel order), capacity P[l] per slot and level
    DevBuf<int> ptsPix;               // ref: pixel index y*w+x of every point (restores the reference's column-major order)
    DevBuf<int> npts;            // [Bmax][L]
    DevBuf<int> solve_order;     // [Bmax] pair slots of the current solve launch, heaviest first
    DevBuf<unsigned char> seq_mask;   // [Bmax] per-slot switch flags of the gated sequence loop (device)
    const unsigned char* active;      // when non-null, kernels skip slots whose flag is 0 (masked key-frame switch pass)
    DevBuf<int> seq_state;       // [Bmax] lastRefFrame per slot (device)
    DevBuf<unsigned> nedge;      // [2][Bmax][L]
    DevBuf<unsigned> maxd2;      // [Bmax][L]
    DevBuf<double> pose0;        // [Bmax][12]
    DevBuf<double> pose;         // [Bmax][12]
    DevBuf<dvo_pair_info> info;  // [Bmax]
    DevBuf<double> trace;        // [Bmax][L][trace_iters][56] or empty
    DevBuf<float> energy;        // [Bmax][L][DVO_ENERGY_ITERS] ||eps|| of every executed iteration of the last solve
    DevBuf<uint32_t> bitmap_scratch;  // candidate / edge bitmaps of every (frame, slot, level): written by sobel_nms_kernel, consumed by canny_kernel
    size_t bitmap_scratch_words; // per slot and frame (the scratch holds 2 x Bmax of them: reference and now CTAs run in one launch)
    long long bm_off[DVO_MAX_LEVELS];   // level region inside a (slot, frame) image of the scratch, in words
    int bm_words[DVO_MAX_LEVELS];       // words per bitmap at the level (the region holds two)
    size_t canny_smem_optin;     // largest dynamic shared-memory opt-in made for canny_kernel so far

    // device staging of dvo_set_frames_raw with host buffers (allocated on first use)
    DevBuf<uint8_t> raw_bgr; DevBuf<float> raw_depth;

    // dvo_pose_graph_optimize: per-graph scratch, and the device copies of host inputs / outputs, grown on demand
    DevBuf<double> pgo_dscr; DevBuf<int> pgo_iscr;
    DevBuf<int> pgo_ref, pgo_now; DevBuf<double> pgo_meas, pgo_cov, pgo_pose, pgo_ncov; DevBuf<dvo_pgo_info> pgo_info;

    bool timing;
    cudaEvent_t ev_a, ev_b;
    float stage_ms[DVO_STAGE_COUNT];
    long long launches;
};

#define DVO_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dvo_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return DVO_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

// ---- stage launchers (each defined next to its kernels) ----
int launch_pyramid(dvo_ctx* c, int first, int count, int frames_mask);
int launch_canny(dvo_ctx* c, int first, int count, int frames_mask);
void canny_scratch_layout(const PyrGeom& g, long long* bm_off, int* bm_words, size_t* words_per_image);
// EDT row pass + packed texels of the now frame (fused up to 800 pixels wide, the row kernels + pack_texel_kernel above that)
int launch_edt_pack(dvo_ctx* c, int first, int count);
// inspection: the dense d2 image of one slot / level into a caller-provided device buffer of P[level] int32
int launch_d2_from_texels(dvo_ctx* c, int slot, int level, int32_t* d_out);
// inspection: {DTn, gx, gy, w} of one slot / level into a caller-provided device buffer of P[level] float4, resolved from the
// packed texels through the solver's own lookup path
int launch_resolve_texels(dvo_ctx* c, int slot, int level, float4* d_out);
int launch_solve(dvo_ctx* c, int first, int count, const dvo_solver_params* p);
// solve of the npairs pairs (c->pair_ref[k], c->pair_now[k]) from c->pair_pose0 into c->pair_pose / c->pair_info
int launch_solve_pairs(dvo_ctx* c, int npairs, const dvo_solver_params* p);
int launch_eval(dvo_ctx* c, int slot, int level, const double* d_pose12, int jac, int weight, int arith, float huber_k, int residual,
                double* d_out /* 6 + 36 + 1 + 1 doubles */, float* d_eps, float* d_w, float* d_u, float* d_v, float* d_J);
// 6x6 pose covariance of slots [first, first+count) at their current pose (c->pose); record k at d_cov + 36 * k * stride.
// With c->active set, slots whose flag is 0 are skipped and keep their records.
int launch_cov(dvo_ctx* c, int first, int count, int level, const dvo_solver_params* p, double* d_cov, dvo_cov_info* d_info, long long stride);
// the same for the pairs of the last launch_solve_pairs, at c->pair_pose; record k at d_cov + 36 * k
int launch_cov_pairs(dvo_ctx* c, int npairs, int level, const dvo_solver_params* p, double* d_cov, dvo_cov_info* d_info);
// d_rel_cov / d_glob_cov: both null, or [nseq][nframes][36] covariances to propagate along the key-frame chain
int launch_gop(dvo_ctx* c, int nseq, int nframes, const int* d_kind, const double* d_rel, double* d_out, const double* d_rel_cov, double* d_glob_cov);
int launch_promote(dvo_ctx* c, int first, int count);
int launch_ingest_raw(dvo_ctx* c, int frame, int first, int count, const uint8_t* d_bgr, const float* d_depth_m);
int launch_copy_bytes(dvo_ctx* c, void* dst, const void* src, size_t n);
// pose-graph optimisation (posegraph.cu): per-graph scratch sizes in doubles / ints, and the one-CTA-per-graph launch on device arrays
int pgo_scratch_size(int nnodes, int nedges, int max_lag, size_t* dbl, size_t* ints);
int launch_pose_graph(dvo_ctx* c, int ngraphs, int nnodes, int nedges, int max_lag, const int* d_ref, const int* d_now, const double* d_meas,
                      const double* d_cov, double* d_poses, const dvo_pgo_params* prm, double* d_node_cov, dvo_pgo_info* d_info, double* d_dscr,
                      int* d_iscr);

// ---- arithmetic policies for the per-point fp32 math ----
// EXACT: one IEEE rounding per written operation, never contracted -> bit-identical to the oracle compiled with
// -ffp-contract=off.  FAST: plain expressions (nvcc contracts to FFMA) and approximate reciprocals.
template <int ARITH> struct Ar;
template <> struct Ar<DVO_ARITH_EXACT> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
    // a*b + c*d and (a*b + c*d) + e*f in the oracle's order
    static __device__ __forceinline__ float dot2(float a, float b, float c, float d) { return __fadd_rn(__fmul_rn(a, b), __fmul_rn(c, d)); }
    static __device__ __forceinline__ float dot3(float a, float b, float c, float d, float e, float f) {
        return __fadd_rn(__fadd_rn(__fmul_rn(a, b), __fmul_rn(c, d)), __fmul_rn(e, f));
    }
    static __device__ __forceinline__ float diff2(float a, float b, float c, float d) { return __fsub_rn(__fmul_rn(a, b), __fmul_rn(c, d)); }
    // getWeightOf: 6.0 / (6.0 + (double)(r*r) / .25)
    static __device__ __forceinline__ float weight_ref(float r) {
        float rr = __fmul_rn(r, r);
        return __double2float_rn(__ddiv_rn(6.0, __dadd_rn(6.0, __dmul_rn((double)rr, 4.0))));
    }
};
template <> struct Ar<DVO_ARITH_FAST> {
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float sub(float a, float b) { return a - b; }
    static __device__ __forceinline__ float div(float a, float b) { return __fdividef(a, b); }
    static __device__ __forceinline__ float dot2(float a, float b, float c, float d) { return fmaf(c, d, a * b); }
    static __device__ __forceinline__ float dot3(float a, float b, float c, float d, float e, float f) { return fmaf(e, f, fmaf(c, d, a * b)); }
    static __device__ __forceinline__ float diff2(float a, float b, float c, float d) { return fmaf(a, b, -(c * d)); }
    static __device__ __forceinline__ float weight_ref(float r) { return __fdividef(1.5f, fmaf(r, r, 1.5f)); }
};
