// rgbd.cu -- RGBDOdometry on the GPU: the reference's semi-dense photometric Gauss-Newton (SURVEY.md §8 F1,
// src/RGBDOdometry.cpp:330-390 pyramids, :407-505 computeJacobian, :514-597 gaussNewtonIterations, :602-700
// computeEpsilon, :707-763 exponentialMap / to_se_3), batched over independent frame pairs.
//
// What the reference stores per level (the N x 6 fp64 Jacobian, the selection mask) is a pure function of the level's
// u8 gray, u16 depth and the pixel index, so nothing of it is materialised: the selection test (forward x-gradient
// >= 5) and the Jacobian row are recomputed per pixel inside the sweeps from 5 bytes per pixel instead of re-reading
// 48-byte rows, and A = J^T J is reduced once per reference frame.  One persistent CTA per pair runs a whole
// gaussNewtonIterations call (epsilon sweep, fp64 reduction to b = -J^T eps and ||eps||, the early exit, the pivoted
// Householder QR solve, exponential map, T <- T exp(psi)^-1) without a host round trip.
//
// Quirks are kept as written (row index paired with cx, depth in raw sensor units, J column 0 = fx*fx/Z, intrinsics
// not scaled per level, signed gradient threshold).  Compiled with -fmad=false: every fp64 expression is evaluated
// in the written order, one rounding per operation, so per-pixel quantities are bit-identical to the CPU oracle.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"

#define RG_MAX_LEVELS DVO_RGBD_MAX_LEVELS
#define RG_THREADS 256

struct RgGeom { int L, Bmax, W, H; int w[RG_MAX_LEVELS], h[RG_MAX_LEVELS], P[RG_MAX_LEVELS]; long long off[RG_MAX_LEVELS]; long long total; };
__host__ __device__ inline long long rg_at(const RgGeom& g, int l, int b) { return g.off[l] + (long long)b * g.P[l]; }
struct RgCam { double fx, fy, cx, cy; };

struct RgState { double T[16]; dvo_rgbd_info info; };

struct dvo_rgbd_ctx {
    dvo_rgbd_config cfg; RgGeom g; RgCam K; bool haveK;
    cudaStream_t own_stream, stream;
    DevBuf<uint8_t> bgr;         // staging: one frame set, [Bmax][H][W][3]
    DevBuf<uint16_t> depth_in;   // staging: [Bmax][H][W]
    DevBuf<uint8_t> gray[2];     // NEAREST pyramid of BGR2GRAY(full), level-major
    DevBuf<uint16_t> depth[2];
    DevBuf<double> A;            // [Bmax][L][36]
    DevBuf<int> npts;            // [Bmax][L]
    DevBuf<RgState> st;          // [Bmax]
    DevBuf<double> pose_stage;   // [Bmax][16] device staging for dvo_rgbd_set_pose
    long long launches;
};

// ------------------------------------------------------------------------------------------------------
// per-pixel quantities (mirror oracle/dvo_oracle.hpp rgbd::compute_jacobian / compute_epsilon line by line)
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void rg_gradients(const uint8_t* __restrict__ g, int rows, int cols, int i, int j, double& gx, double& gy) {
    const int j1 = (j + 1 < cols) ? j + 1 : (cols > 1 ? cols - 2 : j), i1 = (i + 1 < rows) ? i + 1 : (rows > 1 ? rows - 2 : i);   // REFLECT_101
    const double c = (double)g[(size_t)i * cols + j];
    gx = (double)g[(size_t)i * cols + j1] - c;                                    // filter2D [0 -1 1] (:419-426)
    gy = (double)g[(size_t)i1 * cols + j] - c;
}

__device__ __forceinline__ void rg_xyz(int i, int j, double Z, const RgCam& K, double& X, double& Y) {
    X = Z * ((double)i - K.cx) / K.fx;                                            // :476-478: the ROW index pairs with cx
    Y = Z * ((double)j - K.cy) / K.fy;
}

__device__ __forceinline__ void rg_jrow(double gx, double gy, double X, double Y, double Z, const RgCam& K, double* r) {
    const double fx = K.fx, fy = K.fy;
    const double invZ = 1 / Z, invZ2 = 1 / (Z * Z);                               // :480-481
    r[0] = fx * fx * invZ;                                                        // :487 (as written)
    r[1] = fy * gy * invZ;
    r[2] = -fy * gy * Y * invZ2 - fx * gx * X * invZ2;
    r[3] = gy * (-fy * Y * Y * invZ2 - fy) - fx * gx * X * Y * invZ2;
    r[4] = gx * (fx * X * X * invZ2 + fx) + fx * gy * X * Y * invZ2;
    r[5] = fy * gy * X * invZ - fx * gy * Y * invZ;
}

__device__ __forceinline__ void rg_inv3(const double* M, double* Mi) {
    const double c00 = M[4] * M[8] - M[5] * M[7], c01 = M[5] * M[6] - M[3] * M[8], c02 = M[3] * M[7] - M[4] * M[6];
    const double det = M[0] * c00 + M[1] * c01 + M[2] * c02, id = 1.0 / det;
    Mi[0] = c00 * id; Mi[1] = (M[2] * M[7] - M[1] * M[8]) * id; Mi[2] = (M[1] * M[5] - M[2] * M[4]) * id;
    Mi[3] = c01 * id; Mi[4] = (M[0] * M[8] - M[2] * M[6]) * id; Mi[5] = (M[2] * M[3] - M[0] * M[5]) * id;
    Mi[6] = c02 * id; Mi[7] = (M[1] * M[6] - M[0] * M[7]) * id; Mi[8] = (M[0] * M[4] - M[1] * M[3]) * id;
}
// Transform<double,3,Affine>::inverse(): [L^-1, -L^-1 t], L inverted as a general 3x3
__device__ __forceinline__ void rg_affine_inverse(const double* T, double* Ti) {
    double L[9] = {T[0], T[1], T[2], T[4], T[5], T[6], T[8], T[9], T[10]}, Li[9];
    rg_inv3(L, Li);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) Ti[4 * r + c] = Li[3 * r + c];
        Ti[4 * r + 3] = -((Li[3 * r] * T[3] + Li[3 * r + 1] * T[7]) + Li[3 * r + 2] * T[11]);
    }
    Ti[12] = Ti[13] = Ti[14] = 0.0; Ti[15] = 1.0;
}

// one selected reference pixel against the now frame (:640-672); returns true when it is seen
__device__ __forceinline__ bool rg_project(int i, int j, double Z, const RgCam& K, const double* Ti, int rows, int cols, int& fu, int& fv) {
    double X, Y; rg_xyz(i, j, Z, K, X, Y);
    const double o0 = ((Ti[0] * X + Ti[1] * Y) + Ti[2] * Z) + Ti[3];
    const double o1 = ((Ti[4] * X + Ti[5] * Y) + Ti[6] * Z) + Ti[7];
    const double o2 = ((Ti[8] * X + Ti[9] * Y) + Ti[10] * Z) + Ti[11];
    const double outu = o0 * K.fx / o2 + K.cx, outv = o1 * K.fy / o2 + K.cy;      // :650-651
    if (!(outu >= 0 && outu < (double)rows && outv >= 0 && outv < (double)cols)) return false;   // :664 (outu is a row coordinate)
    fu = (int)floor(outu); fv = (int)floor(outv);
    return true;
}

// exponentialMap (:707-745)
__device__ __forceinline__ void rg_exponential_map(const double* psi, double* out16) {
    const double* t = psi; const double* w = psi + 3;
    const double theta = sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
    for (int k = 0; k < 16; ++k) out16[k] = (k % 5 == 0) ? 1.0 : 0.0;
    if (theta < 1E-12) return;
    const double wx[9] = {0, -w[2], w[1], w[2], 0, -w[0], -w[1], w[0], 0};
    double wx2[9];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) wx2[3 * r + c] = (wx[3 * r] * wx[c] + wx[3 * r + 1] * wx[3 + c]) + wx[3 * r + 2] * wx[6 + c];
    const double a = sin(theta) / theta, b = (1.0 - cos(theta)) / (theta * theta), c3 = (theta - sin(theta)) / (theta * theta * theta);
    double V[9];
    for (int k = 0; k < 9; ++k) {
        const double I = (k % 4 == 0) ? 1.0 : 0.0;
        out16[4 * (k / 3) + (k % 3)] = (I + a * wx[k]) + b * wx2[k];
        V[k] = (I + b * wx[k]) + c3 * wx2[k];
    }
    for (int r = 0; r < 3; ++r) out16[4 * r + 3] = (V[3 * r] * t[0] + V[3 * r + 1] * t[1]) + V[3 * r + 2] * t[2];
}

// A.colPivHouseholderQr().solve(b) (:563), 6x6: Householder QR with column pivoting on the largest remaining column norm
__device__ void rg_qr_solve6(const double* Ain, const double* bin, double* x) {
    double A[36], b[6]; int perm[6];
    for (int k = 0; k < 36; ++k) A[k] = Ain[k];
    for (int k = 0; k < 6; ++k) { b[k] = bin[k]; perm[k] = k; }
    for (int k = 0; k < 6; ++k) {
        int piv = k; double best = -1.0;
        for (int c = k; c < 6; ++c) { double n2 = 0; for (int r = k; r < 6; ++r) n2 += A[6 * r + c] * A[6 * r + c]; if (n2 > best) { best = n2; piv = c; } }
        if (piv != k) { for (int r = 0; r < 6; ++r) { const double t = A[6 * r + k]; A[6 * r + k] = A[6 * r + piv]; A[6 * r + piv] = t; } const int t = perm[k]; perm[k] = perm[piv]; perm[piv] = t; }
        const double nrm = sqrt(best);
        if (nrm == 0.0) continue;
        const double alpha = (A[6 * k + k] > 0) ? -nrm : nrm;
        double v[6] = {0, 0, 0, 0, 0, 0};
        for (int r = k; r < 6; ++r) v[r] = A[6 * r + k];
        v[k] -= alpha;
        double vv = 0; for (int r = k; r < 6; ++r) vv += v[r] * v[r];
        if (vv == 0.0) continue;
        for (int c = k; c < 6; ++c) { double d = 0; for (int r = k; r < 6; ++r) d += v[r] * A[6 * r + c]; d = 2.0 * d / vv; for (int r = k; r < 6; ++r) A[6 * r + c] -= d * v[r]; }
        { double d = 0; for (int r = k; r < 6; ++r) d += v[r] * b[r]; d = 2.0 * d / vv; for (int r = k; r < 6; ++r) b[r] -= d * v[r]; }
    }
    double y[6];
    for (int r = 5; r >= 0; --r) {
        double sacc = b[r]; for (int c = r + 1; c < 6; ++c) sacc -= A[6 * r + c] * y[c];
        y[r] = (A[6 * r + r] != 0.0) ? sacc / A[6 * r + r] : 0.0;
    }
    for (int k = 0; k < 6; ++k) x[perm[k]] = y[k];
}

__device__ __forceinline__ void rg_mat4_mul(const double* A, const double* B, double* C) {
    double r[16];
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) r[4 * i + j] = ((A[4 * i] * B[j] + A[4 * i + 1] * B[4 + j]) + A[4 * i + 2] * B[8 + j]) + A[4 * i + 3] * B[12 + j];
    for (int k = 0; k < 16; ++k) C[k] = r[k];
}

// fixed-order block reduction of NV doubles per thread (shuffle tree, then warp partials in warp order)
template <int NV>
__device__ __forceinline__ void rg_block_reduce(double* v, double (*s_red)[NV], double* s_tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (lane == 0) s_red[warp][k] = x;
    }
    __syncthreads();
    if (threadIdx.x < NV) { double x = 0.0; for (int w = 0; w < RG_THREADS / 32; ++w) x += s_red[w][threadIdx.x]; s_tot[threadIdx.x] = x; }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------
// setRefFrame / setNowFrame (:330-390): gray = BGR2GRAY(full); level l = INTER_NEAREST(2^-l) of gray and depth.  One thread
// per output pixel of every level; the 15-bit BGR2GRAY is evaluated at the source pixel (same value as resizing the gray).
__global__ void __launch_bounds__(256) rg_pyramid_kernel(RgGeom g, const uint8_t* __restrict__ bgr, const uint16_t* __restrict__ depth_in,
                                                         uint8_t* __restrict__ gray, uint16_t* __restrict__ depth, int first) {
    const int l = blockIdx.z, b = first + blockIdx.y, slot_in = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.P[l]) return;
    const int w = g.w[l], s = 1 << l;
    const int y = p / w, x = p - y * w;
    const int sy = min(y * s, g.H - 1), sx = min(x * s, g.W - 1);
    const long long src = ((long long)slot_in * g.H + sy) * g.W + sx;
    const uint8_t* q = bgr + 3 * src;
    gray[rg_at(g, l, b) + p] = (uint8_t)((q[0] * 3735 + q[1] * 19235 + q[2] * 9798 + (1 << 14)) >> 15);
    const uint16_t d = depth_in[src];
    depth[rg_at(g, l, b) + p] = d ? d : (uint16_t)1;                              // imageArrivedCallBack: dframe.setTo(1, dframe == 0) (:232)
}

// computeJacobianAllLevels (:393-415): A = J^T J and the number of selected pixels for levels 1..L-1; one CTA per (pair, level)
__global__ void __launch_bounds__(RG_THREADS) rg_jacobian_kernel(RgGeom g, RgCam K, const uint8_t* __restrict__ gray, const uint16_t* __restrict__ depth,
                                                                 double* __restrict__ A, int* __restrict__ npts, int first, int thresh) {
    __shared__ double s_red[RG_THREADS / 32][22];
    __shared__ double s_tot[22];
    const int l = 1 + blockIdx.y, b = first + blockIdx.x;
    const int rows = g.h[l], cols = g.w[l];
    const uint8_t* G = gray + rg_at(g, l, b); const uint16_t* D = depth + rg_at(g, l, b);
    double acc[22];
#pragma unroll
    for (int k = 0; k < 22; ++k) acc[k] = 0.0;
    for (int p = threadIdx.x; p < rows * cols; p += RG_THREADS) {
        const int i = p / cols, j = p - i * cols;
        double gx, gy; rg_gradients(G, rows, cols, i, j, gx, gy);
        if (gx < (double)thresh) continue;                                        // :465
        const double Z = (double)D[p];
        double X, Y; rg_xyz(i, j, Z, K, X, Y);
        double r[6]; rg_jrow(gx, gy, X, Y, Z, K, r);
        int idx = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int c = a; c < 6; ++c) { acc[idx] += r[a] * r[c]; ++idx; }
        acc[21] += 1.0;
    }
    rg_block_reduce<22>(acc, s_red, s_tot);
    if (threadIdx.x == 0) {
        double* Ao = A + ((long long)b * g.L + l) * 36;
        int idx = 0;
        for (int a = 0; a < 6; ++a) for (int c = a; c < 6; ++c) { Ao[6 * a + c] = s_tot[idx]; Ao[6 * c + a] = s_tot[idx]; ++idx; }
        npts[(long long)b * g.L + l] = (int)s_tot[21];
    }
}

struct RgGnArgs {
    RgGeom g; RgCam K;
    const uint8_t *ref_gray, *now_gray; const uint16_t* ref_depth;
    const double* A; const int* npts; RgState* st;
    int first, level, iters, thresh, min_pts, max_pts; double eps_exit;
};

// gaussNewtonIterations(level, T) (:514-597) for one pair per CTA
__global__ void __launch_bounds__(RG_THREADS) rg_gn_kernel(RgGnArgs a) {
    __shared__ double s_red[RG_THREADS / 32][8];
    __shared__ double s_tot[8];
    __shared__ double s_Ti[16];
    __shared__ int s_stop;
    const int b = a.first + blockIdx.x, l = a.level;
    const int rows = a.g.h[l], cols = a.g.w[l];
    const uint8_t* G = a.ref_gray + rg_at(a.g, l, b); const uint16_t* D = a.ref_depth + rg_at(a.g, l, b);
    const uint8_t* N = a.now_gray + rg_at(a.g, l, b);
    RgState& S = a.st[b];
    const int n = a.npts[(long long)b * a.g.L + l];
    if (threadIdx.x == 0) {
        S.info.npts[l] = n; S.info.iters_run[l] = 0; S.info.updates[l] = 0; S.info.nvis_last[l] = 0; S.info.eps_norm_first[l] = 0.0; S.info.eps_norm_last[l] = 0.0;
        if (n <= a.min_pts) S.info.status |= 1;                                   // the reference asserts (:497)
        if (n > a.max_pts) S.info.status |= 2;                                    // (:463)
    }
    for (int itr = 0; itr < a.iters; ++itr) {
        if (threadIdx.x == 0) { double Ti[16]; rg_affine_inverse(S.T, Ti); for (int k = 0; k < 16; ++k) s_Ti[k] = Ti[k]; }
        __syncthreads();
        double Ti[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) Ti[k] = s_Ti[k];
        double acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.0;
        for (int p = threadIdx.x; p < rows * cols; p += RG_THREADS) {
            const int i = p / cols, j = p - i * cols;
            double gx, gy; rg_gradients(G, rows, cols, i, j, gx, gy);
            if (gx < (double)a.thresh) continue;
            const double Z = (double)D[p];
            int fu, fv;
            if (!rg_project(i, j, Z, a.K, Ti, rows, cols, fu, fv)) continue;      // unseen: eps = 0 (:664-669)
            const double e = (double)G[p] - (double)N[(size_t)fu * cols + fv];
            double X, Y; rg_xyz(i, j, Z, a.K, X, Y);
            double r[6]; rg_jrow(gx, gy, X, Y, Z, a.K, r);
#pragma unroll
            for (int c = 0; c < 6; ++c) acc[c] -= r[c] * e;                       // b = -J^T eps (:562)
            acc[6] += e * e; acc[7] += 1.0;
        }
        rg_block_reduce<8>(acc, s_red, s_tot);
        if (threadIdx.x == 0) {
            const double nrm = sqrt(s_tot[6]);
            if (itr == 0) S.info.eps_norm_first[l] = nrm;
            S.info.eps_norm_last[l] = nrm; S.info.nvis_last[l] = (int)s_tot[7]; S.info.iters_run[l] = itr + 1;
            int stop = 0;
            if (nrm < a.eps_exit) stop = 1;                                       // :556
            else {
                double b6[6], psi[6];
                for (int k = 0; k < 6; ++k) b6[k] = s_tot[k];
                rg_qr_solve6(a.A + ((long long)b * a.g.L + l) * 36, b6, psi);     // :563
                double E[16], Ei[16];
                rg_exponential_map(psi, E); rg_affine_inverse(E, Ei);
                rg_mat4_mul(S.T, Ei, S.T);                                        // :579
                S.info.updates[l] += 1;
            }
            s_stop = stop;
        }
        __syncthreads();
        if (s_stop) break;
    }
}

// inspection: dense per-pixel view of one (slot, level) at pose T: selection flag, Jacobian row, residual, floor(u, v)
__global__ void __launch_bounds__(256) rg_eval_kernel(RgGeom g, RgCam K, const uint8_t* __restrict__ ref_gray, const uint16_t* __restrict__ ref_depth,
                                                      const uint8_t* __restrict__ now_gray, int slot, int level, const double* __restrict__ T16, int thresh,
                                                      uint8_t* __restrict__ sel, double* __restrict__ J, double* __restrict__ eps, int* __restrict__ uv) {
    const int rows = g.h[level], cols = g.w[level];
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= rows * cols) return;
    const uint8_t* G = ref_gray + rg_at(g, level, slot); const uint16_t* D = ref_depth + rg_at(g, level, slot);
    const uint8_t* N = now_gray + rg_at(g, level, slot);
    const int i = p / cols, j = p - i * cols;
    double gx, gy; rg_gradients(G, rows, cols, i, j, gx, gy);
    sel[p] = 0; eps[p] = 0.0; uv[2 * p] = -1; uv[2 * p + 1] = -1;
    for (int k = 0; k < 6; ++k) J[6 * (size_t)p + k] = 0.0;
    if (gx < (double)thresh) return;
    sel[p] = 1;
    const double Z = (double)D[p];
    double X, Y; rg_xyz(i, j, Z, K, X, Y);
    double r[6]; rg_jrow(gx, gy, X, Y, Z, K, r);
    for (int k = 0; k < 6; ++k) J[6 * (size_t)p + k] = r[k];
    double T[16], Ti[16];
    for (int k = 0; k < 16; ++k) T[k] = T16[k];
    rg_affine_inverse(T, Ti);
    int fu, fv;
    if (rg_project(i, j, Z, K, Ti, rows, cols, fu, fv)) {
        eps[p] = (double)G[p] - (double)N[(size_t)fu * cols + fv];
        uv[2 * p] = fu; uv[2 * p + 1] = fv;
    }
}

__global__ void rg_set_pose_kernel(RgState* st, int first, int count, const double* __restrict__ T16) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    RgState& S = st[first + k];
    for (int q = 0; q < 16; ++q) S.T[q] = T16 ? T16[16 * (size_t)k + q] : ((q % 5 == 0) ? 1.0 : 0.0);
    S.info.status = 0;
}

// ------------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------------
namespace {
bool rg_range_ok(dvo_rgbd_ctx* c, int first, int count) { return c && first >= 0 && count >= 0 && first + count <= c->cfg.max_batch; }
int rg_level_dim(int dim, int level) { return (int)nearbyint((double)dim * ldexp(1.0, -level)); }     // cv::resize: cvRound(dim * scale)
}  // namespace

extern "C" {

int dvo_rgbd_create(const dvo_rgbd_config* cfg, dvo_rgbd_ctx** out) {
    if (!cfg || !out || cfg->width < 8 || cfg->height < 8 || cfg->levels < 2 || cfg->levels > RG_MAX_LEVELS || cfg->max_batch < 1 || cfg->max_batch > 65535) {
        dvo_set_error("dvo_rgbd_create: bad configuration"); return DVO_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { dvo_set_error("dvo_rgbd_create: no usable CUDA device (there is no CPU fallback)"); return DVO_ERR_CUDA; }
    DVO_CUDA(cudaSetDevice(cfg->device));
    dvo_rgbd_ctx* c = new (std::nothrow) dvo_rgbd_ctx();
    if (!c) return DVO_ERR_NOMEM;
    c->cfg = *cfg;
    RgGeom& g = c->g;
    g.L = cfg->levels; g.Bmax = cfg->max_batch; g.W = cfg->width; g.H = cfg->height;
    long long off = 0;
    for (int l = 0; l < g.L; ++l) { g.w[l] = rg_level_dim(g.W, l); g.h[l] = rg_level_dim(g.H, l); g.P[l] = g.w[l] * g.h[l]; g.off[l] = off; off += (long long)g.P[l] * g.Bmax; }
    g.total = off;
    cudaError_t e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    c->stream = c->own_stream;
    const size_t B = (size_t)g.Bmax, P0 = (size_t)g.P[0];
    int rc = DVO_OK;
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    if (e == cudaSuccess) {
        A(c->bgr.reserve(B * P0 * 3)); A(c->depth_in.reserve(B * P0));
        for (int f = 0; f < 2; ++f) { A(c->gray[f].reserve((size_t)g.total)); A(c->depth[f].reserve((size_t)g.total)); }
        A(c->A.reserve(B * g.L * 36)); A(c->npts.reserve(B * g.L)); A(c->st.reserve(B)); A(c->pose_stage.reserve(B * 16));
        if (rc) { dvo_rgbd_destroy(c); return rc; }
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(c->npts, 0, sizeof(int) * B * g.L, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->st, 0, sizeof(RgState) * B, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->A, 0, sizeof(double) * B * g.L * 36, c->stream);
    if (e != cudaSuccess) { dvo_set_error("dvo_rgbd_create: %s", cudaGetErrorString(e)); dvo_rgbd_destroy(c); return DVO_ERR_CUDA; }
    *out = c;
    return DVO_OK;
}

int dvo_rgbd_destroy(dvo_rgbd_ctx* c) {
    if (!c) return DVO_OK;
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return DVO_OK;
}

int dvo_rgbd_set_stream(dvo_rgbd_ctx* c, void* s) { if (!c) return DVO_ERR_ARG; c->stream = s ? (cudaStream_t)s : c->own_stream; return DVO_OK; }
int dvo_rgbd_synchronize(dvo_rgbd_ctx* c) { if (!c) return DVO_ERR_ARG; DVO_CUDA(cudaStreamSynchronize(c->stream)); return DVO_OK; }
long long dvo_rgbd_launch_count(dvo_rgbd_ctx* c) { return c ? c->launches : 0; }

int dvo_rgbd_set_intrinsics(dvo_rgbd_ctx* c, double fx, double fy, double cx, double cy) {
    if (!c) return DVO_ERR_ARG;
    c->K.fx = fx; c->K.fy = fy; c->K.cx = cx; c->K.cy = cy; c->haveK = true;
    return DVO_OK;
}

// setRefFrame / setNowFrame (:330-390) for slots [first, first + count): BGR u8 HWC + depth u16 (0 is replaced by 1 at
// ingest like imageArrivedCallBack :232 does)
int dvo_rgbd_set_frames(dvo_rgbd_ctx* c, int frame, int first, int count, const uint8_t* bgr, const uint16_t* depth, int mem) {
    if (!rg_range_ok(c, first, count) || (frame != 0 && frame != 1) || !bgr || !depth) { dvo_set_error("dvo_rgbd_set_frames: bad argument"); return DVO_ERR_ARG; }
    if (count == 0) return DVO_OK;
    const RgGeom& g = c->g;
    const size_t P0 = (size_t)g.P[0];
    const cudaMemcpyKind kind = (mem == DVO_MEM_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    DVO_CUDA(cudaMemcpyAsync(c->bgr, bgr, P0 * 3 * count, kind, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->depth_in, depth, P0 * 2 * count, kind, c->stream));
    dim3 grid((unsigned)((g.P[0] + 255) / 256), (unsigned)count, (unsigned)g.L);
    rg_pyramid_kernel<<<grid, 256, 0, c->stream>>>(g, c->bgr, c->depth_in, c->gray[frame], c->depth[frame], first);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_rgbd_compute_jacobians(dvo_rgbd_ctx* c, int first, int count, int gradient_threshold) {
    if (!rg_range_ok(c, first, count)) { dvo_set_error("dvo_rgbd_compute_jacobians: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_rgbd_compute_jacobians: intrinsics not set"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    dim3 grid((unsigned)count, (unsigned)(c->g.L - 1));
    rg_jacobian_kernel<<<grid, RG_THREADS, 0, c->stream>>>(c->g, c->K, c->gray[0], c->depth[0], c->A, c->npts, first, gradient_threshold);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_rgbd_set_pose(dvo_rgbd_ctx* c, int first, int count, const double* T16) {
    if (!rg_range_ok(c, first, count)) return DVO_ERR_ARG;
    if (count == 0) return DVO_OK;
    double* d = nullptr;
    if (T16) {      // pageable host memory: the copy is staged by the runtime before the call returns, so T16 may be reused at once
        d = c->pose_stage + 16 * (size_t)first;
        DVO_CUDA(cudaMemcpyAsync(d, T16, sizeof(double) * 16 * count, cudaMemcpyHostToDevice, c->stream));
    }
    rg_set_pose_kernel<<<(count + 127) / 128, 128, 0, c->stream>>>(c->st, first, count, d);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_rgbd_gauss_newton(dvo_rgbd_ctx* c, int first, int count, int level, const dvo_rgbd_params* p) {
    if (!rg_range_ok(c, first, count) || !p) { dvo_set_error("dvo_rgbd_gauss_newton: bad argument"); return DVO_ERR_ARG; }
    if (level < 1 || level >= c->g.L) { dvo_set_error("dvo_rgbd_gauss_newton: level must be in [1, levels) -- Jacobians at level 0 are not computed (src/RGBDOdometry.cpp:518)"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_rgbd_gauss_newton: intrinsics not set"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    RgGnArgs a;
    a.g = c->g; a.K = c->K; a.ref_gray = c->gray[0]; a.now_gray = c->gray[1]; a.ref_depth = c->depth[0]; a.A = c->A; a.npts = c->npts; a.st = c->st;
    a.first = first; a.level = level; a.iters = p->iterations; a.thresh = p->gradient_threshold; a.min_pts = p->min_points; a.max_pts = p->max_points;
    a.eps_exit = p->eps_norm_exit;
    rg_gn_kernel<<<count, RG_THREADS, 0, c->stream>>>(a);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_rgbd_get_poses(dvo_rgbd_ctx* c, int first, int count, double* T16, dvo_rgbd_info* info) {
    if (!rg_range_ok(c, first, count)) return DVO_ERR_ARG;
    if (count == 0) return DVO_OK;
    std::vector<RgState> h((size_t)count);
    DVO_CUDA(cudaMemcpyAsync(h.data(), c->st + first, sizeof(RgState) * count, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    for (int k = 0; k < count; ++k) {
        if (T16) memcpy(T16 + 16 * (size_t)k, h[k].T, sizeof(double) * 16);
        if (info) info[k] = h[k].info;
    }
    return DVO_OK;
}

int dvo_rgbd_level_dims(dvo_rgbd_ctx* c, int level, int* rows, int* cols) {
    if (!c || level < 0 || level >= c->g.L) return DVO_ERR_ARG;
    if (rows) *rows = c->g.h[level];
    if (cols) *cols = c->g.w[level];
    return DVO_OK;
}

int dvo_rgbd_get_level(dvo_rgbd_ctx* c, int slot, int frame, int level, uint8_t* gray, uint16_t* depth) {
    if (!rg_range_ok(c, slot, 1) || (frame != 0 && frame != 1) || level < 0 || level >= c->g.L) return DVO_ERR_ARG;
    const size_t P = (size_t)c->g.P[level];
    if (gray) DVO_CUDA(cudaMemcpyAsync(gray, c->gray[frame] + rg_at(c->g, level, slot), P, cudaMemcpyDeviceToHost, c->stream));
    if (depth) DVO_CUDA(cudaMemcpyAsync(depth, c->depth[frame] + rg_at(c->g, level, slot), P * 2, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_rgbd_get_A(dvo_rgbd_ctx* c, int slot, int level, double* A36, int* npts) {
    if (!rg_range_ok(c, slot, 1) || level < 1 || level >= c->g.L) return DVO_ERR_ARG;
    if (A36) DVO_CUDA(cudaMemcpyAsync(A36, c->A + ((size_t)slot * c->g.L + level) * 36, sizeof(double) * 36, cudaMemcpyDeviceToHost, c->stream));
    if (npts) DVO_CUDA(cudaMemcpyAsync(npts, c->npts + (size_t)slot * c->g.L + level, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// computeJacobian + computeEpsilon of one slot / level at pose T, returned in the reference's enumeration order (column
// outer, row inner, :459-462): ij (row, col), J (n x 6), eps, uv = floor(outu, outv) or -1.  Returns the count in *n.
int dvo_rgbd_eval(dvo_rgbd_ctx* c, int slot, int level, const double* T16, int gradient_threshold, int capacity, int* n, int* ij, double* J,
                  double* eps, int* uv, double* b6, double* sumsq, int* nvis) {
    if (!rg_range_ok(c, slot, 1) || level < 1 || level >= c->g.L || !T16 || !n) { dvo_set_error("dvo_rgbd_eval: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_rgbd_eval: intrinsics not set"); return DVO_ERR_STATE; }
    const int rows = c->g.h[level], cols = c->g.w[level];
    const size_t P = (size_t)rows * cols;
    DevBuf<uint8_t> d_sel; DevBuf<double> d_J, d_eps, d_T; DevBuf<int> d_uv;
    int rc;
    if ((rc = d_sel.reserve(P)) || (rc = d_J.reserve(6 * P)) || (rc = d_eps.reserve(P)) || (rc = d_uv.reserve(2 * P)) || (rc = d_T.reserve(16))) return rc;
    cudaError_t e = cudaMemcpyAsync(d_T, T16, sizeof(double) * 16, cudaMemcpyHostToDevice, c->stream);
    std::vector<uint8_t> h_sel(P); std::vector<double> h_J(6 * P), h_eps(P); std::vector<int> h_uv(2 * P);
    if (e == cudaSuccess) {
        rg_eval_kernel<<<(unsigned)((P + 255) / 256), 256, 0, c->stream>>>(c->g, c->K, c->gray[0], c->depth[0], c->gray[1], slot, level, d_T, gradient_threshold,
                                                                          d_sel, d_J, d_eps, d_uv);
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_sel.data(), d_sel, P, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_J.data(), d_J, sizeof(double) * 6 * P, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_eps.data(), d_eps, sizeof(double) * P, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_uv.data(), d_uv, sizeof(int) * 2 * P, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { dvo_set_error("dvo_rgbd_eval: %s", cudaGetErrorString(e)); return DVO_ERR_CUDA; }
    int k = 0, seen = 0; double ss = 0.0, b[6] = {0, 0, 0, 0, 0, 0};
    for (int j = 0; j < cols; ++j)
        for (int i = 0; i < rows; ++i) {
            const size_t p = (size_t)i * cols + j;
            if (!h_sel[p]) continue;
            if (k < capacity) {
                if (ij) { ij[2 * k] = i; ij[2 * k + 1] = j; }
                if (J) memcpy(J + 6 * (size_t)k, &h_J[6 * p], sizeof(double) * 6);
                if (eps) eps[k] = h_eps[p];
                if (uv) { uv[2 * k] = h_uv[2 * p]; uv[2 * k + 1] = h_uv[2 * p + 1]; }
            }
            if (h_uv[2 * p] >= 0) { ++seen; ss += h_eps[p] * h_eps[p]; for (int q = 0; q < 6; ++q) b[q] -= h_J[6 * p + q] * h_eps[p]; }
            ++k;
        }
    *n = k;
    if (b6) memcpy(b6, b, sizeof(b));
    if (sumsq) *sumsq = ss;
    if (nvis) *nvis = seen;
    return DVO_OK;
}

}  // extern "C"
