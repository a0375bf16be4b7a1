// photometric.cu -- EPoseEstimator / PyramidalStorageStruct on the GPU (SURVEY.md §8 rows R12-R17).
//
// Dense photometric estimator with a reference-frame Jacobian (src/EPoseEstimator.cpp).  Everything the reference
// caches per level in PyramidalStorageStruct (X, Y, Z, J, gray / colour arrays; src/PyramidalStorage.cpp:38-102) is a
// pure function of the level's u8 gray, u16 depth and the pixel index, so the kernels recompute it on the fly from
// ~5 bytes per pixel instead of re-reading 48-byte fp64 Jacobian rows; dvo_photo_get_level materialises any of those
// arrays on demand for callers that want the storage view.
//
// `compat` = 1 reproduces the reference bug for bug (SURVEY Appendix C: duplicated Jacobian column, row index paired
// with cx, unscaled fx, residual flattened row-major against column-major J rows, holes count as residuals);
// `compat` = 0 is the corrected formulation with Huber weights and LM damping (BASELINE config 3).
//
// This translation unit is compiled with -fmad=false: every fp64 expression is evaluated in the written order with one
// rounding per operation, exactly like the CPU oracle (-ffp-contract=off), so per-pixel quantities are bit-identical.
#include <math.h>
#include <stdlib.h>

#include <new>
#include <vector>

#include "common.cuh"

#define PH_MAX_LEVELS 5
#define PH_NACC 30          // b[6], sumsq, nused, 21 upper-triangle entries of A, nreproj(unused slot)
#define PH_THREADS 256

struct PhGeom { int L, Bmax, W, H; int w[PH_MAX_LEVELS], h[PH_MAX_LEVELS], P[PH_MAX_LEVELS]; long long off[PH_MAX_LEVELS]; long long total; };
__host__ __device__ inline long long ph_at(const PhGeom& g, int l, int b) { return g.off[l] + (long long)b * g.P[l]; }

struct PhCam { double fx, fy, cx, cy; double ifx, ify; };     // ifx / ify: 1 / (sf fx), 1 / (sf fy) of the level a launch works on

// per-pair solver state (global memory)
struct PhState {
    double Tr[16], accTr[16], accA[36], accb[6];
    double accE, lambda, sumsq_first, sumsq_last, visible;
    int have, status, iters_run, stop, nreproj;
    int nreproj_last;      // nReprojected of the last warp an estimate() consumed (nreproj itself is the running counter)
};

struct dvo_photo_ctx {
    dvo_photo_config cfg; PhGeom g; PhCam K; bool haveK;
    cudaStream_t own_stream, stream;
    DevBuf<uint8_t> bgr[2];      // full resolution, [Bmax][H][W][3]
    DevBuf<uint8_t> gray[2];     // AREA pyramid of the full-resolution gray
    DevBuf<uint16_t> depth[2];   // AREA pyramid of depth (now: stored for API completeness)
    DevBuf<int> winner;          // [Bmax][P0]: per target cell the winning source pixel as (column << 16) | row, -1 = hole
    DevBuf<double> partial;      // [Bmax][maxblk][PH_NACC]
    DevBuf<double> A;            // [Bmax][L][36]   J^T J of the reference frame
    DevBuf<PhState> st;          // [Bmax]
    int maxblk;
    long long launches;
};

// ------------------------------------------------------------------------------------------------------
// per-pixel quantities (mirror oracle/dvo_oracle.hpp photo::build_ref_level line by line)
// ------------------------------------------------------------------------------------------------------
struct PixGeom { double X, Y, Z; };

__device__ __forceinline__ PixGeom ph_xyz(int r, int c, double Zmm, double sf, const PhCam& K, bool compat) {
    PixGeom o;
    if (compat) {                                   // src/EPoseEstimator.cpp:466-472
        double X = Zmm / K.fx * ((double)r - sf * K.cx), Y = Zmm / K.fy * ((double)c - sf * K.cy);
        o.X = X / 1000.; o.Y = Y / 1000.; o.Z = Zmm / 1000.;
    } else {
        // corrected formulation (oracle photo::build_ref_level): reciprocal focal lengths once per level (K.ifx / K.ify are
        // 1 / (sf fx), 1 / (sf fy) of THIS level, set by ph_args), metres by a multiply -- no division per pixel
        o.Z = Zmm * 1.0e-3;
        o.X = (o.Z * ((double)c - sf * K.cx)) * K.ifx; o.Y = (o.Z * ((double)r - sf * K.cy)) * K.ify;
    }
    return o;
}

// forward differences with REFLECT_101 (:331-339)
__device__ __forceinline__ void ph_grad(const uint8_t* __restrict__ g, int rows, int cols, int r, int c, double& gx, double& gy) {
    const int c1 = (c + 1 < cols) ? c + 1 : cols - 2, r1 = (r + 1 < rows) ? r + 1 : rows - 2;
    const double v = (double)g[r * cols + c];
    gx = (double)g[r * cols + (cols > 1 ? c1 : c)] - v;
    gy = (double)g[(rows > 1 ? r1 : r) * cols + c] - v;
}

// Jacobian row of pixel (r,c)  (:390-395, :415) from its depth and forward differences
__device__ __forceinline__ void ph_jrow_vals(double Zmm, double egx, double egy, int r, int c, double sf, const PhCam& K, bool compat, double* J) {
    const PixGeom p = ph_xyz(r, c, Zmm, sf, K, compat);
    const double fx = K.fx, fy = K.fy, X = p.X, Y = p.Y, Z = p.Z;
    if (compat) {
        const double Z_inv = 1.0 / Z, Z2_inv = 1.0 / (Z * Z);
        const double J1 = fx * egx * Z_inv;
        const double J2 = fy * egy * Z_inv;
        const double J3 = -fy * egy * Y * Z2_inv - fx * egx * X * Z2_inv;
        const double J4 = egy * (-fy * Y * Y * Z2_inv - fy) - fx * egx * X * Y * Z2_inv;
        const double J6 = fy * egy * X * Z_inv - fx * egy * Y * Z_inv;
        J[0] = J1; J[1] = J2; J[2] = J3; J[3] = J4; J[4] = J4; J[5] = J6;
    } else if (Zmm > 0.0) {
        const double fxs = sf * fx, fys = sf * fy, Z_inv = 1.0 / Z;
        const double J1 = fxs * egx * Z_inv, J2 = fys * egy * Z_inv, J3 = -(J1 * X + J2 * Y) * Z_inv;
        J[0] = J1; J[1] = J2; J[2] = J3; J[3] = J3 * Y - J2 * Z; J[4] = J1 * Z - J3 * X; J[5] = J2 * X - J1 * Y;
    } else { for (int k = 0; k < 6; ++k) J[k] = 0.0; }
}
__device__ __forceinline__ void ph_jrow(const uint8_t* __restrict__ g, const uint16_t* __restrict__ d, int rows, int cols, int r, int c,
                                        double sf, const PhCam& K, bool compat, double* J) {
    double egx, egy; ph_grad(g, rows, cols, r, c, egx, egy);
    ph_jrow_vals((double)d[r * cols + c], egx, egy, r, c, sf, K, compat, J);
}

// deterministic block reduction of PH_NACC doubles into partial[blockIdx]
__device__ __forceinline__ void ph_block_reduce(double* acc, double* out) {
    __shared__ double s_red[PH_THREADS / 32][PH_NACC];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < PH_NACC; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) s_red[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < PH_NACC) {
        double v = 0.0;
#pragma unroll
        for (int wv = 0; wv < PH_THREADS / 32; ++wv) v += s_red[wv][threadIdx.x];
        out[threadIdx.x] = v;
    }
}

// ------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ph_gray_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int b = bgr[3 * i], g = bgr[3 * i + 1], r = bgr[3 * i + 2];
    gray[i] = (uint8_t)((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15);       // OpenCV 4.x BGR2GRAY (SURVEY B.7)
}

// INTER_AREA with integer scale 2^l from full resolution (SURVEY B.5)
template <typename T, int CH>
__global__ void __launch_bounds__(256) ph_area_kernel(const T* __restrict__ src, T* __restrict__ dst, int W, int H, int l, long long src_stride,
                                                       long long dst_stride) {
    const int s = 1 << l, w = W >> l, h = H >> l;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= w * h) return;
    const T* sp = src + (long long)blockIdx.y * src_stride;
    T* dp = dst + (long long)blockIdx.y * dst_stride;
    const int y = q / w, x = q - y * w;
    const float inv_area = (float)(1.0 / (double)(s * s));
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        int sum = 0;
        for (int dy = 0; dy < s; ++dy)
            for (int dx = 0; dx < s; ++dx) sum += (int)sp[((long long)(y * s + dy) * W + (x * s + dx)) * CH + c];
        int o;
        if (l == 1) o = (sum + 2) >> 2;
        else o = __float2int_rn(__fmul_rn((float)sum, inv_area));                  // rint half-to-even
        dp[(long long)q * CH + c] = (T)o;
    }
}

struct PhArgs {
    PhGeom g; PhCam K; double sf;
    const uint8_t* gray_ref; const uint16_t* depth_ref; const uint8_t* gray_now;   // level regions (slot 0)
    int* winner; double* partial; double* A; PhState* st;
    int level, rows, cols, P, first, compat, nblk, maxblk; double huber_k, lambda0;
    int reset_winner;      // ph_accum_kernel hands the winner map back cleared (the estimate loop then needs no clear pass per iteration)
};

// A = J^T J over the reference level (setPyramidalImages :229)
__global__ void __launch_bounds__(PH_THREADS) ph_A_kernel(PhArgs a) {
    const int b = a.first + blockIdx.y;
    const uint8_t* g = a.gray_ref + (long long)b * a.P; const uint16_t* d = a.depth_ref + (long long)b * a.P;
    double acc[PH_NACC];
#pragma unroll
    for (int k = 0; k < PH_NACC; ++k) acc[k] = 0.0;
    for (int i = blockIdx.x * PH_THREADS + threadIdx.x; i < a.P; i += gridDim.x * PH_THREADS) {
        const int r = i / a.cols, c = i - r * a.cols;
        double J[6]; ph_jrow(g, d, a.rows, a.cols, r, c, a.sf, a.K, a.compat != 0, J);
        int idx = 8;
#pragma unroll
        for (int p = 0; p < 6; ++p)
#pragma unroll
            for (int q = p; q < 6; ++q) { acc[idx] += J[p] * J[q]; ++idx; }
    }
    ph_block_reduce(acc, a.partial + ((long long)b * a.maxblk + blockIdx.x) * PH_NACC);
}

__global__ void __launch_bounds__(64) ph_A_final_kernel(PhArgs a) {
    const int b = a.first + blockIdx.x;
    __shared__ double tot[PH_NACC];
    if (threadIdx.x < PH_NACC) {
        double v = 0.0;
        for (int k = 0; k < a.nblk; ++k) v += a.partial[((long long)b * a.maxblk + k) * PH_NACC + threadIdx.x];
        tot[threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double* A = a.A + ((long long)b * a.g.L + a.level) * 36;
        int idx = 8;
        for (int p = 0; p < 6; ++p) for (int q = p; q < 6; ++q) { A[6 * p + q] = tot[idx]; A[6 * q + p] = tot[idx]; ++idx; }
    }
}

__global__ void __launch_bounds__(256) ph_clear_kernel(PhArgs a) {
    const int b = a.first + blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.P) a.winner[(long long)b * a.g.P[0] + i] = -1;
    if (i == 0) a.st[b].nreproj = 0;
}

// warpImage (:490-553): forward splat; "last writer wins" in column-major pixel order == max source index per cell.
// PH_SPLAT_PX pixels per thread (256 apart, so every load and the sources of a warp stay coalesced): the depth loads of all of
// them are issued before the first projection, and the pair's state and inverse transform are read once per thread.  With one
// pixel per thread the kernel sat at 22 % of its issue slots with 80 % of the stall samples on those dependent loads.
#ifndef PH_SPLAT_PX
#define PH_SPLAT_PX 8
#endif
__global__ void __launch_bounds__(256) ph_splat_kernel(PhArgs a) {
    const int b = a.first + blockIdx.y;
    const int base = blockIdx.x * (256 * PH_SPLAT_PX) + threadIdx.x;
    PhState& S = a.st[b];
    if (S.stop) return;
    const int rows = a.rows, cols = a.cols;
    unsigned dzv[PH_SPLAT_PX];
#pragma unroll
    for (int j = 0; j < PH_SPLAT_PX; ++j) { const int i = base + j * 256; dzv[j] = (i < a.P) ? (unsigned)a.depth_ref[(long long)b * a.P + i] : 0u; }
    // Tr^-1 = [R^T, -R^T t]
    const double* Tr = S.Tr;
    double Ti[12];
    for (int u = 0; u < 3; ++u) for (int v = 0; v < 3; ++v) Ti[4 * u + v] = Tr[4 * v + u];
    for (int u = 0; u < 3; ++u) Ti[4 * u + 3] = -((Ti[4 * u] * Tr[3] + Ti[4 * u + 1] * Tr[7]) + Ti[4 * u + 2] * Tr[11]);
    int* wn = a.winner + (long long)b * a.g.P[0];
    int hits = 0;
#pragma unroll
    for (int j = 0; j < PH_SPLAT_PX; ++j) {
        const int i = base + j * 256;
        if (i >= a.P || !(a.compat || dzv[j] > 0u)) continue;
        const int r = i / cols, c = i - r * cols;
        const PixGeom p = ph_xyz(r, c, (double)dzv[j], a.sf, a.K, a.compat != 0);
        const double px = ((Ti[0] * p.X + Ti[1] * p.Y) + Ti[2] * p.Z) + Ti[3] * 1.0;
        const double py = ((Ti[4] * p.X + Ti[5] * p.Y) + Ti[6] * p.Z) + Ti[7] * 1.0;
        const double pz = ((Ti[8] * p.X + Ti[9] * p.Y) + Ti[10] * p.Z) + Ti[11] * 1.0;
        int tR = -1, tC = -1;
        if (a.compat) {                               // :526-527: u is a ROW coordinate, fx unscaled
            const double u = a.K.fx * px / pz + a.sf * a.K.cx, v = a.K.fy * py / pz + a.sf * a.K.cy;
            if (u > -1.0e9 && u < 1.0e9 && v > -1.0e9 && v < 1.0e9) { tR = (int)floor(u); tC = (int)floor(v); }
        } else if (pz > 0.0) {
            const double ipz = 1.0 / pz;
            const double uc = ((a.sf * a.K.fx) * px) * ipz + a.sf * a.K.cx, vr = ((a.sf * a.K.fy) * py) * ipz + a.sf * a.K.cy;
            if (uc > -1.0e9 && uc < 1.0e9 && vr > -1.0e9 && vr < 1.0e9) { tC = (int)floor(uc); tR = (int)floor(vr); }
        }
        if (tR >= 0 && tR < rows - 1 && tC >= 0 && tC < cols - 1) {
            ++hits;
            const int k = (c << 16) | r;              // column-major order of the source (c * rows + r) as a packed key: same maximum, no division to decode
            atomicMax(&wn[tR * cols + tC], k); atomicMax(&wn[tR * cols + tC + 1], k);
            atomicMax(&wn[(tR + 1) * cols + tC], k); atomicMax(&wn[(tR + 1) * cols + tC + 1], k);
        }
    }
    hits = __reduce_add_sync(0xffffffffu, hits);
    if ((threadIdx.x & 31) == 0 && hits) atomicAdd(&S.nreproj, hits);
}

#ifndef PH_ACCUM_MIN_BLOCKS
#define PH_ACCUM_MIN_BLOCKS 2
#endif
// residual + normal equations (:176-182): partial sums per block
__global__ void __launch_bounds__(PH_THREADS, PH_ACCUM_MIN_BLOCKS) ph_accum_kernel(PhArgs a) {
    const int b = a.first + blockIdx.y;
    PhState& S = a.st[b];
    // Huber weights: the residual is a difference of two 8-bit intensities, so |e| is an integer in 0..255 and k / |e| takes 256
    // values -- one IEEE division per table entry instead of one per pixel, same values as the oracle's huber_w
    __shared__ double s_hw[256];
    s_hw[threadIdx.x] = (a.huber_k > 0.0 && (double)threadIdx.x > a.huber_k) ? a.huber_k / (double)threadIdx.x : 1.0;
    __syncthreads();
    double acc[PH_NACC];
#pragma unroll
    for (int k = 0; k < PH_NACC; ++k) acc[k] = 0.0;
    if (!S.stop) {
        const uint8_t* g = a.gray_ref + (long long)b * a.P; const uint16_t* d = a.depth_ref + (long long)b * a.P;
        const uint8_t* gn = a.gray_now + (long long)b * a.P;
        int* wn = a.winner + (long long)b * a.g.P[0];
        const int rows = a.rows, cols = a.cols;
        const int stride = gridDim.x * PH_THREADS, k0 = blockIdx.x * PH_THREADS + threadIdx.x;
        if (a.compat) {
            for (int k = k0; k < a.P; k += stride) {
                // flattened index k: eps is row-major (cell k), J row k is the column-major pixel k (quirk 5); holes give -I_now
                const int wk = wn[k];
                if (a.reset_winner) wn[k] = -1;
                const double cv = (wk >= 0) ? (double)g[(wk & 0xFFFF) * cols + (wk >> 16)] : 0.0;
                const double e = cv - (double)gn[k];
                const int r = k % rows, c = k / rows;
                double J[6]; ph_jrow(g, d, rows, cols, r, c, a.sf, a.K, true, J);
#pragma unroll
                for (int q = 0; q < 6; ++q) acc[q] += J[q] * e;
                acc[6] += e * e; acc[7] += 1.0;
            }
        } else {
            // Software pipeline over the thread's cells: the winner of cell k + 2 strides is loaded while the five gathers its
            // predecessor's winner addresses (source intensity, two forward-difference taps, depth, now intensity) are in flight
            // and the cell before that is accumulated -- two dependent memory latencies per cell are otherwise exposed at the
            // two CTAs per SM that 29 fp64 accumulators leave.
            struct Taps { int rs, cs; unsigned gv, gr, gd, gnv, dz; };
            auto gather = [&](int wk, int k) {
                Taps t; t.rs = -1; t.cs = 0; t.gv = t.gr = t.gd = t.gnv = t.dz = 0u;
                if (wk >= 0) {
                    const int rs = wk & 0xFFFF, cs = wk >> 16;     // source pixel that owns this cell
                    const int c1 = (cs + 1 < cols) ? cs + 1 : cols - 2, r1 = (rs + 1 < rows) ? rs + 1 : rows - 2;   // ph_grad's REFLECT_101 taps
                    t.rs = rs; t.cs = cs;
                    t.gv = g[rs * cols + cs]; t.gr = g[rs * cols + (cols > 1 ? c1 : cs)]; t.gd = g[(rows > 1 ? r1 : rs) * cols + cs];
                    t.dz = d[rs * cols + cs]; t.gnv = gn[k];
                }
                return t;
            };
            int wk1 = (k0 + stride < a.P) ? wn[k0 + stride] : -1;
            Taps t0 = gather((k0 < a.P) ? wn[k0] : -1, k0);
            for (int k = k0; k < a.P; k += stride) {
                const int wk2 = (k + 2 * stride < a.P) ? wn[k + 2 * stride] : -1;
                const Taps t1 = gather(wk1, k + stride);
                if (t0.rs >= 0) {
                    if (a.reset_winner) wn[k] = -1;
                    const double v = (double)t0.gv;
                    const double e = v - (double)t0.gnv;
                    const double w = s_hw[(int)fabs(e)];
                    double J[6]; ph_jrow_vals((double)t0.dz, (double)t0.gr - v, (double)t0.gd - v, t0.rs, t0.cs, a.sf, a.K, false, J);
                    int idx = 8;
#pragma unroll
                    for (int p = 0; p < 6; ++p) {
                        const double jw = J[p] * w;
                        acc[p] += jw * e;
#pragma unroll
                        for (int q = p; q < 6; ++q) { acc[idx] += jw * J[q]; ++idx; }
                    }
                    acc[6] += e * e; acc[7] += 1.0;
                }
                t0 = t1; wk1 = wk2;
            }
        }
    }
    ph_block_reduce(acc, a.partial + ((long long)b * a.maxblk + blockIdx.x) * PH_NACC);
}

__device__ __forceinline__ bool ph_chol6(const double* H, const double* b, double* x) {
    double Lm[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = H[6 * j + i];
            for (int k = 0; k < j; ++k) s -= Lm[6 * i + k] * Lm[6 * j + k];
            if (i == j) { if (!(s > 0)) return false; Lm[6 * i + i] = sqrt(s); }
            else Lm[6 * i + j] = s / Lm[6 * j + j];
        }
    double y[6];
    for (int i = 0; i < 6; ++i) { double s = b[i]; for (int k = 0; k < i; ++k) s -= Lm[6 * i + k] * y[k]; y[i] = s / Lm[6 * i + i]; }
    for (int i = 5; i >= 0; --i) { double s = y[i]; for (int k = i + 1; k < 6; ++k) s -= Lm[6 * k + i] * x[k]; x[i] = s / Lm[6 * i + i]; }
    return true;
}

// exponentialMap (:570-597), guarded for small angles
__device__ __forceinline__ void ph_exp(const double* psi, double* T4) {
    const double w0 = psi[3], w1 = psi[4], w2 = psi[5];
    const double th = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
    const double wx[9] = {0, -w2, w1, w2, 0, -w0, -w1, w0, 0};
    double wx2[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) wx2[3 * i + j] = wx[3 * i] * wx[j] + wx[3 * i + 1] * wx[3 + j] + wx[3 * i + 2] * wx[6 + j];
    double ca, cb, cc;
    if (th < 1e-8) { ca = 1.0; cb = 0.5; cc = 1.0 / 6.0; }
    else { ca = sin(th) / th; cb = (1.0 - cos(th)) / (th * th); cc = (th - sin(th)) / (th * th * th); }
    for (int i = 0; i < 3; ++i) {
        double vt = 0.0;
        for (int j = 0; j < 3; ++j) {
            const double I = (i == j) ? 1.0 : 0.0;
            T4[4 * i + j] = I + ca * wx[3 * i + j] + cb * wx2[3 * i + j];
            vt += (I + cb * wx[3 * i + j] + cc * wx2[3 * i + j]) * psi[j];
        }
        T4[4 * i + 3] = vt;
    }
    T4[12] = T4[13] = T4[14] = 0.0; T4[15] = 1.0;
}

// one thread block per pair: final reduction (fixed order), LM bookkeeping, 6x6 solve, Tr <- Tr * exp(-delta)
__global__ void __launch_bounds__(64) ph_solve_kernel(PhArgs a, int itr) {
    const int b = a.first + blockIdx.x;
    __shared__ double tot[PH_NACC];
    PhState& S = a.st[b];
    if (S.stop) return;
    if (threadIdx.x < PH_NACC) {
        double v = 0.0;
        for (int k = 0; k < a.nblk; ++k) v += a.partial[((long long)b * a.maxblk + k) * PH_NACC + threadIdx.x];
        tot[threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const double sumsq = tot[6];
    S.visible = (double)S.nreproj / ((double)a.rows * (double)a.cols);
    S.nreproj_last = S.nreproj; S.nreproj = 0;               // the next splat counts from zero
    if (itr == 0) S.sumsq_first = sumsq;
    S.sumsq_last = sumsq; S.iters_run = itr + 1;
    double Aev[36];
    if (a.compat) {
        // A = J^T J of the reference level is singular by construction (duplicated column): the normal equations are
        // produced for inspection (accA, accb) and no step is taken
        const double* A = a.A + ((long long)b * a.g.L + a.level) * 36;
        for (int k = 0; k < 36; ++k) S.accA[k] = A[k];
        for (int k = 0; k < 6; ++k) S.accb[k] = tot[k];
        S.accE = sumsq; S.status = 2; S.stop = 1;
        return;
    }
    int idx = 8;
    for (int p = 0; p < 6; ++p) for (int q = p; q < 6; ++q) { Aev[6 * p + q] = tot[idx]; Aev[6 * q + p] = tot[idx]; ++idx; }
    const bool accept = !S.have || a.lambda0 <= 0.0 || sumsq <= S.accE;
    if (accept) {
        for (int k = 0; k < 16; ++k) S.accTr[k] = S.Tr[k];
        for (int k = 0; k < 36; ++k) S.accA[k] = Aev[k];
        for (int k = 0; k < 6; ++k) S.accb[k] = tot[k];
        S.accE = sumsq;
        if (S.have && a.lambda0 > 0.0) S.lambda = (S.lambda * 0.1 < 1e-9) ? 1e-9 : S.lambda * 0.1;
        S.have = 1;
    } else {
        S.lambda *= 10.0;
        if (S.lambda > 1e8) { S.stop = 1; for (int k = 0; k < 16; ++k) S.Tr[k] = S.accTr[k]; return; }
        for (int k = 0; k < 16; ++k) S.Tr[k] = S.accTr[k];
    }
    double Am[36], rhs[6], dl[6];
    for (int k = 0; k < 36; ++k) Am[k] = S.accA[k];
    for (int k = 0; k < 6; ++k) { Am[7 * k] += (a.lambda0 > 0.0 ? S.lambda : 0.0) * S.accA[7 * k] + 1e-9; rhs[k] = S.accb[k]; }
    if (!ph_chol6(Am, rhs, dl)) { S.status = 1; S.stop = 1; for (int k = 0; k < 16; ++k) S.Tr[k] = S.accTr[k]; return; }
    for (int k = 0; k < 6; ++k) dl[k] = -dl[k];
    double E4[16], Tn[16];
    ph_exp(dl, E4);
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j)
        Tn[4 * i + j] = ((S.Tr[4 * i] * E4[j] + S.Tr[4 * i + 1] * E4[4 + j]) + S.Tr[4 * i + 2] * E4[8 + j]) + S.Tr[4 * i + 3] * E4[12 + j];
    for (int k = 0; k < 16; ++k) S.Tr[k] = Tn[k];
}

// end of estimate(): keep the last accepted transform
__global__ void ph_finish_kernel(PhState* st, int first, int count, int compat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    PhState& S = st[first + i];
    if (S.have && !compat) for (int k = 0; k < 16; ++k) S.Tr[k] = S.accTr[k];
}

// pose12 != null: the given poses; identity != 0: the identity; neither: the pose is kept
__global__ void ph_init_state_kernel(PhState* st, int first, int count, const double* pose12, double lambda0, int identity = 0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    PhState& S = st[first + i];
    if (pose12) {
        const double* p = pose12 + 12 * (long long)i;
        for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) S.Tr[4 * r + c] = p[3 * r + c]; S.Tr[4 * r + 3] = p[9 + r]; }
        S.Tr[12] = S.Tr[13] = S.Tr[14] = 0.0; S.Tr[15] = 1.0;
    } else if (identity) {
        for (int k = 0; k < 16; ++k) S.Tr[k] = (k % 5 == 0) ? 1.0 : 0.0;
    }
    S.have = 0; S.status = 0; S.iters_run = 0; S.stop = 0; S.nreproj = 0; S.nreproj_last = 0; S.lambda = lambda0; S.accE = 0.0;
    S.sumsq_first = S.sumsq_last = 0.0; S.visible = 0.0;
}

// materialise the PyramidalStorageStruct arrays of one slot / level as doubles (getLevel, src/PyramidalStorage.cpp:71-102)
__global__ void __launch_bounds__(256) ph_materialize_kernel(PhArgs a, int which, const uint8_t* __restrict__ bgr_level, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.P) return;
    const int b = a.first;
    const uint8_t* g = a.gray_ref + (long long)b * a.P; const uint16_t* d = a.depth_ref + (long long)b * a.P;
    const int r = i / a.cols, c = i - r * a.cols;
    if (which == DVO_PHOTO_J) {
        double J[6]; ph_jrow(g, d, a.rows, a.cols, r, c, a.sf, a.K, a.compat != 0, J);
        double* o = out + ((long long)c * a.rows + r) * 6;                      // row = column-major pixel index (:398-410)
        for (int k = 0; k < 6; ++k) o[k] = J[k];
        return;
    }
    const PixGeom p = ph_xyz(r, c, (double)d[i], a.sf, a.K, a.compat != 0);
    double v = 0.0;
    switch (which) {
        case DVO_PHOTO_X: v = p.X; break;
        case DVO_PHOTO_Y: v = p.Y; break;
        case DVO_PHOTO_Z: v = p.Z; break;
        case DVO_PHOTO_GRAYVALS: v = (double)g[i]; break;
        case DVO_PHOTO_BLUEVALS: v = (double)bgr_level[3 * i]; break;
        case DVO_PHOTO_GREENVALS: v = (double)bgr_level[3 * i + 1]; break;
        case DVO_PHOTO_REDVALS: v = (double)bgr_level[3 * i + 2]; break;
        default: break;
    }
    out[i] = v;
}

// canvas of the current warp (inspection)
__global__ void __launch_bounds__(256) ph_canvas_kernel(PhArgs a, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.P) return;
    const int b = a.first;
    const int wk = a.winner[(long long)b * a.g.P[0] + i];
    out[i] = (wk >= 0) ? (double)a.gray_ref[(long long)b * a.P + (wk & 0xFFFF) * a.cols + (wk >> 16)] : 0.0;
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
namespace {
bool ph_range_ok(dvo_photo_ctx* c, int first, int count) { return c && first >= 0 && count >= 0 && first + count <= c->cfg.max_batch; }

PhArgs ph_args(dvo_photo_ctx* c, int level, int first, int compat, double huber_k, double lambda0) {
    PhArgs a;
    a.g = c->g; a.K = c->K; a.sf = ldexp(1.0, -level);
    a.K.ifx = 1.0 / (a.sf * a.K.fx); a.K.ify = 1.0 / (a.sf * a.K.fy);
    a.gray_ref = c->gray[0] + c->g.off[level]; a.depth_ref = c->depth[0] + c->g.off[level]; a.gray_now = c->gray[1] + c->g.off[level];
    a.winner = c->winner; a.partial = c->partial; a.A = c->A; a.st = c->st;
    a.level = level; a.rows = c->g.h[level]; a.cols = c->g.w[level]; a.P = c->g.P[level]; a.first = first; a.compat = compat;
    int nblk = (a.P + PH_THREADS * 8 - 1) / (PH_THREADS * 8); if (nblk < 1) nblk = 1; if (nblk > c->maxblk) nblk = c->maxblk;
    a.nblk = nblk; a.maxblk = c->maxblk; a.huber_k = huber_k; a.lambda0 = lambda0; a.reset_winner = 0;
    return a;
}
}  // namespace

extern "C" {

#define PH_CREATE_CUDA(call)                                                                    \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dvo_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            dvo_photo_destroy(c);                                                               \
            return DVO_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

int dvo_photo_create(const dvo_photo_config* cfg, dvo_photo_ctx** out) {
    if (!cfg || !out) { dvo_set_error("dvo_photo_create: null argument"); return DVO_ERR_ARG; }
    if (cfg->levels < 1 || cfg->levels > PH_MAX_LEVELS || cfg->max_batch < 1 || cfg->max_batch > 65535 || cfg->width < 8 || cfg->height < 8 ||
        cfg->width > 32767 || cfg->height > 65535 ||          /* the winner map packs (column << 16) | row into an int */
        (cfg->width % (1 << (cfg->levels - 1))) || (cfg->height % (1 << (cfg->levels - 1)))) {
        dvo_set_error("dvo_photo_create: bad config %dx%d levels=%d (dimensions must be divisible by 2^(levels-1))", cfg->width, cfg->height, cfg->levels);
        return DVO_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        dvo_set_error("dvo_photo_create: no usable CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
        cudaGetLastError();
        return DVO_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { dvo_set_error("dvo_photo_create: device %d out of range", cfg->device); return DVO_ERR_ARG; }
    DVO_CUDA(cudaSetDevice(cfg->device));
    dvo_photo_ctx* c = new (std::nothrow) dvo_photo_ctx();
    if (!c) return DVO_ERR_NOMEM;
    c->cfg = *cfg;
    PhGeom& g = c->g; g.L = cfg->levels; g.Bmax = cfg->max_batch; g.W = cfg->width; g.H = cfg->height;
    long long acc = 0;
    for (int l = 0; l < g.L; ++l) { g.w[l] = cfg->width >> l; g.h[l] = cfg->height >> l; g.P[l] = g.w[l] * g.h[l]; g.off[l] = acc * g.Bmax; acc += g.P[l]; }
    g.total = acc * g.Bmax;
    PH_CREATE_CUDA(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    c->maxblk = (g.P[0] + PH_THREADS * 8 - 1) / (PH_THREADS * 8);
    const size_t B = g.Bmax, P0 = g.P[0];
    int rc = DVO_OK;
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    for (int f = 0; f < 2; ++f) { A(c->bgr[f].reserve(B * P0 * 3)); A(c->gray[f].reserve((size_t)g.total)); A(c->depth[f].reserve((size_t)g.total)); }
    A(c->winner.reserve(B * P0)); A(c->partial.reserve(B * c->maxblk * PH_NACC)); A(c->A.reserve(B * g.L * 36)); A(c->st.reserve(B));
    if (rc != DVO_OK) { dvo_photo_destroy(c); return rc; }
    PH_CREATE_CUDA(cudaMemsetAsync(c->st, 0, sizeof(PhState) * B, c->stream));
    PH_CREATE_CUDA(cudaMemsetAsync(c->A, 0, sizeof(double) * B * g.L * 36, c->stream));
    dvo_photo_set_pose(c, 0, g.Bmax, nullptr);
    PH_CREATE_CUDA(cudaStreamSynchronize(c->stream));
    *out = c;
    return DVO_OK;
}

int dvo_photo_destroy(dvo_photo_ctx* c) {
    if (!c) return DVO_OK;
    cudaSetDevice(c->cfg.device);
    if (c->own_stream) cudaStreamSynchronize(c->own_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return DVO_OK;
}

int dvo_photo_set_stream(dvo_photo_ctx* c, void* s) { if (!c) return DVO_ERR_ARG; c->stream = s ? (cudaStream_t)s : c->own_stream; return DVO_OK; }
int dvo_photo_synchronize(dvo_photo_ctx* c) { if (!c) return DVO_ERR_ARG; DVO_CUDA(cudaStreamSynchronize(c->stream)); return DVO_OK; }
long long dvo_photo_launch_count(dvo_photo_ctx* c) { return c ? c->launches : 0; }

int dvo_photo_set_intrinsics(dvo_photo_ctx* c, double fx, double fy, double cx, double cy) {
    if (!c) return DVO_ERR_ARG;
    c->K.fx = fx; c->K.fy = fy; c->K.cx = cx; c->K.cy = cy; c->haveK = true;
    return DVO_OK;
}

// setRefFrame / setNowFrame (:68-126): copy, BGR2GRAY at full resolution, INTER_AREA pyramids of gray and depth
int dvo_photo_set_frames(dvo_photo_ctx* c, int frame, int first, int count, const uint8_t* bgr, const uint16_t* depth, int mem) {
    if (!ph_range_ok(c, first, count) || (frame != 0 && frame != 1) || !bgr) { dvo_set_error("dvo_photo_set_frames: bad argument"); return DVO_ERR_ARG; }
    if (frame == DVO_FRAME_REF && !depth) { dvo_set_error("dvo_photo_set_frames: the reference frame needs depth"); return DVO_ERR_ARG; }
    if (count == 0) return DVO_OK;
    const PhGeom& g = c->g;
    const size_t P0 = g.P[0];
    const cudaMemcpyKind k = mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    DVO_CUDA(cudaMemcpyAsync(c->bgr[frame] + (size_t)first * P0 * 3, bgr, P0 * 3 * count, k, c->stream));
    if (depth) DVO_CUDA(cudaMemcpyAsync(c->depth[frame] + ph_at(g, 0, first), depth, P0 * 2 * count, k, c->stream));
    const long long n = (long long)P0 * count;
    ph_gray_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->bgr[frame] + (size_t)first * P0 * 3, c->gray[frame] + ph_at(g, 0, first), n);
    c->launches++;
    for (int l = 1; l < g.L; ++l) {
        dim3 grid((g.P[l] + 255) / 256, count);
        ph_area_kernel<uint8_t, 1><<<grid, 256, 0, c->stream>>>(c->gray[frame] + ph_at(g, 0, first), c->gray[frame] + ph_at(g, l, first), g.W, g.H, l, (long long)P0, (long long)g.P[l]);
        c->launches++;
        if (depth) {
            ph_area_kernel<uint16_t, 1><<<grid, 256, 0, c->stream>>>(c->depth[frame] + ph_at(g, 0, first), c->depth[frame] + ph_at(g, l, first), g.W, g.H, l, (long long)P0, (long long)g.P[l]);
            c->launches++;
        }
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// evaluateJacobian for every level + A = J^T J (:88-102, :229)
int dvo_photo_prepare_ref(dvo_photo_ctx* c, int first, int count, int compat) {
    if (!ph_range_ok(c, first, count)) return DVO_ERR_ARG;
    if (!c->haveK) { dvo_set_error("dvo_photo_prepare_ref: intrinsics not set (cameraIntrinsicsReady)"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    for (int l = 0; l < c->g.L; ++l) {
        PhArgs a = ph_args(c, l, first, compat, 0.0, 0.0);
        ph_A_kernel<<<dim3(a.nblk, count), PH_THREADS, 0, c->stream>>>(a);
        ph_A_final_kernel<<<count, 64, 0, c->stream>>>(a);
        c->launches += 2;
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_photo_set_pose(dvo_photo_ctx* c, int first, int count, const double* R9T3) {
    if (!ph_range_ok(c, first, count)) return DVO_ERR_ARG;
    if (count == 0) return DVO_OK;
    if (!R9T3) {                                   // identity: set on the device, no copy and no synchronisation
        ph_init_state_kernel<<<(count + 127) / 128, 128, 0, c->stream>>>(c->st, first, count, nullptr, 0.0, 1);
        c->launches++;
        DVO_CUDA(cudaGetLastError());
        return DVO_OK;
    }
    DevBuf<double> d;
    if (const int rc = d.reserve(12 * (size_t)count)) return rc;
    DVO_CUDA(cudaMemcpyAsync(d, R9T3, sizeof(double) * 12 * count, cudaMemcpyHostToDevice, c->stream));
    ph_init_state_kernel<<<(count + 127) / 128, 128, 0, c->stream>>>(c->st, first, count, d, 0.0);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// setPyramidalImages(level) + estimate(R, T) (:216-260, :135-209)
int dvo_photo_estimate(dvo_photo_ctx* c, int first, int count, int level, int iters, int compat, double huber_k, double lambda0) {
    if (!ph_range_ok(c, first, count) || level < 0 || level >= c->g.L || iters < 1) { dvo_set_error("dvo_photo_estimate: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_photo_estimate: intrinsics not set"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    PhArgs a = ph_args(c, level, first, compat, huber_k, lambda0);
    ph_init_state_kernel<<<(count + 127) / 128, 128, 0, c->stream>>>(c->st, first, count, nullptr, lambda0);
    c->launches++;
    const dim3 gpix((a.P + 255) / 256, count);
    // the winner map is cleared once; every accumulation pass hands it back cleared (cells of stopped pairs are never written)
    a.reset_winner = 1;
    ph_clear_kernel<<<gpix, 256, 0, c->stream>>>(a);
    c->launches++;
    for (int itr = 0; itr < iters; ++itr) {
        ph_splat_kernel<<<dim3((a.P + 256 * PH_SPLAT_PX - 1) / (256 * PH_SPLAT_PX), count), 256, 0, c->stream>>>(a);
        ph_accum_kernel<<<dim3(a.nblk, count), PH_THREADS, 0, c->stream>>>(a);
        ph_solve_kernel<<<count, 64, 0, c->stream>>>(a, itr);
        c->launches += 3;
    }
    ph_finish_kernel<<<(count + 127) / 128, 128, 0, c->stream>>>(c->st, first, count, compat);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int dvo_photo_get_poses(dvo_photo_ctx* c, int first, int count, double* R9T3, dvo_photo_info* info) {
    if (!ph_range_ok(c, first, count)) return DVO_ERR_ARG;
    std::vector<PhState> st(count);
    DVO_CUDA(cudaMemcpyAsync(st.data(), c->st + first, sizeof(PhState) * count, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < count; ++i) {
        if (R9T3) { double* p = R9T3 + 12 * (size_t)i; for (int r = 0; r < 3; ++r) { for (int q = 0; q < 3; ++q) p[3 * r + q] = st[i].Tr[4 * r + q]; p[9 + r] = st[i].Tr[4 * r + 3]; } }
        if (info) {
            info[i].status = st[i].status; info[i].iters_run = st[i].iters_run; info[i].nreproj = st[i].nreproj_last;
            info[i].sumsq_first = st[i].sumsq_first; info[i].sumsq_last = st[i].sumsq_last; info[i].visible = st[i].visible;
            memcpy(info[i].A, st[i].accA, sizeof(double) * 36); memcpy(info[i].b, st[i].accb, sizeof(double) * 6);
        }
    }
    return DVO_OK;
}

// PyramidalStorageStruct::getLevel (src/PyramidalStorage.cpp:71-102)
int dvo_photo_get_level(dvo_photo_ctx* c, int slot, int frame, int level, int which, void* dst, size_t bytes, int compat) {
    if (!ph_range_ok(c, slot, 1) || level < 0 || level >= c->g.L || (frame != 0 && frame != 1) || !dst) { dvo_set_error("dvo_photo_get_level: bad argument"); return DVO_ERR_ARG; }
    const PhGeom& g = c->g;
    const size_t P = g.P[level];
    if (which == DVO_PHOTO_GRAY || which == DVO_PHOTO_DEPTH) {
        const size_t es = which == DVO_PHOTO_GRAY ? 1 : 2;
        if (bytes < P * es) { dvo_set_error("dvo_photo_get_level: destination too small"); return DVO_ERR_ARG; }
        const void* src = which == DVO_PHOTO_GRAY ? (const void*)(c->gray[frame] + ph_at(g, level, slot)) : (const void*)(c->depth[frame] + ph_at(g, level, slot));
        DVO_CUDA(cudaMemcpyAsync(dst, src, P * es, cudaMemcpyDeviceToHost, c->stream));
        DVO_CUDA(cudaStreamSynchronize(c->stream));
        return DVO_OK;
    }
    // colour level (im_r_color): INTER_AREA of the full-resolution BGR, built on demand
    DevBuf<uint8_t> d_bgr;
    const bool need_bgr = (which == DVO_PHOTO_BGR || which == DVO_PHOTO_BLUEVALS || which == DVO_PHOTO_GREENVALS || which == DVO_PHOTO_REDVALS);
    if (need_bgr) {
        if (const int rc = d_bgr.reserve(P * 3)) return rc;
        const uint8_t* src = c->bgr[frame] + (size_t)slot * g.P[0] * 3;
        if (level == 0) DVO_CUDA(cudaMemcpyAsync(d_bgr, src, P * 3, cudaMemcpyDeviceToDevice, c->stream));
        else { ph_area_kernel<uint8_t, 3><<<dim3((unsigned)((P + 255) / 256), 1), 256, 0, c->stream>>>(src, d_bgr, g.W, g.H, level, 0, 0); c->launches++; }
        if (which == DVO_PHOTO_BGR) {
            if (bytes < P * 3) { dvo_set_error("dvo_photo_get_level: destination too small"); return DVO_ERR_ARG; }
            DVO_CUDA(cudaMemcpyAsync(dst, d_bgr, P * 3, cudaMemcpyDeviceToHost, c->stream));
            DVO_CUDA(cudaStreamSynchronize(c->stream));
            return DVO_OK;
        }
    }
    if (!c->haveK) { dvo_set_error("dvo_photo_get_level: intrinsics not set"); return DVO_ERR_STATE; }
    if (frame != DVO_FRAME_REF) { dvo_set_error("dvo_photo_get_level: X/Y/Z/J/colour arrays exist for the reference frame only"); return DVO_ERR_ARG; }
    const size_t n = (which == DVO_PHOTO_J) ? P * 6 : P;
    if (bytes < n * sizeof(double)) { dvo_set_error("dvo_photo_get_level: destination too small"); return DVO_ERR_ARG; }
    DevBuf<double> d_out;
    if (const int rc = d_out.reserve(n)) return rc;
    PhArgs a = ph_args(c, level, slot, compat, 0.0, 0.0);
    ph_materialize_kernel<<<(unsigned)((P + 255) / 256), 256, 0, c->stream>>>(a, which, d_bgr, d_out);
    c->launches++;
    DVO_CUDA(cudaMemcpyAsync(dst, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// PyramidalStorageStruct::addLevel with caller-provided images (src/PyramidalStorage.cpp:38-65): replaces one stored level image.
// The derived members (X, Y, Z, J, *Vals) are functions of (im_r, dim_r, K, level) and are re-evaluated by the kernels;
// follow with dvo_photo_prepare_ref to refresh A = J^T J.
int dvo_photo_put_level(dvo_photo_ctx* c, int slot, int frame, int level, int which, const void* src, size_t bytes) {
    if (!ph_range_ok(c, slot, 1) || level < 0 || level >= c->g.L || (frame != 0 && frame != 1) || !src) { dvo_set_error("dvo_photo_put_level: bad argument"); return DVO_ERR_ARG; }
    const PhGeom& g = c->g;
    const size_t P = g.P[level];
    void* dst = nullptr; size_t need = 0;
    if (which == DVO_PHOTO_GRAY) { dst = c->gray[frame] + ph_at(g, level, slot); need = P; }
    else if (which == DVO_PHOTO_DEPTH) { dst = c->depth[frame] + ph_at(g, level, slot); need = P * 2; }
    else if (which == DVO_PHOTO_BGR && level == 0) { dst = c->bgr[frame] + (size_t)slot * g.P[0] * 3; need = P * 3; }
    else { dvo_set_error("dvo_photo_put_level: only GRAY / DEPTH (any level) and BGR (level 0) are stored on the device"); return DVO_ERR_ARG; }
    if (bytes != need) { dvo_set_error("dvo_photo_put_level: expected %zu bytes, got %zu", need, bytes); return DVO_ERR_ARG; }
    DVO_CUDA(cudaMemcpyAsync(dst, src, need, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// A = J^T J of a reference level (setPyramidalImages :229)
int dvo_photo_get_A(dvo_photo_ctx* c, int slot, int level, double* A36) {
    if (!ph_range_ok(c, slot, 1) || level < 0 || level >= c->g.L || !A36) return DVO_ERR_ARG;
    DVO_CUDA(cudaMemcpyAsync(A36, c->A + ((size_t)slot * c->g.L + level) * 36, sizeof(double) * 36, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// one evaluation of the loop body of estimate() at a given pose: warp canvas, b = J^T eps, (weighted) A, sum eps^2
int dvo_photo_eval(dvo_photo_ctx* c, int slot, int level, const double* R9T3, int compat, double huber_k, double* b6, double* A36, double* sumsq,
                   int* nreproj, int* nused, double* canvas) {
    if (!ph_range_ok(c, slot, 1) || level < 0 || level >= c->g.L || !R9T3) return DVO_ERR_ARG;
    int rc = dvo_photo_set_pose(c, slot, 1, R9T3);
    if (rc) return rc;
    PhArgs a = ph_args(c, level, slot, compat, huber_k, 0.0);
    const dim3 gpix((a.P + 255) / 256, 1);
    ph_clear_kernel<<<gpix, 256, 0, c->stream>>>(a);
    ph_splat_kernel<<<dim3((a.P + 256 * PH_SPLAT_PX - 1) / (256 * PH_SPLAT_PX), 1), 256, 0, c->stream>>>(a);
    ph_accum_kernel<<<dim3(a.nblk, 1), PH_THREADS, 0, c->stream>>>(a);
    c->launches += 3;
    std::vector<double> part((size_t)a.nblk * PH_NACC);
    DVO_CUDA(cudaMemcpyAsync(part.data(), c->partial + (size_t)slot * c->maxblk * PH_NACC, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, c->stream));
    PhState st;
    DVO_CUDA(cudaMemcpyAsync(&st, c->st + slot, sizeof(PhState), cudaMemcpyDeviceToHost, c->stream));
    DevBuf<double> d_cv;
    if (canvas) {
        if ((rc = d_cv.reserve(a.P))) return rc;
        ph_canvas_kernel<<<(a.P + 255) / 256, 256, 0, c->stream>>>(a, d_cv);
        c->launches++;
        DVO_CUDA(cudaMemcpyAsync(canvas, d_cv, sizeof(double) * a.P, cudaMemcpyDeviceToHost, c->stream));
    }
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    double tot[PH_NACC];
    for (int k = 0; k < PH_NACC; ++k) { double v = 0.0; for (int j = 0; j < a.nblk; ++j) v += part[(size_t)j * PH_NACC + k]; tot[k] = v; }
    if (b6) memcpy(b6, tot, sizeof(double) * 6);
    if (sumsq) *sumsq = tot[6];
    if (nused) *nused = (int)tot[7];
    if (nreproj) *nreproj = st.nreproj;
    if (A36) {
        if (compat) return dvo_photo_get_A(c, slot, level, A36);
        int idx = 8;
        for (int p = 0; p < 6; ++p) for (int q = p; q < 6; ++q) { A36[6 * p + q] = tot[idx]; A36[6 * q + p] = tot[idx]; ++idx; }
    }
    return DVO_OK;
}

}  // extern "C"
