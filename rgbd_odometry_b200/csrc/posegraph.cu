// posegraph.cu -- batched windowed SE(3) pose-graph optimisation (dvo_pose_graph_optimize): one persistent CTA per graph runs
// the whole Levenberg-Marquardt loop, and optionally the marginal covariances of the returned poses, with no host round trip.
//
// Problem (include/dvo_b200.h): nodes G_i (12-double records, G_a G_b = (R_a R_b, T_a + R_a T_b)), node 0 fixed; edge e = (a, b,
// Z, Sigma) with residual r = log(Z^-1 G_a^-1 G_b), information Omega = Sigma^-1, cost F = 1/2 sum r^T Omega r; right perturbations
// G <- G exp(d), dr/dd_b = Jinv(r) = I + 1/2 ad(r), dr/dd_a = -Jinv(r) Ad(G_b^-1 G_a).
//
// Structure.  Every edge joins nodes at most max_lag apart, so grouping max_lag consecutive nodes of the reduced system (node 0
// removed) into a super-node of s = 6 max_lag unknowns makes H block-tridiagonal: diagonal blocks HD[j] and couplings HR[j] =
// H(j, j+1), M = ceil((N-1) / max_lag) super-nodes, the last one padded with identity rows.
//   - edge pass: threads take edges; r, the two Jacobians and the Omega-weighted blocks H_aa, H_bb, H_ab, g_a, g_b go to per-edge
//     scratch.  Omega comes once per call from a Cholesky factor of Sigma, which also decides whether the edge is used.
//   - assembly, no atomics: every entry of a node block (i, i+o), 0 <= o <= max_lag, and of g_i is summed by one thread over
//     node i's incidence list (valid edges in edge-index order, built once per call), so the sums are bit-reproducible.
//   - solve: odd-even block cyclic reduction.  Level l eliminates the super-nodes at odd multiples of 2^l, all in parallel (one
//     warp each), then every survivor gathers the Schur updates of its two eliminated neighbours in a fixed order.  The factor is
//     the block Cholesky factor of H in that elimination order, so back substitution and the selected inverse (Takahashi) walk
//     the same tree top-down.  ceil(log2 M) levels instead of the M dependent steps of a banded Cholesky.
//   - connectivity: min-label propagation with pointer jumping over the valid edges, once, before iterating.
// Nothing depends on the graph's position in the batch or on the number of graphs: each CTA reads its own inputs and scratch.
#include "common.cuh"

#include <math_constants.h>

namespace {

constexpr int PGO_THREADS = 256;
constexpr int PGO_WARPS = PGO_THREADS / 32;
constexpr double PGO_LAMBDA_MAX = 1e16;   // the LM loop stops when lambda grows past this (DVO_PGO_LAMBDA_MAX in the header)
constexpr int EC_STRIDE = 3 * 36 + 12;    // per-edge H_aa, H_bb, H_ab, g_a, g_b

// per-graph scratch layout, offsets in elements of the double and int regions
struct PgoLayout {
    int N, E, L, s, M;
    long long X, Xt, Om, EC, HD, HR, D, R, Wl, SD, SL, SR, gv, bv, dbl;
    long long valid, deg, off, cur, inc, label, ints;
};

PgoLayout pgo_layout(int nnodes, int nedges, int max_lag) {
    PgoLayout l;
    l.N = nnodes; l.E = nedges; l.L = max_lag; l.s = 6 * max_lag; l.M = (nnodes - 1 + max_lag - 1) / max_lag;
    const long long blk = (long long)l.s * l.s, mb = blk * l.M;
    long long o = 0;
    auto take = [&](long long n) { const long long r = o; o += (n + 1) & ~1LL; return r; };
    l.X = take(12LL * nnodes); l.Xt = take(12LL * nnodes); l.Om = take(36LL * nedges); l.EC = take((long long)EC_STRIDE * nedges);
    l.HD = take(mb); l.HR = take(mb); l.D = take(mb); l.R = take(mb); l.Wl = take(mb); l.SD = take(mb); l.SL = take(mb); l.SR = take(mb);
    l.gv = take((long long)l.s * l.M); l.bv = take((long long)l.s * l.M);
    l.dbl = o;
    o = 0;
    l.valid = take(nedges); l.deg = take(nnodes); l.off = take(nnodes + 1LL); l.cur = take(nnodes); l.inc = take(2LL * nedges);
    l.label = take(nnodes);
    l.ints = o;
    return l;
}

// ------------------------------------------------------------------ fp64 3x3 / SE(3) helpers: the closed forms of solver.cu
__device__ __forceinline__ void m3_mul(const double* A, const double* B, double* C) {
    double r[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) r[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
#pragma unroll
    for (int i = 0; i < 9; ++i) C[i] = r[i];
}
__device__ __forceinline__ void m3t_mul(const double* A, const double* B, double* C) {   // C = A^T B
    double r[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) r[3 * i + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
#pragma unroll
    for (int i = 0; i < 9; ++i) C[i] = r[i];
}
__device__ __forceinline__ void m3_vec(const double* A, const double* v, double* o) {
    const double a = A[0] * v[0] + A[1] * v[1] + A[2] * v[2];
    const double b = A[3] * v[0] + A[4] * v[1] + A[5] * v[2];
    const double c = A[6] * v[0] + A[7] * v[1] + A[8] * v[2];
    o[0] = a; o[1] = b; o[2] = c;
}
__device__ __forceinline__ void m3t_vec(const double* A, const double* v, double* o) {   // o = A^T v
    const double a = A[0] * v[0] + A[3] * v[1] + A[6] * v[2];
    const double b = A[1] * v[0] + A[4] * v[1] + A[7] * v[2];
    const double c = A[2] * v[0] + A[5] * v[1] + A[8] * v[2];
    o[0] = a; o[1] = b; o[2] = c;
}

__device__ __forceinline__ void se3_exp_dev(const double* psi, double* R, double* t) {
    const double wx = psi[3], wy = psi[4], wz = psi[5];
    const double th2 = wx * wx + wy * wy + wz * wz, th = sqrt(th2);
    double A, B, C;
    if (th < 1e-5) { A = 1.0 - th2 / 6.0; B = 0.5 - th2 / 24.0; C = 1.0 / 6.0 - th2 / 120.0; }
    else { double s, c; sincos(th, &s, &c); const double ith = 1.0 / th, ith2 = ith * ith; A = s * ith; B = (1.0 - c) * ith2; C = (th - s) * (ith2 * ith); }
    const double O[9] = {0, -wz, wy, wz, 0, -wx, -wy, wx, 0};
    double O2[9]; m3_mul(O, O, O2);
    double V[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const double I = (i % 4 == 0) ? 1.0 : 0.0;
        R[i] = I + A * O[i] + B * O2[i];
        V[i] = I + B * O[i] + C * O2[i];
    }
    m3_vec(V, psi, t);
}

__device__ __forceinline__ void rot_to_quat_dev(const double* R, double* q) {
    const double tr = R[0] + R[4] + R[8];
    if (tr > 0) {
        double s = sqrt(tr + 1.0); q[3] = 0.5 * s; s = 0.5 / s;
        q[0] = (R[7] - R[5]) * s; q[1] = (R[2] - R[6]) * s; q[2] = (R[3] - R[1]) * s;
    } else {
        int i = 0; if (R[4] > R[0]) i = 1; if (R[8] > R[4 * i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        double s = sqrt(R[4 * i] - R[4 * j] - R[4 * k] + 1.0);
        q[i] = 0.5 * s; s = 0.5 / s;
        q[3] = (R[3 * k + j] - R[3 * j + k]) * s;
        q[j] = (R[3 * j + i] + R[3 * i + j]) * s;
        q[k] = (R[3 * k + i] + R[3 * i + k]) * s;
    }
}

__device__ __forceinline__ void se3_log_dev(const double* R, const double* t, double* psi) {
    double q[4]; rot_to_quat_dev(R, q);
    const double qn = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    double sgn = (q[3] < 0 ? -1.0 : 1.0) / qn;
    const double x = q[0] * sgn, y = q[1] * sgn, z = q[2] * sgn, w = q[3] * sgn;
    const double n2 = x * x + y * y + z * z, n = sqrt(n2);
    const double k = (n < 1e-10) ? (2.0 / w - 2.0 * n2 / (3.0 * w * w * w)) : (2.0 * atan2(n, w) / n);
    const double ox = k * x, oy = k * y, oz = k * z;
    const double th2 = ox * ox + oy * oy + oz * oz, th = sqrt(th2);
    const double O[9] = {0, -oz, oy, oz, 0, -ox, -oy, ox, 0};
    double O2[9]; m3_mul(O, O, O2);
    const double D = (th < 1e-5) ? (1.0 / 12.0 + th2 / 720.0) : ((1.0 - th * sin(th) / (2.0 * (1.0 - cos(th)))) / th2);
    double Vi[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) Vi[i] = ((i % 4 == 0) ? 1.0 : 0.0) - 0.5 * O[i] + D * O2[i];
    m3_vec(Vi, t, psi);
    psi[3] = ox; psi[4] = oy; psi[5] = oz;
}

// r = log(Z^-1 G_a^-1 G_b)
__device__ __forceinline__ void edge_residual(const double* Ga, const double* Gb, const double* Z, double* r) {
    double Rab[9], d[3], tab[3], ER[9], Et[3];
    m3t_mul(Ga, Gb, Rab);
    d[0] = Gb[9] - Ga[9]; d[1] = Gb[10] - Ga[10]; d[2] = Gb[11] - Ga[11];
    m3t_vec(Ga, d, tab);
    m3t_mul(Z, Rab, ER);
    d[0] = tab[0] - Z[9]; d[1] = tab[1] - Z[10]; d[2] = tab[2] - Z[11];
    m3t_vec(Z, d, Et);
    se3_log_dev(ER, Et, r);
}

__device__ __forceinline__ double edge_cost(const double* r, const double* __restrict__ Om) {
    double c = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double w = 0.0;
#pragma unroll
        for (int j = 0; j < 6; ++j) w += Om[6 * i + j] * r[j];
        c += r[i] * w;
    }
    return 0.5 * c;
}

// the edge's Omega-weighted blocks at (G_a, G_b): out = H_aa, H_bb, H_ab (row-major 6x6), g_a, g_b; returns its cost
__device__ double edge_linearize(const double* Ga, const double* Gb, const double* Z, const double* __restrict__ Om, double* __restrict__ out) {
    double r[6];
    edge_residual(Ga, Gb, Z, r);
    // Jb = I + 1/2 ad(r), ad(rho, omega) = [[omega x, rho x], [0, omega x]]
    double Jb[36];
    {
        const double p0 = 0.5 * r[0], p1 = 0.5 * r[1], p2 = 0.5 * r[2], w0 = 0.5 * r[3], w1 = 0.5 * r[4], w2 = 0.5 * r[5];
        const double Wx[9] = {0, -w2, w1, w2, 0, -w0, -w1, w0, 0}, Px[9] = {0, -p2, p1, p2, 0, -p0, -p1, p0, 0};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double I = i == j ? 1.0 : 0.0;
                Jb[6 * i + j] = I + Wx[3 * i + j]; Jb[6 * i + 3 + j] = Px[3 * i + j];
                Jb[6 * (i + 3) + j] = 0.0; Jb[6 * (i + 3) + 3 + j] = I + Wx[3 * i + j];
            }
    }
    // Ja = -Jb Ad(G_b^-1 G_a), Ad(R, t) = [[R, [t]x R], [0, R]]
    double Ja[36];
    {
        double Rba[9], d[3], tba[3], TR[9];
        m3t_mul(Gb, Ga, Rba);
        d[0] = Ga[9] - Gb[9]; d[1] = Ga[10] - Gb[10]; d[2] = Ga[11] - Gb[11];
        m3t_vec(Gb, d, tba);
        const double tx[9] = {0, -tba[2], tba[1], tba[2], 0, -tba[0], -tba[1], tba[0], 0};
        m3_mul(tx, Rba, TR);
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                double v = 0.0;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const double ad = k < 3 ? (j < 3 ? Rba[3 * k + j] : TR[3 * k + j - 3]) : (j < 3 ? 0.0 : Rba[3 * (k - 3) + j - 3]);
                    v += Jb[6 * i + k] * ad;
                }
                Ja[6 * i + j] = -v;
            }
    }
    double w[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < 6; ++j) v += Om[6 * i + j] * r[j];
        w[i] = v;
    }
    // Y = Omega Jb, column by column: H_bb = Jb^T Y, H_ab = Ja^T Y
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        double y[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) v += Om[6 * i + k] * Jb[6 * k + c];
            y[i] = v;
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            double hb = 0.0, ha = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) { hb += Jb[6 * k + i] * y[k]; ha += Ja[6 * k + i] * y[k]; }
            out[36 + 6 * i + c] = hb; out[72 + 6 * i + c] = ha;
        }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        double y[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) v += Om[6 * i + k] * Ja[6 * k + c];
            y[i] = v;
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            double h = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) h += Ja[6 * k + i] * y[k];
            out[6 * i + c] = h;
        }
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double ga = 0.0, gb = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) { ga += Ja[6 * k + i] * w[k]; gb += Jb[6 * k + i] * w[k]; }
        out[108 + i] = ga; out[114 + i] = gb;
    }
    double c = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) c += r[i] * w[i];
    return 0.5 * c;
}

// Omega = Sigma^-1 from the Cholesky factor of Sigma's lower triangle; false if an entry is not finite or Sigma is not positive
// definite (the edge is then not used)
__device__ bool information_from_cov(const double* __restrict__ S, double* __restrict__ Om) {
    for (int i = 0; i < 36; ++i) if (!isfinite(S[i])) return false;
    double L[36], Li[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double v = S[6 * i + j];
            for (int k = 0; k < j; ++k) v -= L[6 * i + k] * L[6 * j + k];
            if (i == j) { if (!(v > 0.0)) return false; L[6 * i + i] = sqrt(v); }
            else L[6 * i + j] = v / L[6 * j + j];
        }
    for (int c = 0; c < 6; ++c)                                   // Li = L^-1, lower triangular
        for (int i = 0; i < 6; ++i) {
            if (i < c) { Li[6 * i + c] = 0.0; continue; }
            double v = i == c ? 1.0 : 0.0;
            for (int k = c; k < i; ++k) v -= L[6 * i + k] * Li[6 * k + c];
            Li[6 * i + c] = v / L[6 * i + i];
        }
    for (int i = 0; i < 6; ++i)                                   // Omega = Li^T Li
        for (int j = 0; j < 6; ++j) {
            double v = 0.0;
            for (int k = 0; k < 6; ++k) v += Li[6 * k + i] * Li[6 * k + j];
            if (!isfinite(v)) return false;
            Om[6 * i + j] = v;
        }
    return true;
}

// ------------------------------------------------------------------ warp-level dense s x s block kernels (row-major, ld = s)
// In-place lower Cholesky (reads and writes the lower triangle); false if not positive definite.  Uniform across the warp.
__device__ bool w_chol(double* A, int s, int lane) {
    for (int j = 0; j < s; ++j) {
        __syncwarp();
        const double d = A[j * s + j];
        if (!(d > 0.0) || !isfinite(d)) return false;
        const double l = sqrt(d), il = 1.0 / l;
        __syncwarp();
        for (int i = j + 1 + lane; i < s; i += 32) A[i * s + j] *= il;
        if (lane == 0) A[j * s + j] = l;
        __syncwarp();
        const int m = s - j - 1;
        for (int q = lane; q < m * m; q += 32) {
            const int i = j + 1 + q / m, k = j + 1 + q % m;
            if (k <= i) A[i * s + k] -= A[i * s + j] * A[k * s + j];
        }
    }
    __syncwarp();
    return true;
}
// B <- L^-1 B (lanes own columns)
__device__ void w_trsm_l(const double* L, double* B, int s, int lane) {
    __syncwarp();
    for (int c = lane; c < s; c += 32)
        for (int i = 0; i < s; ++i) {
            double v = B[i * s + c];
            for (int k = 0; k < i; ++k) v -= L[i * s + k] * B[k * s + c];
            B[i * s + c] = v / L[i * s + i];
        }
    __syncwarp();
}
// B <- L^-T B
__device__ void w_trsm_lt(const double* L, double* B, int s, int lane) {
    __syncwarp();
    for (int c = lane; c < s; c += 32)
        for (int i = s - 1; i >= 0; --i) {
            double v = B[i * s + c];
            for (int k = i + 1; k < s; ++k) v -= L[k * s + i] * B[k * s + c];
            B[i * s + c] = v / L[i * s + i];
        }
    __syncwarp();
}
// C <- beta C + alpha op(A) op(B); C must not alias A or B
__device__ void w_gemm(double* C, const double* A, bool ta, const double* B, bool tb, double alpha, double beta, int s, int lane) {
    __syncwarp();
    for (int q = lane; q < s * s; q += 32) {
        const int i = q / s, j = q % s;
        double v = 0.0;
        for (int k = 0; k < s; ++k) v += (ta ? A[k * s + i] : A[i * s + k]) * (tb ? B[j * s + k] : B[k * s + j]);
        C[q] = beta == 0.0 ? alpha * v : beta * C[q] + alpha * v;
    }
    __syncwarp();
}
// dst <- src^T (or src)
__device__ void w_copy(double* dst, const double* src, bool tr, int s, int lane) {
    __syncwarp();
    for (int q = lane; q < s * s; q += 32) { const int i = q / s, j = q % s; dst[q] = tr ? src[j * s + i] : src[q]; }
    __syncwarp();
}
__device__ void w_identity(double* A, int s, int lane) {
    __syncwarp();
    for (int q = lane; q < s * s; q += 32) A[q] = (q / s == q % s) ? 1.0 : 0.0;
    __syncwarp();
}
// b <- L^-1 b, b <- L^-T b (lane 0), b <- b - op(A) x (lanes own rows)
__device__ void w_trsv_l(const double* L, double* b, int s, int lane) {
    __syncwarp();
    if (lane == 0)
        for (int i = 0; i < s; ++i) { double v = b[i]; for (int k = 0; k < i; ++k) v -= L[i * s + k] * b[k]; b[i] = v / L[i * s + i]; }
    __syncwarp();
}
__device__ void w_trsv_lt(const double* L, double* b, int s, int lane) {
    __syncwarp();
    if (lane == 0)
        for (int i = s - 1; i >= 0; --i) { double v = b[i]; for (int k = i + 1; k < s; ++k) v -= L[k * s + i] * b[k]; b[i] = v / L[i * s + i]; }
    __syncwarp();
}
__device__ void w_gemv_sub(double* b, const double* A, bool ta, const double* x, int s, int lane) {
    __syncwarp();
    for (int i = lane; i < s; i += 32) {
        double v = 0.0;
        for (int k = 0; k < s; ++k) v += (ta ? A[k * s + i] : A[i * s + k]) * x[k];
        b[i] -= v;
    }
    __syncwarp();
}

// deterministic block sum: thread t holds its own partial; fixed tree over the CTA
__device__ double block_sum(double v, double* red) {
    red[threadIdx.x] = v;
    __syncthreads();
    for (int h = PGO_THREADS / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

struct PgoArgs {
    int ngraphs, nedges;
    const int *ref, *now;
    const double *meas, *cov;
    double* poses;
    double* node_cov;
    dvo_pgo_info* info;
    dvo_pgo_params prm;
    double* dscr;
    int* iscr;
};

// Factor D/R (block tridiagonal, M super-nodes) by odd-even cyclic reduction in place: D[k] <- L_k, Wl[k] <- L_k^-1 A(k, left),
// R[k] <- L_k^-1 A(k, right) for every eliminated k; survivors receive the Schur updates.  Returns false (CTA-uniform) if a
// pivot block is not positive definite.
__device__ bool cr_factor(double* D, double* R, double* Wl, int s, int M, int warp, int lane) {
    const long long blk = (long long)s * s;
    int bad = 0;
    for (int h = 1; h < M; h <<= 1) {
        for (int k = h * (2 * warp + 1); k < M; k += 2 * h * PGO_WARPS) {
            if (!w_chol(D + k * blk, s, lane)) { bad = 1; continue; }
            w_copy(Wl + k * blk, R + (k - h) * blk, true, s, lane);                  // A(k, l) = R[l]^T
            w_trsm_l(D + k * blk, Wl + k * blk, s, lane);
            if (k + h < M) w_trsm_l(D + k * blk, R + k * blk, s, lane);
        }
        if (__syncthreads_or(bad)) return false;
        for (int j = 2 * h * warp; j < M; j += 2 * h * PGO_WARPS) {
            if (j - h >= 0) w_gemm(D + j * blk, R + (j - h) * blk, true, R + (j - h) * blk, false, -1.0, 1.0, s, lane);
            if (j + h < M) {
                w_gemm(D + j * blk, Wl + (j + h) * blk, true, Wl + (j + h) * blk, false, -1.0, 1.0, s, lane);
                if (j + 2 * h < M) w_gemm(R + j * blk, Wl + (j + h) * blk, true, R + (j + h) * blk, false, -1.0, 0.0, s, lane);
            }
        }
        __syncthreads();
    }
    if (warp == 0 && !w_chol(D, s, lane)) bad = 1;
    return !__syncthreads_or(bad);
}

// x = A^-1 b in place on b with the factor of cr_factor
__device__ void cr_solve(const double* D, const double* R, const double* Wl, double* b, int s, int M, int warp, int lane) {
    const long long blk = (long long)s * s;
    int top = 1;
    for (int h = 1; h < M; h <<= 1) {
        for (int k = h * (2 * warp + 1); k < M; k += 2 * h * PGO_WARPS) w_trsv_l(D + k * blk, b + k * s, s, lane);
        __syncthreads();
        for (int j = 2 * h * warp; j < M; j += 2 * h * PGO_WARPS) {
            if (j - h >= 0) w_gemv_sub(b + j * s, R + (j - h) * blk, true, b + (j - h) * s, s, lane);
            if (j + h < M) w_gemv_sub(b + j * s, Wl + (j + h) * blk, true, b + (j + h) * s, s, lane);
        }
        __syncthreads();
        top = 2 * h;
    }
    if (warp == 0) { w_trsv_l(D, b, s, lane); w_trsv_lt(D, b, s, lane); }
    __syncthreads();
    for (int h = top / 2; h >= 1; h >>= 1) {
        for (int k = h * (2 * warp + 1); k < M; k += 2 * h * PGO_WARPS) {
            w_gemv_sub(b + k * s, Wl + k * blk, false, b + (k - h) * s, s, lane);
            if (k + h < M) w_gemv_sub(b + k * s, R + k * blk, false, b + (k + h) * s, s, lane);
            w_trsv_lt(D + k * blk, b + k * s, s, lane);
        }
        __syncthreads();
    }
}

// diagonal blocks SD[k] of A^-1 (and the neighbour blocks SL[k] = Sigma(k, left), SR[k] = Sigma(k, right)) from the factor,
// top of the reduction tree down
__device__ void cr_selinv(const double* D, const double* R, const double* Wl, double* SD, double* SL, double* SR, int s, int M, int warp,
                          int lane) {
    const long long blk = (long long)s * s;
    int top = 1, levels = 0;
    while (top < M) { top <<= 1; ++levels; }
    if (warp == 0) { w_identity(SD, s, lane); w_trsm_l(D, SD, s, lane); w_trsm_lt(D, SD, s, lane); }
    __syncthreads();
    for (int lev = levels - 1; lev >= 0; --lev) {
        const int h = 1 << lev;
        for (int k = h * (2 * warp + 1); k < M; k += 2 * h * PGO_WARPS) {
            const int l = k - h, r = k + h;
            const double* Lk = D + k * blk;
            const bool has_r = r < M, l_elim = (l >> (lev + 1)) & 1;     // which of l, r holds Sigma(l, r) as a neighbour block
            double* sl = SL + k * blk; double* sr = SR + k * blk; double* sd = SD + k * blk;
            w_gemm(sl, Wl + k * blk, false, SD + l * blk, false, -1.0, 0.0, s, lane);               // -(W_kl S_ll + W_kr S_rl)
            if (has_r) {
                if (l_elim) w_gemm(sl, R + k * blk, false, SR + l * blk, true, -1.0, 1.0, s, lane);  // S_rl = SR[l]^T
                else w_gemm(sl, R + k * blk, false, SL + r * blk, false, -1.0, 1.0, s, lane);        // S_rl = SL[r]
                if (l_elim) w_gemm(sr, Wl + k * blk, false, SR + l * blk, false, -1.0, 0.0, s, lane); // -(W_kl S_lr + W_kr S_rr)
                else w_gemm(sr, Wl + k * blk, false, SL + r * blk, true, -1.0, 0.0, s, lane);
                w_gemm(sr, R + k * blk, false, SD + r * blk, false, -1.0, 1.0, s, lane);
                w_trsm_lt(Lk, sr, s, lane);
            }
            w_trsm_lt(Lk, sl, s, lane);
            w_identity(sd, s, lane);                                                             // L_k^-T (L_k^-1 - W_kl S_kl^T - W_kr S_kr^T)
            w_trsm_l(Lk, sd, s, lane);
            w_gemm(sd, Wl + k * blk, false, sl, true, -1.0, 1.0, s, lane);
            if (has_r) w_gemm(sd, R + k * blk, false, sr, true, -1.0, 1.0, s, lane);
            w_trsm_lt(Lk, sd, s, lane);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(PGO_THREADS) pgo_kernel(PgoArgs A, PgoLayout Ly) {
    const int g = blockIdx.x, tid = threadIdx.x, warp = tid / 32, lane = tid % 32;
    const int N = Ly.N, E = Ly.E, L = Ly.L, s = Ly.s, M = Ly.M;
    const long long blk = (long long)s * s;
    double* dq = A.dscr + (long long)g * Ly.dbl;
    int* iq = A.iscr + (long long)g * Ly.ints;
    const int* ea = A.ref + (long long)g * E;
    const int* eb = A.now + (long long)g * E;
    const double* Z = A.meas + (long long)g * E * 12;
    const double* S = A.cov + (long long)g * E * 36;
    double* P = A.poses + (long long)g * N * 12;
    double* X = dq + Ly.X; double* Xt = dq + Ly.Xt; double* Om = dq + Ly.Om; double* EC = dq + Ly.EC;
    double* HD = dq + Ly.HD; double* HR = dq + Ly.HR; double* D = dq + Ly.D; double* R = dq + Ly.R; double* Wl = dq + Ly.Wl;
    double* gv = dq + Ly.gv; double* bv = dq + Ly.bv;
    int* valid = iq + Ly.valid; int* deg = iq + Ly.deg; int* off = iq + Ly.off; int* cur = iq + Ly.cur; int* inc = iq + Ly.inc;
    int* label = iq + Ly.label;
    __shared__ double red[PGO_THREADS];
    __shared__ int sh_used;

    // ---- argument check (device indices): bit 0
    int bad = 0;
    for (int e = tid; e < E; e += PGO_THREADS) {
        const int a = ea[e], b = eb[e];
        if (a < 0 || a >= N || b < 0 || b >= N || a == b || abs(a - b) > L) bad = 1;
    }
    int status = __syncthreads_or(bad) ? 1 : 0;
    int used = 0;
    if (!status) {
        // ---- information matrices, validity, incidence lists, connectivity
        for (int i = tid; i < N; i += PGO_THREADS) { deg[i] = 0; label[i] = i; }
        if (tid == 0) sh_used = 0;
        __syncthreads();
        for (int e = tid; e < E; e += PGO_THREADS) {
            const int ok = information_from_cov(S + 36LL * e, Om + 36LL * e) ? 1 : 0;
            valid[e] = ok;
            if (ok) { atomicAdd(&deg[ea[e]], 1); atomicAdd(&deg[eb[e]], 1); atomicAdd(&sh_used, 1); }
        }
        __syncthreads();
        used = sh_used;
        if (tid == 0) { int o = 0; for (int i = 0; i < N; ++i) { off[i] = o; cur[i] = o; o += deg[i]; } off[N] = o; }
        __syncthreads();
        for (int e = tid; e < E; e += PGO_THREADS)
            if (valid[e]) { inc[atomicAdd(&cur[ea[e]], 1)] = e; inc[atomicAdd(&cur[eb[e]], 1)] = e; }
        __syncthreads();
        for (int i = tid; i < N; i += PGO_THREADS)                  // edge-index order within each list
            for (int p = off[i] + 1; p < off[i + 1]; ++p) {
                const int v = inc[p]; int q = p - 1;
                while (q >= off[i] && inc[q] > v) { inc[q + 1] = inc[q]; --q; }
                inc[q + 1] = v;
            }
        for (;;) {
            int changed = 0;
            for (int e = tid; e < E; e += PGO_THREADS) {
                if (!valid[e]) continue;
                const int la = label[ea[e]], lb = label[eb[e]];
                if (la != lb) { const int m = min(la, lb); atomicMin(&label[ea[e]], m); atomicMin(&label[eb[e]], m); changed = 1; }
            }
            __syncthreads();
            for (int i = tid; i < N; i += PGO_THREADS) {
                const int l = label[i], ll = label[l];
                if (ll < l) { atomicMin(&label[i], ll); changed = 1; }
            }
            if (!__syncthreads_or(changed)) break;
        }
        int disc = 0;
        for (int i = tid; i < N; i += PGO_THREADS) if (label[i] != 0) disc = 1;
        if (__syncthreads_or(disc)) status |= 2;
    }

    double F = CUDART_NAN, F0 = CUDART_NAN;
    int iters = 0, accepted = 0;
    const bool want_cov = A.node_cov != nullptr;
    if (!status) {
        for (int q = tid; q < 12 * N; q += PGO_THREADS) { X[q] = P[q]; Xt[q] = P[q]; }
        for (long long q = tid; q < M * blk; q += PGO_THREADS) {    // structural zeros and the identity rows of the padding
            const int j = (int)(q / blk), rr = (int)((q % blk) / s), cc = (int)(q % s);
            const bool pad = 1 + j * L + rr / 6 >= N;
            HD[q] = (pad && rr == cc) ? 1.0 : 0.0; HR[q] = 0.0;
        }
        for (int q = tid; q < M * s; q += PGO_THREADS) gv[q] = 0.0;
        __syncthreads();

        // linearise at X: per-edge blocks, then the node blocks of H and g (one thread per entry, incidence order); returns F
        auto linearize = [&]() -> double {
            double part = 0.0;
            for (int e = tid; e < E; e += PGO_THREADS) {
                if (!valid[e]) continue;
                part += edge_linearize(X + 12 * ea[e], X + 12 * eb[e], Z + 12LL * e, Om + 36LL * e, EC + (long long)EC_STRIDE * e);
            }
            const double f = block_sum(part, red);
            const int nb = (N - 1) * (L + 1) * 36;
            for (int w = tid; w < nb + (N - 1) * 6; w += PGO_THREADS) {
                if (w < nb) {
                    const int i = 1 + w / ((L + 1) * 36), o = (w / 36) % (L + 1), rc = w % 36, r = rc / 6, c = rc % 6, k = i + o;
                    if (k >= N) continue;
                    double v = 0.0;
                    for (int p = off[i]; p < off[i + 1]; ++p) {
                        const int e = inc[p], a = ea[e], b = eb[e];
                        const double* ec = EC + (long long)EC_STRIDE * e;
                        if (o == 0) v += a == i ? ec[rc] : ec[36 + rc];
                        else if (a == i && b == k) v += ec[72 + 6 * r + c];
                        else if (b == i && a == k) v += ec[72 + 6 * c + r];
                    }
                    const int j = (i - 1) / L, pi = (i - 1) % L, jk = (k - 1) / L, pk = (k - 1) % L;
                    if (jk == j) {
                        HD[j * blk + (6 * pi + r) * s + 6 * pk + c] = v;
                        if (o) HD[j * blk + (6 * pk + c) * s + 6 * pi + r] = v;
                    } else {
                        HR[j * blk + (6 * pi + r) * s + 6 * pk + c] = v;
                    }
                } else {
                    const int q = w - nb, i = 1 + q / 6, r = q % 6;
                    double v = 0.0;
                    for (int p = off[i]; p < off[i + 1]; ++p) {
                        const int e = inc[p];
                        v += EC[(long long)EC_STRIDE * e + (ea[e] == i ? 108 : 114) + r];
                    }
                    gv[((i - 1) / L) * s + 6 * ((i - 1) % L) + r] = v;
                }
            }
            __syncthreads();
            return f;
        };
        auto cost_at = [&](const double* Y) -> double {
            double part = 0.0;
            for (int e = tid; e < E; e += PGO_THREADS) {
                if (!valid[e]) continue;
                double r[6];
                edge_residual(Y + 12 * ea[e], Y + 12 * eb[e], Z + 12LL * e, r);
                part += edge_cost(r, Om + 36LL * e);
            }
            return block_sum(part, red);
        };

        F = F0 = linearize();
        double lambda = A.prm.lambda0;
        while (iters < A.prm.max_iterations) {
            ++iters;
            // (H + lambda diag(H)) delta = -g
            for (long long q = tid; q < M * blk; q += PGO_THREADS) {
                const long long rr = (q % blk) / s, cc = q % s;
                D[q] = rr == cc ? HD[q] + lambda * HD[q] : HD[q];
                R[q] = HR[q];
            }
            for (int q = tid; q < M * s; q += PGO_THREADS) bv[q] = -gv[q];
            __syncthreads();
            const bool ok = cr_factor(D, R, Wl, s, M, warp, lane);
            double Ft = CUDART_INF;
            if (ok) {
                cr_solve(D, R, Wl, bv, s, M, warp, lane);
                for (int i = 1 + tid; i < N; i += PGO_THREADS) {          // X_t = X exp(delta)
                    const double* d = bv + ((i - 1) / L) * s + 6 * ((i - 1) % L);
                    double dR[9], dt[3], t2[3];
                    se3_exp_dev(d, dR, dt);
                    const double* x = X + 12 * i; double* y = Xt + 12 * i;
                    m3_mul(x, dR, y);
                    m3_vec(x, dt, t2);
                    y[9] = x[9] + t2[0]; y[10] = x[10] + t2[1]; y[11] = x[11] + t2[2];
                }
                __syncthreads();
                Ft = cost_at(Xt);
            }
            if (ok && Ft < F) {
                ++accepted;
                const double rel = F > 0.0 ? (F - Ft) / F : 0.0;
                for (int q = tid; q < 12 * N; q += PGO_THREADS) X[q] = Xt[q];
                __syncthreads();
                F = Ft;
                lambda /= 10.0;
                if (rel < A.prm.rel_tol) break;
                linearize();
            } else {
                lambda *= 10.0;
                if (lambda > PGO_LAMBDA_MAX) break;
            }
        }
        for (int q = tid; q < 12 * N; q += PGO_THREADS) P[q] = X[q];
        if (want_cov) {                                                   // H at the returned poses, lambda = 0
            linearize();
            for (long long q = tid; q < M * blk; q += PGO_THREADS) { D[q] = HD[q]; R[q] = HR[q]; }
            __syncthreads();
            if (cr_factor(D, R, Wl, s, M, warp, lane)) {
                double* SD = dq + Ly.SD;
                cr_selinv(D, R, Wl, SD, dq + Ly.SL, dq + Ly.SR, s, M, warp, lane);
                double* nc = A.node_cov + (long long)g * N * 36;
                for (int q = tid; q < 36 * N; q += PGO_THREADS) {
                    const int i = q / 36, r = (q % 36) / 6, c = q % 6;
                    nc[q] = i == 0 ? 0.0 : SD[((i - 1) / L) * blk + (6 * ((i - 1) % L) + r) * s + 6 * ((i - 1) % L) + c];
                }
            } else {
                status |= 4;
            }
        }
    }
    if (want_cov && status) {
        double* nc = A.node_cov + (long long)g * N * 36;
        for (int q = tid; q < 36 * N; q += PGO_THREADS) nc[q] = CUDART_NAN;
    }
    if (A.info && tid == 0) {
        dvo_pgo_info I;
        I.status = status; I.iterations = iters; I.accepted = accepted; I.edges_used = used;
        I.cost_initial = F0; I.cost_final = F;
        A.info[g] = I;
    }
}

}  // namespace

int pgo_scratch_size(int nnodes, int nedges, int max_lag, size_t* dbl, size_t* ints) {
    const PgoLayout l = pgo_layout(nnodes, nedges, max_lag);
    *dbl = (size_t)l.dbl; *ints = (size_t)l.ints;
    return DVO_OK;
}

int launch_pose_graph(dvo_ctx* c, int ngraphs, int nnodes, int nedges, int max_lag, const int* d_ref, const int* d_now, const double* d_meas,
                      const double* d_cov, double* d_poses, const dvo_pgo_params* prm, double* d_node_cov, dvo_pgo_info* d_info, double* d_dscr,
                      int* d_iscr) {
    PgoArgs a;
    a.ngraphs = ngraphs; a.nedges = nedges; a.ref = d_ref; a.now = d_now; a.meas = d_meas; a.cov = d_cov; a.poses = d_poses;
    a.node_cov = d_node_cov; a.info = d_info; a.prm = *prm; a.dscr = d_dscr; a.iscr = d_iscr;
    pgo_kernel<<<ngraphs, PGO_THREADS, 0, c->stream>>>(a, pgo_layout(nnodes, nedges, max_lag));
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}
