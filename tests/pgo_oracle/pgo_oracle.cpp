// pgo_oracle.cpp -- CPU oracle of the windowed pose-graph optimisation (dvo_pose_graph_optimize, include/dvo_b200.h) and its C
// shim for ctypes (tests/pgo_oracle_lib.py).  TEST INFRASTRUCTURE ONLY: nothing under rgbd_odometry_b200/ includes, links or
// calls it.  It builds on the SE(3) closed forms of oracle/dvo_oracle.hpp (se3_exp, se3_log, mat3_*), included as is.
//
// Build: g++ -O3 -ffp-contract=off -std=c++17 -fPIC -shared (tests/pgo_oracle_lib.py does it on first use).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "../../oracle/dvo_oracle.hpp"

namespace orc {

// ------------------------------------------------------------------------------------------------------
// Windowed pose-graph optimisation (dvo_pose_graph_optimize, include/dvo_b200.h).  Same problem and the same LM decisions as
// the device, but the damped system is factored by a SEQUENTIAL banded Cholesky of the scalar matrix (the device uses block
// cyclic reduction), and the marginals are columns of H^-1 from that factor, so the two eliminations are independent.
// ------------------------------------------------------------------------------------------------------
namespace pgo {
struct Params { int max_iterations; double lambda0, rel_tol; };
struct Info { int status, iterations, accepted, edges_used; double cost_initial, cost_final; };
constexpr double LAMBDA_MAX = 1e16;

// Omega = Sigma^-1 from the Cholesky factor of Sigma's lower triangle; false if non-finite or not positive definite
inline bool information(const double* S, double* Om) {
    for (int i = 0; i < 36; ++i) if (!std::isfinite(S[i])) return false;
    double L[36] = {0}, Li[36] = {0};
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double v = S[6 * i + j];
            for (int k = 0; k < j; ++k) v -= L[6 * i + k] * L[6 * j + k];
            if (i == j) { if (!(v > 0.0)) return false; L[6 * i + i] = std::sqrt(v); }
            else L[6 * i + j] = v / L[6 * j + j];
        }
    for (int c = 0; c < 6; ++c)
        for (int i = c; i < 6; ++i) {
            double v = i == c ? 1.0 : 0.0;
            for (int k = c; k < i; ++k) v -= L[6 * i + k] * Li[6 * k + c];
            Li[6 * i + c] = v / L[6 * i + i];
        }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            double v = 0.0;
            for (int k = 0; k < 6; ++k) v += Li[6 * k + i] * Li[6 * k + j];
            if (!std::isfinite(v)) return false;
            Om[6 * i + j] = v;
        }
    return true;
}

// r = log(Z^-1 Ga^-1 Gb); records are R[9] T[3]
inline void residual(const double* Ga, const double* Gb, const double* Z, double* r) {
    double RaT[9], RzT[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { RaT[3 * i + j] = Ga[3 * j + i]; RzT[3 * i + j] = Z[3 * j + i]; }
    double Rab[9], tab[3], d[3], ER[9], Et[3];
    mat3_mul(RaT, Gb, Rab);
    for (int i = 0; i < 3; ++i) d[i] = Gb[9 + i] - Ga[9 + i];
    mat3_vec(RaT, d, tab);
    mat3_mul(RzT, Rab, ER);
    for (int i = 0; i < 3; ++i) d[i] = tab[i] - Z[9 + i];
    mat3_vec(RzT, d, Et);
    se3_log(ER, Et, r);
}

// Jb = I + 1/2 ad(r), Ja = -Jb Ad(Gb^-1 Ga)
inline void jacobians(const double* Ga, const double* Gb, const double* r, double* Ja, double* Jb) {
    const double p[3] = {0.5 * r[0], 0.5 * r[1], 0.5 * r[2]}, w[3] = {0.5 * r[3], 0.5 * r[4], 0.5 * r[5]};
    const double Wx[9] = {0, -w[2], w[1], w[2], 0, -w[0], -w[1], w[0], 0}, Px[9] = {0, -p[2], p[1], p[2], 0, -p[0], -p[1], p[0], 0};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double I = i == j ? 1.0 : 0.0;
            Jb[6 * i + j] = I + Wx[3 * i + j]; Jb[6 * i + 3 + j] = Px[3 * i + j];
            Jb[6 * (i + 3) + j] = 0.0; Jb[6 * (i + 3) + 3 + j] = I + Wx[3 * i + j];
        }
    double RbT[9], Rba[9], tba[3], d[3], TR[9], Ad[36];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) RbT[3 * i + j] = Gb[3 * j + i];
    mat3_mul(RbT, Ga, Rba);
    for (int i = 0; i < 3; ++i) d[i] = Ga[9 + i] - Gb[9 + i];
    mat3_vec(RbT, d, tba);
    const double tx[9] = {0, -tba[2], tba[1], tba[2], 0, -tba[0], -tba[1], tba[0], 0};
    mat3_mul(tx, Rba, TR);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            Ad[6 * i + j] = Rba[3 * i + j]; Ad[6 * i + 3 + j] = TR[3 * i + j];
            Ad[6 * (i + 3) + j] = 0.0; Ad[6 * (i + 3) + 3 + j] = Rba[3 * i + j];
        }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            double v = 0.0;
            for (int k = 0; k < 6; ++k) v += Jb[6 * i + k] * Ad[6 * k + j];
            Ja[6 * i + j] = -v;
        }
}

inline double quad(const double* r, const double* Om) {
    double c = 0.0;
    for (int i = 0; i < 6; ++i) { double w = 0.0; for (int j = 0; j < 6; ++j) w += Om[6 * i + j] * r[j]; c += r[i] * w; }
    return 0.5 * c;
}

// symmetric band matrix, lower band stored: a[i][i - j] for 0 <= i - j <= w
struct Band {
    int n = 0, w = 0; std::vector<double> a;
    void reset(int n_, int w_) { n = n_; w = w_; a.assign((size_t)n * (w + 1), 0.0); }
    double& at(int i, int j) { return a[(size_t)i * (w + 1) + (i - j)]; }
    double get(int i, int j) const { if (i < j) std::swap(i, j); return i - j > w ? 0.0 : a[(size_t)i * (w + 1) + (i - j)]; }
};
// in-place banded Cholesky, row by row
inline bool band_chol(Band& B) {
    for (int i = 0; i < B.n; ++i)
        for (int j = std::max(0, i - B.w); j <= i; ++j) {
            double v = B.at(i, j);
            for (int k = std::max(0, i - B.w); k < j; ++k) v -= B.at(i, k) * B.at(j, k);
            if (i == j) { if (!(v > 0.0) || !std::isfinite(v)) return false; B.at(i, i) = std::sqrt(v); }
            else B.at(i, j) = v / B.at(j, j);
        }
    return true;
}
inline void band_solve(Band& L, double* x, int first = 0) {     // x <- (L L^T)^-1 x; x[0 .. first) must be zero
    for (int i = first; i < L.n; ++i) {
        double v = x[i];
        for (int k = std::max(first, i - L.w); k < i; ++k) v -= L.at(i, k) * x[k];
        x[i] = v / L.at(i, i);
    }
    for (int i = L.n - 1; i >= 0; --i) {
        double v = x[i];
        for (int k = i + 1; k <= std::min(L.n - 1, i + L.w); ++k) v -= L.at(k, i) * x[k];
        x[i] = v / L.at(i, i);
    }
}

struct Graph {
    int N, E, L; const int *a, *b; const double *Z; std::vector<double> Om; std::vector<char> ok;
};
inline double cost(const Graph& G, const double* X) {
    double F = 0.0;
    for (int e = 0; e < G.E; ++e) {
        if (!G.ok[e]) continue;
        double r[6]; residual(X + 12 * G.a[e], X + 12 * G.b[e], G.Z + 12 * e, r);
        F += quad(r, &G.Om[36 * e]);
    }
    return F;
}
// H (band, unknowns 6 (i - 1) + k of nodes i >= 1) and g at X, edges in index order; returns F
inline double linearize(const Graph& G, const double* X, Band& H, std::vector<double>& g) {
    const int n = 6 * (G.N - 1);
    H.reset(n, 6 * G.L + 5); g.assign(n, 0.0);
    double F = 0.0;
    for (int e = 0; e < G.E; ++e) {
        if (!G.ok[e]) continue;
        const int a = G.a[e], b = G.b[e];
        const double* Om = &G.Om[36 * e];
        double r[6], Ja[36], Jb[36], w[6];
        residual(X + 12 * a, X + 12 * b, G.Z + 12 * e, r);
        jacobians(X + 12 * a, X + 12 * b, r, Ja, Jb);
        F += quad(r, Om);
        for (int i = 0; i < 6; ++i) { double v = 0.0; for (int j = 0; j < 6; ++j) v += Om[6 * i + j] * r[j]; w[i] = v; }
        const double* J[2] = {Ja, Jb}; const int node[2] = {a, b};
        for (int u = 0; u < 2; ++u) {
            if (node[u] == 0) continue;
            const int ou = 6 * (node[u] - 1);
            for (int i = 0; i < 6; ++i) { double v = 0.0; for (int k = 0; k < 6; ++k) v += J[u][6 * k + i] * w[k]; g[ou + i] += v; }
            for (int v2 = 0; v2 < 2; ++v2) {
                if (node[v2] == 0) continue;
                const int ov = 6 * (node[v2] - 1);
                for (int i = 0; i < 6; ++i)
                    for (int j = 0; j < 6; ++j) {
                        if (ou + i < ov + j) continue;                          // lower triangle only
                        double v = 0.0;
                        for (int k = 0; k < 6; ++k) { double y = 0.0; for (int q = 0; q < 6; ++q) y += Om[6 * k + q] * J[v2][6 * q + j]; v += J[u][6 * k + i] * y; }
                        H.at(ou + i, ov + j) += v;
                    }
            }
        }
    }
    return F;
}
inline void retract(const double* x, const double* d, double* y) {
    double dR[9], dt[3], t2[3];
    se3_exp(d, dR, dt);
    mat3_mul(x, dR, y);
    mat3_vec(x, dt, t2);
    for (int i = 0; i < 3; ++i) y[9 + i] = x[9 + i] + t2[i];
}
// (H + lambda diag H) delta = -g by the banded factor; false if not positive definite
inline bool damped_step(const Band& H, const std::vector<double>& g, double lambda, std::vector<double>& delta) {
    Band D = H;
    for (int i = 0; i < D.n; ++i) D.at(i, i) += lambda * H.a[(size_t)i * (H.w + 1)];
    if (!band_chol(D)) return false;
    delta.resize(g.size());
    for (size_t i = 0; i < g.size(); ++i) delta[i] = -g[i];
    band_solve(D, delta.data());
    return true;
}

inline Info optimize(int N, int E, int L, const int* a, const int* b, const double* Z, const double* S, double* poses, const Params& prm,
                     double* node_cov) {
    Info info{0, 0, 0, 0, NAN, NAN};
    for (int e = 0; e < E; ++e)
        if (a[e] < 0 || a[e] >= N || b[e] < 0 || b[e] >= N || a[e] == b[e] || std::abs(a[e] - b[e]) > L) info.status |= 1;
    Graph G{N, E, L, a, b, Z, std::vector<double>(36 * (size_t)E), std::vector<char>(E, 0)};
    if (!info.status) {
        std::vector<int> comp(N);
        for (int i = 0; i < N; ++i) comp[i] = i;
        auto find = [&](int x) { while (comp[x] != x) x = comp[x] = comp[comp[x]]; return x; };
        for (int e = 0; e < E; ++e) {
            G.ok[e] = information(S + 36 * e, &G.Om[36 * e]);
            if (G.ok[e]) { ++info.edges_used; const int ra = find(a[e]), rb = find(b[e]); comp[std::max(ra, rb)] = std::min(ra, rb); }
        }
        for (int i = 0; i < N; ++i) if (find(i) != 0) info.status |= 2;
    }
    if (info.status) {
        if (node_cov) for (size_t q = 0; q < 36 * (size_t)N; ++q) node_cov[q] = NAN;
        return info;
    }
    std::vector<double> X(poses, poses + 12 * (size_t)N), Xt = X, g, delta;
    Band H;
    double F = linearize(G, X.data(), H, g);
    info.cost_initial = F;
    double lambda = prm.lambda0;
    while (info.iterations < prm.max_iterations) {
        ++info.iterations;
        const bool ok = damped_step(H, g, lambda, delta);
        double Ft = INFINITY;
        if (ok) {
            for (int i = 1; i < N; ++i) retract(&X[12 * i], &delta[6 * (i - 1)], &Xt[12 * i]);
            Ft = cost(G, Xt.data());
        }
        if (ok && Ft < F) {
            ++info.accepted;
            const double rel = F > 0.0 ? (F - Ft) / F : 0.0;
            X = Xt; F = Ft; lambda /= 10.0;
            if (rel < prm.rel_tol) break;
            linearize(G, X.data(), H, g);
        } else {
            lambda *= 10.0;
            if (lambda > LAMBDA_MAX) break;
        }
    }
    info.cost_final = F;
    std::memcpy(poses, X.data(), sizeof(double) * 12 * N);
    if (node_cov) {
        linearize(G, X.data(), H, g);
        if (!band_chol(H)) {
            info.status |= 4;
            for (size_t q = 0; q < 36 * (size_t)N; ++q) node_cov[q] = NAN;
        } else {
            for (int q = 0; q < 36; ++q) node_cov[q] = 0.0;
            std::vector<double> x(H.n);
            for (int i = 1; i < N; ++i)
                for (int c = 0; c < 6; ++c) {
                    const int col = 6 * (i - 1) + c;
                    std::fill(x.begin(), x.end(), 0.0); x[col] = 1.0;
                    band_solve(H, x.data(), col);
                    for (int r = 0; r < 6; ++r) node_cov[36 * (size_t)i + 6 * r + c] = x[6 * (i - 1) + r];
                }
        }
    }
    return info;
}
}  // namespace pgo
}  // namespace orc

using namespace orc;

extern "C" {

// ---- windowed pose-graph optimisation (pgo::optimize): graphs one after another; info6 per graph: status, iterations, accepted,
// edges_used, cost_initial, cost_final ----
void orc_pose_graph(int ngraphs, int N, int E, int L, const int* a, const int* b, const double* Z, const double* S, double* poses,
                    int max_iterations, double lambda0, double rel_tol, double* node_cov, double* info6) {
    for (int gi = 0; gi < ngraphs; ++gi) {
        const size_t e0 = (size_t)gi * E, n0 = (size_t)gi * N;
        const pgo::Info I = pgo::optimize(N, E, L, a + e0, b + e0, Z + 12 * e0, S + 36 * e0, poses + 12 * n0, pgo::Params{max_iterations, lambda0, rel_tol},
                                          node_cov ? node_cov + 36 * n0 : nullptr);
        if (info6) { double* o = info6 + 6 * gi; o[0] = I.status; o[1] = I.iterations; o[2] = I.accepted; o[3] = I.edges_used; o[4] = I.cost_initial; o[5] = I.cost_final; }
    }
}
// one graph at poses X: per-edge residuals r (E x 6) and validity, the dense H (n x n, n = 6 (N - 1)), g, F, and the damped step
// (H + lambda diag H) delta = -g through the banded factor (returns -1 if that is not positive definite)
int orc_pgo_system(int N, int E, int L, const int* a, const int* b, const double* Z, const double* S, const double* X, double lambda,
                   double* r, int* valid, double* Hdense, double* g, double* F, double* delta) {
    pgo::Graph G{N, E, L, a, b, Z, std::vector<double>(36 * (size_t)E), std::vector<char>(E, 0)};
    for (int e = 0; e < E; ++e) {
        G.ok[e] = pgo::information(S + 36 * e, &G.Om[36 * e]);
        if (valid) valid[e] = G.ok[e];
        if (r) pgo::residual(X + 12 * a[e], X + 12 * b[e], Z + 12 * e, r + 6 * e);
    }
    pgo::Band H; std::vector<double> gv, d;
    const double f = pgo::linearize(G, X, H, gv);
    if (F) *F = f;
    const int n = H.n;
    if (Hdense) for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) Hdense[(size_t)i * n + j] = H.get(i, j);
    if (g) std::memcpy(g, gv.data(), sizeof(double) * n);
    if (!pgo::damped_step(H, gv, lambda, d)) return -1;
    if (delta) std::memcpy(delta, d.data(), sizeof(double) * n);
    return 0;
}

}  // extern "C"
