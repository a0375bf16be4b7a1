// solver.cu -- the batched coarse-to-fine edge-alignment solve: one persistent CTA per frame pair runs every
// level and iteration on the device (warp, gather, Jacobian, weights, fp64 reduction to g = J^T W eps and
// H = J^T W J, the 6-vector step / 6x6 solve, SE(3) update, best-iterate tracking, termination) with no host
// round trip.  Follows SolveDVO::runIterations (src/SolveDVO.cpp:619-1017), computeJacobianOfNowFrame
// (:306-414) and getReprojectedEpsilons (:425-462); see SURVEY.md Appendix A for the restated arithmetic.
#include "common.cuh"
#include "se3.cuh"

namespace {

constexpr int EVAL_THREADS = 256;     // inspection kernel

// SolveDVO::rotationize (src/SolveDVO.cpp:1269-1282) returns U V^T of the SVD, i.e. the orthogonal polar factor.
// Computed here by Newton's iteration X <- (X + X^-T)/2, which converges quadratically; the input is within
// ~1e-15 of a rotation on every call the solver makes, so one or two steps suffice.
__device__ __forceinline__ void rotationize_dev(double* R) {
    for (int it = 0; it < 40; ++it) {
        const double c00 = R[4] * R[8] - R[5] * R[7], c01 = R[5] * R[6] - R[3] * R[8], c02 = R[3] * R[7] - R[4] * R[6];
        const double c10 = R[2] * R[7] - R[1] * R[8], c11 = R[0] * R[8] - R[2] * R[6], c12 = R[1] * R[6] - R[0] * R[7];
        const double c20 = R[1] * R[5] - R[2] * R[4], c21 = R[2] * R[3] - R[0] * R[5], c22 = R[0] * R[4] - R[1] * R[3];
        const double det = R[0] * c00 + R[1] * c01 + R[2] * c02;
        if (fabs(det) < 1e-300) break;
        const double id = 1.0 / det;
        const double Xit[9] = {c00 * id, c01 * id, c02 * id, c10 * id, c11 * id, c12 * id, c20 * id, c21 * id, c22 * id};   // X^-T
        double delta = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) { const double nv = 0.5 * (R[i] + Xit[i]); delta = fmax(delta, fabs(nv - R[i])); R[i] = nv; }
        if (delta < 4e-16) break;
    }
}

// 6x6 SPD solve by Cholesky; reads the upper triangle of H (row-major).  Returns false if not positive definite.
// The solver's serial step runs on one thread per pair while the CTA waits, so its dependent fp64 chain is what
// counts: the factor is kept as L with the reciprocal diagonal (one rsqrt per column, no division or square root
// anywhere else) and everything stays in registers.  Agrees with the oracle's sqrt/divide form to a few ulps.
__device__ __forceinline__ bool chol6_dev(const double* H, const double* b, double* x) {
    double Lm[6][6], inv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double d = H[6 * j + j];
#pragma unroll
        for (int k = 0; k < j; ++k) d = fma(-Lm[j][k], Lm[j][k], d);
        if (!(d > 0)) return false;
        const double r = rsqrt(d);
        inv[j] = r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double v = H[6 * j + i];
#pragma unroll
            for (int k = 0; k < j; ++k) v = fma(-Lm[i][k], Lm[j][k], v);
            Lm[i][j] = v * r;
        }
    }
    double y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double v = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) v = fma(-Lm[i][k], y[k], v);
        y[i] = v * inv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double v = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) v = fma(-Lm[k][i], x[k], v);
        x[i] = v * inv[i];
    }
    return true;
}

// ------------------------------------------------------------------ per-point evaluation
struct PoseF { float R[9], T[3]; };
struct LevelCam { float M00, M02, M11, M12; int w, h; float wf, hf, M00_lo, M11_lo; int tw; };

// Where the solver reads the now frame's distance transform from: packed 8-byte texels (common.cuh) + per-level lookup
// tables in shared memory, lut[d2] = DTn = sqrtf(d2) * scale, lut[LUT_N + d2] = getWeightOf(DTn), d2 < LUT_N; larger d2 (a
// point more than 63 pixels from every edge) are evaluated directly with the same operations.
constexpr int LUT_N = 4096;
constexpr int LUT_BYTES = 2 * LUT_N * (int)sizeof(float);
struct TexSrc {
    const uint2* tex8;       // level / slot base
    const int32_t* d2;       // row-major d2 of the level / slot (escaped texels only)
    const float* lut;        // shared-memory tables
    float scale;             // (float)(255 / sqrt(max d2))
};

// normalize(0,255,MINMAX) scale of one now-frame level image (src/SolveDVO.cpp:1774; SURVEY B.3)
__device__ __forceinline__ float dtn_scale(unsigned mx2, unsigned ne) {
    if (ne == 0u) return 0.0f;
    const double smax = (double)__fsqrt_rn((float)mx2);          // smin = 0 whenever an edge exists
    const double sc = 255.0 * ((smax > 2.220446049250313e-16) ? __ddiv_rn(1.0, smax) : 0.0);
    return __double2float_rn(sc);
}
__device__ __forceinline__ float dtn_direct(int d2, float scale) { return __fmul_rn(__fsqrt_rn((float)d2), scale); }

template <int THREADS>
__device__ __forceinline__ void build_lut(float* lut, unsigned mx2, float scale) {
    const int n = (int)min(mx2, (unsigned)(LUT_N - 1));
    for (int i = threadIdx.x; i <= n; i += THREADS) {
        const float v = dtn_direct(i, scale);
        lut[i] = v; lut[LUT_N + i] = Ar<DVO_ARITH_EXACT>::weight_ref(v);
    }
}

// the five d2 values of a packed texel; false when the texel is escaped
struct Stencil { int c, l, r, u, d; };
__device__ __forceinline__ bool unpack_texel(const uint2 t, Stencil& s) {
    s.c = (int)(t.x & 0xFFFFu);
    s.l = s.c + ((int)(t.x << 6) >> 22);
    s.r = s.c + ((int)(t.y << 22) >> 22);
    s.u = s.c + ((int)(t.y << 12) >> 22);
    s.d = s.c + ((int)(t.y << 2) >> 22);
    return (int)t.x >= 0;
}
__device__ __forceinline__ void stencil_from_d2(const int32_t* __restrict__ d2, int w, int h, int x, int y, Stencil& s) {
    const int32_t* d = d2 + y * w + x;
    s.c = __ldg(d);
    const bool bx = (x == 0 || x == w - 1), by = (y == 0 || y == h - 1);
    s.l = bx ? s.c : __ldg(d - 1); s.r = bx ? s.c : __ldg(d + 1);
    s.u = by ? s.c : __ldg(d - w); s.d = by ? s.c : __ldg(d + w);
}
// {DTn, gx, gy, getWeightOf(DTn)} of the pixel: DTn = sqrtf(d2) * scale, REFLECT_101 central differences (exactly 0 on the
// border, where the taps coincide), getWeightOf(DTn) (src/SolveDVO.cpp:1774, 1063-1098, 1047-1053)
__device__ __forceinline__ float4 texel_values(const Stencil& s, const float* __restrict__ lut, float scale) {
    float c, l, r, u, d, wt;
    if (max(max(max(s.c, s.l), max(s.r, s.u)), s.d) < LUT_N) {
        c = lut[s.c]; l = lut[s.l]; r = lut[s.r]; u = lut[s.u]; d = lut[s.d]; wt = lut[LUT_N + s.c];
    } else {
        c = dtn_direct(s.c, scale); l = dtn_direct(s.l, scale); r = dtn_direct(s.r, scale);
        u = dtn_direct(s.u, scale); d = dtn_direct(s.d, scale); wt = Ar<DVO_ARITH_EXACT>::weight_ref(c);
    }
    float4 t;
    t.x = c;
    t.y = __fadd_rn(__fmul_rn(-0.5f, l), __fmul_rn(0.5f, r));
    t.z = __fadd_rn(__fmul_rn(-0.5f, u), __fmul_rn(0.5f, d));
    t.w = wt;
    return t;
}

// Z = p'_z * RN(1/p'_z) (:339-341) can only round to 1 or to the float just below 1 (the reciprocal is correctly
// rounded, so the product lies within 2^-24 of 1).  The four IEEE divisions of the reference's A1 matrix (:388-393)
// therefore have closed forms: c/Z is a per-level constant, and a/(Z*Z) = a/(1-2^-23) is the float rounding of
// double(a) * RN64(1/(1-2^-23)) -- checked against a/Z for all 2^32 float inputs (DESIGN.md).  Any other Z takes
// the generic IEEE division.
#define DVO_Z_BELOW_ONE 0x3F7FFFFF
__device__ __forceinline__ LevelCam make_level_cam(const Intr& K, const PyrGeom& geom, int l) {
    LevelCam cam;
    const float scaleFac = (float)ldexp(1.0, -l);                                       // :334
    cam.M00 = __fmul_rn(scaleFac, K.fx); cam.M02 = __fmul_rn(scaleFac, K.cx);            // scaleMatrix * K (:344)
    cam.M11 = __fmul_rn(scaleFac, K.fy); cam.M12 = __fmul_rn(scaleFac, K.cy);
    cam.w = geom.w[l]; cam.h = geom.h[l]; cam.wf = (float)cam.w; cam.hf = (float)cam.h;
    cam.M00_lo = __fdiv_rn(cam.M00, __int_as_float(DVO_Z_BELOW_ONE));
    cam.M11_lo = __fdiv_rn(cam.M11, __int_as_float(DVO_Z_BELOW_ONE));
    cam.tw = geom.tw[l];
    return cam;
}

// The frames every solver kernel reads: the reference slots' edge points and the now slots' distance transforms.
struct FrameArgs {
    PyrGeom geom; Intr K;
    const float *X, *Y, *Z; const int* npts; const unsigned* nedge_now;
    const uint2* tex8; const int32_t* d2; const unsigned* maxd2;
};

// Level l of the reference points of slot rb against the now frame of slot nb.  Builds the now frame's lookup tables into
// lut; they are visible after the caller's next barrier.
struct LevelSrc { const float *X, *Y, *Z; LevelCam cam; TexSrc tex; };
template <int THREADS>
__device__ __forceinline__ LevelSrc level_source(const FrameArgs& f, int l, int rb, int nb, float* lut) {
    LevelSrc o;
    const long long base = lvl_at(f.geom, l, rb);
    o.X = f.X + base; o.Y = f.Y + base; o.Z = f.Z + base;
    o.cam = make_level_cam(f.K, f.geom, l);
    o.tex.tex8 = f.tex8 + tex_at(f.geom, l, nb); o.tex.d2 = f.d2 + lvl_at(f.geom, l, nb); o.tex.lut = lut;
    const long long at = (long long)nb * f.geom.L + l;
    const unsigned mx2 = f.maxd2[at];
    o.tex.scale = dtn_scale(mx2, f.nedge_now[at]);
    build_lut<THREADS>(lut, mx2, o.tex.scale);
    return o;
}

// Reprojection of one reference edge point (computeJacobianOfNowFrame "Step 2/3", src/SolveDVO.cpp:327-345).
// idx < 0 when the reprojection falls outside the now image (J = eps = w = 0, :371-374).
struct Proj { float px, py, pz, inv, X, Y, Z, u, v; int idx; };

__device__ __forceinline__ Proj project_point(float Xp, float Yp, float Zp, const PoseF& P, const LevelCam& cam) {
    typedef Ar<DVO_ARITH_EXACT> E;   // always IEEE-exact so that FAST arithmetic gathers the same texel
    const float* R = P.R;
    Proj o;
    // p' = cR^T (P - cT)                                                       (:330)
    const float d0 = E::sub(Xp, P.T[0]), d1 = E::sub(Yp, P.T[1]), d2 = E::sub(Zp, P.T[2]);
    o.px = E::dot3(R[0], d0, R[3], d1, R[6], d2);
    o.py = E::dot3(R[1], d0, R[4], d1, R[7], d2);
    o.pz = E::dot3(R[2], d0, R[5], d1, R[8], d2);
    o.inv = E::div(1.0f, o.pz);                                                  // :339
    o.X = E::mul(o.px, o.inv); o.Y = E::mul(o.py, o.inv); o.Z = E::mul(o.pz, o.inv);   // :340-341
    o.u = E::dot2(cam.M00, o.X, cam.M02, o.Z);                                   // :344
    o.v = E::dot2(cam.M11, o.Y, cam.M12, o.Z);
    const bool vis = (o.u >= 0.0f && o.u < cam.wf && o.v >= 0.0f && o.v < cam.hf);
    o.idx = vis ? tex_index(__float2int_rz(o.u), __float2int_rz(o.v), cam.tw) : -1;   // :376-377
    return o;
}

// Jacobian row, residual and weight from the gathered texel {DTn, gx, gy, getWeightOf(DTn)} (:383-406, :446-450).
template <int ARITH, int JAC, int WMODE>
__device__ __forceinline__ void finish_point(const Proj& q, const float4 t, const PoseF& P, const LevelCam& cam,
                                             int weight_mode_rt, float huber_k, float* Jr, float& e, float& wgt) {
    const int weight_mode = (WMODE >= 0) ? WMODE : weight_mode_rt;
    typedef Ar<ARITH> A;
    const float* R = P.R;
    const float G0 = t.y, G1 = t.z;
    if (JAC == DVO_JAC_REFERENCE) {
        const float X = q.X, Y = q.Y, Z = q.Z;
        float A00, A02, A11, A12;
        const bool one = (Z == 1.0f), lo = (__float_as_int(Z) == DVO_Z_BELOW_ONE);
        if (ARITH == DVO_ARITH_EXACT && (one || lo)) {
            const double rzz = one ? 1.0 : 0x1.000002000004p+0;                          // RN64(1 / (1 - 2^-23))
            A00 = one ? cam.M00 : cam.M00_lo; A11 = one ? cam.M11 : cam.M11_lo;          // :388, :392
            A02 = -(float)((double)A::mul(cam.M00, X) * rzz);                            // :390
            A12 = -(float)((double)A::mul(cam.M11, Y) * rzz);                            // :393
        } else {
            const float ZZ = A::mul(Z, Z);
            A00 = A::div(cam.M00, Z); A02 = -A::div(A::mul(cam.M00, X), ZZ);
            A11 = A::div(cam.M11, Z); A12 = -A::div(A::mul(cam.M11, Y), ZZ);
        }
        const float w0 = A::dot3(R[0], X, R[3], Y, R[6], Z);                             // :399
        const float w1 = A::dot3(R[1], X, R[4], Y, R[7], Z);
        const float w2 = A::dot3(R[2], X, R[5], Y, R[8], Z);
        const float a = A::mul(G0, A00), b = A::mul(G1, A11), c = A::dot2(G0, A02, G1, A12);
        Jr[0] = -A::dot3(a, R[0], b, R[1], c, R[2]);                                     // :397-405
        Jr[1] = -A::dot3(a, R[3], b, R[4], c, R[5]);
        Jr[2] = -A::dot3(a, R[6], b, R[7], c, R[8]);
        Jr[3] = A::diff2(b, w2, c, w1);
        Jr[4] = A::diff2(c, w0, a, w2);
        Jr[5] = A::diff2(a, w1, b, w0);
    } else {
        const float a = A::mul(A::mul(G0, cam.M00), q.inv), b = A::mul(A::mul(G1, cam.M11), q.inv);
        const float c = -A::mul(A::dot2(a, q.px, b, q.py), q.inv);
        Jr[0] = -a; Jr[1] = -b; Jr[2] = -c;
        Jr[3] = A::diff2(b, q.pz, c, q.py);
        Jr[4] = A::diff2(c, q.px, a, q.pz);
        Jr[5] = A::diff2(a, q.py, b, q.px);
    }
    e = t.x;                                                                     // :446
    if (weight_mode == DVO_WEIGHT_REF_CAUCHY) wgt = (ARITH == DVO_ARITH_EXACT) ? t.w : A::weight_ref(e);
    else if (weight_mode == DVO_WEIGHT_HUBER) { const float ae = fabsf(e); wgt = ae <= huber_k ? 1.0f : A::div(huber_k, ae); }
    else wgt = 1.0f;
}

// raw gathered texel, and its resolution to {DTn, gx, gy, w}
__device__ __forceinline__ uint2 load_texel(const TexSrc& S, int idx) { return __ldg(S.tex8 + idx); }
__device__ __forceinline__ float4 resolve_texel(const TexSrc& S, const LevelCam& cam, const Proj& q, const uint2 raw) {
    Stencil s;
    if (!unpack_texel(raw, s)) stencil_from_d2(S.d2, cam.w, cam.h, __float2int_rz(q.u), __float2int_rz(q.v), s);
    return texel_values(s, S.lut, S.scale);
}

// DTn of pixel (x, y)
__device__ __forceinline__ float dtn_at(const TexSrc& S, const LevelCam& cam, int x, int y) {
    const unsigned w0 = __ldg(&S.tex8[tex_index(x, y, cam.tw)].x);
    int d2 = (int)(w0 & 0xFFFFu);
    if ((int)w0 < 0) d2 = __ldg(S.d2 + y * cam.w + x);
    return d2 < LUT_N ? S.lut[d2] : dtn_direct(d2, S.scale);
}

// SolveDVO::interpolate (src/SolveDVO.cpp:1285-1308) at the reprojection (v = row, u = column): "squared-bilinear"
// lookup of the normalised DT, fp32, products left to right; ceil indices clamped to the image (the reference would
// trip its own bound assert there).  Three extra gathers next to the texel already fetched.
__device__ __forceinline__ float interpolate_dt(const TexSrc& S, const LevelCam& cam, const Proj& q, float Fdd) {
    const int rx_d = __float2int_rz(q.u), ry_d = __float2int_rz(q.v);               // u, v >= 0 here: floor == trunc
    const float fx_d = (float)rx_d, fy_d = (float)ry_d;
    const float inc_x = __fsub_rn(q.u, fx_d), inc_y = __fsub_rn(q.v, fy_d);
    const int rx_u = min(rx_d + (q.u > fx_d ? 1 : 0), cam.w - 1), ry_u = min(ry_d + (q.v > fy_d ? 1 : 0), cam.h - 1);
    const float Fdu = dtn_at(S, cam, rx_u, ry_d);
    const float Fud = dtn_at(S, cam, rx_d, ry_u), Fuu = dtn_at(S, cam, rx_u, ry_u);
    const float ax = __fsub_rn(1.0f, inc_x), ay = __fsub_rn(1.0f, inc_y);
    const float f1 = __fsqrt_rn(__fadd_rn(__fmul_rn(__fmul_rn(ax, Fdd), Fdd), __fmul_rn(__fmul_rn(inc_x, Fdu), Fdu)));
    const float f2 = __fsqrt_rn(__fadd_rn(__fmul_rn(__fmul_rn(ax, Fud), Fud), __fmul_rn(__fmul_rn(inc_x, Fuu), Fuu)));
    return __fsqrt_rn(__fadd_rn(__fmul_rn(__fmul_rn(ay, f1), f1), __fmul_rn(__fmul_rn(inc_y, f2), f2)));
}

// Accumulator layout: [0..5] g, [6] sum eps^2, [7] sum eps, then (NEED_H) 21 upper-triangle entries of H row by row.
template <bool NEED_H> struct AccN { static constexpr int N = NEED_H ? 29 : 8; };
// The covariance sweep (WSQ) appends [29] sum w eps^2 to the Gauss-Newton layout.
constexpr int COV_NACC = AccN<true>::N + 1;

// One visible point's terms (:714-720, :777): g += J w eps, sum eps^2, sum eps, (NEED_H) H += J w J^T, (WSQ) sum w eps^2.
template <int ARITH, bool NEED_H, bool WSQ>
__device__ __forceinline__ void accumulate_point(const float* Jr, float e, float wgt, double* acc, int& nvis) {
    typedef Ar<ARITH> A;
    ++nvis;
    const double de = (double)e;
    acc[6] = fma(de, de, acc[6]);
    acc[7] += de;
    if constexpr (WSQ) acc[COV_NACC - 1] = fma((double)wgt * de, de, acc[COV_NACC - 1]);   // double(w) * double(eps) is exact
    double Jw[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) { Jw[k] = (double)A::mul(Jr[k], wgt); acc[k] = fma(Jw[k], de, acc[k]); }
    if (NEED_H) {
        int idx = 8;
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
            for (int c = r; c < 6; ++c) { acc[idx] = fma(Jw[r], (double)Jr[c], acc[idx]); ++idx; }
    }
}

// Software-pipelined sweep over a thread's points: the coordinates are loaded two points ahead and the (random)
// texel gather of the next point is in flight while the current point's Jacobian / fp64 accumulation executes.
// (A counted loop with unconditional look-ahead loads into slack behind the arrays, unrolled by 1 / 2 / 3, was measured slower:
// 4.51 / 4.32 / 4.84 ms per 1024 pairs against 4.01 for this guarded form -- DESIGN.md "measured and rejected".)
template <int ARITH, int JAC, bool NEED_H, int THREADS, bool OUT, int RES, int WMODE, bool WSQ = false>
__device__ __forceinline__ void accumulate_points(const float* __restrict__ X, const float* __restrict__ Y,
                                                  const float* __restrict__ Z, int N, const PoseF& P, const LevelCam& cam,
                                                  const TexSrc& S, int weight_mode_rt, float huber_k,
                                                  double* acc, int& nvis, float* o_eps, float* o_w, float* o_u, float* o_v,
                                                  float* o_J) {
    constexpr int stride = THREADS;
    typedef Ar<ARITH> A;
    const int weight_mode = (WMODE >= 0) ? WMODE : weight_mode_rt;
    int i = threadIdx.x;
    if (i >= N) return;
    float cx = __ldg(X + i), cy = __ldg(Y + i), cz = __ldg(Z + i);
    Proj q = project_point(cx, cy, cz, P, cam);
    uint2 t = make_uint2(0u, 0u);
    if (q.idx >= 0) t = load_texel(S, q.idx);
    int i1 = i + stride;
    if (i1 < N) { cx = __ldg(X + i1); cy = __ldg(Y + i1); cz = __ldg(Z + i1); }
    for (;;) {
        const int i2 = i1 + stride;
        float nx = 0.f, ny = 0.f, nz = 1.f;
        if (i2 < N) { nx = __ldg(X + i2); ny = __ldg(Y + i2); nz = __ldg(Z + i2); }       // coordinates two ahead
        Proj qn; qn.idx = -1;
        uint2 tn = make_uint2(0u, 0u);
        if (i1 < N) { qn = project_point(cx, cy, cz, P, cam); if (qn.idx >= 0) tn = load_texel(S, qn.idx); }   // gather one ahead
        // ---- consume point i
        float Jr[6], e = 0.f, wgt = 0.f;
        if (q.idx >= 0) {
            const float4 tv = resolve_texel(S, cam, q, t);
            finish_point<ARITH, JAC, WMODE>(q, tv, P, cam, weight_mode_rt, huber_k, Jr, e, wgt);
            if (RES == DVO_RESIDUAL_DT_INTERP) {                                     // :443-444, weight from the interpolated value (:450)
                e = interpolate_dt(S, cam, q, tv.x);
                if (weight_mode == DVO_WEIGHT_REF_CAUCHY) wgt = A::weight_ref(e);
                else if (weight_mode == DVO_WEIGHT_HUBER) { const float ae = fabsf(e); wgt = ae <= huber_k ? 1.0f : A::div(huber_k, ae); }
            }
            accumulate_point<ARITH, NEED_H, WSQ>(Jr, e, wgt, acc, nvis);
        } else {
#pragma unroll
            for (int k = 0; k < 6; ++k) Jr[k] = 0.f;
        }
        if (OUT) {
            if (o_u) { o_u[i] = q.u; o_v[i] = q.v; }
            if (o_eps) { o_eps[i] = e; o_w[i] = wgt; }
            if (o_J) {
#pragma unroll
                for (int k = 0; k < 6; ++k) o_J[6 * i + k] = Jr[k]; }
        }
        if (i1 >= N) break;
        i = i1; i1 = i2; q = qn; t = tn; cx = nx; cy = ny; cz = nz;
    }
}

// ---- sweep with a shared-memory ring (PIPE = ring depth D): the shipped configuration only (EXACT arithmetic, reference Jacobian,
// floor residual, packed texels, getWeightOf weights).  A point is projected D-1 steps before it is consumed; its normalised
// coordinates, reprojection and texel index go to the thread's own ring slot and the 8-byte texel follows with cp.async (no
// destination register, no scoreboard wait), so up to D-1 gathers per thread are in flight instead of one.  With 16-byte row-major
// texels the sweep was bound by DRAM transactions and a deeper ring did not pay (round 1); with packed Morton texels DRAM runs at
// 20 % and the first use of a gathered texel is the top stall.
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int JAC, bool NEED_H, int THREADS, int D>
__device__ __forceinline__ void accumulate_points_ring(const float* __restrict__ X, const float* __restrict__ Y, const float* __restrict__ Z, int N,
                                                       const PoseF& P, const LevelCam& cam, const TexSrc& S, double* acc, int& nvis,
                                                       unsigned char* ring) {
    static_assert((D & (D - 1)) == 0 && D >= 2, "ring depth must be a power of two");
    float4* ringP = reinterpret_cast<float4*>(ring);                               // [D][THREADS] {X, Y, Z, texel index}
    float2* ringUV = reinterpret_cast<float2*>(ring + D * THREADS * 16);            // [D][THREADS] reprojection (escape path only)
    uint2* ringT = reinterpret_cast<uint2*>(ring + D * THREADS * 24);               // [D][THREADS] texel, filled by cp.async
    const int tid = threadIdx.x;
    if (tid >= N) return;
    const int n_iter = (N - tid + THREADS - 1) / THREADS;
    const float* __restrict__ px = X + tid; const float* __restrict__ py = Y + tid; const float* __restrict__ pz = Z + tid;
    float cx = __ldg(px), cy = __ldg(py), cz = __ldg(pz);
    auto issue = [&](int k) {                      // project point k (coordinates in cx, cy, cz), start its gather, fetch the next coordinates
        const int slot = (k & (D - 1)) * THREADS + tid;
        const Proj q = project_point(cx, cy, cz, P, cam);
        ringP[slot] = make_float4(q.X, q.Y, q.Z, __int_as_float(q.idx));
        ringUV[slot] = make_float2(q.u, q.v);
        if (q.idx >= 0) cp_async8(&ringT[slot], S.tex8 + q.idx);
        if (k + 1 < n_iter) { px += THREADS; py += THREADS; pz += THREADS; cx = __ldg(px); cy = __ldg(py); cz = __ldg(pz); }
    };
#pragma unroll
    for (int k = 0; k < D - 1; ++k) { if (k < n_iter) issue(k); cp_async_commit(); }
    for (int k = 0; k < n_iter; ++k) {
        if (k + D - 1 < n_iter) issue(k + D - 1);
        cp_async_commit();
        cp_async_wait<D - 1>();                    // the group of point k has landed
        const int slot = (k & (D - 1)) * THREADS + tid;
        const float4 pr = ringP[slot];
        Proj q; q.X = pr.x; q.Y = pr.y; q.Z = pr.z; q.idx = __float_as_int(pr.w);
        if (q.idx >= 0) {
            const float2 uv = ringUV[slot]; q.u = uv.x; q.v = uv.y;
            const float4 tv = resolve_texel(S, cam, q, ringT[slot]);
            float Jr[6], e, wgt;
            finish_point<DVO_ARITH_EXACT, JAC, DVO_WEIGHT_REF_CAUCHY>(q, tv, P, cam, DVO_WEIGHT_REF_CAUCHY, 0.f, Jr, e, wgt);
            accumulate_point<DVO_ARITH_EXACT, NEED_H, false>(Jr, e, wgt, acc, nvis);
        }
    }
    cp_async_wait<0>();
}

// Deterministic block reduction of NACC fp64 accumulators per thread.
// Stage 1 (per warp).  TRANSPOSED (the 29-accumulator Gauss-Newton case): eight accumulators at a time are parked
// in a [8][36] shared tile (row = accumulator, column = lane); lane (r, q) = (lane / 4, lane % 4) sums columns
// q, q+4, .. of row r and two xor-shuffles combine the four quarters -- 1 store + 1 load per value instead of the
// 5-level shuffle tree (15 instructions per value), which was a third of the fixed per-iteration cost.  The row
// stride of 36 doubles makes both the stores and the strided loads bank-conflict free.  The small tile (2.3 KB per
// warp) is deliberate: a full [29][33] tile cost 61 KB per CTA of L1 capacity and slowed the gather-bound sweep.
// The 8-accumulator sub-gradient case keeps the shuffle tree (its tile pass would not be shorter).
// Stage 2: thread k sums the warp partials in warp order.
// The covariance's serial tail reuses scr as its 6x6 workspace.
template <int NACC, int THREADS> struct ReduceScratch {
    static constexpr bool TRANSPOSED = (NACC > 8);
    static constexpr int WARPS = THREADS / 32, ROW = 36, PER_WARP = TRANSPOSED ? 8 * ROW : 1;
    double scr[TRANSPOSED ? WARPS * PER_WARP : 0];   // per-warp transposed tile (none for the shuffle tree)
    double red[WARPS][NACC];        // warp partials
    double tot[NACC];               // block sums
    int nv[WARPS], nvtot;           // visible points per warp, per block
    int stop;                       // solve: the lead's stop decision, read by every thread after the iteration's barrier
                                    // (it fills the slot after nvtot: a flag of its own would move SolverState by 8 bytes and change
                                    // how ptxas vectorises its stores)
};

template <int NACC, int THREADS>
__device__ __forceinline__ void block_reduce(double* acc, int nvis, ReduceScratch<NACC, THREADS>& R) {
    typedef ReduceScratch<NACC, THREADS> RS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (RS::TRANSPOSED) {
        double* ws = R.scr + warp * RS::PER_WARP;
        const int r = lane >> 2, q = lane & 3;
#pragma unroll
        for (int p0 = 0; p0 < NACC; p0 += 8) {
#pragma unroll
            for (int k = 0; k < 8; ++k) if (p0 + k < NACC) ws[k * RS::ROW + lane] = acc[p0 + k];
            __syncwarp();
            double v = 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) v += ws[r * RS::ROW + 4 * j + q];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (q == 0 && p0 + r < NACC) R.red[warp][p0 + r] = v;
            __syncwarp();
        }
    } else {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
            double v = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) R.red[warp][k] = v;
        }
    }
    for (int o = 16; o > 0; o >>= 1) nvis += __shfl_down_sync(0xffffffffu, nvis, o);
    if (lane == 0) R.nv[warp] = nvis;
    __syncthreads();
    if (threadIdx.x < NACC) {
        double v = 0.0;
#pragma unroll
        for (int wv = 0; wv < RS::WARPS; ++wv) v += R.red[wv][threadIdx.x];
        R.tot[threadIdx.x] = v;
    }
    if (threadIdx.x == 32) { int n = 0; for (int wv = 0; wv < RS::WARPS; ++wv) n += R.nv[wv]; R.nvtot = n; }
    __syncthreads();
}

// ------------------------------------------------------------------ solver state (thread 0, in shared memory)
struct SolverState {
    double cR[9], cT[3], bestR[9], bestT[3], descent[6];
    double accR[9], accT[3], accH[36], accg[6];
    double lambda, bestSumEps;
    float accE, bestE, bestRatio;
    int have_acc, bestItr;
};

struct SolveArgs {
    FrameArgs f;
    const double* pose0; double* pose; dvo_pair_info* info; double* trace; int trace_iters; const int* order; const unsigned char* active;
    float* energy;
    dvo_solver_params prm; int first;
    // pair launches (solve_pairs_kernel) only: reference / now slot of each pair.  Appended so that the parameter offsets of the
    // slot kernels stay where they were.
    const int* ref_slot; const int* now_slot;
};

// One iteration's serial tail (thread 0): best tracking, step computation, pose update.  Returns 1 to stop the level.
// ENERGY: record energyAtEachIteration in energy_rec (slot launches; pair launches keep no per-iteration state).
template <bool ENERGY>
__device__ __forceinline__ int solver_step(SolverState& S, const double* tot, int nvis, int N, int itr, const dvo_solver_params& prm,
                                        bool need_h, dvo_pair_info* info, int level, double* trace_rec, float* energy_rec) {
    const float ratio = (float)nvis / (float)N;                                   // :457
    const float energy = (float)sqrt(tot[6]);                                      // :1310-1312
    info->iterations_run[level] = itr + 1;
    if constexpr (ENERGY) { if (itr < DVO_ENERGY_ITERS) energy_rec[itr] = energy; }   // energyAtEachIteration (:634, :690)
    double Hf[36];
    if (need_h) {
        int idx = 8;
        for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { Hf[6 * r + c] = tot[idx]; Hf[6 * c + r] = tot[idx]; ++idx; }
    } else { for (int k = 0; k < 36; ++k) Hf[k] = 0.0; }
    if (trace_rec) {
        for (int k = 0; k < 6; ++k) trace_rec[k] = tot[k];
        for (int k = 0; k < 36; ++k) trace_rec[6 + k] = Hf[k];
        trace_rec[42] = energy; trace_rec[43] = nvis;
        for (int k = 0; k < 9; ++k) trace_rec[44 + k] = S.cR[k];
        for (int k = 0; k < 3; ++k) trace_rec[53 + k] = S.cT[k];
    }
    if (energy <= S.bestE) {                                                      // :696-705
        S.bestE = energy; S.bestRatio = ratio; S.bestItr = itr; S.bestSumEps = tot[7];
        for (int k = 0; k < 9; ++k) S.bestR[k] = S.cR[k];
        for (int k = 0; k < 3; ++k) S.bestT[k] = S.cT[k];
    }
    double psi[6];
    if (prm.solver == DVO_SOLVER_SUBGRAD_REF) {
        double g[6]; for (int k = 0; k < 6; ++k) g[k] = tot[k];
        double cPsi[6]; se3_log_dev(S.cR, S.cT, cPsi);                            // :736-739
        double cn = 0; for (int k = 0; k < 6; ++k) cn += cPsi[k] * cPsi[k]; cn = sqrt(cn);
        if (cn > 0) { const double icn = 1.0 / cn; for (int k = 0; k < 6; ++k) cPsi[k] *= icn; }   // :740-741 (one reciprocal instead of six divisions)
        const double stepLength = 9.0 * 1.0E-2 / ((itr > 5) ? (double)(itr - 4) : 1.0);   // :773
        for (int k = 0; k < 6; ++k) g[k] += 0.05 * cPsi[k];                       // :796
        for (int k = 0; k < 6; ++k) S.descent[k] = 0.5 * g[k] + 0.5 * S.descent[k];      // :799
        const double Pv[6] = {1.0, 1.0, 1.0, 0.5, 0.5, 0.5};                      // :729
        double nrm = 0;
        for (int k = 0; k < 6; ++k) { psi[k] = -stepLength * Pv[k] * S.descent[k]; nrm += psi[k] * psi[k]; }   // :821
        nrm = sqrt(nrm);
        const double radius = (double)0.003f;                                     // :25, :835
        if (nrm > radius) { const double sc = radius / nrm; for (int k = 0; k < 6; ++k) psi[k] *= sc; }
        else if (nrm < (double)1.0E-7f) return 1;                                 // :840 -> :872
    } else {
        const bool accept = (prm.solver == DVO_SOLVER_GN) || !S.have_acc || (energy <= S.accE);
        if (accept) {
            for (int k = 0; k < 9; ++k) S.accR[k] = S.cR[k];
            for (int k = 0; k < 3; ++k) S.accT[k] = S.cT[k];
            for (int k = 0; k < 36; ++k) S.accH[k] = Hf[k];
            for (int k = 0; k < 6; ++k) S.accg[k] = tot[k];
            S.accE = energy;
            if (prm.solver == DVO_SOLVER_LM && S.have_acc) S.lambda = (S.lambda * 0.1 < 1e-9) ? 1e-9 : S.lambda * 0.1;
            S.have_acc = 1;
        } else {
            S.lambda *= 10.0;
            if (S.lambda > 1e8) return 1;
            for (int k = 0; k < 9; ++k) S.cR[k] = S.accR[k];
            for (int k = 0; k < 3; ++k) S.cT[k] = S.accT[k];
        }
        double Am[36], nb[6];
        for (int k = 0; k < 36; ++k) Am[k] = S.accH[k];
        const double lam = (prm.solver == DVO_SOLVER_LM) ? S.lambda : 0.0;
        for (int k = 0; k < 6; ++k) { Am[7 * k] += lam * S.accH[7 * k] + 1e-9; nb[k] = -S.accg[k]; }
        if (!chol6_dev(Am, nb, psi)) return 1;
        double n2 = 0; for (int k = 0; k < 6; ++k) n2 += psi[k] * psi[k];
        if (sqrt(n2) < (double)1.0E-7f) return 1;
    }
    double xR[9], xt[3], Rt[3];
    se3_exp_dev(psi, xR, xt);                                                     // :905-907
    m3_vec(S.cR, xt, Rt);
    S.cT[0] += Rt[0]; S.cT[1] += Rt[1]; S.cT[2] += Rt[2];                         // :916
    m3_mul(S.cR, xR, S.cR);                                                       // :917
    rotationize_dev(S.cR);                                                        // :919
    return 0;
}

// Launch order: heaviest pairs first (longest-processing-time-first).  A pair occupies its CTA for the whole schedule
// (~1 ms), so with B / (CTAs resident) only a few "waves" the makespan is set by what the last-started CTAs still
// have to do; starting the big pairs first leaves the short ones for the tail.  Work = sum_l iters[l] * npts[l],
// bucketed into 256 classes by a single CTA (counting sort; the order inside a class is irrelevant to the results).
// work(i) is the work of launch entry i, id(i) what the order list holds for it.
template <typename Work, typename Id>
__device__ __forceinline__ void order_heaviest_first(int count, Work work, Id id, int* __restrict__ order) {
    __shared__ unsigned s_max, s_cnt[256], s_base[256];
    const int tid = threadIdx.x;
    if (tid == 0) s_max = 1u;
    if (tid < 256) s_cnt[tid] = 0u;
    __syncthreads();
    unsigned m = 0;
    for (int i = tid; i < count; i += blockDim.x) m = max(m, work(i));
    atomicMax(&s_max, m);
    __syncthreads();
    const float scale = 255.0f / (float)s_max;
    for (int i = tid; i < count; i += blockDim.x) atomicAdd(&s_cnt[255 - min(255, (int)((float)work(i) * scale))], 1u);
    __syncthreads();
    if (tid == 0) { unsigned run = 0; for (int k = 0; k < 256; ++k) { s_base[k] = run; run += s_cnt[k]; } }
    __syncthreads();
    for (int i = tid; i < count; i += blockDim.x) {
        const int cls = 255 - min(255, (int)((float)work(i) * scale));
        order[atomicAdd(&s_base[cls], 1u)] = id(i);
    }
}

// work of a launch entry whose reference data is slot s: sum_l iters[l] * npts[s][l]
__device__ __forceinline__ unsigned slot_work(const int* __restrict__ npts, int L, const dvo_solver_params& prm, int s) {
    unsigned wk = 0;
    for (int l = 0; l < L; ++l) wk += (unsigned)max(prm.iters[l], 0) * (unsigned)npts[(long long)s * L + l];
    return wk;
}

__global__ void __launch_bounds__(1024) solve_order_kernel(const int* __restrict__ npts, int L, dvo_solver_params prm, int first, int count,
                                                           int* __restrict__ order) {
    order_heaviest_first(count, [&](int i) { return slot_work(npts, L, prm, first + i); }, [&](int i) { return first + i; }, order);
}

// Pairs: the work of pair k is that of its reference slot (out-of-range slots weigh nothing); the list holds pair indices.
__global__ void __launch_bounds__(1024) pair_order_kernel(const int* __restrict__ npts, int L, dvo_solver_params prm, int Bmax, int count,
                                                          const int* __restrict__ ref_slot, int* __restrict__ order) {
    auto work = [&](int k) {
        const int s = ref_slot[k];
        return (s < 0 || s >= Bmax) ? 0u : slot_work(npts, L, prm, s);
    };
    order_heaviest_first(count, work, [](int k) { return k; }, order);
}

// One CTA owns a frame pair for the whole coarse-to-fine schedule.  (A thread-block-cluster variant that striped a
// pair's points over 2/4/8 CTAs and combined partial sums through distributed shared memory was measured slower --
// 4.29 ms -> 4.58 / 5.53 / 8.62 ms per 1024 pairs -- and removed; so was a cp.async shared-memory ring that kept 2..8
// texel gathers in flight per thread: 4.56 .. 4.72 ms.  See DESIGN.md "measured and rejected".)
//
// PAIRS (solve_pairs_kernel, dvo_align_pairs): the order list holds pair indices b; the reference data (edge points, npts) come
// from slot a.ref_slot[b], the now data (texels, d2, max d2, edge counts) from slot a.now_slot[b]; pose0 / pose / info are indexed
// by pair, and no trace or energies are written.  Otherwise b is a slot and both slots are b.  The flag is a template parameter
// so that the slot kernels compile exactly as they would without it.
template <int ARITH, int JAC, bool NEED_H, int THREADS, int RES, int WMODE, int PIPE, bool PAIRS>
__device__ __forceinline__ void solve_body(const SolveArgs& a) {
    extern __shared__ float s_lut[];          // 2 * LUT_N floats, then the sweep's ring (PIPE > 0)
    constexpr int NACC = AccN<NEED_H>::N;
    __shared__ ReduceScratch<NACC, THREADS> R;
    __shared__ PoseF s_pose;
    __shared__ SolverState S;
    __shared__ dvo_pair_info s_info;

    const int b = a.order[blockIdx.x];
    if (!PAIRS && a.active && !a.active[b]) return;       // masked pass (gated key-frame switch): pose / info of the slot stay as they are
    const int L = a.f.geom.L;
    const bool lead = (threadIdx.x == 0);
    int rb = b, nb = b;                                   // slot of the reference data, slot of the now data
    if constexpr (PAIRS) {
        rb = a.ref_slot[b]; nb = a.now_slot[b];
        if (rb < 0 || rb >= a.f.geom.Bmax || nb < 0 || nb >= a.f.geom.Bmax) {                     // status bit 1, NaN pose
            if (lead) {
                const double qnan = __longlong_as_double(0x7ff8000000000000ll);
                for (int k = 0; k < 12; ++k) a.pose[12 * (long long)b + k] = qnan;
                dvo_pair_info inf;
                inf.status = 2; inf.laplacian_b = 0.f;
                for (int l = 0; l < DVO_MAX_LEVELS; ++l) {
                    inf.npts[l] = 0; inf.best_index[l] = -1; inf.iterations_run[l] = 0; inf.best_energy[l] = 0.f; inf.visible_ratio[l] = 0.f;
                }
                a.info[b] = inf;
            }
            return;
        }
    }
    if (lead) {
        for (int k = 0; k < 9; ++k) S.cR[k] = a.pose0[12 * (long long)b + k];
        for (int k = 0; k < 3; ++k) S.cT[k] = a.pose0[12 * (long long)b + 9 + k];
        s_info.status = 0; s_info.laplacian_b = 0.f;
        for (int l = 0; l < DVO_MAX_LEVELS; ++l) {
            s_info.npts[l] = (l < L) ? a.f.npts[(long long)rb * L + l] : 0; s_info.best_index[l] = -1; s_info.iterations_run[l] = 0;
            s_info.best_energy[l] = 0.f; s_info.visible_ratio[l] = 0.f;
        }
    }
    __syncthreads();

    for (int l = L - 1; l >= 0; --l) {
        const int iters = a.prm.iters[l];
        if (iters <= 0) continue;
        const int N = a.f.npts[(long long)rb * L + l];
        const unsigned ne = a.f.nedge_now[(long long)nb * L + l];
        if (N <= 0 || ne == 0u) { if (lead) s_info.status |= 1; continue; }                  // reference asserts (:282)
        // level_source spelled out: with d2 taken at lvl_at(l, nb) for slot launches too, ptxas allocates the slot kernels'
        // registers differently and their spills change
        const long long base = lvl_at(a.f.geom, l, rb);
        LevelSrc lv; lv.X = a.f.X + base; lv.Y = a.f.Y + base; lv.Z = a.f.Z + base;
        lv.cam = make_level_cam(a.f.K, a.f.geom, l);
        lv.tex.tex8 = a.f.tex8 + tex_at(a.f.geom, l, nb); lv.tex.lut = s_lut;
        if constexpr (PAIRS) lv.tex.d2 = a.f.d2 + lvl_at(a.f.geom, l, nb);
        else lv.tex.d2 = a.f.d2 + base;
        const unsigned mx2 = a.f.maxd2[(long long)nb * L + l];
        lv.tex.scale = dtn_scale(mx2, ne);
        build_lut<THREADS>(s_lut, mx2, lv.tex.scale);
        if (lead) {
            S.bestE = 1.0E10f; S.bestRatio = 1.0f; S.bestItr = -1; S.bestSumEps = 0.0;        // :642-650
            for (int k = 0; k < 9; ++k) S.bestR[k] = (k % 4 == 0) ? 1.0 : 0.0;
            for (int k = 0; k < 3; ++k) S.bestT[k] = 0.0;
            for (int k = 0; k < 6; ++k) S.descent[k] = 0.0;                                   // :654
            S.have_acc = 0; S.lambda = a.prm.lm_lambda0; S.accE = 0.f;
            for (int k = 0; k < 9; ++k) s_pose.R[k] = (float)S.cR[k];                          // :673-674
            for (int k = 0; k < 3; ++k) s_pose.T[k] = (float)S.cT[k];
            R.stop = 0;
        }
        __syncthreads();
        for (int itr = 0; itr < iters; ++itr) {
            PoseF P = s_pose;
            double acc[NACC];
#pragma unroll
            for (int k = 0; k < NACC; ++k) acc[k] = 0.0;
            int nvis = 0;
            if constexpr (PIPE > 0 && JAC == DVO_JAC_REFERENCE)
                accumulate_points_ring<JAC, NEED_H, THREADS, PIPE>(lv.X, lv.Y, lv.Z, N, P, lv.cam, lv.tex, acc, nvis,
                                                                   reinterpret_cast<unsigned char*>(s_lut) + LUT_BYTES);
            else
                accumulate_points<ARITH, JAC, NEED_H, THREADS, false, RES, WMODE>(lv.X, lv.Y, lv.Z, N, P, lv.cam, lv.tex, a.prm.weight, a.prm.huber_k,
                                                                                  acc, nvis, nullptr, nullptr, nullptr, nullptr, nullptr);
            block_reduce<NACC, THREADS>(acc, nvis, R);
            if (lead) {
                double* tr = nullptr;
                if (!PAIRS && a.trace && itr < a.trace_iters)
                    tr = a.trace + (((long long)b * L + l) * a.trace_iters + itr) * DVO_TRACE_DOUBLES;
                R.stop = solver_step<!PAIRS>(S, R.tot, R.nvtot, N, itr, a.prm, NEED_H, &s_info, l, tr, a.energy + ((long long)b * L + l) * DVO_ENERGY_ITERS);
                for (int k = 0; k < 9; ++k) s_pose.R[k] = (float)S.cR[k];                      // pose of the next iteration (:673-674)
                for (int k = 0; k < 3; ++k) s_pose.T[k] = (float)S.cT[k];
            }
            __syncthreads();
            if (R.stop) break;
        }
        if (lead) {
            for (int k = 0; k < 9; ++k) S.cR[k] = S.bestR[k];                                  // :997-1001
            rotationize_dev(S.cR);
            for (int k = 0; k < 3; ++k) S.cT[k] = S.bestT[k];
            s_info.best_index[l] = S.bestItr; s_info.best_energy[l] = S.bestE; s_info.visible_ratio[l] = S.bestRatio;
            s_info.laplacian_b = (float)(S.bestSumEps / (double)N);                            // :1466-1472 at the finest level run
        }
        __syncthreads();
    }
    if (lead) {
        for (int k = 0; k < 9; ++k) a.pose[12 * (long long)b + k] = S.cR[k];
        for (int k = 0; k < 3; ++k) a.pose[12 * (long long)b + 9 + k] = S.cT[k];
        a.info[b] = s_info;
    }
}

template <int ARITH, int JAC, bool NEED_H, int THREADS, int RES, int WMODE, int PIPE>
__global__ void __launch_bounds__(THREADS, (NEED_H ? 512 : 768) / THREADS) solve_kernel(SolveArgs a) {
    solve_body<ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE, false>(a);
}
template <int ARITH, int JAC, bool NEED_H, int THREADS, int RES, int WMODE, int PIPE>
__global__ void __launch_bounds__(THREADS, (NEED_H ? 512 : 768) / THREADS) solve_pairs_kernel(SolveArgs a) {
    solve_body<ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE, true>(a);
}

// ------------------------------------------------------------------ single evaluation (parity inspection)
// The normal equations at pose P of the N reference points of slot rb against the now frame of slot nb at level l, with the
// run-time weight mode: one sweep with H (plus sum w eps^2 when WSQ), then the block reduction.  The sums are in R.tot and
// R.nvtot on every thread after the return.
template <int ARITH, int JAC, int THREADS, int RES, bool OUT, bool WSQ>
__device__ __forceinline__ void eval_normal_equations(const FrameArgs& f, int l, int rb, int nb, int N, const PoseF& P, int weight,
                                                      float huber_k, float* lut, ReduceScratch<WSQ ? COV_NACC : AccN<true>::N, THREADS>& R,
                                                      float* o_eps, float* o_w, float* o_u, float* o_v, float* o_J) {
    constexpr int NACC = WSQ ? COV_NACC : AccN<true>::N;
    const LevelSrc lv = level_source<THREADS>(f, l, rb, nb, lut);
    __syncthreads();
    double acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = 0.0;
    int nvis = 0;
    accumulate_points<ARITH, JAC, true, THREADS, OUT, RES, -1, WSQ>(lv.X, lv.Y, lv.Z, N, P, lv.cam, lv.tex, weight, huber_k, acc, nvis,
                                                                     o_eps, o_w, o_u, o_v, o_J);
    block_reduce<NACC, THREADS>(acc, nvis, R);
}

struct EvalArgs {
    FrameArgs f;
    const double* pose; int slot, level, weight; float huber_k;
    double* out;            // g[6], H[36], sumsq, nvis
    float *eps, *w, *u, *v, *J;
};

template <int ARITH, int JAC, int RES>
__global__ void __launch_bounds__(EVAL_THREADS) eval_kernel(EvalArgs a) {
    extern __shared__ float s_lut[];
    __shared__ ReduceScratch<AccN<true>::N, EVAL_THREADS> R;
    const int b = a.slot, l = a.level;
    PoseF P;
    for (int k = 0; k < 9; ++k) P.R[k] = (float)a.pose[k];
    for (int k = 0; k < 3; ++k) P.T[k] = (float)a.pose[9 + k];
    eval_normal_equations<ARITH, JAC, EVAL_THREADS, RES, true, false>(a.f, l, b, b, a.f.npts[(long long)b * a.f.geom.L + l], P, a.weight,
                                                                      a.huber_k, s_lut, R, a.eps, a.w, a.u, a.v, a.J);
    if (threadIdx.x == 0) {
        for (int k = 0; k < 6; ++k) a.out[k] = R.tot[k];
        int idx = 8;
        for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { a.out[6 + 6 * r + c] = R.tot[idx]; a.out[6 + 6 * c + r] = R.tot[idx]; ++idx; }
        a.out[42] = R.tot[6]; a.out[43] = (double)R.nvtot;
    }
}

// ------------------------------------------------------------------ pose covariance (dvo_pose_covariance)
// One CTA per slot evaluates the normal equations at the slot's returned pose c->pose with the EXACT Jacobian and EXACT
// arithmetic (the derivative of the residual wrt T <- T exp(psi), psi = (rho, omega)), the caller's weight / Huber k /
// residual, plus sum w eps^2; thread 0 then forms Sigma = sigma^2 H^-1 from a Cholesky factor of H.  The CTA shape is
// fixed (COV_THREADS), so a slot's result never depends on how many slots share the launch.  Reads c->pose only.
constexpr int COV_THREADS = 256;
struct CovArgs {
    FrameArgs f;
    const double* pose; int first, level, weight; float huber_k;
    double* cov;            // 36 doubles per slot, record of CTA k at cov + 36 * k * stride
    dvo_cov_info* info;     // optional, same indexing
    long long stride;
    const unsigned char* active;   // optional per-slot mask: a slot whose flag is 0 keeps its record as it is
    // pair launches (cov_pairs_kernel) only, appended as in SolveArgs: reference / now slot of each pair
    const int* ref_slot; const int* now_slot;
};

// Serial tail on thread 0: H (full symmetric, row-major, in shared memory M[0..35]) -> Sigma = s2 H^-1 into out, log det H.
// The factor overwrites M's lower triangle, L^-1 goes to M + 36.  Returns false when H is not positive definite.
__device__ __forceinline__ bool cov_from_normal_matrix(double* M, double s2, double* out, double* logdetH) {
    double* Li = M + 36;
    double ld = 0.0;
    for (int j = 0; j < 6; ++j) {
        double d = M[6 * j + j];
        for (int k = 0; k < j; ++k) d -= M[6 * j + k] * M[6 * j + k];
        if (!(d > 0.0)) return false;
        ld += log(d);
        const double r = sqrt(d);
        M[6 * j + j] = r;
        for (int i = j + 1; i < 6; ++i) {
            double v = M[6 * i + j];
            for (int k = 0; k < j; ++k) v -= M[6 * i + k] * M[6 * j + k];
            M[6 * i + j] = v / r;
        }
    }
    for (int j = 0; j < 6; ++j) {                         // L^-1 (lower triangular), column by column
        for (int i = 0; i < j; ++i) Li[6 * i + j] = 0.0;
        Li[6 * j + j] = 1.0 / M[6 * j + j];
        for (int i = j + 1; i < 6; ++i) {
            double v = 0.0;
            for (int k = j; k < i; ++k) v += M[6 * i + k] * Li[6 * k + j];
            Li[6 * i + j] = -v / M[6 * i + i];
        }
    }
    for (int i = 0; i < 6; ++i)                           // H^-1 = L^-T L^-1
        for (int j = i; j < 6; ++j) {
            double v = 0.0;
            for (int k = j; k < 6; ++k) v += Li[6 * k + i] * Li[6 * k + j];
            out[6 * i + j] = s2 * v; out[6 * j + i] = s2 * v;
        }
    *logdetH = ld;
    return true;
}

// PAIRS: CTA k evaluates pair k (a.first = 0) at its pose a.pose[k] on reference slot a.ref_slot[k] and now slot
// a.now_slot[k]; a pair with a slot outside [0, Bmax) gets status bit 0.  As solve_body, a template flag.
template <int RES, bool PAIRS>
__device__ __forceinline__ void cov_body(const CovArgs& a) {
    extern __shared__ float s_lut[];
    __shared__ ReduceScratch<COV_NACC, COV_THREADS> R;
    const int b = a.first + blockIdx.x, l = a.level, L = a.f.geom.L;
    if (!PAIRS && a.active && !a.active[b]) return;       // masked pass (key-frame switch): the slot's record stays as it is
    int rb = b, nb = b;                                   // slot of the reference data, slot of the now data
    bool in_range = true;
    if constexpr (PAIRS) {
        rb = a.ref_slot[b]; nb = a.now_slot[b];
        in_range = rb >= 0 && rb < a.f.geom.Bmax && nb >= 0 && nb < a.f.geom.Bmax;
    }
    const int N = in_range ? a.f.npts[(long long)rb * L + l] : 0;
    const unsigned ne = in_range ? a.f.nedge_now[(long long)nb * L + l] : 0u;
    double* out = a.cov + 36 * (long long)blockIdx.x * a.stride;
    dvo_cov_info* inf = a.info ? a.info + (long long)blockIdx.x * a.stride : nullptr;
    int status = 0, nvis = 0;
    double sigma2 = 0.0, logdet = 0.0;
    if (N > 0 && ne != 0u) {                              // block-uniform
        PoseF P;
        for (int k = 0; k < 9; ++k) P.R[k] = (float)a.pose[12 * (long long)b + k];
        for (int k = 0; k < 3; ++k) P.T[k] = (float)a.pose[12 * (long long)b + 9 + k];
        eval_normal_equations<DVO_ARITH_EXACT, DVO_JAC_EXACT, COV_THREADS, RES, false, true>(a.f, l, rb, nb, N, P, a.weight, a.huber_k, s_lut, R,
                                                                                           nullptr, nullptr, nullptr, nullptr, nullptr);
        if (threadIdx.x != 0) return;
        nvis = R.nvtot;
        if (nvis < 7) status |= 2;
        else {
            double* M = R.scr;                            // the reduction scratch is free again
            int idx = 8;
            for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { M[6 * r + c] = R.tot[idx]; M[6 * c + r] = R.tot[idx]; ++idx; }
            sigma2 = R.tot[COV_NACC - 1] / (double)(nvis - 6);
            double ldH = 0.0;
            if (cov_from_normal_matrix(M, sigma2, out, &ldH)) logdet = 6.0 * log(sigma2) - ldH;
            else status |= 4;
        }
    } else {
        if (threadIdx.x != 0) return;
        status = 1;
    }
    if (status) {
        const double qnan = __longlong_as_double(0x7ff8000000000000ll);
        for (int k = 0; k < 36; ++k) out[k] = qnan;
        sigma2 = qnan; logdet = qnan;
    }
    if (inf) { inf->status = status; inf->level = l; inf->nvis = nvis; inf->sigma2 = sigma2; inf->logdet = logdet; }
}

template <int RES>
__global__ void __launch_bounds__(COV_THREADS) cov_kernel(CovArgs a) { cov_body<RES, false>(a); }
template <int RES>
__global__ void __launch_bounds__(COV_THREADS) cov_pairs_kernel(CovArgs a) { cov_body<RES, true>(a); }

// ------------------------------------------------------------------ packed texels -> float images (parity inspection)
// {DTn, gx, gy, w} of every pixel of one slot / level through exactly the code path the solver uses (packed texel or
// escaped d2 stencil, lookup table or direct evaluation), so that dvo_get_level_buffer checks that path pixel by pixel.
struct ResolveArgs { FrameArgs f; int slot, level; float4* out; };

__global__ void __launch_bounds__(256) resolve_texels_kernel(ResolveArgs a) {
    extern __shared__ float s_lut[];
    const LevelSrc lv = level_source<256>(a.f, a.level, a.slot, a.slot, s_lut);
    __syncthreads();
    const int w = lv.cam.w, h = lv.cam.h;
    const uint2* __restrict__ tex = lv.tex.tex8;
    const int32_t* __restrict__ d2 = lv.tex.d2;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < w * h; i += gridDim.x * 256) {
        const int y = i / w, x = i - y * w;
        Stencil s;
        if (!unpack_texel(__ldg(tex + tex_index(x, y, lv.cam.tw)), s)) stencil_from_d2(d2, w, h, x, y, s);
        a.out[i] = texel_values(s, s_lut, lv.tex.scale);
    }
}

// Sigma_g = Ad(Tr^-1) Sigma_key Ad(Tr^-1)^T + Sigma_rel for tangent psi = (rho, omega) and T <- T exp(psi):
// T_key exp(dk) Tr exp(dr) = T_key Tr exp(Ad(Tr^-1) dk) exp(dr), Ad(R, t) = [[R, [t]x R], [0, R]], Tr^-1 = (R^T, -R^T t).
// Sigma_key == nullptr stands for a zero key-frame covariance.
__device__ __forceinline__ void propagate_cov(const double* r, const double* __restrict__ Skey, const double* __restrict__ Srel, double* __restrict__ Sg) {
    double A[36];
    const double Rt[9] = {r[0], r[3], r[6], r[1], r[4], r[7], r[2], r[5], r[8]};
    double u[3]; m3_vec(Rt, r + 9, u);
    u[0] = -u[0]; u[1] = -u[1]; u[2] = -u[2];
    const double ux[9] = {0, -u[2], u[1], u[2], 0, -u[0], -u[1], u[0], 0};
    double UR[9]; m3_mul(ux, Rt, UR);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A[6 * i + j] = Rt[3 * i + j]; A[6 * i + 3 + j] = UR[3 * i + j];
            A[6 * (i + 3) + j] = 0.0; A[6 * (i + 3) + 3 + j] = Rt[3 * i + j];
        }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double row[6];                                    // row i of A Sigma_key
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            double v = 0.0;
            if (Skey) {
#pragma unroll
                for (int p = 0; p < 6; ++p) v += A[6 * i + p] * Skey[6 * p + q];
            }
            row[q] = v;
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            double v = 0.0;
#pragma unroll
            for (int q = 0; q < 6; ++q) v += row[q] * A[6 * j + q];
            Sg[6 * i + j] = v + Srel[6 * i + j];
        }
    }
}

// ------------------------------------------------------------------ GOP composition (src/GOP.cpp:138-196)
// With rel_cov / glob_cov (both or neither) the covariance of every global pose is propagated alongside; the pose arithmetic is
// the same instructions either way, so the composed poses do not depend on whether covariances are requested.
__global__ void gop_kernel(int nseq, int nframes, const int* __restrict__ kind, const double* __restrict__ rel, double* __restrict__ out,
                           const double* __restrict__ rel_cov, double* glob_cov) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseq) return;
    double kR[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kT[3] = {0, 0, 0};
    long long key = -1;                                                            // record holding Sigma_key (-1: zero)
    for (int f = 0; f < nframes; ++f) {
        const long long i = (long long)s * nframes + f;
        const double* r = rel + 12 * i;
        double gR[9], gT[3], RT[3];
        m3_vec(kR, r + 9, RT);
        gT[0] = kT[0] + RT[0]; gT[1] = kT[1] + RT[1]; gT[2] = kT[2] + RT[2];      // :144, :172
        m3_mul(kR, r, gR);                                                         // :145, :173
        double* o = out + 19 * i;
        for (int k = 0; k < 9; ++k) o[k] = gR[k];
        for (int k = 0; k < 3; ++k) { o[9 + k] = gT[k]; o[12 + k] = gT[k]; }
        rot_to_quat_dev(gR, o + 15);                                               // :103-114
        if (glob_cov) propagate_cov(r, key >= 0 ? glob_cov + 36 * key : nullptr, rel_cov + 36 * i, glob_cov + 36 * i);
        if (kind[i] != 0) {                                                        // :184-185, :192-193
            for (int k = 0; k < 9; ++k) kR[k] = gR[k]; for (int k = 0; k < 3; ++k) kT[k] = gT[k];
            key = i;
        }
    }
}

}  // namespace

// Kernels that use the lookup tables need 32 KB of dynamic shared memory on top of their static reduction scratch:
// opt in once per kernel and device.
template <typename KArgs, void (*KERN)(KArgs)>
static cudaError_t optin_lut_smem(int device, int bytes = LUT_BYTES) {
    static unsigned long long done = 0ull;
    const unsigned long long bit = 1ull << (device & 63);
    if (done & bit) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done |= bit;
    return e;
}

// PAIRS selects solve_pairs_kernel, the same configuration launched over pairs (dvo_align_pairs)
template <int ARITH, int JAC, bool NEED_H, int THREADS, int RES, int WMODE, bool PAIRS>
static cudaError_t launch_solve_w(dvo_ctx* c, const SolveArgs& a, int count) {
    // the shipped configuration (reference Jacobian, getWeightOf weights) takes the ring sweep, 4 deep for the 29-accumulator
    // kernel and 2 deep for the 8-accumulator (sub-gradient) one; every other configuration the register pipeline
    constexpr int PIPE = (WMODE == DVO_WEIGHT_REF_CAUCHY && JAC == DVO_JAC_REFERENCE) ? (NEED_H ? 4 : 2) : 0;
    constexpr int SMEM = LUT_BYTES + PIPE * THREADS * 32;
    constexpr auto kern = PAIRS ? solve_pairs_kernel<ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE> : solve_kernel<ARITH, JAC, NEED_H, THREADS, RES, WMODE, PIPE>;
    const cudaError_t e = optin_lut_smem<SolveArgs, kern>(c->cfg.device, SMEM);
    if (e != cudaSuccess) return e;
    kern<<<count, THREADS, SMEM, c->stream>>>(a);
    return cudaGetLastError();
}

// the shipped weight (getWeightOf, REF_CAUCHY) on the shipped residual gets its own instantiation with the weight mode fixed at
// compile time; every other combination takes the generic kernel that branches on the run-time value
template <int ARITH, int JAC, bool NEED_H, int THREADS, int RES, bool PAIRS>
static cudaError_t launch_solve_inst(dvo_ctx* c, const SolveArgs& a, int count) {
    if (ARITH == DVO_ARITH_EXACT && RES == DVO_RESIDUAL_DT_FLOOR && a.prm.weight == DVO_WEIGHT_REF_CAUCHY)
        return launch_solve_w<ARITH, JAC, NEED_H, THREADS, RES, (ARITH == DVO_ARITH_EXACT && RES == DVO_RESIDUAL_DT_FLOOR) ? DVO_WEIGHT_REF_CAUCHY : -1, PAIRS>(c, a, count);
    return launch_solve_w<ARITH, JAC, NEED_H, THREADS, RES, -1, PAIRS>(c, a, count);
}

template <int ARITH, int JAC, bool PAIRS>
static cudaError_t launch_solve_t(dvo_ctx* c, const SolveArgs& a, int count, bool need_h) {
    constexpr int THREADS = 256;
    constexpr int F = DVO_RESIDUAL_DT_FLOOR, I = DVO_RESIDUAL_DT_INTERP;
    if (a.prm.residual == I) {
        if (ARITH != DVO_ARITH_EXACT) return cudaErrorNotSupported;      // the interpolated variant is built for EXACT arithmetic only
        if (need_h) return launch_solve_inst<DVO_ARITH_EXACT, JAC, true, THREADS, I, PAIRS>(c, a, count);
        return launch_solve_inst<DVO_ARITH_EXACT, JAC, false, THREADS, I, PAIRS>(c, a, count);
    }
    // Up to one pair per SM there is nothing to overlap a CTA with, so a pair gets 512 threads: the sweeps run twice as
    // wide and a pair's latency drops by a third (148 pairs, GN: 0.91 -> 0.62 ms).  At full load the two shapes tie
    // (3.76 vs 3.80 ms per 1024 pairs), so larger launches keep two 256-thread CTAs per SM.
    // The shape is fixed per context (dvo_create: max_batch <= SM count -> 512), never per launch: the two shapes group the
    // fp64 partial sums differently, and a pair's pose must not depend on how many pairs happen to share a launch.
    const bool wide = (ARITH == DVO_ARITH_EXACT) && c->solve_shape == 512;
    if (wide && need_h) return launch_solve_inst<DVO_ARITH_EXACT, JAC, true, 512, F, PAIRS>(c, a, count);
    if (wide) return launch_solve_inst<DVO_ARITH_EXACT, JAC, false, 512, F, PAIRS>(c, a, count);
    if (need_h) return launch_solve_inst<ARITH, JAC, true, THREADS, F, PAIRS>(c, a, count);
    return launch_solve_inst<ARITH, JAC, false, THREADS, F, PAIRS>(c, a, count);
}

// The kernel choice of every solve launch, slots (dvo_run) and pairs (dvo_align_pairs) alike.
template <bool PAIRS>
static cudaError_t dispatch_solve(dvo_ctx* c, const SolveArgs& a, int count, const dvo_solver_params* p) {
    // H is needed by GN / LM, and by SUBGRAD_REF only when a trace is kept (parity tests on J^T W J).  Pair launches keep no trace
    // but follow the same rule: H selects the reduction, and with it how the partial sums of g are grouped.
    const bool need_h = (p->solver != DVO_SOLVER_SUBGRAD_REF) || (c->trace != nullptr);
    const bool ex = p->arithmetic != DVO_ARITH_FAST, rj = p->jacobian != DVO_JAC_EXACT;
    if (ex && rj) return launch_solve_t<DVO_ARITH_EXACT, DVO_JAC_REFERENCE, PAIRS>(c, a, count, need_h);
    if (ex) return launch_solve_t<DVO_ARITH_EXACT, DVO_JAC_EXACT, PAIRS>(c, a, count, need_h);
    if (rj) return launch_solve_t<DVO_ARITH_FAST, DVO_JAC_REFERENCE, PAIRS>(c, a, count, need_h);
    return launch_solve_t<DVO_ARITH_FAST, DVO_JAC_EXACT, PAIRS>(c, a, count, need_h);
}

static FrameArgs frame_args(const dvo_ctx* c) {
    FrameArgs f;
    f.geom = c->geom; f.K = c->K; f.X = c->ptsX; f.Y = c->ptsY; f.Z = c->ptsZ; f.npts = c->npts;
    f.nedge_now = c->nedge + (size_t)DVO_FRAME_NOW * c->geom.Bmax * c->geom.L;
    f.tex8 = c->tex8; f.d2 = c->d2; f.maxd2 = c->maxd2;
    return f;
}

static SolveArgs solve_args(dvo_ctx* c, const dvo_solver_params* p) {
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.f = frame_args(c);
    a.prm = *p;
    return a;
}

int launch_solve(dvo_ctx* c, int first, int count, const dvo_solver_params* p) {
    SolveArgs a = solve_args(c, p);
    a.pose0 = c->pose0; a.pose = c->pose; a.info = c->info; a.trace = c->trace; a.trace_iters = c->cfg.trace_iters; a.energy = c->energy;
    a.first = first;
    if (c->trace) DVO_CUDA(cudaMemsetAsync(c->trace + (size_t)first * c->geom.L * c->cfg.trace_iters * DVO_TRACE_DOUBLES, 0,
                                           sizeof(double) * (size_t)count * c->geom.L * c->cfg.trace_iters * DVO_TRACE_DOUBLES, c->stream));
    // the order list of slots [first, first + count) lives at solve_order + first, so launches on disjoint ranges never share it
    solve_order_kernel<<<1, 1024, 0, c->stream>>>(c->npts, c->geom.L, *p, first, count, c->solve_order + first);
    a.order = c->solve_order + first; a.active = c->active;
    DVO_CUDA(dispatch_solve<false>(c, a, count, p));
    c->launches++;
    c->launches++;
    return DVO_OK;
}

int launch_solve_pairs(dvo_ctx* c, int npairs, const dvo_solver_params* p) {
    SolveArgs a = solve_args(c, p);
    a.pose0 = c->pair_pose0; a.pose = c->pair_pose; a.info = c->pair_info;
    a.ref_slot = c->pair_ref; a.now_slot = c->pair_now;
    pair_order_kernel<<<1, 1024, 0, c->stream>>>(c->npts, c->geom.L, *p, c->geom.Bmax, npairs, c->pair_ref, c->pair_order);
    a.order = c->pair_order;
    DVO_CUDA(dispatch_solve<true>(c, a, npairs, p));
    c->launches += 2;
    return DVO_OK;
}

template <int ARITH, int JAC, int RES>
static cudaError_t launch_eval_inst(dvo_ctx* c, const EvalArgs& a) {
    const cudaError_t e = optin_lut_smem<EvalArgs, eval_kernel<ARITH, JAC, RES>>(c->cfg.device);
    if (e != cudaSuccess) return e;
    eval_kernel<ARITH, JAC, RES><<<1, EVAL_THREADS, LUT_BYTES, c->stream>>>(a);
    return cudaGetLastError();
}

int launch_eval(dvo_ctx* c, int slot, int level, const double* d_pose12, int jac, int weight, int arith, float huber_k, int residual,
                double* d_out, float* d_eps, float* d_w, float* d_u, float* d_v, float* d_J) {
    EvalArgs a;
    a.f = frame_args(c);
    a.pose = d_pose12; a.slot = slot; a.level = level; a.weight = weight; a.huber_k = huber_k; a.out = d_out;
    a.eps = d_eps; a.w = d_w; a.u = d_u; a.v = d_v; a.J = d_J;
    const bool ex = arith != DVO_ARITH_FAST, rj = jac != DVO_JAC_EXACT;
    constexpr int F = DVO_RESIDUAL_DT_FLOOR, I = DVO_RESIDUAL_DT_INTERP;
    cudaError_t e;
    if (residual == I) {
        if (!ex) { dvo_set_error("the interpolated-DT residual is built for EXACT arithmetic only"); return DVO_ERR_ARG; }
        e = rj ? launch_eval_inst<DVO_ARITH_EXACT, DVO_JAC_REFERENCE, I>(c, a) : launch_eval_inst<DVO_ARITH_EXACT, DVO_JAC_EXACT, I>(c, a);
    } else if (ex && rj) e = launch_eval_inst<DVO_ARITH_EXACT, DVO_JAC_REFERENCE, F>(c, a);
    else if (ex) e = launch_eval_inst<DVO_ARITH_EXACT, DVO_JAC_EXACT, F>(c, a);
    else if (rj) e = launch_eval_inst<DVO_ARITH_FAST, DVO_JAC_REFERENCE, F>(c, a);
    else e = launch_eval_inst<DVO_ARITH_FAST, DVO_JAC_EXACT, F>(c, a);
    c->launches++;
    DVO_CUDA(e);
    return DVO_OK;
}

int launch_resolve_texels(dvo_ctx* c, int slot, int level, float4* d_out) {
    ResolveArgs a;
    a.f = frame_args(c); a.slot = slot; a.level = level; a.out = d_out;
    DVO_CUDA((optin_lut_smem<ResolveArgs, resolve_texels_kernel>(c->cfg.device)));
    const int blocks = (c->geom.P[level] + 255) / 256;
    resolve_texels_kernel<<<blocks < 64 ? blocks : 64, 256, LUT_BYTES, c->stream>>>(a);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

template <int RES, bool PAIRS>
static cudaError_t launch_cov_inst(dvo_ctx* c, const CovArgs& a, int count) {
    constexpr auto kern = PAIRS ? cov_pairs_kernel<RES> : cov_kernel<RES>;
    const cudaError_t e = optin_lut_smem<CovArgs, kern>(c->cfg.device);
    if (e != cudaSuccess) return e;
    kern<<<count, COV_THREADS, LUT_BYTES, c->stream>>>(a);
    return cudaGetLastError();
}

template <bool PAIRS>
static int launch_cov_t(dvo_ctx* c, int first, int count, int level, const dvo_solver_params* p, double* d_cov, dvo_cov_info* d_info, long long stride) {
    if (count == 0) return DVO_OK;
    CovArgs a;
    memset(&a, 0, sizeof(a));
    a.f = frame_args(c);
    a.pose = c->pose; a.first = first; a.level = level; a.weight = p->weight; a.huber_k = p->huber_k;
    a.cov = d_cov; a.info = d_info; a.stride = stride;
    if (PAIRS) { a.pose = c->pair_pose; a.ref_slot = c->pair_ref; a.now_slot = c->pair_now; }
    else a.active = c->active;
    const cudaError_t e = p->residual == DVO_RESIDUAL_DT_INTERP ? launch_cov_inst<DVO_RESIDUAL_DT_INTERP, PAIRS>(c, a, count)
                                                                : launch_cov_inst<DVO_RESIDUAL_DT_FLOOR, PAIRS>(c, a, count);
    c->launches++;
    DVO_CUDA(e);
    return DVO_OK;
}

int launch_cov(dvo_ctx* c, int first, int count, int level, const dvo_solver_params* p, double* d_cov, dvo_cov_info* d_info, long long stride) {
    return launch_cov_t<false>(c, first, count, level, p, d_cov, d_info, stride);
}

int launch_cov_pairs(dvo_ctx* c, int npairs, int level, const dvo_solver_params* p, double* d_cov, dvo_cov_info* d_info) {
    return launch_cov_t<true>(c, 0, npairs, level, p, d_cov, d_info, 1);
}

int launch_gop(dvo_ctx* c, int nseq, int nframes, const int* d_kind, const double* d_rel, double* d_out, const double* d_rel_cov, double* d_glob_cov) {
    gop_kernel<<<(nseq + 127) / 128, 128, 0, c->stream>>>(nseq, nframes, d_kind, d_rel, d_out, d_rel_cov, d_glob_cov);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}
