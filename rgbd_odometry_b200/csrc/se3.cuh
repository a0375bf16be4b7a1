// se3.cuh -- fp64 3x3 / SE(3) closed forms of the solver (solver.cu) and the pose-graph optimiser (posegraph.cu).
// Both files build with the same flags, so one source gives both the same bits.  photometric.cu and rgbd.cu build with
// -fmad=false and keep their own operation orders: they must not use these.
#pragma once
#include <cuda_runtime.h>

namespace {

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

// SE(3) exponential, tangent = (upsilon, omega), translation first (Sophus::SE3d::exp, src/SolveDVO.cpp:905).
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

// rotation matrix -> unit quaternion (x,y,z,w), Shepperd's branches
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

// SE(3) logarithm (Sophus::SE3d::log of setRotationMatrix(cR), translation cT; src/SolveDVO.cpp:736-739)
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

}  // namespace
