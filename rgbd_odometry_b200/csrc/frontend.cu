// frontend.cu -- the publisher's undistortion front-end (src/camTopic2PublisherPyD.cpp:86-117: cv::undistort of the BGR
// frame and of the 16-bit depth frame before the pyramid is built).  cv::undistort = initUndistortRectifyMap (fp64
// forward distortion model; map quantised to 1/32 pixel) + remap(INTER_LINEAR, BORDER_CONSTANT 0): a pure gather, one
// thread per output pixel, batched over `count` images.  8-bit: 15-bit fixed-point weights, (sum + 2^14) >> 15;
// 16-bit: fp32 weights, products added left to right, cvRound + saturate.  Compiled with -fmad=false like the oracle
// (-ffp-contract=off); bit-exact against cv2.undistort 4.13 through the oracle (tests/golden/undistort_*.npz).
#include <math.h>
#include <string.h>

#include "common.cuh"

struct UndArgs { double fx, fy, cx, cy, k1, k2, p1, p2, k3; int W, H, cn; };

template <typename T>
__global__ void __launch_bounds__(256) undistort_kernel(UndArgs a, const T* __restrict__ src, T* __restrict__ dst) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.W * a.H) return;
    const int i = p / a.W, j = p - i * a.W;
    const size_t img = (size_t)blockIdx.y * a.W * a.H * a.cn;
    src += img; dst += img;
    const double ir0 = 1.0 / a.fx, ir2 = -a.cx / a.fx, ir4 = 1.0 / a.fy, ir5 = -a.cy / a.fy;
    const double x = (double)j * ir0 + ir2, y = (double)i * ir4 + ir5;
    const double x2 = x * x, y2 = y * y, r2 = x2 + y2, _2xy = 2 * x * y;
    const double kr = 1 + ((a.k3 * r2 + a.k2) * r2 + a.k1) * r2;
    const double xd = x * kr + a.p1 * _2xy + a.p2 * (r2 + 2 * x2), yd = y * kr + a.p1 * (r2 + 2 * y2) + a.p2 * _2xy;
    const double u = a.fx * xd + a.cx, v = a.fy * yd + a.cy;
    const long long iu = (long long)rint(u * 32.0), iv = (long long)rint(v * 32.0);
    const long long sx = iu >> 5, sy = iv >> 5;
    const int fa = (int)(iu & 31), fb = (int)(iv & 31);
    const bool x0 = sx >= 0 && sx < a.W, x1 = sx + 1 >= 0 && sx + 1 < a.W, y0 = sy >= 0 && sy < a.H, y1 = sy + 1 >= 0 && sy + 1 < a.H;
    const size_t o00 = ((size_t)(y0 ? sy : 0) * a.W + (size_t)(x0 ? sx : 0)) * a.cn, o01 = ((size_t)(y0 ? sy : 0) * a.W + (size_t)(x1 ? sx + 1 : 0)) * a.cn;
    const size_t o10 = ((size_t)(y1 ? sy + 1 : 0) * a.W + (size_t)(x0 ? sx : 0)) * a.cn, o11 = ((size_t)(y1 ? sy + 1 : 0) * a.W + (size_t)(x1 ? sx + 1 : 0)) * a.cn;
    for (int c = 0; c < a.cn; ++c) {
        const T s00 = (y0 && x0) ? src[o00 + c] : (T)0, s01 = (y0 && x1) ? src[o01 + c] : (T)0;
        const T s10 = (y1 && x0) ? src[o10 + c] : (T)0, s11 = (y1 && x1) ? src[o11 + c] : (T)0;
        if (sizeof(T) == 1) {
            const int w00 = (32 - fa) * (32 - fb) * 32, w01 = fa * (32 - fb) * 32, w10 = (32 - fa) * fb * 32, w11 = fa * fb * 32;
            int r = ((int)s00 * w00 + (int)s01 * w01 + (int)s10 * w10 + (int)s11 * w11 + (1 << 14)) >> 15;
            dst[(size_t)p * a.cn + c] = (T)min(max(r, 0), 255);
        } else {
            const float w00 = (float)((32 - fa) * (32 - fb)) / 1024.f, w01 = (float)(fa * (32 - fb)) / 1024.f;
            const float w10 = (float)((32 - fa) * fb) / 1024.f, w11 = (float)(fa * fb) / 1024.f;
            const float f = (((float)s00 * w00 + (float)s01 * w01) + (float)s10 * w10) + (float)s11 * w11;
            const int r = (int)rintf(f);
            dst[(size_t)p * a.cn + c] = (T)min(max(r, 0), 65535);
        }
    }
}

extern "C" int dvo_undistort(const void* src, void* dst, int width, int height, int type, int count, const double* K4, const double* D5, int mem,
                             void* cuda_stream) {
    if (!src || !dst || width < 2 || height < 2 || count < 0 || !K4 || !D5 || (type != DVO_IMG_U8C1 && type != DVO_IMG_U8C3 && type != DVO_IMG_U16C1)) {
        dvo_set_error("dvo_undistort: bad argument"); return DVO_ERR_ARG;
    }
    if (count == 0) return DVO_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { dvo_set_error("dvo_undistort: no usable CUDA device (there is no CPU fallback)"); return DVO_ERR_CUDA; }
    UndArgs a;
    a.fx = K4[0]; a.fy = K4[1]; a.cx = K4[2]; a.cy = K4[3]; a.k1 = D5[0]; a.k2 = D5[1]; a.p1 = D5[2]; a.p2 = D5[3]; a.k3 = D5[4];
    a.W = width; a.H = height; a.cn = (type == DVO_IMG_U8C3) ? 3 : 1;
    const size_t bytes = (size_t)width * height * a.cn * (type == DVO_IMG_U16C1 ? 2 : 1) * count;
    const cudaStream_t s = (cudaStream_t)cuda_stream;
    const void* d_src = src; void* d_dst = dst;
    DevBuf<uint8_t> t_src, t_dst;
    if (mem != DVO_MEM_DEVICE) {
        int rc;
        if ((rc = t_src.reserve(bytes)) || (rc = t_dst.reserve(bytes))) return rc;
        DVO_CUDA(cudaMemcpyAsync(t_src, src, bytes, cudaMemcpyHostToDevice, s));
        d_src = t_src; d_dst = t_dst;
    }
    dim3 grid((unsigned)(((size_t)width * height + 255) / 256), (unsigned)count);
    if (type == DVO_IMG_U16C1) undistort_kernel<uint16_t><<<grid, 256, 0, s>>>(a, (const uint16_t*)d_src, (uint16_t*)d_dst);
    else undistort_kernel<uint8_t><<<grid, 256, 0, s>>>(a, (const uint8_t*)d_src, (uint8_t*)d_dst);
    cudaError_t e = cudaGetLastError();
    if (mem != DVO_MEM_DEVICE) {
        if (e == cudaSuccess) e = cudaMemcpyAsync(dst, t_dst, bytes, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    }
    if (e != cudaSuccess) { dvo_set_error("dvo_undistort: %s", cudaGetErrorString(e)); return DVO_ERR_CUDA; }
    return DVO_OK;
}

// =====================================================================================================
// Raw-frame ingest (src/camTopic2PublisherPyD.cpp:65-80, :338-348): the publisher receives a bgr8 frame and a 32FC1 depth
// frame in metres.  depth16 = convertTo(CV_16UC1) of 1000.0 * depth (fp32 product, cvRound = round half to even,
// saturate), then setTo(1, depth16 == 0); framemono = cvtColor(BGR2GRAY) of the NEAREST-resized BGR -- BGR2GRAY is
// per pixel, so gray(level i) = NEAREST level i of the full-resolution gray, which the pyramid kernels already build.
// One fused pass writes the context's level-0 gray / depth regions: 7 B read, 3 B written per pixel.
// =====================================================================================================
__device__ __forceinline__ unsigned gray_of(unsigned b, unsigned g, unsigned r) { return (b * 3735u + g * 19235u + r * 9798u + (1u << 14)) >> 15; }
__device__ __forceinline__ unsigned mm_of(float m) {
    const float v = m * 1000.0f;                                     // -fmad=false: one rounding
    if (!(fabsf(v) <= 3.0e38f)) return 1u;                           // NaN / inf -> cvRound gives INT_MIN -> saturates to 0 -> 1
    const int r = __float2int_rn(fminf(fmaxf(v, -1.0e9f), 1.0e9f));
    const int s = min(max(r, 0), 65535);
    return s == 0 ? 1u : (unsigned)s;
}

__global__ void __launch_bounds__(256) ingest_raw_kernel(const uint8_t* __restrict__ bgr, const float* __restrict__ depth_m, uint8_t* __restrict__ gray,
                                                         uint16_t* __restrict__ depth, long long P0, long long slot_stride_px, int vec) {
    // grid.y = image; source images are tightly packed (P0 pixels each), destinations are the level-0 regions of consecutive slots
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (q >= P0) return;
    const uint8_t* sb = bgr + ((long long)blockIdx.y * P0 + q) * 3;
    const float* sd = depth_m ? depth_m + (long long)blockIdx.y * P0 + q : nullptr;
    uint8_t* dg = gray + (long long)blockIdx.y * slot_stride_px + q;
    uint16_t* dd = depth ? depth + (long long)blockIdx.y * slot_stride_px + q : nullptr;
    if (vec && q + 4 <= P0) {
        const uint32_t* s32 = reinterpret_cast<const uint32_t*>(sb);
        const uint32_t w0 = s32[0], w1 = s32[1], w2 = s32[2];        // B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
        const unsigned g0 = gray_of(w0 & 255u, (w0 >> 8) & 255u, (w0 >> 16) & 255u);
        const unsigned g1 = gray_of(w0 >> 24, w1 & 255u, (w1 >> 8) & 255u);
        const unsigned g2 = gray_of((w1 >> 16) & 255u, w1 >> 24, w2 & 255u);
        const unsigned g3 = gray_of((w2 >> 8) & 255u, (w2 >> 16) & 255u, w2 >> 24);
        *reinterpret_cast<uint32_t*>(dg) = g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
        if (sd && dd) {
            const float4 m = *reinterpret_cast<const float4*>(sd);
            *reinterpret_cast<uint2*>(dd) = make_uint2(mm_of(m.x) | (mm_of(m.y) << 16), mm_of(m.z) | (mm_of(m.w) << 16));
        }
    } else {
        for (int k = 0; k < 4 && q + k < P0; ++k) {
            dg[k] = (uint8_t)gray_of(sb[3 * k], sb[3 * k + 1], sb[3 * k + 2]);
            if (sd && dd) dd[k] = (uint16_t)mm_of(sd[k]);
        }
    }
}

int launch_ingest_raw(dvo_ctx* c, int frame, int first, int count, const uint8_t* d_bgr, const float* d_depth_m) {
    const long long P0 = c->geom.P[0];
    // 4-pixel vector path: every image's pixel count and the source pointers must keep 4-byte / 16-byte alignment
    const int vec = (P0 % 4 == 0) && ((reinterpret_cast<uintptr_t>(d_bgr) & 3) == 0) && (!d_depth_m || (reinterpret_cast<uintptr_t>(d_depth_m) & 15) == 0);
    uint8_t* gray = c->gray[frame] + lvl_at(c->geom, 0, first);
    uint16_t* depth = (d_depth_m && c->depth[frame]) ? c->depth[frame] + lvl_at(c->geom, 0, first) : nullptr;
    for (int z0 = 0; z0 < count; z0 += 32768) {
        const int nz = (count - z0 < 32768) ? count - z0 : 32768;
        dim3 grid((unsigned)((P0 / 4 + 1 + 255) / 256), (unsigned)nz);
        ingest_raw_kernel<<<grid, 256, 0, c->stream>>>(d_bgr + (long long)z0 * P0 * 3, d_depth_m ? d_depth_m + (long long)z0 * P0 : nullptr,
                                                       gray + (long long)z0 * P0, depth ? depth + (long long)z0 * P0 : nullptr, P0, P0, vec);
        c->launches++;
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// Device-to-device byte copy as a kernel.  The sequence pipeline moves a staged frame into the level-0 regions while the next
// frame's host-to-device copy is in flight: a cudaMemcpyAsync D2D can be scheduled on the same copy engine as that upload (the
// end-to-end sequence rate then varied 3x between runs); a kernel leaves the copy engines to the host link.
__global__ void __launch_bounds__(256) copy_bytes_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, size_t n16, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride)
        reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
    for (size_t i = (n16 << 4) + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i];
}
int launch_copy_bytes(dvo_ctx* c, void* dst, const void* src, size_t n) {
    if (n == 0) return DVO_OK;
    const bool vec = ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15) == 0;
    const size_t n16 = vec ? (n >> 4) : 0;
    size_t blocks = ((vec ? n16 : n) + 255) / 256;
    const size_t cap = (size_t)c->sm_count * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    copy_bytes_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(static_cast<uint8_t*>(dst), static_cast<const uint8_t*>(src), n16, n);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}
