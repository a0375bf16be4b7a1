// preprocess.cu -- pyramid, Canny (Sobel + NMS kernel; hysteresis kernel with the fused EDT column pass / reference point list),
// EDT row pass + packed distance texels, d2 read-back from the texels (inspection only).  All stages are bit-exact against
// oracle/dvo_oracle.hpp.
#include "common.cuh"

// =====================================================================================================
// NEAREST pyramid (src/camTopic2PublisherPyD.cpp:338-348): level l pixel (y,x) = level-0 pixel (y<<l, x<<l),
// always taken from full resolution.  Depth zeros become 1 on levels >= 1 here; level 0 keeps the caller's
// bytes and the zero fix (src/SolveDVO.cpp:512) is applied where depth is consumed / read back.
// =====================================================================================================
struct PyrArgs {
    PyrGeom g;
    uint8_t* gray;
    uint16_t* depth;   // may be null
    int first;
    int sub_total;     // sum_{l>=l0} P[l]
    int l0;            // first level this launch produces
    const unsigned char* active;   // optional per-slot mask
};

__global__ void __launch_bounds__(256) pyramid_nearest_kernel(PyrArgs a) {
    const int b = a.first + blockIdx.y;
    if (a.active && !a.active[b]) return;
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.sub_total) return;
    int l = a.l0;
    while (l < a.g.L - 1 && q >= a.g.P[l]) { q -= a.g.P[l]; ++l; }
    const int w = a.g.w[l], W0 = a.g.w[0], H0 = a.g.h[0];
    const int y = q / w, x = q - y * w;
    const int sy = min(y << l, H0 - 1), sx = min(x << l, W0 - 1);
    const long long src = lvl_at(a.g, 0, b) + (long long)sy * W0 + sx;
    const long long dst = lvl_at(a.g, l, b) + q;
    a.gray[dst] = a.gray[src];
    if (a.depth) { uint16_t d = a.depth[src]; a.depth[dst] = d == 0 ? (uint16_t)1 : d; }
}

// Level 1 holds three quarters of the pyramid's pixels below level 0.  When the widths allow it (W0 = 2 w1, w1 % 4 == 0)
// a thread produces four consecutive level-1 pixels from one 8-byte gray load and one 16-byte depth load and writes
// them with one 4-byte / one 8-byte store, instead of four byte-wide round trips.
__global__ void __launch_bounds__(256) pyramid_level1_vec4_kernel(PyrArgs a) {
    const int b = a.first + blockIdx.y;
    if (a.active && !a.active[b]) return;
    const int w1 = a.g.w[1], W0 = a.g.w[0], H0 = a.g.h[0];
    const int q4 = blockIdx.x * blockDim.x + threadIdx.x;          // group of 4 output pixels
    if (q4 * 4 >= a.g.P[1]) return;
    const int y = (q4 * 4) / w1, x = q4 * 4 - y * w1;
    const int sy = min(2 * y, H0 - 1);
    const long long src = lvl_at(a.g, 0, b) + (long long)sy * W0 + 2 * x;
    const long long dst = lvl_at(a.g, 1, b) + (long long)q4 * 4;
    const uint2 gv = *reinterpret_cast<const uint2*>(a.gray + src);
    const uint32_t gout = (gv.x & 0xFFu) | ((gv.x >> 8) & 0xFF00u) | ((gv.y & 0xFFu) << 16) | ((gv.y << 8) & 0xFF000000u);   // bytes 0, 2, 4, 6
    *reinterpret_cast<uint32_t*>(a.gray + dst) = gout;
    if (a.depth) {
        const uint4 dv = *reinterpret_cast<const uint4*>(a.depth + src);
        uint32_t d0 = dv.x & 0xFFFFu, d1 = dv.y & 0xFFFFu, d2 = dv.z & 0xFFFFu, d3 = dv.w & 0xFFFFu;                        // elements 0, 2, 4, 6
        d0 = d0 ? d0 : 1u; d1 = d1 ? d1 : 1u; d2 = d2 ? d2 : 1u; d3 = d3 ? d3 : 1u;
        *reinterpret_cast<uint2*>(a.depth + dst) = make_uint2(d0 | (d1 << 16), d2 | (d3 << 16));
    }
}

// The same with eight level-1 pixels per thread (w1 % 8 == 0): one 16-byte gray load, two 16-byte depth loads.
__global__ void __launch_bounds__(256) pyramid_level1_vec8_kernel(PyrArgs a) {
    const int b = a.first + blockIdx.y;
    if (a.active && !a.active[b]) return;
    const int w1 = a.g.w[1], W0 = a.g.w[0], H0 = a.g.h[0];
    const int q8 = blockIdx.x * blockDim.x + threadIdx.x;          // group of 8 output pixels
    if (q8 * 8 >= a.g.P[1]) return;
    const int y = (q8 * 8) / w1, x = q8 * 8 - y * w1;
    const int sy = min(2 * y, H0 - 1);
    const long long src = lvl_at(a.g, 0, b) + (long long)sy * W0 + 2 * x;
    const long long dst = lvl_at(a.g, 1, b) + (long long)q8 * 8;
    const uint4 gv = *reinterpret_cast<const uint4*>(a.gray + src);
    uint4 d0, d1;
    if (a.depth) { d0 = *reinterpret_cast<const uint4*>(a.depth + src); d1 = *reinterpret_cast<const uint4*>(a.depth + src + 8); }
    auto even_bytes = [](uint32_t lo, uint32_t hi) { return __byte_perm(lo, hi, 0x6420); };                                 // bytes 0, 2 of lo and hi
    *reinterpret_cast<uint2*>(a.gray + dst) = make_uint2(even_bytes(gv.x, gv.y), even_bytes(gv.z, gv.w));
    if (a.depth) {
        auto fix = [](uint32_t v) { v &= 0xFFFFu; return v ? v : 1u; };                                                     // element 0 of the pair, 0 -> 1
        *reinterpret_cast<uint4*>(a.depth + dst) = make_uint4(fix(d0.x) | (fix(d0.y) << 16), fix(d0.z) | (fix(d0.w) << 16),
                                                              fix(d1.x) | (fix(d1.y) << 16), fix(d1.z) | (fix(d1.w) << 16));
    }
}

// Levels >= 2 when every width is a multiple of 4: a thread produces four consecutive pixels of one level row (four independent
// loads, one 4-byte / one 8-byte store) instead of one pixel per thread -- the one-pixel kernel is latency-bound, not traffic-bound.
__global__ void __launch_bounds__(256) pyramid_nearest_vec4_kernel(PyrArgs a) {
    const int b = a.first + blockIdx.y;
    if (a.active && !a.active[b]) return;
    int q = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (q >= a.sub_total) return;
    int l = a.l0;
    while (l < a.g.L - 1 && q >= a.g.P[l]) { q -= a.g.P[l]; ++l; }
    const int w = a.g.w[l], W0 = a.g.w[0], H0 = a.g.h[0];
    const int y = q / w, x = q - y * w;
    const int sy = min(y << l, H0 - 1);
    const long long row = lvl_at(a.g, 0, b) + (long long)sy * W0;
    const long long dst = lvl_at(a.g, l, b) + q;
    int sx[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) sx[j] = min((x + j) << l, W0 - 1);
    uint32_t gv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) gv[j] = a.gray[row + sx[j]];
    if (a.depth) {
        uint32_t dv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { dv[j] = a.depth[row + sx[j]]; }
#pragma unroll
        for (int j = 0; j < 4; ++j) dv[j] = dv[j] ? dv[j] : 1u;
        *reinterpret_cast<uint2*>(a.depth + dst) = make_uint2(dv[0] | (dv[1] << 16), dv[2] | (dv[3] << 16));
    }
    *reinterpret_cast<uint32_t*>(a.gray + dst) = gv[0] | (gv[1] << 8) | (gv[2] << 16) | (gv[3] << 24);
}

int launch_pyramid(dvo_ctx* c, int first, int count, int frames_mask) {
    const PyrGeom& g = c->geom;
    if (g.L < 2) return DVO_OK;
    const bool vec1 = (g.w[0] == 2 * g.w[1]) && (g.w[1] % 4 == 0);
    const int l0 = vec1 ? 2 : 1;
    int sub = 0;
    bool vec_rest = true;                                  // 4-pixel groups never straddle a row or a level, stores stay aligned
    for (int l = l0; l < g.L; ++l) { sub += g.P[l]; vec_rest = vec_rest && (g.w[l] % 4 == 0) && (g.off[l] % 4 == 0) && (g.P[l] % 4 == 0); }
    for (int f = 0; f < 2; ++f) {
        if (!(frames_mask & (1 << f))) continue;
        PyrArgs a; a.g = g; a.gray = c->gray[f]; a.depth = c->depth[f]; a.first = first; a.sub_total = sub; a.l0 = l0; a.active = c->active;
        if (vec1 && g.w[1] % 8 == 0 && g.off[1] % 8 == 0 && g.P[1] % 8 == 0 && g.P[0] % 16 == 0) {
            dim3 grid1((g.P[1] / 8 + 255) / 256, count);
            pyramid_level1_vec8_kernel<<<grid1, 256, 0, c->stream>>>(a);
            c->launches++;
        } else if (vec1) {
            dim3 grid1((g.P[1] / 4 + 255) / 256, count);
            pyramid_level1_vec4_kernel<<<grid1, 256, 0, c->stream>>>(a);
            c->launches++;
        }
        if (sub > 0 && vec_rest) {
            dim3 grid((sub / 4 + 255) / 256, count);
            pyramid_nearest_vec4_kernel<<<grid, 256, 0, c->stream>>>(a);
            c->launches++;
        } else if (sub > 0) {
            dim3 grid((sub + 255) / 256, count);
            pyramid_nearest_kernel<<<grid, 256, 0, c->stream>>>(a);
            c->launches++;
        }
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// =====================================================================================================
// Canny (cv::Canny(img,150,100,3,true), src/SolveDVO.cpp:1705,1767; SURVEY Appendix B.1).
// One CTA per (slot, frame) image at one level.  Candidate / edge sets live as bitmaps (1 bit per pixel,
// bit i of word wx <-> x = 32*wx + i) with a one-word / one-row zero border, in shared memory when they fit
// (640x480: 2 x 42 KB) or in a global scratch otherwise.
//
//  phase 1  Sobel + NMS + double threshold: sobel_nms_kernel above (its own launch over every level and both frames); this
//           kernel starts from the candidate and strong bitmaps it left in the scratch.
//  phase 2  Hysteresis = monotone fixed point E <- C & dilate3x3(E) from E = strong.  Its closure equals the
//           reference's stack traversal regardless of order, hence bit-exact.  Thread <-> (word column, row
//           strip): each iteration sweeps the strip down and up so information crosses a whole strip per
//           iteration; strips whose 3x3 strip neighbourhood did not change are skipped.
//  phase 3  edge bytes 0/255 (128-bit stores) + edge count.
//  phase 4  (now) the edge bitmap is transposed (32x32 ballot transposes) so that a column is a bit string, and
//           every pixel gets its distance to the nearest edge pixel above/below with clz/ffs -- EDT phase 1.
//           (ref) selected = edge && depth > 100 bitmap: popcounts + a block scan give a stable enumeration of
//           selectedPts/enlistRefEdgePts (src/SolveDVO.cpp:1230-1264, 224-264), emitted row-major (see phase 4).
// =====================================================================================================
struct CannyArgs {
    const uint8_t* gray[2];   // level region of the reference / now frame (slot 0)
    uint8_t* edge[2];
    const uint16_t* depth; // ref
    uint16_t* gcol;        // now
    float *X, *Y, *Z;      // ref, level region
    int* pix;              // ref, level region: pixel index y*w+x of every emitted point
    int* npts;             // + level, stride L
    unsigned* nedge[2];    // + level, stride L (per frame)
    int w, h, P, L;
    int frame0;            // frame of blocks [0, count): 0 = reference, 1 = now
    int count;             // blocks [count, 2 count) process the now frame of the same slots (one launch for both frames)
    long long gscratch_frame_stride;   // global bitmaps: offset of the now frame's scratch
    float tmpfx, tmpfy, tmpcx, tmpcy;
    uint32_t* gscratch;    // this level's region of the bitmap scratch (slot 0, reference frame): source of the bitmaps, and their home when they do not fit in shared memory
    long long gscratch_stride;
    int first;
    int bm_words;          // words per bitmap region
    const unsigned char* active;   // optional per-slot mask
};

__device__ __forceinline__ void sobel3(const uint8_t* __restrict__ g, int w, int h, int y, int x, int& dx, int& dy) {
    const int ym = max(y - 1, 0), yp = min(y + 1, h - 1), xm = max(x - 1, 0), xp = min(x + 1, w - 1);
    const uint8_t* r0 = g + ym * w; const uint8_t* r1 = g + y * w; const uint8_t* r2 = g + yp * w;
    const int a = r0[xm], b = r0[x], c = r0[xp], d = r1[xm], f = r1[xp], p = r2[xm], q = r2[x], r = r2[xp];
    dx = (c + 2 * f + r) - (a + 2 * d + p);
    dy = (p + 2 * q + r) - (a + 2 * b + c);
}
__device__ __forceinline__ int mag_at(const uint8_t* __restrict__ g, int w, int h, int y, int x) {
    if ((unsigned)y >= (unsigned)h || (unsigned)x >= (unsigned)w) return 0;   // zero-padded magnitude border
    int dx, dy; sobel3(g, w, h, y, x, dx, dy);
    return dx * dx + dy * dy;
}

__device__ __forceinline__ uint32_t expand4(uint32_t nib) { return (((nib & 0xFu) * 0x00204081u) & 0x01010101u) * 0xFFu; }

// horizontal Sobel partial sums of one gray row at column x: hs = g(x+1) - g(x-1), hb = g(x-1) + 2 g(x) + g(x+1),
// BORDER_REPLICATE.  Row index already clamped by the caller.
__device__ __forceinline__ void row_sums(const uint8_t* __restrict__ grow, int w, int x, int lane, int& hs, int& hb) {
    const int v = (x < w) ? (int)grow[x] : 0;
    int l = __shfl_up_sync(0xffffffffu, v, 1), r = __shfl_down_sync(0xffffffffu, v, 1);
    if (lane == 0) l = (x > 0 && x < w) ? (int)grow[x - 1] : v;
    if (lane == 31) r = (x + 1 < w) ? (int)grow[x + 1] : v;
    if (x + 1 >= w) r = v;
    hs = r - l; hb = l + 2 * v + r;
}

// =====================================================================================================
// Canny phase 1: Sobel + non-maximum suppression + double threshold, every pyramid level and both frames in ONE launch.
// Output: the candidate bitmap (m > low, local maximum along the gradient) and the strong bitmap (candidate and m > high) of
// every image, in the padded layout canny_kernel works on (word (y + 1) * pitch + wx + 1), in the bitmap scratch.
//
// Warp task = (image, 128-column chunk, NMS_ROWS-row strip).  A lane owns FOUR adjacent columns (one aligned 32-bit load per
// row), so three of the four horizontal neighbours of a pixel are already in the lane's registers and a row costs 4 shuffles
// instead of 16; the chunk's two outside columns are carried by lanes 0 / 31 as one extra (halo) column each, so chunks are
// word aligned and the bitmap words are plain stores.  The arithmetic is fp32 on purpose: every value (gray <= 255, Sobel
// sums <= 1020, squared magnitude <= 2 080 800, tan(22.5) products < 2^24) is an integer that fp32 represents exactly, so
// the result is bit-identical to OpenCV's integer code, but adds / multiplies run on the FMA pipe and |x| is a free operand
// modifier -- on sm_100 the integer ALU pipe (half rate) was the limiter of the integer version (ncu: 70 % ALU pipe).
//   OpenCV:  horizontal  <=>  |dy| * 2^15 <  |dx| * 13573            <=>  |dy| < |dx| * (13573 / 2^15)
//            vertical    <=>  |dy| * 2^15 >  |dx| * (13573 + 2^16)   <=>  |dy| - 2 |dx| > |dx| * (13573 / 2^15)
//   (13573 / 2^15 is a dyadic rational: the products are exact.)  "m >= nb" on integers is "m > nb - 0.5".
// =====================================================================================================
#ifndef DVO_NMS_L2_AHEAD
#define DVO_NMS_L2_AHEAD 4           // rows prefetched into L2 ahead of the register prefetch (0 = off)
#endif
#ifndef DVO_NMS_MIN_BLOCKS
#define DVO_NMS_MIN_BLOCKS 2
#endif
#ifndef DVO_NMS_ROWS
#define DVO_NMS_ROWS 48
#endif
#ifndef DVO_NMS_WARPS
#define DVO_NMS_WARPS 8
#endif
constexpr int NMS_ROWS = DVO_NMS_ROWS, NMS_WARPS = DVO_NMS_WARPS;
struct NmsArgs {
    const uint8_t* gray[2];
    uint32_t* scratch;                 // bitmap scratch: [slot][frame] regions of slot_stride / frame_stride words
    long long slot_stride, frame_stride;
    long long off[DVO_MAX_LEVELS];     // gray: level offset
    long long bm_off[DVO_MAX_LEVELS];  // scratch: level offset inside a (slot, frame) region
    int w[DVO_MAX_LEVELS], h[DVO_MAX_LEVELS], P[DVO_MAX_LEVELS], bm_words[DVO_MAX_LEVELS];
    int chunks[DVO_MAX_LEVELS], strips[DVO_MAX_LEVELS], task_end[DVO_MAX_LEVELS];   // warp tasks of levels 0..l
    int L, first, count, frame0;
    float low, high;                   // squared thresholds (10000, 22500)
    const unsigned char* active;
};
struct NmsSums { float s[4], b[4], sH, bH; };     // horizontal Sobel sums of one gray row: s = g(x+1) - g(x-1), b = g(x-1) + 2 g(x) + g(x+1); H = halo column
struct NmsMags { float m[4], L, R; };             // squared gradient magnitudes of one row: own four columns, left and right neighbour
struct NmsGrad { float dx[4], dy[4]; };

template <bool VEC>       // VEC: width a multiple of 4 and 4-byte aligned rows -> one 32-bit load per lane and row
__global__ void __launch_bounds__(NMS_WARPS * 32, DVO_NMS_MIN_BLOCKS) sobel_nms_kernel(NmsArgs a) {
    const int lane = threadIdx.x & 31;
    int task = blockIdx.x * NMS_WARPS + (threadIdx.x >> 5);
    int l = 0;
    while (l < a.L && task >= a.task_end[l]) ++l;
    if (l >= a.L) return;
    if (l) task -= a.task_end[l - 1];
    const int chunks = a.chunks[l], strips = a.strips[l];
    const int chunk = task % chunks, t2 = task / chunks, strip = t2 % strips, img = t2 / strips;
    const int second = (img >= a.count) ? 1 : 0;
    const int frame = second ? DVO_FRAME_NOW : a.frame0;
    const int b = a.first + img - second * a.count;
    if (a.active && !a.active[b]) return;
    const int w = a.w[l], h = a.h[l];
    const int wd = (w + 31) >> 5, pitch = wd + 2;
    const uint8_t* __restrict__ g = a.gray[frame] + a.off[l] + (long long)b * a.P[l];
    uint32_t* Cb = a.scratch + (long long)b * a.slot_stride + (long long)frame * a.frame_stride + a.bm_off[l];
    const int bmw = a.bm_words[l];
    const int c0 = chunk << 7, xb = c0 + (lane << 2);
    const int y0 = strip * NMS_ROWS, y1 = min(h, y0 + NMS_ROWS);
    const bool first_lane = (lane == 0), last_lane = (lane == 31);
    const bool halo_valid = first_lane ? (c0 > 0) : (last_lane && c0 + 128 < w);        // the halo column lies inside the image
    const bool self_left = (xb == 0), self_right = (xb + 4 >= w);                       // BORDER_REPLICATE at the image border
    const int hx0 = first_lane ? c0 - 2 : c0 + 128;                                      // the two halo bytes: columns hx0, hx0 + 1
    const uint32_t sel_near = 0x7440u + (first_lane ? 1u : 0u), sel_far = 0x7440u + (first_lane ? 0u : 1u);
    const float lowt = (xb < w) ? a.low : 3.0e38f, high = a.high;
    const float K = 13573.0f / 32768.0f;

    // raw gray row r (clamped to the image): the lane's four bytes + the two halo bytes
    const bool in_image = (xb < w);
    const uint8_t* __restrict__ gx = g + (in_image ? xb : 0);
    const uint8_t* __restrict__ gh = g + (halo_valid ? hx0 : 0);
    const unsigned roff_max = (unsigned)((h - 1) * w);
    auto load_row = [&](unsigned roff, uint32_t& wv, uint32_t& hv) {      // roff = clamped row * w
        if (VEC) {
            wv = in_image ? *reinterpret_cast<const uint32_t*>(gx + roff) : 0u;
            hv = halo_valid ? (uint32_t)*reinterpret_cast<const uint16_t*>(gh + roff) : 0u;
        } else {
            const uint8_t* __restrict__ row = g + roff;
            wv = 0u;
#pragma unroll
            for (int j = 0; j < 4; ++j) wv |= (uint32_t)row[min(xb + j, w - 1)] << (8 * j);
            hv = halo_valid ? ((uint32_t)row[hx0] | ((uint32_t)row[min(hx0 + 1, w - 1)] << 8)) : 0u;
        }
    };
    auto byte_f = [](uint32_t wv, uint32_t sel) { return __uint_as_float(__byte_perm(wv, 0x4B000000u, sel)) - 8388608.0f; };
    auto sums = [&](uint32_t wv, uint32_t hv, NmsSums& S) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = byte_f(wv, 0x7440u + j);
        const float hn = byte_f(hv, sel_near), hf = byte_f(hv, sel_far);
        float lft = __shfl_up_sync(0xffffffffu, v[3], 1), rgt = __shfl_down_sync(0xffffffffu, v[0], 1);
        if (first_lane) lft = hn;
        if (last_lane) rgt = hn;
        if (self_left) lft = v[0];
        if (self_right) rgt = v[3];
        S.s[0] = v[1] - lft;  S.s[1] = v[2] - v[0]; S.s[2] = v[3] - v[1]; S.s[3] = rgt - v[2];
        S.b[0] = fmaf(2.0f, v[0], lft) + v[1];  S.b[1] = fmaf(2.0f, v[1], v[0]) + v[2];
        S.b[2] = fmaf(2.0f, v[2], v[1]) + v[3]; S.b[3] = fmaf(2.0f, v[3], v[2]) + rgt;
        const float gm1 = first_lane ? hf : v[3], gp1 = first_lane ? v[0] : hf;          // halo column's left / right neighbour
        S.sH = gp1 - gm1; S.bH = fmaf(2.0f, hn, gm1) + gp1;
    };
    // gradient and squared magnitude of an image row from the sums of the gray rows above (A), on (B) and below it (Cs); a row
    // outside the image (inside == false, warp-uniform) has magnitude zero
    auto grad_mag = [&](bool inside, const NmsSums& A, const NmsSums& B, const NmsSums& Cs, NmsGrad& G, NmsMags& M) {
        float mH;
        if (inside) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                G.dx[j] = fmaf(2.0f, B.s[j], A.s[j]) + Cs.s[j]; G.dy[j] = Cs.b[j] - A.b[j];
                M.m[j] = fmaf(G.dx[j], G.dx[j], G.dy[j] * G.dy[j]);
            }
            const float dxH = fmaf(2.0f, B.sH, A.sH) + Cs.sH, dyH = Cs.bH - A.bH;
            mH = halo_valid ? fmaf(dxH, dxH, dyH * dyH) : 0.0f;
            if (!VEC) {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (xb + j >= w) M.m[j] = 0.0f;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) { G.dx[j] = 0.0f; G.dy[j] = 0.0f; M.m[j] = 0.0f; }
            mH = 0.0f;
        }
        M.L = __shfl_up_sync(0xffffffffu, M.m[3], 1); M.R = __shfl_down_sync(0xffffffffu, M.m[0], 1);
        if (first_lane) M.L = mH;
        if (last_lane) M.R = mH;
        if (self_right) M.R = 0.0f;
    };

    uint32_t wv, hv;
    NmsSums S0, S1, S2;
    NmsMags M0, M1, M2;
    NmsGrad G0, G1;
    auto row_off = [&](int r) { return min((unsigned)max(r, 0) * (unsigned)w, roff_max); };
    load_row(row_off(y0 - 2), wv, hv); sums(wv, hv, S0);
    load_row(row_off(y0 - 1), wv, hv); sums(wv, hv, S1);
    load_row(row_off(y0), wv, hv);     sums(wv, hv, S2);
    grad_mag(y0 > 0, S0, S1, S2, G0, M0);                                               // magnitude row y0 - 1
    load_row(row_off(y0 + 1), wv, hv); sums(wv, hv, S0);                                 // S0 <- gray row y0 + 1
    grad_mag(true, S1, S2, S0, G0, M1);                                                  // magnitude row y0, its gradient in G0
    uint32_t wvn, hvn;
    load_row(row_off(y0 + 2), wvn, hvn);                                                 // one row ahead in registers ...
    unsigned roff_next = row_off(y0 + 3);
    unsigned roff_l2 = row_off(y0 + 3 + DVO_NMS_L2_AHEAD);                               // ... and DVO_NMS_L2_AHEAD more rows ahead into L2

    const int widx = (c0 >> 5) + (lane >> 3);
    const bool writer = ((lane & 7) == 0) && widx < wd;
    uint32_t* Cp = Cb + (long long)(y0 + 1) * pitch + 1 + widx;
    const int sh = (lane & 3) << 2;

    // non-maximum suppression + thresholds of one row (magnitude rows P above, C on, N below; Gc = gradient on the row) -> bitmap words
    auto nms_row = [&](const NmsMags& P, const NmsMags& C, const NmsMags& N, const NmsGrad& Gc) {
        float crm[4], ncm[4];                       // "m >= nb" on integers is "m > nb - 0.5"
#pragma unroll
        for (int j = 0; j < 4; ++j) { crm[j] = ((j < 3) ? C.m[j < 3 ? j + 1 : 3] : C.R) - 0.5f; ncm[j] = N.m[j] - 0.5f; }
        uint32_t bits = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float m = C.m[j];
            const float cl = j ? C.m[j > 0 ? j - 1 : 0] : C.L;
            const float pl = j ? P.m[j > 0 ? j - 1 : 0] : P.L, pr = (j < 3) ? P.m[j < 3 ? j + 1 : 3] : P.R;
            const float nl = j ? N.m[j > 0 ? j - 1 : 0] : N.L, nr = (j < 3) ? N.m[j < 3 ? j + 1 : 3] : N.R;
            const float adx = fabsf(Gc.dx[j]), ady = fabsf(Gc.dy[j]);
            const float t = adx * K, u = fmaf(adx, -2.0f, ady);
            const bool horiz = ady < t, vert = u > t;
            const bool neg = Gc.dx[j] * Gc.dy[j] < 0.0f;                                 // only read in the diagonal case, where dx, dy != 0
            const float da = neg ? pr : pl, db = neg ? nl : nr;
            const float na = horiz ? cl : (vert ? P.m[j] : da);
            const float nb = horiz ? crm[j] : (vert ? ncm[j] : db);
            const bool cand = (m > na) && (m > nb) && (m > lowt);
            const bool strong = cand && (m > high);
            bits |= (cand ? (1u << j) : 0u) | (strong ? (0x10000u << j) : 0u);
        }
        // candidate nibbles of a lane quad -> low half-word, strong nibbles -> high half-word; two quads make the 32-bit words
        bits <<= sh;
        bits |= __shfl_xor_sync(0xffffffffu, bits, 1);
        bits |= __shfl_xor_sync(0xffffffffu, bits, 2);
        const uint32_t hi = __shfl_down_sync(0xffffffffu, bits, 4);
        if (writer) {
            Cp[0] = __byte_perm(bits, hi, 0x5410);
            Cp[bmw] = __byte_perm(bits, hi, 0x7632);
        }
        Cp += pitch;
    };
    // One row: roles are passed by reference so that the caller rotates names, not registers.  A, B = sums of gray rows y, y+1;
    // Cs receives row y+2.  P, C = magnitude rows y-1, y; N receives y+1.  Gc = gradient at row y, Gn receives row y+1.
    auto row_step = [&](const NmsSums& A, const NmsSums& B, NmsSums& Cs, const NmsMags& P, const NmsMags& C, NmsMags& N,
                        const NmsGrad& Gc, NmsGrad& Gn) {
        wv = wvn; hv = hvn;
        load_row(roff_next, wvn, hvn); roff_next = min(roff_next + (unsigned)w, roff_max);   // gray row y + 3
        if (DVO_NMS_L2_AHEAD > 0) {
            if (in_image) asm volatile("prefetch.global.L2 [%0];" :: "l"(gx + roff_l2));
            roff_l2 = min(roff_l2 + (unsigned)w, roff_max);
        }
        sums(wv, hv, Cs);                                                                // gray row y + 2
        grad_mag(true, A, B, Cs, Gn, N);
        nms_row(P, C, N, Gc);
    };
    // rows whose lower neighbour row lies inside the image; the image's last row is done after the loops
    const int yend = (y1 == h) ? y1 - 1 : y1;
    // roles on entry: sums A = row y0 (S2), B = row y0 + 1 (S0), free = S1; magnitudes P = M0, C = M1, free = M2
    int y = y0;
    for (; y + 6 <= yend; y += 6) {               // six steps = a whole number of rotations of the sums / magnitudes (3) and of the gradient pair (2)
        row_step(S2, S0, S1, M0, M1, M2, G0, G1);
        row_step(S0, S1, S2, M1, M2, M0, G1, G0);
        row_step(S1, S2, S0, M2, M0, M1, G0, G1);
        row_step(S2, S0, S1, M0, M1, M2, G1, G0);
        row_step(S0, S1, S2, M1, M2, M0, G0, G1);
        row_step(S1, S2, S0, M2, M0, M1, G1, G0);
    }
    for (; y < yend; ++y) {                        // remainder: plain step, roles rotated by moves
        row_step(S2, S0, S1, M0, M1, M2, G0, G1);
        S2 = S0; S0 = S1; M0 = M1; M1 = M2; G0 = G1;
    }
    if (y1 == h) {                                 // last image row: the magnitude row below it is the zero padding
        grad_mag(false, S2, S0, S1, G1, M2);
        nms_row(M0, M1, M2, G0);
    }
}

constexpr int CANNY_MAX_WARPS = 24;
#ifndef DVO_CANNY_INTERLEAVE
#define DVO_CANNY_INTERLEAVE 1
#endif
#ifndef DVO_CANNY_STOP_AFTER
#define DVO_CANNY_STOP_AFTER 0
#endif

// The hysteresis sweep is a chaotic relaxation on purpose: within a round a thread reads neighbouring words their owners may be
// updating (bits only ever get set, every word has one writer, the loop ends after a round without changes).  In shared memory
// those reads go through a volatile pointer, so the compiler neither caches nor merges them and the behaviour is defined; the
// global-scratch variant keeps plain (L1-cached) accesses, ordered by the block barrier between rounds.
template <bool GLOBAL_BITMAPS> struct HystPtr { typedef volatile uint32_t* type; };
template <> struct HystPtr<true> { typedef uint32_t* type; };

template <bool GLOBAL_BITMAPS>
__global__ void __launch_bounds__(768, 2) canny_kernel(CannyArgs a) {
    extern __shared__ uint32_t smem_u32[];
    __shared__ int s_scan[CANNY_MAX_WARPS + 1];
    __shared__ int s_base;
    __shared__ unsigned s_cnt;
    __shared__ unsigned char s_chg[2][768];
    const int T = blockDim.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // one launch covers the reference AND the now frame of every slot: 2 x count CTAs leave a much fuller last wave than two
    // launches of count CTAs each (1024 CTAs at 296 resident = 3.46 waves)
#if DVO_CANNY_INTERLEAVE
    // both frames in one launch (count < 0x7fffffff): even blocks take the reference frame, odd blocks the now frame of the same
    // slot, so that every SM works on a mix of the two kinds of CTA (their last phases differ)
    const bool both = a.count != 0x7fffffff;
    const int second = both ? (int)(blockIdx.x & 1u) : 0;
    const int frame = second ? DVO_FRAME_NOW : a.frame0;
    const int b = a.first + (both ? (int)(blockIdx.x >> 1) : (int)blockIdx.x);
#else
    const int second = (blockIdx.x >= (unsigned)a.count) ? 1 : 0;
    const int frame = second ? DVO_FRAME_NOW : a.frame0;
    const int b = a.first + (int)blockIdx.x - second * a.count;
#endif
    const bool do_points = (frame == DVO_FRAME_REF), do_cols = (frame == DVO_FRAME_NOW);
    if (a.active && !a.active[b]) return;
    const int w = a.w, h = a.h;
    const int wd = (w + 31) >> 5, pitch = wd + 2;
    const int nwords = a.bm_words;
    // bitmaps: shared memory (LDS/STS/ATOMS) or, for images too large for it, a global scratch
    // (the global scratch is indexed by SLOT, not by block: launches on different streams own disjoint slot ranges)
    uint32_t* C = GLOBAL_BITMAPS ? a.gscratch + (long long)b * a.gscratch_stride + (long long)frame * a.gscratch_frame_stride : smem_u32;   // gscratch already points at this level's region
    uint32_t* E = C + nwords;

    // phase 1 (Sobel + NMS) ran in sobel_nms_kernel: it left the candidate and the strong bitmap of this image in the scratch.
    if (GLOBAL_BITMAPS) {      // bitmaps stay where they are; the transposed layout of the previous pass may have touched the border
        for (int i = tid; i < pitch; i += T) { C[i] = 0u; E[i] = 0u; C[(h + 1) * pitch + i] = 0u; E[(h + 1) * pitch + i] = 0u; }
        for (int y = tid; y < h; y += T) {
            C[(y + 1) * pitch] = 0u; E[(y + 1) * pitch] = 0u; C[(y + 1) * pitch + wd + 1] = 0u; E[(y + 1) * pitch + wd + 1] = 0u;
        }
    } else {
        const uint32_t* __restrict__ src = a.gscratch + (long long)b * a.gscratch_stride + (long long)frame * a.gscratch_frame_stride;
        if ((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (nwords & 1) == 0) {
            const uint4* s4 = reinterpret_cast<const uint4*>(src); uint4* d4 = reinterpret_cast<uint4*>(C);
            for (int i = tid; i < (nwords >> 1); i += T) d4[i] = s4[i];
        } else {
            for (int i = tid; i < 2 * nwords; i += T) C[i] = src[i];
        }
    }
    if (tid == 0) { s_cnt = 0u; s_base = 0; }
    __syncthreads();

#if DVO_CANNY_STOP_AFTER == 1
    return;        // phase timing probe (tools/prepare_variants.sh); never defined in a shipped build
#endif
    // ------------------------------------------------------------------ phase 2: hysteresis closure
    {
        const int Hs = max(1, min(h, min(T, 768) / wd));    // row strips
        const int Rh = (h + Hs - 1) / Hs;
        const int items = wd * Hs;
        const int sh = tid / wd, wx = tid - sh * wd;
        const bool owner = tid < items;
        const int ya = sh * Rh, yb = min(h, ya + Rh);
        for (int i = tid; i < 2 * 768; i += T) (&s_chg[0][0])[i] = (i < 768) ? 1 : 0;     // everything active at first
        __syncthreads();
        int cur = 0;
        for (;;) {
            int changed = 0;
            bool active = false;
            if (owner && ya < yb) {
                for (int dsy = -1; dsy <= 1 && !active; ++dsy)
                    for (int dwx = -1; dwx <= 1; ++dwx) {
                        const int s2 = sh + dsy, w2 = wx + dwx;
                        if (s2 >= 0 && s2 < Hs && w2 >= 0 && w2 < wd && s_chg[cur][s2 * wd + w2]) { active = true; break; }
                    }
            }
            if (active) {
                // Sweep the strip down, then up, with the 3x3 word neighbourhood in a sliding register window: one step loads
                // the three words of the incoming row and the candidate word (4 LDS; 11 before).  Words of the neighbouring
                // columns are as old as the step that loaded them -- harmless for a monotone relaxation.  Inside a word the
                // seeds are extended to whole runs of candidates with two carry chains instead of a shift-and-or loop.
                auto spread = [](uint32_t l, uint32_t c, uint32_t r) { return c | (c << 1) | (c >> 1) | (l >> 31) | (r << 31); };
                auto flood = [](uint32_t f, uint32_t c) {          // f subset of c: every seed grows to its run of ones of c
                    const uint32_t up = ((c + f) ^ c) & c;
                    const uint32_t cr = __brev(c), fr = __brev(f);
                    return f | up | __brev(((cr + fr) ^ cr) & cr);
                };
                typename HystPtr<GLOBAL_BITMAPS>::type Ev = E;
                const uint32_t* Cv = C;                            // candidates are read-only in this phase
                {   // down
                    int idx = (ya + 1) * pitch + wx + 1;
                    uint32_t sp = spread(Ev[idx - pitch - 1], Ev[idx - pitch], Ev[idx - pitch + 1]);
                    uint32_t el = Ev[idx - 1], ec = Ev[idx], er = Ev[idx + 1];
                    for (int y = ya; y < yb; ++y, idx += pitch) {
                        const uint32_t nl = Ev[idx + pitch - 1], nc = Ev[idx + pitch], nr = Ev[idx + pitch + 1];
                        const uint32_t c = Cv[idx];
                        uint32_t f = ec;
                        if (c != 0u && ec != c) {
                            f = flood(ec | (c & (sp | spread(el, ec, er) | spread(nl, nc, nr))), c);
                            if (f != ec) { Ev[idx] = f; changed = 1; }
                        }
                        sp = spread(el, f, er); el = nl; ec = nc; er = nr;
                    }
                }
                {   // up
                    int idx = yb * pitch + wx + 1;                 // row yb - 1
                    uint32_t sp = spread(Ev[idx + pitch - 1], Ev[idx + pitch], Ev[idx + pitch + 1]);
                    uint32_t el = Ev[idx - 1], ec = Ev[idx], er = Ev[idx + 1];
                    for (int y = yb - 1; y >= ya; --y, idx -= pitch) {
                        const uint32_t nl = Ev[idx - pitch - 1], nc = Ev[idx - pitch], nr = Ev[idx - pitch + 1];
                        const uint32_t c = Cv[idx];
                        uint32_t f = ec;
                        if (c != 0u && ec != c) {
                            f = flood(ec | (c & (sp | spread(el, ec, er) | spread(nl, nc, nr))), c);
                            if (f != ec) { Ev[idx] = f; changed = 1; }
                        }
                        sp = spread(el, f, er); el = nl; ec = nc; er = nr;
                    }
                }
            }
            if (owner) s_chg[cur ^ 1][tid] = (unsigned char)changed;
            cur ^= 1;
            if (!__syncthreads_or(changed)) break;
        }
    }

#if DVO_CANNY_STOP_AFTER == 2
    return;        // phase timing probe (tools/prepare_variants.sh); never defined in a shipped build
#endif
    // ------------------------------------------------------------------ phase 3: edge bytes (0/255) + edge count
    const int nw = h * wd;
    {
        uint8_t* eo = a.edge[frame] + (long long)b * a.P;
        unsigned cnt = 0;
        const bool vec_ok = (w % 16 == 0) && ((reinterpret_cast<uintptr_t>(eo) & 15) == 0);
        for (int q = tid; q < nw; q += T) {
            const int y = q / wd, wx = q - y * wd;
            const uint32_t e = E[(y + 1) * pitch + wx + 1];
            cnt += __popc(e);
            const int x0 = wx << 5;
            if (vec_ok && x0 + 32 <= w) {
                uint4 v0, v1;
                v0.x = expand4(e); v0.y = expand4(e >> 4); v0.z = expand4(e >> 8); v0.w = expand4(e >> 12);
                v1.x = expand4(e >> 16); v1.y = expand4(e >> 20); v1.z = expand4(e >> 24); v1.w = expand4(e >> 28);
                uint4* dst = reinterpret_cast<uint4*>(eo + (long long)y * w + x0);
                dst[0] = v0; dst[1] = v1;
            } else {
                for (int i = 0; i < 32 && x0 + i < w; ++i) eo[(long long)y * w + x0 + i] = ((e >> i) & 1u) ? 255 : 0;
            }
        }
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
        if (lane == 0 && cnt) atomicAdd(&s_cnt, cnt);
    }

#if DVO_CANNY_STOP_AFTER == 3
    return;        // phase timing probe (tools/prepare_variants.sh); never defined in a shipped build
#endif
    // ------------------------------------------------------------------ phase 4 (ref): selected = edge && depth > 100, in place
    if (do_points) {
        const uint16_t* __restrict__ dep = a.depth + (long long)b * a.P;
        for (int q = tid; q < nw; q += T) {
            const int y = q / wd, wx = q - y * wd;
            const int idx = (y + 1) * pitch + wx + 1;
            uint32_t e = E[idx], sel = 0u;
            const uint16_t* __restrict__ dr = dep + (long long)y * w + (wx << 5);
            while (e) {                               // four edge pixels per round: their depth loads are in flight together
                const int i0 = __ffs(e) - 1; e &= e - 1;
                const int i1 = e ? __ffs(e) - 1 : i0; e &= e - 1;        // 0 & (0 - 1) == 0: an exhausted word repeats i0
                const int i2 = e ? __ffs(e) - 1 : i0; e &= e - 1;
                const int i3 = e ? __ffs(e) - 1 : i0; e &= e - 1;
                const unsigned d0 = dr[i0], d1 = dr[i1], d2 = dr[i2], d3 = dr[i3];
                sel |= (d0 > 100u ? 1u << i0 : 0u) | (d1 > 100u ? 1u << i1 : 0u) | (d2 > 100u ? 1u << i2 : 0u) | (d3 > 100u ? 1u << i3 : 0u);
            }
            E[idx] = sel;
        }
    }
    __syncthreads();
    if (tid == 0) a.nedge[frame][(long long)b * a.L] = s_cnt;

    // ------------------------------------------------------------------ transpose E -> Et (into C's storage): Et[x * hwp + (y >> 5)], bit y & 31
    const int hw = (h + 31) >> 5, hwp = hw | 1;
    uint32_t* Et = C;
    if (do_cols) {
        const int nwarps = T >> 5;
        for (int blk = warp; blk < hw * wd; blk += nwarps) {
            const int wy = blk / wd, wx = blk - wy * wd;
            const int y = (wy << 5) + lane;
            const uint32_t word = (y < h) ? E[(y + 1) * pitch + wx + 1] : 0u;
            uint32_t mine = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) { const uint32_t bt = __ballot_sync(0xffffffffu, (word >> j) & 1u); if (lane == j) mine = bt; }
            Et[((wx << 5) + lane) * hwp + wy] = mine;
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------ phase 4 (now): EDT phase 1 from the column bit strings
    // thread <-> column; per 32-row word the nearest edge above / below comes from clz / ffs on the masked word, with
    // carries (last edge row above the word, first edge row below it) tracked incrementally.
    if (do_cols) {
        uint16_t* gc = a.gcol + (long long)b * a.P;
        const int BIG = 1 << 20;
        for (int x = tid; x < w; x += T) {
            const uint32_t* col = Et + x * hwp;
            int lastrow = -BIG;                 // last edge row in words < wy
            int nextrow = -1;                   // first edge row in words > wy (valid while >= 32*(wy+1)), BIG if none
            for (int wy = 0; wy < hw; ++wy) {
                const uint32_t Wd = col[wy];
                const int base = wy << 5;
                if (nextrow < base + 32) {      // recompute (amortised: each word is scanned once)
                    nextrow = BIG;
                    for (int kk = wy + 1; kk < hw; ++kk) { const uint32_t vv = col[kk]; if (vv) { nextrow = (kk << 5) + __ffs(vv) - 1; break; } }
                }
                uint16_t* o = gc + (long long)base * w + x;
#pragma unroll
                for (int bt = 0; bt < 32; ++bt) {
                    if (base + bt < h) {
                        const uint32_t mle = Wd & (0xffffffffu >> (31 - bt));
                        const uint32_t mge = Wd & (0xffffffffu << bt);
                        const int dn = mle ? bt - (31 - __clz(mle)) : base + bt - lastrow;
                        const int up = mge ? (__ffs(mge) - 1) - bt : nextrow - (base + bt);
                        o[(long long)bt * w] = (uint16_t)min(min(dn, up), DVO_EDT_INF_1D);
                    }
                }
                if (Wd) lastrow = base + 31 - __clz(Wd);
            }
        }
    }

    // ------------------------------------------------------------------ phase 4 (ref): stable compaction + back-projection
    // selectedPts / enlistRefEdgePts (src/SolveDVO.cpp:1230-1264, 224-264).  The reference enumerates column-major; the
    // list is emitted ROW-major here because the solver gathers from row-major texels: 32 consecutive points of a
    // horizontal contour then share 8 DRAM atoms inside one warp instruction.  Every sum over points is order
    // independent up to fp64 rounding; the pixel index of each point is kept so that the reference's order can be
    // restored wherever a per-point list is exposed (dvo_get_points, dvo_eval_normal_equations).
    if (do_points) {
        const uint16_t* __restrict__ dep = a.depth + (long long)b * a.P;
        float* X = a.X + (long long)b * a.P; float* Y = a.Y + (long long)b * a.P; float* Z = a.Z + (long long)b * a.P;
        int* pix = a.pix + (long long)b * a.P;
        const int per = (nw + T - 1) / T;
        const int q0 = min(nw, tid * per), q1 = min(nw, q0 + per);
        int mycnt = 0;
        for (int q = q0; q < q1; ++q) { const int y = q / wd, wx = q - y * wd; mycnt += __popc(E[(y + 1) * pitch + wx + 1]); }
        int incl = mycnt;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        if (tid < 32) {
            const int nwp = T >> 5;
            const int v = (tid < nwp) ? s_scan[tid] : 0;
            int iv = v;
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, iv, o); if (lane >= o) iv += t; }
            if (tid < nwp) s_scan[tid] = iv - v;               // exclusive warp offsets
            if (tid == 31) s_scan[CANNY_MAX_WARPS] = iv;       // total
        }
        __syncthreads();
        int off = s_scan[warp] + (incl - mycnt);
        for (int q = q0; q < q1; ++q) {
            const int y = q / wd, wx = q - y * wd;
            uint32_t v = E[(y + 1) * pitch + wx + 1];
            const uint16_t* __restrict__ dr = dep + (long long)y * w;
            while (v) {                               // four points per round: their depth loads are in flight together
                int xs[4], n = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (v) { xs[k] = (wx << 5) + __ffs(v) - 1; v &= v - 1; n = k + 1; } else xs[k] = xs[0];
                }
                unsigned dv[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) dv[k] = dr[xs[k]];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (k < n) {
                        const int x = xs[k];
                        const float z = __fdiv_rn((float)dv[k], 1000.0f);                                    // :248
                        X[off + k] = __fmul_rn(__fmul_rn(z, __fsub_rn((float)x, a.tmpcx)), a.tmpfx);        // :249
                        Y[off + k] = __fmul_rn(__fmul_rn(z, __fsub_rn((float)y, a.tmpcy)), a.tmpfy);        // :250
                        Z[off + k] = z;
                        pix[off + k] = y * w + x;
                    }
                }
                off += n;
            }
        }
        if (tid == 0) a.npts[(long long)b * a.L] = s_scan[CANNY_MAX_WARPS];
    }
}

static int canny_bitmap_words(int w, int h) {
    const int wd = (w + 31) >> 5;
    const int a = (wd + 2) * (h + 2);
    const int t = (wd << 5) * (((h + 31) >> 5) | 1);       // transposed layout reuses the candidate bitmap's storage
    return a > t ? a : t;
}

// Bitmap scratch geometry (context creation): per (slot, frame) one region per level holding the candidate and the edge bitmap.
void canny_scratch_layout(const PyrGeom& g, long long* bm_off, int* bm_words, size_t* words_per_image) {
    long long o = 0;
    for (int l = 0; l < g.L; ++l) { bm_off[l] = o; bm_words[l] = canny_bitmap_words(g.w[l], g.h[l]); o += 2LL * ((bm_words[l] + 3) & ~3); }
    *words_per_image = (size_t)o;
}

int launch_canny(dvo_ctx* c, int first, int count, int frames_mask) {
    const PyrGeom& g = c->geom;
    if (!(frames_mask & 3)) return DVO_OK;
    if ((frames_mask & 1) && !c->depth[0]) { dvo_set_error("canny: reference depth missing"); return DVO_ERR_STATE; }
    if (!c->bitmap_scratch) { dvo_set_error("canny: bitmap scratch missing"); return DVO_ERR_STATE; }
    const bool both = (frames_mask & 3) == 3;
    const int frame0 = (frames_mask & 1) ? DVO_FRAME_REF : DVO_FRAME_NOW;
    const long long slot_stride = (long long)c->bitmap_scratch_words, frame_stride = slot_stride * g.Bmax;
    {   // phase 1 of every level and frame: one launch
        NmsArgs n;
        n.gray[0] = c->gray[0]; n.gray[1] = c->gray[1];
        n.scratch = c->bitmap_scratch; n.slot_stride = slot_stride; n.frame_stride = frame_stride;
        long long tasks = 0;
        for (int l = 0; l < g.L; ++l) {
            n.off[l] = g.off[l]; n.bm_off[l] = c->bm_off[l]; n.w[l] = g.w[l]; n.h[l] = g.h[l]; n.P[l] = g.P[l]; n.bm_words[l] = c->bm_words[l];
            n.chunks[l] = (g.w[l] + 127) >> 7; n.strips[l] = (g.h[l] + NMS_ROWS - 1) / NMS_ROWS;
            tasks += (long long)n.chunks[l] * n.strips[l] * count * (both ? 2 : 1);
            if (tasks > 0x7fffffff - NMS_WARPS) { dvo_set_error("canny: too many tiles in one launch"); return DVO_ERR_ARG; }
            n.task_end[l] = (int)tasks;
        }
        n.L = g.L; n.first = first; n.count = both ? count : 0x7fffffff; n.frame0 = frame0;
        n.low = 10000.0f; n.high = 22500.0f; n.active = c->active;
        bool vec = true;          // every level: width a multiple of 4, rows 4-byte aligned (level offsets and image sizes are then multiples of 4 too)
        for (int l = 0; l < g.L; ++l) vec = vec && (g.w[l] % 4 == 0) && (g.off[l] % 4 == 0) && (g.P[l] % 4 == 0);
        const unsigned grid = (unsigned)((tasks + NMS_WARPS - 1) / NMS_WARPS);
        if (vec) sobel_nms_kernel<true><<<grid, NMS_WARPS * 32, 0, c->stream>>>(n);
        else sobel_nms_kernel<false><<<grid, NMS_WARPS * 32, 0, c->stream>>>(n);
        c->launches++;
    }
    for (int l = 0; l < g.L; ++l) {
        const int words = c->bm_words[l];
        const size_t smem = (size_t)2 * words * sizeof(uint32_t);
        const bool use_global = smem + 8192 > c->smem_optin;
        // hysteresis: thread <-> (word column, row strip), up to 24 warps per CTA (two CTAs per SM); the column pass wants a thread per column
        const int wdl = (g.w[l] + 31) >> 5;
        int strips = (CANNY_MAX_WARPS * 32) / wdl; if (strips > g.h[l]) strips = g.h[l]; if (strips < 1) strips = 1;
        int threads = wdl * strips; if (threads < g.w[l]) threads = g.w[l];
        int warps = (threads + 31) / 32; if (warps > CANNY_MAX_WARPS) warps = CANNY_MAX_WARPS; if (warps < 4) warps = 4;
        // smaller levels: smaller CTAs, more of them per SM (their phases are short and barrier-separated)
        constexpr int cap[DVO_MAX_LEVELS] = {24, 12, 8, 4, 4, 4};      // 640x480, 1024 pairs: 4.14 ms with 24 warps everywhere, 3.95 ms so
        if (warps > cap[l]) warps = cap[l];
        const int T = warps * 32;
        CannyArgs a;
        for (int f = 0; f < 2; ++f) {
            a.gray[f] = c->gray[f] + g.off[l]; a.edge[f] = c->edge[f] + g.off[l];
            a.nedge[f] = c->nedge + (size_t)f * g.Bmax * g.L + l;
        }
        a.depth = c->depth[0] ? c->depth[0] + g.off[l] : nullptr;
        a.gcol = c->gcol + g.off[l];
        a.X = c->ptsX + g.off[l]; a.Y = c->ptsY + g.off[l]; a.Z = c->ptsZ + g.off[l]; a.pix = c->ptsPix + g.off[l];
        a.npts = c->npts + l;
        a.w = g.w[l]; a.h = g.h[l]; a.P = g.P[l]; a.L = g.L;
        a.frame0 = frame0;
        a.count = both ? count : 0x7fffffff;                                           // single frame: no block is "second"
        const float scaleFac = (float)ldexp(1.0, -l);                                  // src/SolveDVO.cpp:231
        a.tmpfx = (float)(1. / (double)(scaleFac * c->K.fx));                          // :232
        a.tmpfy = (float)(1. / (double)(scaleFac * c->K.fy));                          // :233
        a.tmpcx = scaleFac * c->K.cx; a.tmpcy = scaleFac * c->K.cy;                    // :234-235
        a.gscratch = c->bitmap_scratch + c->bm_off[l];                                 // this level's region of slot 0, reference frame
        a.gscratch_stride = slot_stride;
        a.gscratch_frame_stride = frame_stride;
        a.first = first; a.bm_words = words; a.active = c->active;
        const int nblocks = both ? 2 * count : count;
        if (use_global) canny_kernel<true><<<nblocks, T, 0, c->stream>>>(a);
        else {
            if (smem > 48 * 1024 && smem > c->canny_smem_optin) {                      // opt in once per size (not per launch)
                DVO_CUDA(cudaFuncSetAttribute(canny_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                c->canny_smem_optin = smem;
            }
            canny_kernel<false><<<nblocks, T, smem, c->stream>>>(a);
        }
        c->launches++;
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// =====================================================================================================
// EDT phase 2 (rows): d2(y,x) = min_x' ( gcol(y,x')^2 + (x-x')^2 ), exact in integers.
// The cost matrix M[x][x'] = f(x') + (x-x')^2 is Monge, so the leftmost argmin is non-decreasing in x.  One
// warp per row resolves positions in breadth-first bisection order: at bisection step s the positions
// p = s*(2j+1) (1-based) are searched only between the argmins of their already-solved neighbours p-s and p+s,
// so each level costs O(w) evaluations and the whole row O(w log w), with no sequential stack as in the
// Meijster/Felzenszwalb scan.  Result is independent of evaluation order (pure min) -> bit-exact.
// =====================================================================================================
#define DVO_EDT_SPARSE_DIV 2048     // an image is "sparse" when nedge * DVO_EDT_SPARSE_DIV < P

struct EdtArgs {
    const uint16_t* gcol; int32_t* d2; unsigned* maxd2;   // level regions; maxd2 + level, stride L
    int w, h, P, L, first;
};

// Shared memory per warp: dv (i32, result), g (u16, column distance), arg (u16, leftmost argmin).
// Every search window is clipped to |x - x'| <= g(x) (the candidate x' = x already gives g(x)^2).  Positions of one
// bisection level are taken 32 at a time: a lane scans its own window when it is short; long windows (rare, but they
// would otherwise stall the other 31 lanes) are scanned cooperatively by the whole warp and reduced with REDUX.
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) edt_rows_kernel(EdtArgs a, const unsigned* __restrict__ nedge) {
    extern __shared__ int smem_i32[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = a.w;
    const int row = blockIdx.x * WARPS + warp;
    const int b = a.first + blockIdx.y;
    if (row >= a.h) return;                      // whole warp exits together; only __syncwarp below
    {   // this kernel only takes the images the window kernel skipped (few edge pixels)
        const unsigned ne = nedge[(long long)b * a.L];
        if (ne == 0u || (unsigned long long)ne * DVO_EDT_SPARSE_DIV >= (unsigned long long)a.P) return;
    }
    const int wp = (w + 1) & ~1;                 // even number of u16 per array
    int* dv = smem_i32 + (size_t)warp * (w + wp);
    unsigned short* gs = reinterpret_cast<unsigned short*>(dv + w);
    unsigned short* arg = gs + wp;
    const uint16_t* __restrict__ gr = a.gcol + (long long)b * a.P + (long long)row * w;
    for (int x = lane; x < w; x += 32) gs[x] = gr[x];
    __syncwarp();
    constexpr int SOLO_MAX = 6;
    int n = 1; while (n < w + 1) n <<= 1;
    for (int step = n >> 1; step >= 1; step >>= 1) {
        const int cnt = ((w / step) + 1) >> 1;   // positions p = step*(2j+1) <= w, j = 0..cnt-1
        for (int j0 = 0; j0 < cnt; j0 += 32) {
            const int j = j0 + lane;
            const bool has = j < cnt;
            int m = 0, lo = 0, hi = -1;
            if (has) {
                const int p = step * (2 * j + 1);
                m = p - 1;
                const int gm = gs[m];
                lo = (p - step >= 1) ? (int)arg[p - step - 1] : 0;
                hi = (p + step <= w) ? (int)arg[p + step - 1] : w - 1;
                lo = max(lo, m - gm); hi = min(hi, m + gm);
            }
            const bool solo = has && (hi - lo < SOLO_MAX);
            if (solo) {
                int best = 0x7fffffff, bx = lo;
                for (int xq = lo; xq <= hi; ++xq) {
                    const int dxx = m - xq, gq = gs[xq]; const int v = gq * gq + dxx * dxx;
                    if (v < best) { best = v; bx = xq; }
                }
                dv[m] = best; arg[m] = (unsigned short)bx;
            }
            unsigned longmask = __ballot_sync(0xffffffffu, has && !solo);
            while (longmask) {
                const int src = __ffs(longmask) - 1; longmask &= longmask - 1;
                const int Lo = __shfl_sync(0xffffffffu, lo, src), Hi = __shfl_sync(0xffffffffu, hi, src), M = __shfl_sync(0xffffffffu, m, src);
                int best = 0x7fffffff, bx = 0x7fffffff;
                for (int xq = Lo + lane; xq <= Hi; xq += 32) {
                    const int dxx = M - xq, gq = gs[xq]; const int v = gq * gq + dxx * dxx;
                    if (v < best) { best = v; bx = xq; }
                }
                const int vmin = __reduce_min_sync(0xffffffffu, best);
                const int xmin = __reduce_min_sync(0xffffffffu, best == vmin ? bx : 0x7fffffff);
                if (lane == 0) { dv[M] = vmin; arg[M] = (unsigned short)xmin; }
            }
        }
        __syncwarp();
    }
    int32_t* out = a.d2 + (long long)b * a.P + (long long)row * w;
    int mx = 0;
    for (int x = lane; x < w; x += 32) { const int v = dv[x]; out[x] = v; mx = max(mx, v); }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) atomicMax(&a.maxd2[(long long)b * a.L], (unsigned)mx);
}

// ---- EDT rows, primary kernel: expanding window with early exit -------------------------------------------------
// d2(x) = min_k ( g(x +- k)^2 + k^2 ).  A warp takes 32 consecutive pixels of a row and grows k while k^2 is still
// smaller than some lane's current best; every later candidate is at least k^2, so stopping is exact.  With contour
// edge maps the loop length is the largest distance inside the 32-pixel segment (a dozen steps at 640x480), every
// step is two conflict-free shared-memory loads and two min's for all 32 lanes -- no divergence, no stack.
// Images with very few edge pixels (loop length ~ image width) are left to the bisection kernel below.
constexpr int EDT16_G = 170, EDT16_PAD = 192, EDT16_BIG = 30000;
#ifndef DVO_EDT_PACKED16
#define DVO_EDT_PACKED16 1
#endif
// per-warp scratch of the window routines in ints: the 32-bit row (w + 2) or the two padded 16-bit copies
__host__ __device__ inline int edt_window_scratch_ints(int w) { return DVO_EDT_PACKED16 ? (w + 2 * EDT16_PAD + 2) : (w + 2); }

// expanding-window row routine of edt_rows_window_kernel for one warp; g2 = this warp's (w + 2)-int scratch + 1
template <typename Emit>
__device__ __forceinline__ void edt_row_window(const uint16_t* __restrict__ gr, int* g2, int w, int lane, Emit emit) {
    for (int x = lane; x < w; x += 32) { const int gv = gr[x]; g2[x] = gv * gv; }
    if (lane == 0) { g2[-1] = 0x3fffffff; g2[w] = 0x3fffffff; }
    __syncwarp();
    for (int x0 = 0; x0 < w; x0 += 32) {
        const int x = x0 + lane;
        int best = (x < w) ? g2[x] : 0;
        const int kint = min(x0, w - 32 - x0);
        const int* gc = g2 + min(x, w - 1);
        int k = 1, kk = 1;
        while (k < w) {
            if (__all_sync(0xffffffffu, kk >= best)) break;
            if (k + 3 <= kint) {
                const int a0 = min(gc[-k], gc[k]), a1 = min(gc[-k - 1], gc[k + 1]), a2 = min(gc[-k - 2], gc[k + 2]), a3 = min(gc[-k - 3], gc[k + 3]);
                const int k1 = kk + 2 * k + 1, k2 = kk + 4 * k + 4, k3 = kk + 6 * k + 9;
                best = min(min(best, a0 + kk), min(a1 + k1, min(a2 + k2, a3 + k3)));
                kk += 8 * k + 16; k += 4;
            } else {
                const int vl = g2[min(max(x - k, -1), w)], vr = g2[min(x + k, w)];
                best = min(best, min(vl, vr) + kk);
                kk += 2 * k + 1; ++k;
            }
        }
        if (x < w) emit(x, best);
    }
    __syncwarp();
}

// The same expanding window on PACKED 16-bit lanes: a lane owns two adjacent pixels and every step is one per-halfword
// min and one per-halfword add-min (VIMNMX.U16x2 / VIADDMNMX.U16x2), i.e. two instructions for two pixels instead of two per
// pixel.  The row lives in shared memory twice -- A[i] = (g2[2i], g2[2i+1]) and B[i] = (g2[2i+1], g2[2i+2]) -- so that the
// pair at any offset is one aligned 32-bit load.  Column distances are clamped to EDT16_G before squaring and both copies
// carry EDT16_PAD halfwords of EDT16_BIG on either side: every sum stays below 2^16 (g2 <= 28 900, k <= 173 + 3, BIG + k^2 <=
// 60 976).  A result below EDT16_G^2 was produced by an unclamped candidate and is therefore the exact minimum; the routine
// returns false if any pixel of the row reached EDT16_G^2, and the caller redoes that row with the 32-bit routine.
// H = this warp's scratch as halfwords: copy A at H[0 ..), copy B at H[EDT16_PAD + w + EDT16_PAD ..); w is even.
__device__ __forceinline__ void edt16_fill_pads(unsigned short* H, int w, int lane) {
    const int n = w + 2 * EDT16_PAD;
    for (int i = lane; i < EDT16_PAD; i += 32) { H[i] = EDT16_BIG; H[EDT16_PAD + w + i] = EDT16_BIG; H[n + i] = EDT16_BIG; H[n + EDT16_PAD + w + i] = EDT16_BIG; }
    __syncwarp();
}
template <typename Emit2>
__device__ __forceinline__ bool edt_row_window16(const uint16_t* __restrict__ gr, unsigned short* H, int w, int lane, Emit2 emit2) {
    const int n = w + 2 * EDT16_PAD;                       // halfwords per copy (even)
    uint32_t* A = reinterpret_cast<uint32_t*>(H);
    uint32_t* B = reinterpret_cast<uint32_t*>(H + n);
    const uint32_t* __restrict__ gr2 = reinterpret_cast<const uint32_t*>(gr);
    for (int p = lane; 2 * p < w; p += 32) {
        const uint32_t gv = gr2[p];
        const uint32_t g0 = min(gv & 0xFFFFu, (uint32_t)EDT16_G), g1 = min(gv >> 16, (uint32_t)EDT16_G);
        A[(EDT16_PAD >> 1) + p] = (g0 * g0) | ((g1 * g1) << 16);
    }
    __syncwarp();
    for (int p = lane - 1; 2 * p < w; p += 32) {          // B[i] = (H[2i+1], H[2i+2]): from p = -1 (left pad | g2[0]) to the last pair (g2[w-1] | right pad)
        const int i = (EDT16_PAD >> 1) + p;
        B[i] = __byte_perm(A[i], A[i + 1], 0x5432);
    }
    __syncwarp();
    bool exact = true;
    for (int x0 = 0; x0 < w; x0 += 64) {
        const int x = x0 + 2 * lane;
        const int i0 = (EDT16_PAD + min(x, w - 2)) >> 1;
        uint32_t best = (x < w) ? A[i0] : 0u;
        const uint32_t* a = A + i0;
        const uint32_t* b = B + i0;
        int k = 1;
        uint32_t kk = 0x00010001u;                         // k^2 in both halfwords
        for (;;) {
            const uint32_t bmax = max(best & 0xFFFFu, best >> 16);
            if (__all_sync(0xffffffffu, (kk & 0xFFFFu) >= bmax)) break;
            // offsets k .. k+3 with k odd: pairs at odd offsets come from copy B, even offsets from copy A
            const int m = k >> 1;
            const uint32_t c0 = __vminu2(b[m], b[-m - 1]), c1 = __vminu2(a[m + 1], a[-m - 1]);
            const uint32_t c2 = __vminu2(b[m + 1], b[-m - 2]), c3 = __vminu2(a[m + 2], a[-m - 2]);
            const uint32_t k1 = kk + (uint32_t)(2 * k + 1) * 0x00010001u, k2 = kk + (uint32_t)(4 * k + 4) * 0x00010001u, k3 = kk + (uint32_t)(6 * k + 9) * 0x00010001u;
            best = __viaddmin_u16x2(c0, kk, best); best = __viaddmin_u16x2(c1, k1, best);
            best = __viaddmin_u16x2(c2, k2, best); best = __viaddmin_u16x2(c3, k3, best);
            kk += (uint32_t)(8 * k + 16) * 0x00010001u; k += 4;
        }
        if (x < w) {
            emit2(x, best);
            if (max(best & 0xFFFFu, best >> 16) >= (uint32_t)(EDT16_G * EDT16_G)) exact = false;
        }
    }
    __syncwarp();
    return __all_sync(0xffffffffu, exact);
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) edt_rows_window_kernel(EdtArgs a, const unsigned* __restrict__ nedge) {
    extern __shared__ int smem_i32[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = a.w;
    const int row = blockIdx.x * WARPS + warp;
    const int b = a.first + blockIdx.y;
    if (row >= a.h) return;
    const unsigned ne = nedge[(long long)b * a.L];
    if (ne != 0u && (unsigned long long)ne * DVO_EDT_SPARSE_DIV < (unsigned long long)a.P) return;   // sparse image: other kernel
    int32_t* out = a.d2 + (long long)b * a.P + (long long)row * w;
    if (ne == 0u) {                                  // no edge pixel at all: d2 is the sentinel everywhere
        for (int x = lane; x < w; x += 32) out[x] = DVO_EDT_INF;
        if (lane == 0) atomicMax(&a.maxd2[(long long)b * a.L], (unsigned)DVO_EDT_INF);
        return;
    }
    int* scratch = smem_i32 + (size_t)warp * edt_window_scratch_ints(w);
    const uint16_t* __restrict__ gr = a.gcol + (long long)b * a.P + (long long)row * w;
    int mx = 0;
    auto emit = [&](int x, int v) { out[x] = v; mx = max(mx, v); };
    const bool packed16 = DVO_EDT_PACKED16 && (w % 2 == 0) && ((reinterpret_cast<uintptr_t>(gr) & 3) == 0) && ((reinterpret_cast<uintptr_t>(out) & 7) == 0);
    bool done = false;
    if (packed16) {
        edt16_fill_pads(reinterpret_cast<unsigned short*>(scratch), w, lane);
        auto emit2 = [&](int x, uint32_t v2) {
            *reinterpret_cast<int2*>(out + x) = make_int2((int)(v2 & 0xFFFFu), (int)(v2 >> 16));
            mx = max(mx, (int)max(v2 & 0xFFFFu, v2 >> 16));
        };
        done = edt_row_window16(gr, reinterpret_cast<unsigned short*>(scratch), w, lane, emit2);
    }
    if (!done) edt_row_window(gr, scratch + 1, w, lane, emit);     // odd width, or a pixel further than EDT16_G from every edge
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) atomicMax(&a.maxd2[(long long)b * a.L], (unsigned)mx);
}

static int launch_edt_rows(dvo_ctx* c, int first, int count) {
    const PyrGeom& g = c->geom;
    constexpr int WARPS = 8;
    DVO_CUDA(cudaMemsetAsync(c->maxd2 + (size_t)first * g.L, 0, sizeof(unsigned) * (size_t)count * g.L, c->stream));
    for (int l = 0; l < g.L; ++l) {
        EdtArgs a; a.gcol = c->gcol + g.off[l]; a.d2 = c->d2 + g.off[l]; a.maxd2 = c->maxd2 + l;
        a.w = g.w[l]; a.h = g.h[l]; a.P = g.P[l]; a.L = g.L; a.first = first;
        const unsigned* ne = c->nedge + (size_t)DVO_FRAME_NOW * g.Bmax * g.L + l;
        const int w = g.w[l];
        dim3 grid((g.h[l] + WARPS - 1) / WARPS, count);
        {   // dense images: expanding-window kernel
            const size_t smem = (size_t)WARPS * edt_window_scratch_ints(w) * sizeof(int);
            static size_t opted_w = 0;                      // largest opt-in so far (one device per process)
            if (smem > 48 * 1024 && smem > opted_w) { DVO_CUDA(cudaFuncSetAttribute(edt_rows_window_kernel<WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); opted_w = smem; }
            edt_rows_window_kernel<WARPS><<<grid, WARPS * 32, smem, c->stream>>>(a, ne);
            c->launches++;
        }
        {   // sparse images: bisection kernel (exits immediately for every other image)
            const int wp = (w + 1) & ~1;
            const size_t smem = (size_t)WARPS * (w + wp) * sizeof(int);
            static size_t opted_b = 0;
            if (smem > 48 * 1024 && smem > opted_b) { DVO_CUDA(cudaFuncSetAttribute(edt_rows_kernel<WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); opted_b = smem; }
            edt_rows_kernel<WARPS><<<grid, WARPS * 32, smem, c->stream>>>(a, ne);
            c->launches++;
        }
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// =====================================================================================================
// packed texels (common.cuh "packed texel"): the exact d2 of every pixel and of its four stencil neighbours in 8 bytes,
// stored in 4x4 Morton tiles: 4 B read + 8 B written per pixel, and the solver's working set per reprojected point is an
// 8-byte texel in a 4x4-pixel line.  DTn / gradient / weight are evaluated in the solver (texel_values) from per-level
// lookup tables: DT = sqrtf(d2), DTn = DT * (float)(255 * (1/(max-min))), gx/gy = 0.5*(next) - 0.5*(prev) with
// REFLECT_101, w = getWeightOf(DTn) (src/SolveDVO.cpp:1774, 1790, 1063-1098, 1047-1053; SURVEY Appendix B.3, B.6).
// Thread <-> texel of the blocked layout (stores are contiguous); the five d2 loads hit L1 / L2.
// =====================================================================================================
struct PackArgs { const int32_t* d2; uint2* tex8; int w, h, P, Pt, tw, th, first; };

// One CTA = a 64x8-pixel region = 16x2 tiles: the d2 values (plus a one-pixel halo) are staged through shared memory with
// row-contiguous loads, every thread assembles two texels, and each warp stores 256 contiguous bytes (two whole tiles).
#ifndef DVO_PACK_RH
#define DVO_PACK_RH 32         // tile rows of pack_texel_kernel: 8 / 16 / 32 rows -> 63.1 / 62.5 / 62.1 ms per 148 x 8 frames of 1280x720 (config 4)
#endif
constexpr int PACK_RW = 64, PACK_RH = DVO_PACK_RH;
__global__ void __launch_bounds__(256) pack_texel_kernel(PackArgs a) {
    __shared__ int tile[PACK_RH + 2][PACK_RW + 2 + 1];
    const int b = a.first + blockIdx.z;
    const int w = a.w, h = a.h;
    const int x0 = blockIdx.x * PACK_RW, y0 = blockIdx.y * PACK_RH;
    const int32_t* __restrict__ d = a.d2 + (long long)b * a.P;
    for (int i = threadIdx.x; i < (PACK_RH + 2) * (PACK_RW + 2); i += 256) {
        const int ry = i / (PACK_RW + 2), rx = i - ry * (PACK_RW + 2);
        const int y = y0 + ry - 1, x = x0 + rx - 1;
        tile[ry][rx] = (x >= 0 && x < w && y >= 0 && y < h) ? __ldg(d + (long long)y * w + x) : 0;
    }
    __syncthreads();
    uint2* __restrict__ out = a.tex8 + (long long)b * a.Pt;
#pragma unroll
    for (int r = 0; r < PACK_RH / 4; ++r) {
        const int ty = blockIdx.y * (PACK_RH / 4) + r, tx = blockIdx.x * (PACK_RW / 4) + (threadIdx.x >> 4);
        if (ty >= a.th || tx >= a.tw) continue;
        const int k = threadIdx.x & 15;
        const int ly = (r << 2) | ((k >> 2) & 2) | ((k >> 1) & 1), lx = ((threadIdx.x >> 4) << 2) | ((k >> 1) & 2) | (k & 1);
        const int y = y0 + ly, x = x0 + lx;
        uint2 t = make_uint2(DVO_TEX_ESCAPE, 0u);
        if (x < w && y < h) {
            const int c = tile[ly + 1][lx + 1];
            const bool bx = (x == 0 || x == w - 1), by = (y == 0 || y == h - 1);
            const int dl = bx ? 0 : tile[ly + 1][lx] - c, dr = bx ? 0 : tile[ly + 1][lx + 2] - c;
            const int du = by ? 0 : tile[ly][lx + 1] - c, dd = by ? 0 : tile[ly + 2][lx + 1] - c;
            const int lo = min(min(dl, dr), min(du, dd)), hi = max(max(dl, dr), max(du, dd));
            if (c < 65536 && lo >= -512 && hi <= 511) {
                t.x = (unsigned)c | (((unsigned)dl & 0x3FFu) << 16);
                t.y = ((unsigned)dr & 0x3FFu) | (((unsigned)du & 0x3FFu) << 10) | (((unsigned)dd & 0x3FFu) << 20);
            }
        }
        out[(((long long)ty * a.tw + tx) << 4) + k] = t;
    }
}

static int launch_pack(dvo_ctx* c, int first, int count) {
    const PyrGeom& g = c->geom;
    for (int l = 0; l < g.L; ++l) {
        PackArgs a; a.d2 = c->d2 + g.off[l]; a.tex8 = c->tex8 + g.offt[l];
        a.w = g.w[l]; a.h = g.h[l]; a.P = g.P[l]; a.Pt = g.Pt[l]; a.tw = g.tw[l]; a.th = (g.h[l] + 3) >> 2;
        for (int z0 = 0; z0 < count; z0 += 32768) {          // gridDim.z limit is 65535
            a.first = first + z0;
            const int nz = (count - z0 < 32768) ? count - z0 : 32768;
            dim3 grid((a.tw + PACK_RW / 4 - 1) / (PACK_RW / 4), (a.th + PACK_RH / 4 - 1) / (PACK_RH / 4), nz);
            pack_texel_kernel<<<grid, 256, 0, c->stream>>>(a);
            c->launches++;
        }
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// =====================================================================================================
// EDT rows + packed texels in one pass (the hot path up to 800 pixels wide).  edt_rows_*_kernel followed by pack_texel_kernel
// writes the 32-bit d2 image (4 B/px) only to read it straight back (4 B/px + halo); here a CTA owns a band of R image
// rows: its warps evaluate the R + 2 rows y0-1 .. y0+R with the same exact row routines (expanding window, or the
// bisection for sparse images) into a 16-bit band buffer in shared memory, and the band's texels are assembled from
// there and stored as whole 128-byte Morton tiles.  The two halo rows are evaluated twice ((R+2)/R of the row work).
// The band holds min(d2, 65535); a texel whose stencil touches a saturated value is escaped (DVO_TEX_ESCAPE), and every
// pixel with d2 >= DVO_D2_SPILL additionally writes its exact value to the 32-bit d2 image.  Neighbours of an escaped
// texel are at most one pixel further from the edge set than a pixel with d >= 254.99, i.e. d2 >= 64 516 >
// DVO_D2_SPILL, so every value the solver's escape path reads (stencil_from_d2) has been written.  The 32-bit image is
// therefore SPARSE in this mode: inspection (dvo_get_level_buffer) takes d2 from the texel where it is not escaped.
// =====================================================================================================
#define DVO_D2_SPILL 64000

struct EdtPackArgs { const uint16_t* gcol; int32_t* d2; uint2* tex8; unsigned* maxd2; int w, h, P, Pt, tw, th, L, first; };

// bisection row routine of edt_rows_kernel for one warp; dv / gs / arg = this warp's scratch
template <typename Emit>
__device__ __forceinline__ void edt_row_bisect(const uint16_t* __restrict__ gr, int* dv, unsigned short* gs, unsigned short* arg, int w, int lane, Emit emit) {
    for (int x = lane; x < w; x += 32) gs[x] = gr[x];
    __syncwarp();
    constexpr int SOLO_MAX = 6;
    int n = 1; while (n < w + 1) n <<= 1;
    for (int step = n >> 1; step >= 1; step >>= 1) {
        const int cnt = ((w / step) + 1) >> 1;
        for (int j0 = 0; j0 < cnt; j0 += 32) {
            const int j = j0 + lane;
            const bool has = j < cnt;
            int m = 0, lo = 0, hi = -1;
            if (has) {
                const int p = step * (2 * j + 1);
                m = p - 1;
                const int gm = gs[m];
                lo = (p - step >= 1) ? (int)arg[p - step - 1] : 0;
                hi = (p + step <= w) ? (int)arg[p + step - 1] : w - 1;
                lo = max(lo, m - gm); hi = min(hi, m + gm);
            }
            const bool solo = has && (hi - lo < SOLO_MAX);
            if (solo) {
                int best = 0x7fffffff, bx = lo;
                for (int xq = lo; xq <= hi; ++xq) {
                    const int dxx = m - xq, gq = gs[xq]; const int v = gq * gq + dxx * dxx;
                    if (v < best) { best = v; bx = xq; }
                }
                dv[m] = best; arg[m] = (unsigned short)bx;
            }
            unsigned longmask = __ballot_sync(0xffffffffu, has && !solo);
            while (longmask) {
                const int src = __ffs(longmask) - 1; longmask &= longmask - 1;
                const int Lo = __shfl_sync(0xffffffffu, lo, src), Hi = __shfl_sync(0xffffffffu, hi, src), M = __shfl_sync(0xffffffffu, m, src);
                int best = 0x7fffffff, bx = 0x7fffffff;
                for (int xq = Lo + lane; xq <= Hi; xq += 32) {
                    const int dxx = M - xq, gq = gs[xq]; const int v = gq * gq + dxx * dxx;
                    if (v < best) { best = v; bx = xq; }
                }
                const int vmin = __reduce_min_sync(0xffffffffu, best);
                const int xmin = __reduce_min_sync(0xffffffffu, best == vmin ? bx : 0x7fffffff);
                if (lane == 0) { dv[M] = vmin; arg[M] = (unsigned short)xmin; }
            }
        }
        __syncwarp();
    }
    for (int x = lane; x < w; x += 32) emit(x, dv[x]);
    __syncwarp();
}

template <int WARPS, int R, bool SPARSE>
__global__ void __launch_bounds__(WARPS * 32) edt_pack_kernel(EdtPackArgs a, const unsigned* __restrict__ nedge) {
    extern __shared__ int smem_i32[];
    static_assert(R % 4 == 0, "a band is a whole number of tile rows");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = a.w, h = a.h;
    const int b = a.first + blockIdx.y;
    const unsigned ne = nedge[(long long)b * a.L];
    const bool sparse = (ne != 0u) && ((unsigned long long)ne * DVO_EDT_SPARSE_DIV < (unsigned long long)a.P);
    if (sparse != SPARSE) return;
    const int y0 = blockIdx.x * R;
    const int bp = (w + 1) & ~1;                                     // band pitch (u16), even
    unsigned short* band = reinterpret_cast<unsigned short*>(smem_i32);
    const int per_warp = SPARSE ? (w + bp) : edt_window_scratch_ints(w);
    int* scratch = smem_i32 + ((R + 2) * bp) / 2 + warp * per_warp;
    int32_t* __restrict__ d2g = a.d2 + (long long)b * a.P;
    int mx = 0;
    const bool packed16 = !SPARSE && DVO_EDT_PACKED16 && (w % 2 == 0) && ne != 0u &&
                          ((reinterpret_cast<uintptr_t>(a.gcol + (long long)b * a.P) & 3) == 0);     // block-uniform; rows are read as 32-bit pairs
    __shared__ int s_next_row;
    if (threadIdx.x == 0) s_next_row = WARPS;
    if (ne != 0u) {      // the band's column distances (contiguous rows y0-1 .. y0+R) towards L2 while the first rows are being set up
        const int ya = max(y0 - 1, 0), yb = min(y0 + R + 1, h);
        const char* base = reinterpret_cast<const char*>(a.gcol + (long long)b * a.P + (long long)ya * w);
        const int nbytes = (yb - ya) * w * 2;
        for (int o = threadIdx.x * 128; o < nbytes; o += WARPS * 32 * 128) asm volatile("prefetch.global.L2 [%0];" :: "l"(base + o));
    }
    if (packed16) edt16_fill_pads(reinterpret_cast<unsigned short*>(scratch), w, lane);
    __syncthreads();
    // rows are handed out dynamically (their cost follows the distance to the nearest edge): first one per warp, then first come first served
    for (int r = warp; r < R + 2; ) {
        const int rcur = r;
        if (lane == 0) r = atomicAdd(&s_next_row, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        const int y = y0 - 1 + rcur;
        if (y < 0 || y >= h) continue;                               // warp-uniform
        unsigned short* brow = band + rcur * bp;
        int32_t* grow = d2g + (long long)y * w;
        auto emit = [&](int x, int v) {
            brow[x] = (unsigned short)min(v, 65535);
            if (v >= DVO_D2_SPILL) grow[x] = v;
            mx = max(mx, v);
        };
        if (ne == 0u) {                                              // no edge pixel at all: d2 is the sentinel everywhere
            for (int x = lane; x < w; x += 32) emit(x, DVO_EDT_INF);
            continue;
        }
        const uint16_t* __restrict__ gr = a.gcol + (long long)b * a.P + (long long)y * w;
        if (SPARSE) {
            unsigned short* gs = reinterpret_cast<unsigned short*>(scratch + w);
            edt_row_bisect(gr, scratch, gs, gs + bp, w, lane, emit);
        } else if (packed16) {
            unsigned* brow2 = reinterpret_cast<unsigned*>(brow);
            auto emit2 = [&](int x, uint32_t v2) { brow2[x >> 1] = v2; mx = max(mx, (int)max(v2 & 0xFFFFu, v2 >> 16)); };   // both values < DVO_D2_SPILL
            if (!edt_row_window16(gr, reinterpret_cast<unsigned short*>(scratch), w, lane, emit2)) {
                edt_row_window(gr, scratch + 1, w, lane, emit);                          // a pixel further than EDT16_G from every edge: exact 32-bit redo
                edt16_fill_pads(reinterpret_cast<unsigned short*>(scratch), w, lane);   // the redo used the scratch
            }
        } else {
            edt_row_window(gr, scratch + 1, w, lane, emit);
        }
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0 && mx > 0) atomicMax(&a.maxd2[(long long)b * a.L], (unsigned)mx);
    __syncthreads();
    // ---- texels of the band: rows y0 .. y0 + R - 1, tile row by tile row (16 * tw contiguous texels each).  A thread assembles
    // one Morton quad = a 2x2 pixel block = 32 contiguous bytes: its 4x4 band neighbourhood takes eight shared-memory loads
    // (the two middle rows: left, aligned pair, right; the outer rows: the pair), the four texels go out as two 16-byte stores.
    uint2* __restrict__ out = a.tex8 + (long long)b * a.Pt;
    const int row_quads = a.tw << 2;
#pragma unroll 1
    for (int tyl = 0; tyl < R / 4; ++tyl) {
        const int ty = (y0 >> 2) + tyl;
        if (ty >= a.th) break;
        for (int q = threadIdx.x; q < row_quads; q += WARPS * 32) {
            const int tx = q >> 2, sub = q & 3;
            const int x = (tx << 2) | ((sub & 1) << 1), ly = (tyl << 2) | (sub & 2), y = y0 + ly;        // top-left pixel of the quad (x even)
            uint2 t[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) t[k] = make_uint2(DVO_TEX_ESCAPE, 0u);
            if (x < w && y < h) {
                const unsigned short* br = band + (ly + 1) * bp + x;                                    // band row of image row y
                // v[r][c]: rows y-1 .. y+2, columns x-1 .. x+2 (corners unused); out-of-image taps are never selected below
                int v[4][4];
                const bool has_r = (x + 1 < w), has_b = (y + 1 < h);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const unsigned short* p = br + (r - 1) * bp;
                    const unsigned pr = *reinterpret_cast<const unsigned*>(p);                          // x is even and bp is even: 4-byte aligned
                    v[r][1] = (int)(pr & 0xFFFFu); v[r][2] = (int)(pr >> 16);
                    if (r == 1 || r == 2) { v[r][0] = (x > 0) ? (int)p[-1] : 0; v[r][3] = (x + 2 < w) ? (int)p[2] : 0; }
                    else { v[r][0] = 0; v[r][3] = 0; }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int dy = k >> 1, dx = k & 1;
                    const int px = x + dx, py = y + dy;
                    if ((dx && !has_r) || (dy && !has_b)) continue;
                    const int c = v[1 + dy][1 + dx];
                    const bool bx = (px == 0 || px == w - 1), by = (py == 0 || py == h - 1);
                    const int l = bx ? c : v[1 + dy][dx], r = bx ? c : v[1 + dy][2 + dx], u = by ? c : v[dy][1 + dx], d = by ? c : v[2 + dy][1 + dx];
                    const int dl = l - c, dr = r - c, du = u - c, dd = d - c;
                    const int lo = min(min(dl, dr), min(du, dd)), hi = max(max(dl, dr), max(du, dd));
                    if (max(max(max(c, l), max(r, u)), d) < 65535 && lo >= -512 && hi <= 511) {
                        t[k].x = (unsigned)c | (((unsigned)dl & 0x3FFu) << 16);
                        t[k].y = ((unsigned)dr & 0x3FFu) | (((unsigned)du & 0x3FFu) << 10) | (((unsigned)dd & 0x3FFu) << 20);
                    }
                }
            }
            uint4* o = reinterpret_cast<uint4*>(out + (long long)ty * (row_quads << 2) + ((long long)q << 2));
            o[0] = make_uint4(t[0].x, t[0].y, t[1].x, t[1].y);
            o[1] = make_uint4(t[2].x, t[2].y, t[3].x, t[3].y);
        }
    }
}

// shared memory the fused kernel needs for a level of width w (the sparse variant is the larger one)
static size_t edt_pack_smem(int warps, int R, int w, bool sparse) {
    const int bp = (w + 1) & ~1;
    return (size_t)(R + 2) * bp * sizeof(unsigned short) + (size_t)warps * (sparse ? (w + bp) : edt_window_scratch_ints(w)) * sizeof(int);
}

template <int WARPS, int R>
static int launch_edt_pack_t(dvo_ctx* c, int first, int count) {
    const PyrGeom& g = c->geom;
    if (edt_pack_smem(WARPS, R, g.w[0], true) > c->smem_optin) {          // image too wide for a band in shared memory: unfused kernels
        const int rc = launch_edt_rows(c, first, count);
        return rc ? rc : launch_pack(c, first, count);
    }
    DVO_CUDA(cudaMemsetAsync(c->maxd2 + (size_t)first * g.L, 0, sizeof(unsigned) * (size_t)count * g.L, c->stream));
    for (int l = 0; l < g.L; ++l) {
        EdtPackArgs a; a.gcol = c->gcol + g.off[l]; a.d2 = c->d2 + g.off[l]; a.tex8 = c->tex8 + g.offt[l]; a.maxd2 = c->maxd2 + l;
        a.w = g.w[l]; a.h = g.h[l]; a.P = g.P[l]; a.Pt = g.Pt[l]; a.tw = g.tw[l]; a.th = (g.h[l] + 3) >> 2; a.L = g.L; a.first = first;
        const unsigned* ne = c->nedge + (size_t)DVO_FRAME_NOW * g.Bmax * g.L + l;
        const int w = g.w[l], bp = (w + 1) & ~1;
        dim3 grid((g.h[l] + R - 1) / R, count);
        const size_t band = (size_t)(R + 2) * bp * sizeof(unsigned short);
        const size_t smem_d = band + (size_t)WARPS * edt_window_scratch_ints(w) * sizeof(int), smem_s = band + (size_t)WARPS * (w + bp) * sizeof(int);
        static size_t opted_d = 0, opted_s = 0;          // largest opt-in so far (per instantiation; one device per process)
        if (smem_d > 48 * 1024 && smem_d > opted_d) { DVO_CUDA(cudaFuncSetAttribute(edt_pack_kernel<WARPS, R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_d)); opted_d = smem_d; }
        if (smem_s > 48 * 1024 && smem_s > opted_s) { DVO_CUDA(cudaFuncSetAttribute(edt_pack_kernel<WARPS, R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s)); opted_s = smem_s; }
        edt_pack_kernel<WARPS, R, false><<<grid, WARPS * 32, smem_d, c->stream>>>(a, ne);
        edt_pack_kernel<WARPS, R, true><<<grid, WARPS * 32, smem_s, c->stream>>>(a, ne);
        c->launches += 2;
    }
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

int launch_edt_pack(dvo_ctx* c, int first, int count) {
    // band height (640x480, 1024 pairs, packed 16-bit window): 20 rows + 2 halo with 11 warps (73 KB of shared memory, three CTAs per
    // SM) 2.65 ms; 24 rows x 13 warps (86 KB, two CTAs per SM) 2.82; 12 x 7: 2.78; 16 x 9: 2.80; 28 x 10: 2.82; also 16 x 8: 2.70,
    // 16 x 10: 2.76, 20 x 9 / 10 / 12 / 14: 2.83 / 2.73 / 2.96 / 3.10.  (With the 32-bit window 24 x 13 was best: 3.83 against 3.85 -
    // 4.00, and 4.41 for the unfused kernels.)  At 1280x720 a band costs twice the shared memory and the fused kernel is no faster
    // than the unfused pair: wide images stay unfused.
    if (c->geom.w[0] > 800) { const int rc = launch_edt_rows(c, first, count); return rc ? rc : launch_pack(c, first, count); }
    return launch_edt_pack_t<11, 20>(c, first, count);
}

// inspection (dvo_get_level_buffer D2): the dense d2 image of one slot / level from the packed texels
// (centre value) and, where a texel is escaped, from the sparse 32-bit image
__global__ void __launch_bounds__(256) d2_from_texels_kernel(const uint2* __restrict__ tex8, const int32_t* __restrict__ d2g, int32_t* __restrict__ out, int w, int h, int tw) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= w * h) return;
    const int y = i / w, x = i - y * w;
    const unsigned w0 = tex8[tex_index(x, y, tw)].x;
    out[i] = ((int)w0 < 0) ? d2g[i] : (int)(w0 & 0xFFFFu);
}

int launch_d2_from_texels(dvo_ctx* c, int slot, int level, int32_t* d_out) {
    const PyrGeom& g = c->geom;
    d2_from_texels_kernel<<<(g.P[level] + 255) / 256, 256, 0, c->stream>>>(c->tex8 + tex_at(g, level, slot), c->d2 + lvl_at(g, level, slot), d_out,
                                                                         g.w[level], g.h[level], g.tw[level]);
    c->launches++;
    DVO_CUDA(cudaGetLastError());
    return DVO_OK;
}

// =====================================================================================================
// setPrevFrameAsRefFrame (src/SolveDVO.cpp:561-584): im_r = p_now_framemono, dim_r = p_now_depth.  The previous now
// frame's level-0 images (saved by dvo_set_frames) become the reference frame's level 0; the caller rebuilds the
// reference pyramid, edges and point list exactly as the reference does (computeDistTransfrmOfRef, preProcessRefFrame).
// =====================================================================================================
__global__ void __launch_bounds__(256) promote_masked_kernel(PyrGeom g, const uint8_t* __restrict__ prev_gray, const uint16_t* __restrict__ prev_depth,
                                                             uint8_t* __restrict__ gray, uint16_t* __restrict__ depth, int first,
                                                             const unsigned char* __restrict__ active) {
    const int b = first + blockIdx.y;
    if (!active[b]) return;
    const int P0 = g.P[0];
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) * 4;          // P0 is a multiple of 4 for every supported size? no: tail handled below
    const long long src = (long long)P0 * b, dst = lvl_at(g, 0, b);
    for (int k = q; k < min(q + 4, P0); ++k) { gray[dst + k] = prev_gray[src + k]; depth[dst + k] = prev_depth[src + k]; }
}

int launch_promote(dvo_ctx* c, int first, int count) {
    const PyrGeom& g = c->geom;
    if (!c->prev_gray) { dvo_set_error("promote: context was created without keep_now_depth"); return DVO_ERR_STATE; }
    for (int i = first; i < first + count; ++i)
        if (!c->prev_valid[i]) { dvo_set_error("promote: slot %d has no previous now frame (isPrevFrameAvailable)", i); return DVO_ERR_STATE; }
    const size_t P0 = g.P[0];
    if (c->active) {
        dim3 grid((unsigned)((P0 + 1023) / 1024), (unsigned)count);
        promote_masked_kernel<<<grid, 256, 0, c->stream>>>(g, c->prev_gray, c->prev_depth, c->gray[0], c->depth[0], first, c->active);
        c->launches++;
        DVO_CUDA(cudaGetLastError());
        return DVO_OK;
    }
    DVO_CUDA(cudaMemcpyAsync(c->gray[0] + lvl_at(g, 0, first), c->prev_gray + P0 * first, P0 * count, cudaMemcpyDeviceToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->depth[0] + lvl_at(g, 0, first), c->prev_depth + P0 * first, P0 * count * 2, cudaMemcpyDeviceToDevice, c->stream));
    return DVO_OK;
}
