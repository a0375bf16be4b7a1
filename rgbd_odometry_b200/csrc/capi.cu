// capi.cu -- the extern "C" boundary declared in include/dvo_b200.h: context lifetime, device memory arena,
// host<->device staging and the stage sequencing.  No CPU compute path exists here: every entry point either
// launches the sm_100a kernels or fails.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <new>
#include <vector>

#include "common.cuh"

static thread_local char g_err[512] = "";

void dvo_set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}

// cv::resize output size: cvRound(dim * 2^-level), round half to even (SURVEY Appendix B.4)
static int level_dim(int dim, int level) { return (int)nearbyint((double)dim * ldexp(1.0, -level)); }

namespace {
struct StageTimer {
    dvo_ctx* c; int stage; bool on;
    StageTimer(dvo_ctx* c_, int s) : c(c_), stage(s), on(c_->timing) { if (on) cudaEventRecord(c->ev_a, c->stream); }
    ~StageTimer() {
        if (!on) return;
        cudaEventRecord(c->ev_b, c->stream); cudaEventSynchronize(c->ev_b);
        float ms = 0.f; cudaEventElapsedTime(&ms, c->ev_a, c->ev_b); c->stage_ms[stage] += ms;
    }
};
bool range_ok(dvo_ctx* c, int first, int count) { return c && first >= 0 && count >= 0 && first + count <= c->cfg.max_batch; }
// make the context stream wait for whatever dvo_process left running on the internal streams
int join_aux(dvo_ctx* c) {
    if (!c || !c->aux_pending) return DVO_OK;
    c->aux_pending = false;
    for (int k = 0; k < 2; ++k) DVO_CUDA(cudaStreamWaitEvent(c->stream, c->ev_aux_done[k], 0));
    return DVO_OK;
}
}  // namespace

extern "C" {

const char* dvo_last_error(void) { return g_err; }

int dvo_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// inside dvo_create: any CUDA failure after the context object exists releases everything acquired so far
#define CREATE_CUDA(call)                                                                       \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dvo_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            dvo_destroy(c);                                                                     \
            return DVO_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

int dvo_create(const dvo_config* cfg, dvo_ctx** out) {
    if (!cfg || !out) { dvo_set_error("dvo_create: null argument"); return DVO_ERR_ARG; }
    // max_batch <= 65535: several kernels carry the slot index in gridDim.y / gridDim.z
    if (cfg->width < 8 || cfg->height < 8 || cfg->levels < 1 || cfg->levels > DVO_MAX_LEVELS || cfg->max_batch < 1 || cfg->max_batch > 65535 ||
        cfg->width >= DVO_EDT_INF_1D || cfg->height >= DVO_EDT_INF_1D) {
        dvo_set_error("dvo_create: bad config %dx%d levels=%d max_batch=%d", cfg->width, cfg->height, cfg->levels, cfg->max_batch);
        return DVO_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        dvo_set_error("dvo_create: no usable CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
        cudaGetLastError();
        return DVO_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { dvo_set_error("dvo_create: device %d out of range (%d devices)", cfg->device, ndev); return DVO_ERR_ARG; }
    DVO_CUDA(cudaSetDevice(cfg->device));
    dvo_ctx* c = new (std::nothrow) dvo_ctx();
    if (!c) return DVO_ERR_NOMEM;
    c->cfg = *cfg;
    PyrGeom& g = c->geom;
    g.L = cfg->levels; g.Bmax = cfg->max_batch;
    long long acc = 0; int maxP = 0;
    for (int l = 0; l < g.L; ++l) {
        g.w[l] = level_dim(cfg->width, l); g.h[l] = level_dim(cfg->height, l);
        if (g.w[l] < 2 || g.h[l] < 2) { dvo_set_error("dvo_create: level %d is %dx%d (too small)", l, g.w[l], g.h[l]); dvo_destroy(c); return DVO_ERR_ARG; }
        g.P[l] = g.w[l] * g.h[l]; g.off[l] = acc * g.Bmax; acc += g.P[l];
        if (g.P[l] > maxP) maxP = g.P[l];
    }
    g.total = acc * g.Bmax;
    long long acct = 0;
    for (int l = 0; l < g.L; ++l) {
        g.tw[l] = (g.w[l] + 3) >> 2; g.Pt[l] = g.tw[l] * ((g.h[l] + 3) >> 2) * 16;
        g.offt[l] = acct * g.Bmax; acct += g.Pt[l];
    }
    g.total_t = acct * g.Bmax;
    cudaDeviceProp prop;
    CREATE_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    c->solve_shape = (cfg->max_batch <= c->sm_count) ? 512 : 256;
    CREATE_CUDA(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CREATE_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 16; ++i) CREATE_CUDA(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&c->ev_entry, cudaEventDisableTiming));
    for (int k = 0; k < 2; ++k) {
        CREATE_CUDA(cudaStreamCreateWithFlags(&c->aux[k], cudaStreamNonBlocking));
        CREATE_CUDA(cudaEventCreateWithFlags(&c->ev_pre[k], cudaEventDisableTiming));
        CREATE_CUDA(cudaEventCreateWithFlags(&c->ev_aux_done[k], cudaEventDisableTiming));
    }
    CREATE_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreate(&c->ev_a));
    CREATE_CUDA(cudaEventCreate(&c->ev_b));

    const size_t T = (size_t)g.total, B = (size_t)g.Bmax;
    int rc = DVO_OK;
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    for (int f = 0; f < 2; ++f) { A(c->gray[f].reserve(T)); A(c->edge[f].reserve(T)); }
    A(c->depth[0].reserve(T));
    if (cfg->keep_now_depth) { A(c->depth[1].reserve(T)); A(c->prev_gray.reserve(B * (size_t)g.P[0])); A(c->prev_depth.reserve(B * (size_t)g.P[0])); }
    A(c->gcol.reserve(T)); A(c->d2.reserve(T));
    A(c->tex8.reserve((size_t)g.total_t));
    A(c->ptsX.reserve(T)); A(c->ptsY.reserve(T)); A(c->ptsZ.reserve(T)); A(c->ptsPix.reserve(T));
    A(c->npts.reserve(B * g.L)); A(c->solve_order.reserve(B)); A(c->seq_mask.reserve(B)); A(c->seq_state.reserve(B)); A(c->nedge.reserve(2 * B * g.L)); A(c->maxd2.reserve(B * g.L));
    A(c->pose0.reserve(B * 12)); A(c->pose.reserve(B * 12)); A(c->info.reserve(B));
    if (cfg->trace_iters > 0) A(c->trace.reserve(B * g.L * cfg->trace_iters * DVO_TRACE_DOUBLES));
    A(c->energy.reserve(B * g.L * DVO_ENERGY_ITERS));
    // candidate / edge bitmaps: sobel_nms_kernel -> canny_kernel (which keeps working in them when they do not fit in shared memory)
    canny_scratch_layout(g, c->bm_off, c->bm_words, &c->bitmap_scratch_words);
    A(c->bitmap_scratch.reserve(c->bitmap_scratch_words * B * 2));
    if (rc != DVO_OK) { dvo_destroy(c); return rc; }
    c->now_valid.reset(new (std::nothrow) unsigned char[B]());
    c->prev_valid.reset(new (std::nothrow) unsigned char[B]());
    if (!c->now_valid || !c->prev_valid) { dvo_set_error("dvo_create: out of host memory"); dvo_destroy(c); return DVO_ERR_NOMEM; }
    CREATE_CUDA(cudaMemsetAsync(c->npts, 0, sizeof(int) * B * g.L, c->stream));
    CREATE_CUDA(cudaMemsetAsync(c->bitmap_scratch, 0, sizeof(uint32_t) * c->bitmap_scratch_words * B * 2, c->stream));   // the bitmaps' zero borders are never written
    CREATE_CUDA(cudaMemsetAsync(c->nedge, 0, sizeof(unsigned) * 2 * B * g.L, c->stream));
    CREATE_CUDA(cudaMemsetAsync(c->maxd2, 0, sizeof(unsigned) * B * g.L, c->stream));
    CREATE_CUDA(cudaMemsetAsync(c->info, 0, sizeof(dvo_pair_info) * B, c->stream));
    dvo_set_initial_pose(c, 0, g.Bmax, nullptr, DVO_MEM_HOST);
    CREATE_CUDA(cudaStreamSynchronize(c->stream));
    *out = c;
    return DVO_OK;
}

int dvo_destroy(dvo_ctx* c) {
    if (!c) return DVO_OK;
    cudaSetDevice(c->cfg.device);
    if (c->own_stream) cudaStreamSynchronize(c->own_stream);
    for (int k = 0; k < 2; ++k) {
        if (c->seq_ev_ready[k]) cudaEventDestroy(c->seq_ev_ready[k]);
        if (c->seq_ev_free[k]) cudaEventDestroy(c->seq_ev_free[k]);
    }
    if (c->ev_a) cudaEventDestroy(c->ev_a);
    if (c->ev_b) cudaEventDestroy(c->ev_b);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    for (int k = 0; k < 2; ++k) {
        if (c->aux[k]) { cudaStreamSynchronize(c->aux[k]); cudaStreamDestroy(c->aux[k]); }
        if (c->ev_pre[k]) cudaEventDestroy(c->ev_pre[k]);
        if (c->ev_aux_done[k]) cudaEventDestroy(c->ev_aux_done[k]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    for (int i = 0; i < 16; ++i) if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
    if (c->ev_entry) cudaEventDestroy(c->ev_entry);
    delete c;                                            // the buffers free themselves
    return DVO_OK;
}

int dvo_set_stream(dvo_ctx* c, void* s) {
    if (!c) return DVO_ERR_ARG;
    { int rc = join_aux(c); if (rc) return rc; }
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return DVO_OK;
}

int dvo_synchronize(dvo_ctx* c) {
    if (!c) return DVO_ERR_ARG;
    { int rc = join_aux(c); if (rc) return rc; }
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_set_intrinsics(dvo_ctx* c, float fx, float fy, float cx, float cy) {
    if (!c) return DVO_ERR_ARG;
    c->K.fx = fx; c->K.fy = fy; c->K.cx = cx; c->K.cy = cy; c->haveK = true;
    return DVO_OK;
}

}  // extern "C"

// Validation and p_now_* bookkeeping shared by dvo_set_frames / dvo_set_frames_raw.  Every argument is checked before any
// copy is enqueued or any flag changes, so an error return leaves the context as it was.
static int begin_set_frames(dvo_ctx* c, const char* who, int frame, int first, int count, bool have_gray, bool have_depth) {
    if (!range_ok(c, first, count) || (frame != DVO_FRAME_REF && frame != DVO_FRAME_NOW) || !have_gray) { dvo_set_error("%s: bad argument", who); return DVO_ERR_ARG; }
    if (frame == DVO_FRAME_REF && !have_depth) { dvo_set_error("%s: the reference frame needs depth", who); return DVO_ERR_ARG; }
    bool rotate = false;
    if (frame == DVO_FRAME_NOW && c->prev_gray) {
        if (!have_depth) { dvo_set_error("%s: a context with keep_now_depth needs the now frame's depth", who); return DVO_ERR_ARG; }
        bool any = false, all = true;
        for (int i = first; i < first + count; ++i) { any |= c->now_valid[i] != 0; all &= c->now_valid[i] != 0; }
        if (any && !all) { dvo_set_error("%s: slots [%d,%d) mix first and subsequent now frames", who, first, first + count); return DVO_ERR_STATE; }
        rotate = all && count > 0;
    }
    const size_t P0 = c->geom.P[0];
    if (rotate) {
        // setRcvdFrameAsNowFrame keeps the outgoing now frame as p_now_* (src/SolveDVO.cpp:594-600)
        DVO_CUDA(cudaMemcpyAsync(c->prev_gray + P0 * first, c->gray[1] + lvl_at(c->geom, 0, first), P0 * count, cudaMemcpyDeviceToDevice, c->stream));
        DVO_CUDA(cudaMemcpyAsync(c->prev_depth + P0 * first, c->depth[1] + lvl_at(c->geom, 0, first), P0 * count * 2, cudaMemcpyDeviceToDevice, c->stream));
        for (int i = first; i < first + count; ++i) c->prev_valid[i] = 1;
    }
    if (frame == DVO_FRAME_NOW) for (int i = first; i < first + count; ++i) c->now_valid[i] = 1;
    return DVO_OK;
}

extern "C" {

int dvo_set_frames(dvo_ctx* c, int frame, int first, int count, const uint8_t* gray, const uint16_t* depth, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    { const int rc = begin_set_frames(c, "dvo_set_frames", frame, first, count, gray != nullptr, depth != nullptr); if (rc) return rc; }
    StageTimer t(c, DVO_STAGE_H2D);
    const size_t P0 = c->geom.P[0];
    const cudaMemcpyKind k = mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    DVO_CUDA(cudaMemcpyAsync(c->gray[frame] + lvl_at(c->geom, 0, first), gray, P0 * count, k, c->stream));
    if (depth && c->depth[frame])
        DVO_CUDA(cudaMemcpyAsync(c->depth[frame] + lvl_at(c->geom, 0, first), depth, P0 * count * sizeof(uint16_t), k, c->stream));
    return DVO_OK;
}

int dvo_set_frames_raw(dvo_ctx* c, int frame, int first, int count, const uint8_t* bgr, const float* depth_m, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    { const int rc = begin_set_frames(c, "dvo_set_frames_raw", frame, first, count, bgr != nullptr, depth_m != nullptr); if (rc) return rc; }
    if (count == 0) return DVO_OK;
    StageTimer t(c, DVO_STAGE_H2D);
    const size_t P0 = c->geom.P[0];
    const uint8_t* d_bgr = bgr; const float* d_dm = depth_m;
    if (mem != DVO_MEM_DEVICE) {
        // staging sized for the largest range seen so far; a copy still in flight may read the buffers a growth replaces
        if (c->raw_bgr.n < (size_t)count * P0 * 3) DVO_CUDA(cudaStreamSynchronize(c->stream));
        int rc = c->raw_bgr.reserve((size_t)count * P0 * 3);
        if (rc == DVO_OK) rc = c->raw_depth.reserve((size_t)count * P0);
        if (rc) return rc;
        DVO_CUDA(cudaMemcpyAsync(c->raw_bgr, bgr, P0 * count * 3, cudaMemcpyHostToDevice, c->stream));
        if (depth_m) DVO_CUDA(cudaMemcpyAsync(c->raw_depth, depth_m, P0 * count * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        d_bgr = c->raw_bgr; d_dm = depth_m ? c->raw_depth.get() : nullptr;
    }
    return launch_ingest_raw(c, frame, first, count, d_bgr, d_dm);
}

int dvo_promote_now_to_ref(dvo_ctx* c, int first, int count) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count)) return DVO_ERR_ARG;
    return launch_promote(c, first, count);
}

int dvo_build_pyramids(dvo_ctx* c, int first, int count, int frames_mask) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count)) { dvo_set_error("dvo_build_pyramids: bad range"); return DVO_ERR_ARG; }
    if (count == 0) return DVO_OK;
    StageTimer t(c, DVO_STAGE_PYRAMID);
    return launch_pyramid(c, first, count, frames_mask);
}

int dvo_prepare(dvo_ctx* c, int first, int count, int frames_mask) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count)) { dvo_set_error("dvo_prepare: bad range"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_prepare: intrinsics not set (SolveDVO asserts isCameraIntrinsicsAvailable)"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    int rc;
    { StageTimer t(c, DVO_STAGE_CANNY); rc = launch_canny(c, first, count, frames_mask); if (rc) return rc; }
    if (frames_mask & 2) {       // EDT rows + texels: the stage slot of the row pass times both (DVO_STAGE_NORMGRAD stays 0)
        StageTimer t(c, DVO_STAGE_EDT_ROWS); rc = launch_edt_pack(c, first, count); if (rc) return rc;
    }
    return DVO_OK;
}

int dvo_set_initial_pose(dvo_ctx* c, int first, int count, const double* R9T3, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count)) return DVO_ERR_ARG;
    if (R9T3) {
        DVO_CUDA(cudaMemcpyAsync(c->pose0 + 12 * (size_t)first, R9T3, sizeof(double) * 12 * count,
                                 mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
        if (mem != DVO_MEM_DEVICE) DVO_CUDA(cudaStreamSynchronize(c->stream));
    } else {
        std::vector<double> id((size_t)12 * count, 0.0);
        for (int i = 0; i < count; ++i) { id[12 * (size_t)i] = 1.0; id[12 * (size_t)i + 4] = 1.0; id[12 * (size_t)i + 8] = 1.0; }
        DVO_CUDA(cudaMemcpyAsync(c->pose0 + 12 * (size_t)first, id.data(), sizeof(double) * 12 * count, cudaMemcpyHostToDevice, c->stream));
        DVO_CUDA(cudaStreamSynchronize(c->stream));
    }
    return DVO_OK;
}

int dvo_run(dvo_ctx* c, int first, int count, const dvo_solver_params* p) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count) || !p) { dvo_set_error("dvo_run: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_run: intrinsics not set"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    StageTimer t(c, DVO_STAGE_SOLVE);
    return launch_solve(c, first, count, p);
}

// pyramids + Canny / EDT + texels + solve of one slot range on the CURRENT c->stream, no stage timers, no join
static int process_range(dvo_ctx* c, int first, int count, const dvo_solver_params* p, cudaEvent_t pre_done) {
    int rc;
    if ((rc = launch_pyramid(c, first, count, 3))) return rc;
    if ((rc = launch_canny(c, first, count, 3))) return rc;
    if ((rc = launch_edt_pack(c, first, count))) return rc;
    if (pre_done) DVO_CUDA(cudaEventRecord(pre_done, c->stream));
    return launch_solve(c, first, count, p);
}

int dvo_process(dvo_ctx* c, int first, int count, const dvo_solver_params* p, double* d_poses) {
    if (!range_ok(c, first, count) || !p) { dvo_set_error("dvo_process: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_process: intrinsics not set"); return DVO_ERR_STATE; }
    if (count == 0) return DVO_OK;
    // Per-stage timers synchronise, and a half batch must still fill the chip for the overlap to pay: otherwise run staged.
    if (c->timing || count < 4 * c->sm_count) {
        int rc = join_aux(c); if (rc) return rc;
        if ((rc = dvo_build_pyramids(c, first, count, 3))) return rc;
        if ((rc = dvo_prepare(c, first, count, 3))) return rc;
        if ((rc = dvo_run(c, first, count, p))) return rc;
        if (d_poses) DVO_CUDA(cudaMemcpyAsync(d_poses, c->pose + 12 * (size_t)first, sizeof(double) * 12 * count, cudaMemcpyDeviceToDevice, c->stream));
        return DVO_OK;
    }
    // Fork: both internal streams start after everything issued on the context stream so far.  Half 1's preprocessing
    // additionally waits for half 0's, so it runs beside half 0's solve; each internal stream is in order with its own
    // work of the previous call, which is all the dependency there is (the halves own disjoint slots).
    // A call whose slot split differs from the one still in flight could touch slots the OTHER internal stream is working
    // on: join first (device-side) in that case.  With the same (first, count) every stream only meets its own slots.
    if (c->aux_pending && (c->proc_first != first || c->proc_count != count)) { const int rc = join_aux(c); if (rc) return rc; }
    c->proc_first = first; c->proc_count = count;
    DVO_CUDA(cudaEventRecord(c->ev_fork, c->stream));
    const cudaStream_t user = c->stream;
    const int n0 = count / 2;
    const int starts[2] = {first, first + n0}, counts[2] = {n0, count - n0};
    int rc = DVO_OK;
    for (int k = 0; k < 2 && rc == DVO_OK; ++k) {
        cudaError_t e = cudaStreamWaitEvent(c->aux[k], c->ev_fork, 0);
        if (e == cudaSuccess && k == 1) e = cudaStreamWaitEvent(c->aux[1], c->ev_pre[0], 0);
        if (e != cudaSuccess) { dvo_set_error("dvo_process: %s", cudaGetErrorString(e)); rc = DVO_ERR_CUDA; break; }
        c->stream = c->aux[k];
        rc = process_range(c, starts[k], counts[k], p, c->ev_pre[k]);
        if (rc == DVO_OK && d_poses && cudaMemcpyAsync(d_poses + 12 * (size_t)(starts[k] - first), c->pose + 12 * (size_t)starts[k], sizeof(double) * 12 * counts[k],
                                                       cudaMemcpyDeviceToDevice, c->aux[k]) != cudaSuccess) rc = DVO_ERR_CUDA;
        if (rc == DVO_OK && cudaEventRecord(c->ev_aux_done[k], c->aux[k]) != cudaSuccess) rc = DVO_ERR_CUDA;
    }
    c->stream = user;
    c->aux_pending = true;
    if (rc != DVO_OK) join_aux(c);
    return rc;
}

int dvo_join(dvo_ctx* c) {
    if (!c) return DVO_ERR_ARG;
    return join_aux(c);
}

int dvo_join_stream(dvo_ctx* c, void* s) {
    if (!c) return DVO_ERR_ARG;
    if (!c->aux_pending) return DVO_OK;
    for (int k = 0; k < 2; ++k) DVO_CUDA(cudaStreamWaitEvent((cudaStream_t)s, c->ev_aux_done[k], 0));
    return DVO_OK;
}

int dvo_get_poses(dvo_ctx* c, int first, int count, double* R9T3, dvo_pair_info* info, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count)) return DVO_ERR_ARG;
    StageTimer t(c, DVO_STAGE_D2H);
    const cudaMemcpyKind k = mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (R9T3) DVO_CUDA(cudaMemcpyAsync(R9T3, c->pose + 12 * (size_t)first, sizeof(double) * 12 * count, k, c->stream));
    if (info) DVO_CUDA(cudaMemcpyAsync(info, c->info + first, sizeof(dvo_pair_info) * count, k, c->stream));
    if (mem != DVO_MEM_DEVICE) DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// frame pairs per upload/compute pipeline stage in dvo_align_batch: 8 stages per 1024 pairs, 25.7 ms per pass against
// 27.2 (256), 30.2 (512), 33.3 (64)
constexpr int E2E_CHUNK = 128;

int dvo_align_batch(dvo_ctx* c, int count, const uint8_t* ref_gray, const uint16_t* ref_depth, const uint8_t* now_gray,
                    const uint16_t* now_depth, const dvo_solver_params* p, double* R9T3, dvo_pair_info* info) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!c || count < 0 || !ref_gray || !ref_depth || !now_gray || !p) { dvo_set_error("dvo_align_batch: bad argument"); return DVO_ERR_ARG; }
    if (!c->haveK) { dvo_set_error("dvo_align_batch: intrinsics not set"); return DVO_ERR_STATE; }
    const size_t P0 = c->geom.P[0];
    const int B = c->cfg.max_batch;
    const bool timing = c->timing;
    c->timing = false;                                   // the per-stage timers synchronise; keep the pipeline asynchronous
    int rc = DVO_OK;
    for (int done = 0; done < count && rc == DVO_OK; done += B) {
        const int n = (count - done < B) ? count - done : B;
        if ((rc = dvo_set_initial_pose(c, 0, n, nullptr, DVO_MEM_HOST))) break;
        // Uploads run on their own stream, chunk by chunk, so that the copy of chunk k+1 overlaps the kernels of chunk k.
        // Every chunk owns its slots, so no buffer is reused inside one pass over the context.
        cudaError_t e = cudaEventRecord(c->ev_entry, c->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(c->copy_stream, c->ev_entry, 0);
        if (e != cudaSuccess) { dvo_set_error("dvo_align_batch: %s", cudaGetErrorString(e)); rc = DVO_ERR_CUDA; break; }
        int nchunks = (n + E2E_CHUNK - 1) / E2E_CHUNK;
        if (nchunks > 16) nchunks = 16;
        const int chunk = (n + nchunks - 1) / nchunks;
        int k = 0;
        for (int c0 = 0; c0 < n && rc == DVO_OK; c0 += chunk, ++k) {
            const int m = (n - c0 < chunk) ? n - c0 : chunk;
            const size_t src = P0 * (size_t)(done + c0);
            const long long dst = lvl_at(c->geom, 0, c0);
            e = cudaMemcpyAsync(c->gray[0] + dst, ref_gray + src, P0 * m, cudaMemcpyHostToDevice, c->copy_stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(c->depth[0] + dst, ref_depth + src, P0 * m * 2, cudaMemcpyHostToDevice, c->copy_stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(c->gray[1] + dst, now_gray + src, P0 * m, cudaMemcpyHostToDevice, c->copy_stream);
            if (e == cudaSuccess && now_depth && c->depth[1])
                e = cudaMemcpyAsync(c->depth[1] + dst, now_depth + src, P0 * m * 2, cudaMemcpyHostToDevice, c->copy_stream);
            if (e == cudaSuccess) e = cudaEventRecord(c->ev_chunk[k], c->copy_stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(c->stream, c->ev_chunk[k], 0);
            if (e != cudaSuccess) { dvo_set_error("dvo_align_batch: %s", cudaGetErrorString(e)); rc = DVO_ERR_CUDA; break; }
            if ((rc = dvo_build_pyramids(c, c0, m, 3))) break;
            if ((rc = dvo_prepare(c, c0, m, 3))) break;
            if ((rc = dvo_run(c, c0, m, p))) break;
        }
        if (rc == DVO_OK)
            rc = dvo_get_poses(c, 0, n, R9T3 ? R9T3 + 12 * (size_t)done : nullptr, info ? info + done : nullptr, DVO_MEM_HOST);
    }
    c->timing = timing;
    return rc;
}

// ---- sequence mode: SolveDVO::loop (src/SolveDVO.cpp:1896-2373) for `nseq` independent sequences in lock step ----
}  // extern "C"

namespace {
// h(Sigma) = 3 (1 + ln 2 pi) + logdet(Sigma) / 2: differential entropy of a 6-D Gaussian pose estimate, in nats
__device__ __forceinline__ double pose_entropy(double logdet) { return 3.0 * (1.0 + log(2.0 * 3.14159265358979323846)) + 0.5 * logdet; }

// cinfo (entropy gate on, else null): per-frame dvo_cov_info [nseq][nframes], frame t holding the covariance of its first solve;
// frames before t hold their final covariance.  ent [nseq][nframes] receives the ratio at every frame the gate evaluates.
__global__ void seq_gate_kernel(int nseq, int nframes, int t, dvo_keyframe_policy pol, int finest, const dvo_pair_info* __restrict__ info,
                                const double* __restrict__ pose, double* __restrict__ pose0, int* __restrict__ lastRef,
                                unsigned char* __restrict__ mask, double* __restrict__ rel, int* __restrict__ kind, int* __restrict__ reason,
                                const dvo_cov_info* __restrict__ cinfo, double ent_thr, double* __restrict__ ent) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseq) return;
    const dvo_pair_info& I = info[s];
    const long long cur = (long long)s * nframes + t;
    int signal = 0, why = 0;
    if (pol.use_quality_gates) {                                                             // :2129-2151, in source order
        if (I.laplacian_b > pol.laplacian_thresh) { signal = 1; why = 2; }
        if (I.visible_ratio[finest] < pol.visible_ratio_thresh) { signal = 1; why = 3; }
        if (I.npts[finest] < pol.min_reprojections) { signal = 1; why = 4; }
    }
    if (cinfo && lastRef[s] != t - 1) {                                                      // entropy ratio (DVO-SLAM, Kerl et al. 2013)
        // h_ref: the final covariance of frame lastRef + 1, the first frame solved against the current key frame
        const double h_ref = pose_entropy(cinfo[(long long)s * nframes + lastRef[s] + 1].logdet);
        const double alpha = pose_entropy(cinfo[cur].logdet) / h_ref;                        // NaN when either covariance is degenerate
        ent[cur] = alpha;
        if (isfinite(alpha) && h_ref < 0.0 && alpha < ent_thr) { signal = 1; why = 6; }     // h_ref >= 0: the ratio means nothing
    }
    if (pol.keyframe_every > 0 && (t - lastRef[s]) == pol.keyframe_every) { signal = 1; why = 5; }   // :2155-2160
    if (signal && lastRef[s] != t - 1) {                                                     // :2192
        mask[s] = 1; lastRef[s] = t - 1;
        kind[cur - 1] = 2; reason[cur - 1] = why;                                            // gop.updateMostRecentToKeyFrame(reasonForChange)
        for (int k = 0; k < 12; ++k) pose0[12 * (long long)s + k] = (k == 0 || k == 4 || k == 8) ? 1.0 : 0.0;   // cR_64 = I, cT_64 = 0 (:2203-2204)
    } else {
        mask[s] = 0;
        for (int k = 0; k < 12; ++k) { const double v = pose[12 * (long long)s + k]; rel[12 * cur + k] = v; pose0[12 * (long long)s + k] = v; }
        kind[cur] = 0; reason[cur] = 0;                                                      // gop.pushAsOrdinaryFrame (:2232)
    }
}
__global__ void seq_finish_kernel(int nseq, int nframes, int t, const unsigned char* __restrict__ mask, const double* __restrict__ pose,
                                  double* __restrict__ pose0, double* __restrict__ rel, int* __restrict__ kind, int* __restrict__ reason) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseq || !mask[s]) return;
    const long long cur = (long long)s * nframes + t;
    for (int k = 0; k < 12; ++k) { const double v = pose[12 * (long long)s + k]; rel[12 * cur + k] = v; pose0[12 * (long long)s + k] = v; }
    kind[cur] = 0; reason[cur] = 0;                                                          // pushAsOrdinaryFrame after the re-run (:2224)
}
__global__ void seq_init_kernel(int nseq, int nframes, double* __restrict__ pose0, int* __restrict__ lastRef, double* __restrict__ rel,
                                int* __restrict__ kind, int* __restrict__ reason) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseq) return;
    lastRef[s] = 0;
    for (int k = 0; k < 12; ++k) { const double v = (k == 0 || k == 4 || k == 8) ? 1.0 : 0.0; pose0[12 * (long long)s + k] = v; rel[12 * (long long)s * nframes + k] = v; }
    kind[(long long)s * nframes] = 1; reason[(long long)s * nframes] = 1;                    // gop.pushAsKeyFrame(nFrame, 1, I, 0) (:2016)
}

// One loop for both entry points.  Frame 0 is the first reference / key frame (:2013-2017); every later frame is aligned against
// the current reference with the previous frame's pose as the initial guess (:1931-1932, :2097-2104); a key-frame signal makes the
// PREVIOUS frame the reference, resets the pose and solves the frame again (:2155-2233).  Everything between frames stays on the
// device: poses, statistics, the per-slot decision (seq_gate_kernel) and the record of relative poses / kinds / reasons.
//
// Uploads are pipelined: frame t+1 of every sequence travels on the copy stream into one of two staging buffers (one strided
// 2-D copy per image plane instead of nseq small ones) while frame t is being solved; the compute stream then moves it into
// the level-0 regions with a device-to-device copy (after saving the outgoing now frame as p_now_*, :594-600).
//
// With the periodic rule alone (the shipped policy) the host knows the switch frames, so (a) the masked switch pass is only
// launched at those frames and (b) the solve against the outgoing key frame, whose result the reference discards
// (:2210-2227), is skipped.  With the quality gates the decision depends on that solve, so it runs and every frame from t = 2
// on is followed by the masked pass (its kernels return at once for unflagged slots).
//
// Covariances (cov: dvo_run_sequences_cov / _entropy): after each frame's final solve one cov_kernel launch evaluates every slot at
// its final relative pose, on the reference it was finally solved against, into the device record at frame t.
//
// Entropy gate (ent_thr > 0, dvo_run_sequences_entropy): the decision depends on the first solve's covariance, so the loop runs like
// the quality-gate loop, and the covariance launch moves before the gate: first solve, cov_kernel over every slot (record and
// dvo_cov_info of frame t), gate, masked switch pass, masked cov_kernel for the re-solved slots only.  The other slots' first-solve
// records already are their final ones.
int run_sequences_core(dvo_ctx* c, const char* who, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem,
                       const dvo_solver_params* p, const dvo_keyframe_policy* pol, double* rel_poses, int* kind, int* reason,
                       double* global_poses, bool cov, double* rel_cov, double* global_cov, double ent_thr = 0.0,
                       double* entropy_ratio = nullptr) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!c || nseq < 1 || nseq > c->cfg.max_batch || nframes < 1 || !gray || !depth || !p || !pol || !rel_poses || !kind || (global_cov && !cov) ||
        isnan(ent_thr)) {
        dvo_set_error("%s: bad argument", who); return DVO_ERR_ARG;
    }
    const bool entropy_on = ent_thr > 0.0;
    if (!c->prev_gray) { dvo_set_error("%s: create the context with keep_now_depth = 1", who); return DVO_ERR_STATE; }
    if (!c->haveK) { dvo_set_error("%s: intrinsics not set", who); return DVO_ERR_STATE; }
    int finest = -1;
    for (int l = 0; l < c->geom.L; ++l) if (p->iters[l] > 0) { finest = l; break; }
    if (finest < 0) { dvo_set_error("%s: no level has iterations", who); return DVO_ERR_ARG; }
    const size_t P0 = c->geom.P[0], n = (size_t)nseq * nframes;
    const bool host_in = (mem != DVO_MEM_DEVICE);
    int rc = DVO_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == DVO_OK) { dvo_set_error("%s: %s", who, cudaGetErrorString(e)); rc = DVO_ERR_CUDA; } return rc != DVO_OK; };

    // ---- buffers: record of the run (device), staging for the uploads -- owned by the context, grown on demand, reused across calls
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    A(c->seq_rel.reserve(12 * n)); A(c->seq_kind.reserve(n)); A(c->seq_reason.reserve(n));
    if (host_in)
        for (int k = 0; k < 2 && rc == DVO_OK; ++k) {
            A(c->seq_stage_g[k].reserve(P0 * nseq)); A(c->seq_stage_d[k].reserve(P0 * nseq));
            if (!c->seq_ev_ready[k]) fail(cudaEventCreateWithFlags(&c->seq_ev_ready[k], cudaEventDisableTiming));
            if (!c->seq_ev_free[k]) fail(cudaEventCreateWithFlags(&c->seq_ev_free[k], cudaEventDisableTiming));
        }
    if (cov) { A(c->seq_cov.reserve(36 * n)); A(c->seq_cov_info.reserve(n)); }
    if (entropy_on) A(c->seq_ent.reserve(n));
    if (rc != DVO_OK) return rc;
    double* d_rel = c->seq_rel; int* d_kind = c->seq_kind; int* d_reason = c->seq_reason; double* d_glob = nullptr;
    uint8_t* stage_g[2] = {c->seq_stage_g[0], c->seq_stage_g[1]}; uint16_t* stage_d[2] = {c->seq_stage_d[0], c->seq_stage_d[1]};
    cudaEvent_t ev_ready[2] = {c->seq_ev_ready[0], c->seq_ev_ready[1]}, ev_free[2] = {c->seq_ev_free[0], c->seq_ev_free[1]};
    fail(cudaMemsetAsync(d_rel, 0, sizeof(double) * 12 * n, c->stream));
    fail(cudaMemsetAsync(d_kind, 0, sizeof(int) * n, c->stream));
    fail(cudaMemsetAsync(d_reason, 0, sizeof(int) * n, c->stream));
    if (cov) fail(cudaMemsetAsync(c->seq_cov, 0, sizeof(double) * 36 * n, c->stream));              // frame 0 anchors the chain: zeros
    if (entropy_on) fail(cudaMemsetAsync(c->seq_ent, 0xff, sizeof(double) * n, c->stream));      // all-ones: NaN where the gate is not evaluated
    if (host_in) { fail(cudaEventRecord(c->ev_entry, c->stream)); fail(cudaStreamWaitEvent(c->copy_stream, c->ev_entry, 0)); }

    // frame t of every sequence: host -> staging buffer t & 1 on the copy stream
    bool staged_before[2] = {false, false};
    auto upload = [&](int t) {
        if (!host_in || t >= nframes || rc != DVO_OK) return;
        const int k = t & 1;
        if (staged_before[k]) fail(cudaStreamWaitEvent(c->copy_stream, ev_free[k], 0));
        fail(cudaMemcpy2DAsync(stage_g[k], P0, gray + (size_t)t * P0, (size_t)nframes * P0, P0, nseq, cudaMemcpyHostToDevice, c->copy_stream));
        fail(cudaMemcpy2DAsync(stage_d[k], P0 * 2, depth + (size_t)t * P0, (size_t)nframes * P0 * 2, P0 * 2, nseq, cudaMemcpyHostToDevice, c->copy_stream));
        fail(cudaEventRecord(ev_ready[k], c->copy_stream));
        staged_before[k] = true;
    };
    // staged (or device-resident) frame t -> level-0 regions of `frame` on the compute stream
    auto ingest = [&](int frame, int t) {
        if (rc != DVO_OK) return;
        uint8_t* dg = c->gray[frame] + lvl_at(c->geom, 0, 0); uint16_t* dd = c->depth[frame] + lvl_at(c->geom, 0, 0);
        if (frame == DVO_FRAME_NOW && c->now_valid[0]) {                                     // setRcvdFrameAsNowFrame keeps the outgoing now frame (:594-600)
            if (rc == DVO_OK) rc = launch_copy_bytes(c, c->prev_gray, dg, P0 * nseq);
            if (rc == DVO_OK) rc = launch_copy_bytes(c, c->prev_depth, dd, P0 * nseq * 2);
            for (int s2 = 0; s2 < nseq; ++s2) c->prev_valid[s2] = 1;
        }
        if (frame == DVO_FRAME_NOW) for (int s2 = 0; s2 < nseq; ++s2) c->now_valid[s2] = 1;
        if (host_in) {
            const int k = t & 1;
            fail(cudaStreamWaitEvent(c->stream, ev_ready[k], 0));
            if (rc == DVO_OK) rc = launch_copy_bytes(c, dg, stage_g[k], P0 * nseq);          // a kernel, not a D2D memcpy: the copy engines stay with the uploads
            if (rc == DVO_OK) rc = launch_copy_bytes(c, dd, stage_d[k], P0 * nseq * 2);
            fail(cudaEventRecord(ev_free[k], c->stream));
        } else {
            fail(cudaMemcpy2DAsync(dg, P0, gray + (size_t)t * P0, (size_t)nframes * P0, P0, nseq, cudaMemcpyDeviceToDevice, c->stream));
            fail(cudaMemcpy2DAsync(dd, P0 * 2, depth + (size_t)t * P0, (size_t)nframes * P0 * 2, P0 * 2, nseq, cudaMemcpyDeviceToDevice, c->stream));
        }
    };

    const int blk = (nseq + 127) / 128;
    const bool timing = c->timing;
    c->timing = false;                                                                       // per-stage timers synchronise; keep the pipeline asynchronous
    for (int s2 = 0; s2 < nseq; ++s2) { c->now_valid[s2] = 0; c->prev_valid[s2] = 0; }
    upload(0); upload(1);
    ingest(DVO_FRAME_REF, 0);
    if (rc == DVO_OK) rc = dvo_build_pyramids(c, 0, nseq, 1);
    if (rc == DVO_OK) rc = dvo_prepare(c, 0, nseq, 1);
    if (rc == DVO_OK) { seq_init_kernel<<<blk, 128, 0, c->stream>>>(nseq, nframes, c->pose0, c->seq_state, d_rel, d_kind, d_reason); c->launches++; fail(cudaGetLastError()); }
    int host_last_ref = 0;                                                                   // mirrors lastRef of every slot under the periodic rule alone
    for (int t = 1; t < nframes && rc == DVO_OK; ++t) {
        ingest(DVO_FRAME_NOW, t);                                                            // setRcvdFrameAsNowFrame
        upload(t + 1);                                                                       // next frame travels while this one is solved
        if (rc != DVO_OK) break;
        if ((rc = dvo_build_pyramids(c, 0, nseq, 2))) break;
        if ((rc = dvo_prepare(c, 0, nseq, 2))) break;
        bool switch_pass = t >= 2, first_solve = true;                                       // a previous now frame exists from t = 2 on
        if (!pol->use_quality_gates && !entropy_on) {
            switch_pass = t >= 2 && pol->keyframe_every > 0 && (t - host_last_ref) == pol->keyframe_every && host_last_ref != t - 1;
            if (switch_pass) { host_last_ref = t - 1; first_solve = false; }
        }
        if (first_solve && (rc = dvo_run(c, 0, nseq, p))) break;                             // warm start: pose0 holds the previous frame's pose (:1931-1932)
        double* const cov_t = cov ? c->seq_cov + 36 * (size_t)t : nullptr;
        dvo_cov_info* const cinfo_t = entropy_on ? c->seq_cov_info + t : nullptr;
        if (entropy_on && (rc = launch_cov(c, 0, nseq, finest, p, cov_t, cinfo_t, nframes))) break;
        seq_gate_kernel<<<blk, 128, 0, c->stream>>>(nseq, nframes, t, *pol, finest, c->info, c->pose, c->pose0, c->seq_state, c->seq_mask, d_rel, d_kind, d_reason,
                                                    entropy_on ? c->seq_cov_info.get() : nullptr, ent_thr, c->seq_ent);
        c->launches++;
        if (fail(cudaGetLastError())) break;
        if (switch_pass) {
            c->active = c->seq_mask;                                                         // only the flagged slots do any work
            rc = dvo_promote_now_to_ref(c, 0, nseq);                                         // setPrevFrameAsRefFrame (:2196)
            if (rc == DVO_OK) rc = dvo_build_pyramids(c, 0, nseq, 1);
            if (rc == DVO_OK) rc = dvo_prepare(c, 0, nseq, 1);                               // computeDistTransfrmOfRef + preProcessRefFrame (:2197)
            if (rc == DVO_OK) rc = dvo_run(c, 0, nseq, p);                                   // re-run from identity (:2213-2220)
            if (rc == DVO_OK && entropy_on) rc = launch_cov(c, 0, nseq, finest, p, cov_t, cinfo_t, nframes);
            c->active = nullptr;
            if (rc != DVO_OK) break;
            seq_finish_kernel<<<blk, 128, 0, c->stream>>>(nseq, nframes, t, c->seq_mask, c->pose, c->pose0, d_rel, d_kind, d_reason);
            c->launches++;
            if (fail(cudaGetLastError())) break;
        }
        // c->pose of every slot is now frame t's final relative pose, and its frames are the pair it was finally solved on
        if (cov && !entropy_on && (rc = launch_cov(c, 0, nseq, finest, p, cov_t, nullptr, nframes))) break;
    }
    c->active = nullptr;
    c->timing = timing;
    if (rc == DVO_OK && (global_poses || global_cov)) {
        A(c->seq_glob.reserve(19 * n));
        if (global_cov && rc == DVO_OK) A(c->seq_gcov.reserve(36 * n));
        d_glob = c->seq_glob;
        if (rc == DVO_OK) {
            rc = launch_gop(c, nseq, nframes, d_kind, d_rel, d_glob, global_cov ? c->seq_cov.get() : nullptr, global_cov ? c->seq_gcov.get() : nullptr);
            if (rc == DVO_OK && global_poses) fail(cudaMemcpyAsync(global_poses, d_glob, sizeof(double) * 19 * n, cudaMemcpyDeviceToHost, c->stream));
            if (rc == DVO_OK && global_cov) fail(cudaMemcpyAsync(global_cov, c->seq_gcov, sizeof(double) * 36 * n, cudaMemcpyDeviceToHost, c->stream));
        }
    }
    if (rc == DVO_OK) {
        fail(cudaMemcpyAsync(rel_poses, d_rel, sizeof(double) * 12 * n, cudaMemcpyDeviceToHost, c->stream));
        fail(cudaMemcpyAsync(kind, d_kind, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
        if (reason) fail(cudaMemcpyAsync(reason, d_reason, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
        if (rel_cov) fail(cudaMemcpyAsync(rel_cov, c->seq_cov, sizeof(double) * 36 * n, cudaMemcpyDeviceToHost, c->stream));
        if (entropy_ratio && entropy_on) fail(cudaMemcpyAsync(entropy_ratio, c->seq_ent, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
        if (entropy_ratio && !entropy_on) std::fill(entropy_ratio, entropy_ratio + n, (double)NAN);
    }
    cudaStreamSynchronize(c->copy_stream);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && rc == DVO_OK) { dvo_set_error("%s: %s", who, cudaGetErrorString(cudaGetLastError())); rc = DVO_ERR_CUDA; }
    return rc;
}
}  // namespace

extern "C" {

int dvo_run_sequences(dvo_ctx* c, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, const dvo_solver_params* p,
                      int keyframe_every, double* rel_poses, int* kind, double* global_poses) {
    dvo_keyframe_policy pol; memset(&pol, 0, sizeof(pol));
    pol.keyframe_every = keyframe_every; pol.use_quality_gates = 0; pol.laplacian_thresh = 3.0f; pol.visible_ratio_thresh = 0.8f; pol.min_reprojections = 50;
    return run_sequences_core(c, "dvo_run_sequences", nseq, nframes, gray, depth, DVO_MEM_HOST, p, &pol, rel_poses, kind, nullptr, global_poses, false,
                              nullptr, nullptr);
}

int dvo_run_sequences_gated(dvo_ctx* c, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, const dvo_solver_params* p,
                            const dvo_keyframe_policy* pol, double* rel_poses, int* kind, int* reason, double* global_poses) {
    return run_sequences_core(c, "dvo_run_sequences", nseq, nframes, gray, depth, DVO_MEM_HOST, p, pol, rel_poses, kind, reason, global_poses, false,
                              nullptr, nullptr);
}

int dvo_run_sequences_mem(dvo_ctx* c, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem, const dvo_solver_params* p,
                          const dvo_keyframe_policy* pol, double* rel_poses, int* kind, int* reason, double* global_poses) {
    return run_sequences_core(c, "dvo_run_sequences", nseq, nframes, gray, depth, mem, p, pol, rel_poses, kind, reason, global_poses, false, nullptr,
                              nullptr);
}

int dvo_run_sequences_cov(dvo_ctx* c, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem, const dvo_solver_params* p,
                          const dvo_keyframe_policy* pol, double* rel_poses, int* kind, int* reason, double* global_poses, double* rel_cov,
                          double* global_cov) {
    if (!rel_cov) { dvo_set_error("dvo_run_sequences_cov: rel_cov is required"); return DVO_ERR_ARG; }
    return run_sequences_core(c, "dvo_run_sequences_cov", nseq, nframes, gray, depth, mem, p, pol, rel_poses, kind, reason, global_poses, true,
                              rel_cov, global_cov);
}

int dvo_run_sequences_entropy(dvo_ctx* c, int nseq, int nframes, const uint8_t* gray, const uint16_t* depth, int mem, const dvo_solver_params* p,
                              const dvo_keyframe_policy* pol, double entropy_ratio_thresh, double* rel_poses, int* kind, int* reason,
                              double* global_poses, double* rel_cov, double* global_cov, double* entropy_ratio) {
    return run_sequences_core(c, "dvo_run_sequences_entropy", nseq, nframes, gray, depth, mem, p, pol, rel_poses, kind, reason, global_poses, true,
                              rel_cov, global_cov, entropy_ratio_thresh, entropy_ratio);
}

}  // extern "C"

extern "C" {

int dvo_pose_covariance(dvo_ctx* c, int first, int count, const dvo_solver_params* p, int level, double* cov36, dvo_cov_info* info, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, first, count) || !p || !cov36 || (mem != DVO_MEM_HOST && mem != DVO_MEM_DEVICE) || level < -1 || level >= c->geom.L ||
        (p->residual != DVO_RESIDUAL_DT_FLOOR && p->residual != DVO_RESIDUAL_DT_INTERP)) {
        dvo_set_error("dvo_pose_covariance: bad argument"); return DVO_ERR_ARG;
    }
    if (!c->haveK) { dvo_set_error("dvo_pose_covariance: intrinsics not set"); return DVO_ERR_STATE; }
    if (level < 0) for (int l = 0; l < c->geom.L; ++l) if (p->iters[l] > 0) { level = l; break; }
    if (level < 0) { dvo_set_error("dvo_pose_covariance: level = -1 and no level has iterations"); return DVO_ERR_ARG; }
    if (count == 0) return DVO_OK;
    if (mem == DVO_MEM_DEVICE) return launch_cov(c, first, count, level, p, cov36, info, 1);
    if (c->cov_buf.n < 36 * (size_t)count) DVO_CUDA(cudaStreamSynchronize(c->stream));   // growth replaces buffers work in flight may use
    int rc;
    if ((rc = c->cov_buf.reserve(36 * (size_t)count)) || (rc = c->cov_info_buf.reserve(count))) return rc;
    if ((rc = launch_cov(c, first, count, level, p, c->cov_buf, c->cov_info_buf, 1))) return rc;
    DVO_CUDA(cudaMemcpyAsync(cov36, c->cov_buf, sizeof(double) * 36 * count, cudaMemcpyDeviceToHost, c->stream));
    if (info) DVO_CUDA(cudaMemcpyAsync(info, c->cov_info_buf, sizeof(dvo_cov_info) * count, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_align_pairs(dvo_ctx* c, int npairs, const int* ref_slot, const int* now_slot, const double* pose0, const dvo_solver_params* p,
                    double* poses, dvo_pair_info* info, double* cov36, dvo_cov_info* cov_info, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!c || npairs < 0 || !ref_slot || !now_slot || !p || !poses || (mem != DVO_MEM_HOST && mem != DVO_MEM_DEVICE) ||
        (cov36 && p->residual != DVO_RESIDUAL_DT_FLOOR && p->residual != DVO_RESIDUAL_DT_INTERP)) {
        dvo_set_error("dvo_align_pairs: bad argument"); return DVO_ERR_ARG;
    }
    if (!c->haveK) { dvo_set_error("dvo_align_pairs: intrinsics not set"); return DVO_ERR_STATE; }
    int level = -1;                                      // covariance level: the finest with iterations, as dvo_pose_covariance's -1
    if (cov36) {
        for (int l = 0; l < c->geom.L; ++l) if (p->iters[l] > 0) { level = l; break; }
        if (level < 0) { dvo_set_error("dvo_align_pairs: covariance requested and no level has iterations"); return DVO_ERR_ARG; }
    }
    const int B = c->cfg.max_batch;
    if (mem == DVO_MEM_HOST)                             // device indices are checked by the kernels (status bit 1)
        for (int k = 0; k < npairs; ++k)
            if (ref_slot[k] < 0 || ref_slot[k] >= B || now_slot[k] < 0 || now_slot[k] >= B) {
                dvo_set_error("dvo_align_pairs: pair %d addresses slots (%d, %d) outside [0, %d)", k, ref_slot[k], now_slot[k], B);
                return DVO_ERR_ARG;
            }
    if (npairs == 0) return DVO_OK;
    const size_t n = (size_t)npairs;
    // per-pair state: one set of buffers per context, grown on demand; growth replaces buffers work in flight may use
    if (c->pair_ref.n < n) DVO_CUDA(cudaStreamSynchronize(c->stream));
    int rc = DVO_OK;
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    A(c->pair_ref.reserve(n)); A(c->pair_now.reserve(n)); A(c->pair_order.reserve(n));
    A(c->pair_pose0.reserve(n * 12)); A(c->pair_pose.reserve(n * 12)); A(c->pair_info.reserve(n));
    if (rc) return rc;
    const cudaMemcpyKind in = mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const cudaMemcpyKind out = mem == DVO_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    DVO_CUDA(cudaMemcpyAsync(c->pair_ref, ref_slot, sizeof(int) * n, in, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->pair_now, now_slot, sizeof(int) * n, in, c->stream));
    std::vector<double> id;
    if (pose0) DVO_CUDA(cudaMemcpyAsync(c->pair_pose0, pose0, sizeof(double) * 12 * n, in, c->stream));
    else {
        id.assign(12 * n, 0.0);
        for (size_t k = 0; k < n; ++k) { id[12 * k] = 1.0; id[12 * k + 4] = 1.0; id[12 * k + 8] = 1.0; }
        DVO_CUDA(cudaMemcpyAsync(c->pair_pose0, id.data(), sizeof(double) * 12 * n, cudaMemcpyHostToDevice, c->stream));
    }
    if ((rc = launch_solve_pairs(c, npairs, p))) return rc;
    double* d_cov = cov36; dvo_cov_info* d_cinfo = cov_info;
    if (cov36 && mem == DVO_MEM_HOST) {
        if (c->cov_buf.n < 36 * n) DVO_CUDA(cudaStreamSynchronize(c->stream));   // as in dvo_pose_covariance
        if ((rc = c->cov_buf.reserve(36 * n)) || (rc = c->cov_info_buf.reserve(n))) return rc;
        d_cov = c->cov_buf; d_cinfo = c->cov_info_buf;
    }
    if (cov36 && (rc = launch_cov_pairs(c, npairs, level, p, d_cov, d_cinfo))) return rc;
    DVO_CUDA(cudaMemcpyAsync(poses, c->pair_pose, sizeof(double) * 12 * n, out, c->stream));
    if (info) DVO_CUDA(cudaMemcpyAsync(info, c->pair_info, sizeof(dvo_pair_info) * n, out, c->stream));
    if (cov36 && mem == DVO_MEM_HOST) {
        DVO_CUDA(cudaMemcpyAsync(cov36, c->cov_buf, sizeof(double) * 36 * n, cudaMemcpyDeviceToHost, c->stream));
        if (cov_info) DVO_CUDA(cudaMemcpyAsync(cov_info, c->cov_info_buf, sizeof(dvo_cov_info) * n, cudaMemcpyDeviceToHost, c->stream));
    }
    if (mem == DVO_MEM_HOST) DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_level_dims(dvo_ctx* c, int level, int* w, int* h) {
    if (!c || level < 0 || level >= c->geom.L) return DVO_ERR_ARG;
    if (w) *w = c->geom.w[level];
    if (h) *h = c->geom.h[level];
    return DVO_OK;
}

int dvo_get_level_buffer(dvo_ctx* c, int slot, int frame, int level, int which, void* dst, size_t bytes) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, slot, 1) || level < 0 || level >= c->geom.L || (frame != 0 && frame != 1) || !dst) { dvo_set_error("dvo_get_level_buffer: bad argument"); return DVO_ERR_ARG; }
    const size_t P = c->geom.P[level];
    const long long o = lvl_at(c->geom, level, slot);
    const void* src = nullptr; size_t es = 0;
    switch (which) {
        case DVO_BUF_GRAY: src = c->gray[frame] + o; es = 1; break;
        case DVO_BUF_DEPTH: if (!c->depth[frame]) { dvo_set_error("depth not stored for this frame"); return DVO_ERR_STATE; } src = c->depth[frame] + o; es = 2; break;
        case DVO_BUF_EDGE: src = c->edge[frame] + o; es = 1; break;
        case DVO_BUF_D2: if (frame != DVO_FRAME_NOW) { dvo_set_error("d2 exists for the now frame only"); return DVO_ERR_ARG; } break;
        case DVO_BUF_DTN: case DVO_BUF_GX: case DVO_BUF_GY:
            if (frame != DVO_FRAME_NOW) { dvo_set_error("DT exists for the now frame only"); return DVO_ERR_ARG; } break;
        default: dvo_set_error("dvo_get_level_buffer: unknown buffer %d", which); return DVO_ERR_ARG;
    }
    if (which == DVO_BUF_D2) {      // the fused EDT + texel kernel leaves the 32-bit image sparse: rebuild the dense one from the texels
        if (bytes < P * 4) { dvo_set_error("dvo_get_level_buffer: destination too small"); return DVO_ERR_ARG; }
        DevBuf<int32_t> d_tmp;
        int rc;
        if ((rc = d_tmp.reserve(P)) || (rc = launch_d2_from_texels(c, slot, level, d_tmp))) return rc;
        DVO_CUDA(cudaMemcpyAsync(dst, d_tmp, P * 4, cudaMemcpyDeviceToHost, c->stream));
        DVO_CUDA(cudaStreamSynchronize(c->stream));
        return DVO_OK;
    }
    if (which >= DVO_BUF_DTN) {      // no float images are kept: evaluate them from the packed texels for this slot / level on demand
        if (bytes < P * 4) { dvo_set_error("dvo_get_level_buffer: destination too small"); return DVO_ERR_ARG; }
        std::vector<float> tmp(P * 4);
        DevBuf<float4> d_tmp;
        int rc;
        if ((rc = d_tmp.reserve(P)) || (rc = launch_resolve_texels(c, slot, level, d_tmp))) return rc;
        DVO_CUDA(cudaMemcpyAsync(tmp.data(), d_tmp, P * 16, cudaMemcpyDeviceToHost, c->stream));
        DVO_CUDA(cudaStreamSynchronize(c->stream));
        const int comp = which - DVO_BUF_DTN;
        float* d = (float*)dst;
        for (size_t i = 0; i < P; ++i) d[i] = tmp[4 * i + comp];
        return DVO_OK;
    }
    if (bytes < P * es) { dvo_set_error("dvo_get_level_buffer: destination too small"); return DVO_ERR_ARG; }
    DVO_CUDA(cudaMemcpyAsync(dst, src, P * es, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    if (which == DVO_BUF_DEPTH && level == 0) {            // level-0 zero fix is applied at read-out (see preprocess.cu)
        uint16_t* d = (uint16_t*)dst;
        for (size_t i = 0; i < P; ++i) if (d[i] == 0) d[i] = 1;
    }
    return DVO_OK;
}

// The device keeps the point list in row-major pixel order; the reference enumerates column-major (xx outer, yy inner,
// src/SolveDVO.cpp:1237-1241).  perm[k] = device index of the k-th point in the reference's order.
static int reference_order(dvo_ctx* c, int slot, int level, int n, std::vector<int>& perm) {
    perm.resize(n);
    if (n == 0) return DVO_OK;
    std::vector<int> pix(n);
    DVO_CUDA(cudaMemcpyAsync(pix.data(), c->ptsPix + lvl_at(c->geom, level, slot), sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    const int w = c->geom.w[level], h = c->geom.h[level];
    std::vector<long long> key(n);
    for (int i = 0; i < n; ++i) { const int y = pix[i] / w, x = pix[i] - y * w; key[i] = ((long long)x * h + y) * (long long)n + i; }
    std::sort(key.begin(), key.end());
    for (int k = 0; k < n; ++k) perm[k] = (int)(key[k] % n);
    return DVO_OK;
}

int dvo_get_points(dvo_ctx* c, int slot, int level, float* X, float* Y, float* Z, int capacity, int* n) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, slot, 1) || level < 0 || level >= c->geom.L || !n) return DVO_ERR_ARG;
    int cnt = 0;
    DVO_CUDA(cudaMemcpyAsync(&cnt, c->npts + (size_t)slot * c->geom.L + level, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    *n = cnt;
    const int m = cnt < capacity ? cnt : capacity;
    if (m <= 0 || !(X || Y || Z)) return DVO_OK;
    std::vector<int> perm;
    int rc = reference_order(c, slot, level, cnt, perm);
    if (rc) return rc;
    const long long o = lvl_at(c->geom, level, slot);
    std::vector<float> tmp(cnt);
    float* dst[3] = {X, Y, Z}; const float* src[3] = {c->ptsX + o, c->ptsY + o, c->ptsZ + o};
    for (int a = 0; a < 3; ++a) {
        if (!dst[a]) continue;
        DVO_CUDA(cudaMemcpyAsync(tmp.data(), src[a], sizeof(float) * cnt, cudaMemcpyDeviceToHost, c->stream));
        DVO_CUDA(cudaStreamSynchronize(c->stream));
        for (int k = 0; k < m; ++k) dst[a][k] = tmp[perm[k]];
    }
    return DVO_OK;
}

int dvo_eval_normal_equations(dvo_ctx* c, int slot, int level, const double* R9T3, int jacobian, int weight, int arithmetic,
                              float huber_k, double* H36, double* g6, double* sumsq, int* nvis, float* eps, float* w, float* u,
                              float* v, float* J) {
    dvo_solver_params prm;
    memset(&prm, 0, sizeof(prm));
    prm.jacobian = jacobian; prm.weight = weight; prm.arithmetic = arithmetic; prm.huber_k = huber_k;
    return dvo_eval_normal_equations_ex(c, slot, level, R9T3, &prm, H36, g6, sumsq, nvis, eps, w, u, v, J);
}

int dvo_eval_normal_equations_ex(dvo_ctx* c, int slot, int level, const double* R9T3, const dvo_solver_params* prm,
                                 double* H36, double* g6, double* sumsq, int* nvis, float* eps, float* w, float* u, float* v, float* J) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!prm) return DVO_ERR_ARG;
    if (!range_ok(c, slot, 1) || level < 0 || level >= c->geom.L || !R9T3) return DVO_ERR_ARG;
    if (!c->haveK) { dvo_set_error("intrinsics not set"); return DVO_ERR_STATE; }
    int N = 0;
    DVO_CUDA(cudaMemcpyAsync(&N, c->npts + (size_t)slot * c->geom.L + level, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    DevBuf<double> d_pose, d_out; DevBuf<float> d_pp;
    const bool pp = eps || w || u || v || J;
    const size_t n1 = (size_t)(N > 0 ? N : 1);
    int rc;
    if ((rc = d_pose.reserve(12)) || (rc = d_out.reserve(44)) || (pp && (rc = d_pp.reserve(n1 * 10)))) return rc;
    DVO_CUDA(cudaMemcpyAsync(d_pose, R9T3, sizeof(double) * 12, cudaMemcpyHostToDevice, c->stream));
    float *de = nullptr, *dw = nullptr, *du = nullptr, *dv = nullptr, *dJ = nullptr;
    if (pp) { de = d_pp; dw = d_pp + n1; du = d_pp + 2 * n1; dv = d_pp + 3 * n1; dJ = d_pp + 4 * n1; }
    if ((rc = launch_eval(c, slot, level, d_pose, prm->jacobian, prm->weight, prm->arithmetic, prm->huber_k, prm->residual, d_out, de, dw, du, dv, dJ)))
        return rc;
    double out[44];
    std::vector<float> host(pp ? n1 * 10 : 0);
    DVO_CUDA(cudaMemcpyAsync(out, d_out, sizeof(out), cudaMemcpyDeviceToHost, c->stream));
    if (pp && N > 0) DVO_CUDA(cudaMemcpyAsync(host.data(), d_pp, sizeof(float) * n1 * 10, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    if (g6) memcpy(g6, out, sizeof(double) * 6);
    if (H36) memcpy(H36, out + 6, sizeof(double) * 36);
    if (sumsq) *sumsq = out[42];
    if (nvis) *nvis = (int)out[43];
    if (pp && N > 0) {                               // per-point arrays are returned in the reference's (column-major) order
        std::vector<int> perm;
        if ((rc = reference_order(c, slot, level, N, perm))) return rc;
        for (int k = 0; k < N; ++k) {
            const size_t i = (size_t)perm[k];
            if (eps) eps[k] = host[i];
            if (w) w[k] = host[n1 + i];
            if (u) u[k] = host[2 * n1 + i];
            if (v) v[k] = host[3 * n1 + i];
            if (J) for (int q = 0; q < 6; ++q) J[6 * (size_t)k + q] = host[4 * n1 + 6 * i + q];
        }
    }
    return DVO_OK;
}

int dvo_get_trace(dvo_ctx* c, int slot, int level, double* trace) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, slot, 1) || level < 0 || level >= c->geom.L || !trace) return DVO_ERR_ARG;
    if (!c->trace) { dvo_set_error("dvo_get_trace: context created with trace_iters = 0"); return DVO_ERR_STATE; }
    const size_t n = (size_t)c->cfg.trace_iters * DVO_TRACE_DOUBLES;
    DVO_CUDA(cudaMemcpyAsync(trace, c->trace + ((size_t)slot * c->geom.L + level) * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_get_energies(dvo_ctx* c, int slot, int level, float* energies, int capacity) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!range_ok(c, slot, 1) || level < 0 || level >= c->geom.L || !energies || capacity < 0) return DVO_ERR_ARG;
    const int n = capacity < DVO_ENERGY_ITERS ? capacity : DVO_ENERGY_ITERS;
    if (n == 0) return DVO_OK;
    DVO_CUDA(cudaMemcpyAsync(energies, c->energy + ((size_t)slot * c->geom.L + level) * DVO_ENERGY_ITERS, sizeof(float) * n, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_enable_timing(dvo_ctx* c, int on) {
    if (!c) return DVO_ERR_ARG;
    c->timing = on != 0;
    for (int i = 0; i < DVO_STAGE_COUNT; ++i) c->stage_ms[i] = 0.f;
    return DVO_OK;
}

int dvo_get_stage_ms(dvo_ctx* c, float* ms) {
    if (!c || !ms) return DVO_ERR_ARG;
    for (int i = 0; i < DVO_STAGE_COUNT; ++i) { ms[i] = c->stage_ms[i]; c->stage_ms[i] = 0.f; }
    return DVO_OK;
}

long long dvo_launch_count(dvo_ctx* c) { return c ? c->launches : 0; }

int dvo_gop_compose(dvo_ctx* c, int nseq, int nframes, const int* kind, const double* rel, double* out, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!c || nseq < 1 || nframes < 1 || !kind || !rel || !out) return DVO_ERR_ARG;
    const size_t n = (size_t)nseq * nframes;
    if (mem == DVO_MEM_DEVICE) return launch_gop(c, nseq, nframes, kind, rel, out, nullptr, nullptr);
    DevBuf<int> d_kind; DevBuf<double> d_rel, d_out;
    int rc;
    if ((rc = d_kind.reserve(n)) || (rc = d_rel.reserve(12 * n)) || (rc = d_out.reserve(19 * n))) return rc;
    DVO_CUDA(cudaMemcpyAsync(d_kind, kind, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(d_rel, rel, sizeof(double) * 12 * n, cudaMemcpyHostToDevice, c->stream));
    if ((rc = launch_gop(c, nseq, nframes, d_kind, d_rel, d_out, nullptr, nullptr))) return rc;
    DVO_CUDA(cudaMemcpyAsync(out, d_out, sizeof(double) * 19 * n, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

int dvo_pose_graph_optimize(dvo_ctx* c, int ngraphs, int nnodes, int nedges, int max_lag, const int* edge_ref, const int* edge_now,
                            const double* meas12, const double* cov36, double* poses12, const dvo_pgo_params* prm, double* node_cov36,
                            dvo_pgo_info* info, int mem) {
    if (c) { const int jr = join_aux(c); if (jr) return jr; }
    if (!c || ngraphs < 0 || nnodes < 2 || nedges < 0 || max_lag < 1 || max_lag > DVO_PGO_MAX_LAG || !poses12 || !prm ||
        (nedges > 0 && (!edge_ref || !edge_now || !meas12 || !cov36)) || (mem != DVO_MEM_HOST && mem != DVO_MEM_DEVICE) ||
        prm->max_iterations < 0 || !(prm->lambda0 > 0.0) || !(prm->rel_tol >= 0.0)) {
        dvo_set_error("dvo_pose_graph_optimize: bad argument"); return DVO_ERR_ARG;
    }
    const size_t G = (size_t)ngraphs, E = (size_t)nedges, N = (size_t)nnodes;
    if (mem == DVO_MEM_HOST)                             // device indices are checked by the kernel (status bit 0)
        for (size_t k = 0; k < G * E; ++k) {
            const int a = edge_ref[k], b = edge_now[k];
            if (a < 0 || a >= nnodes || b < 0 || b >= nnodes || a == b || abs(a - b) > max_lag) {
                dvo_set_error("dvo_pose_graph_optimize: graph %zu edge %zu joins nodes (%d, %d): outside [0, %d), equal, or more than %d apart",
                              k / (E ? E : 1), k % (E ? E : 1), a, b, nnodes, max_lag);
                return DVO_ERR_ARG;
            }
        }
    if (ngraphs == 0) return DVO_OK;
    size_t dbl = 0, ints = 0;
    pgo_scratch_size(nnodes, nedges, max_lag, &dbl, &ints);
    int rc = DVO_OK;
    auto A = [&](int r) { if (rc == DVO_OK) rc = r; };
    // growth replaces buffers work in flight may use
    if (c->pgo_dscr.n < G * dbl || c->pgo_iscr.n < G * ints) DVO_CUDA(cudaStreamSynchronize(c->stream));
    A(c->pgo_dscr.reserve(G * dbl)); A(c->pgo_iscr.reserve(G * ints));
    if (rc) return rc;
    if (mem == DVO_MEM_DEVICE)
        return launch_pose_graph(c, ngraphs, nnodes, nedges, max_lag, edge_ref, edge_now, meas12, cov36, poses12, prm, node_cov36, info,
                                 c->pgo_dscr, c->pgo_iscr);
    if (c->pgo_ref.n < G * E || c->pgo_meas.n < 12 * G * E || c->pgo_cov.n < 36 * G * E || c->pgo_pose.n < 12 * G * N ||
        (node_cov36 && c->pgo_ncov.n < 36 * G * N) || c->pgo_info.n < G)
        DVO_CUDA(cudaStreamSynchronize(c->stream));
    A(c->pgo_ref.reserve(G * E)); A(c->pgo_now.reserve(G * E)); A(c->pgo_meas.reserve(12 * G * E)); A(c->pgo_cov.reserve(36 * G * E));
    A(c->pgo_pose.reserve(12 * G * N)); A(c->pgo_info.reserve(G));
    if (node_cov36) A(c->pgo_ncov.reserve(36 * G * N));
    if (rc) return rc;
    DVO_CUDA(cudaMemcpyAsync(c->pgo_ref, edge_ref, sizeof(int) * G * E, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->pgo_now, edge_now, sizeof(int) * G * E, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->pgo_meas, meas12, sizeof(double) * 12 * G * E, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->pgo_cov, cov36, sizeof(double) * 36 * G * E, cudaMemcpyHostToDevice, c->stream));
    DVO_CUDA(cudaMemcpyAsync(c->pgo_pose, poses12, sizeof(double) * 12 * G * N, cudaMemcpyHostToDevice, c->stream));
    if ((rc = launch_pose_graph(c, ngraphs, nnodes, nedges, max_lag, c->pgo_ref, c->pgo_now, c->pgo_meas, c->pgo_cov, c->pgo_pose, prm,
                                node_cov36 ? c->pgo_ncov.get() : nullptr, c->pgo_info, c->pgo_dscr, c->pgo_iscr)))
        return rc;
    DVO_CUDA(cudaMemcpyAsync(poses12, c->pgo_pose, sizeof(double) * 12 * G * N, cudaMemcpyDeviceToHost, c->stream));
    if (node_cov36) DVO_CUDA(cudaMemcpyAsync(node_cov36, c->pgo_ncov, sizeof(double) * 36 * G * N, cudaMemcpyDeviceToHost, c->stream));
    if (info) DVO_CUDA(cudaMemcpyAsync(info, c->pgo_info, sizeof(dvo_pgo_info) * G, cudaMemcpyDeviceToHost, c->stream));
    DVO_CUDA(cudaStreamSynchronize(c->stream));
    return DVO_OK;
}

// ---- device-resident storage blobs (PyramidalStorageStruct keeps caller-provided level arrays on the device) ----
struct dvo_blob { DevBuf<unsigned char> d; size_t bytes; int device; };

int dvo_blob_create(size_t bytes, int device, dvo_blob** out) {
    if (!out || bytes == 0) { dvo_set_error("dvo_blob_create: bad argument"); return DVO_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { cudaGetLastError(); dvo_set_error("dvo_blob_create: no usable CUDA device (there is no CPU fallback)"); return DVO_ERR_CUDA; }
    if (device < 0 || device >= ndev) { dvo_set_error("dvo_blob_create: device %d out of range", device); return DVO_ERR_ARG; }
    DVO_CUDA(cudaSetDevice(device));
    dvo_blob* b = new (std::nothrow) dvo_blob();
    if (!b) return DVO_ERR_NOMEM;
    b->bytes = bytes; b->device = device;
    if (const int rc = b->d.reserve(bytes)) { cudaGetLastError(); delete b; return rc; }
    *out = b;
    return DVO_OK;
}
int dvo_blob_upload(dvo_blob* b, const void* host_src, size_t bytes) {
    if (!b || !host_src || bytes > b->bytes) { dvo_set_error("dvo_blob_upload: bad argument"); return DVO_ERR_ARG; }
    DVO_CUDA(cudaSetDevice(b->device));
    DVO_CUDA(cudaMemcpy(b->d, host_src, bytes, cudaMemcpyHostToDevice));
    return DVO_OK;
}
int dvo_blob_download(dvo_blob* b, void* host_dst, size_t bytes) {
    if (!b || !host_dst || bytes > b->bytes) { dvo_set_error("dvo_blob_download: bad argument"); return DVO_ERR_ARG; }
    DVO_CUDA(cudaSetDevice(b->device));
    DVO_CUDA(cudaMemcpy(host_dst, b->d, bytes, cudaMemcpyDeviceToHost));
    return DVO_OK;
}
void* dvo_blob_device_ptr(dvo_blob* b) { return b ? b->d.get() : nullptr; }
size_t dvo_blob_bytes(dvo_blob* b) { return b ? b->bytes : 0; }
int dvo_blob_destroy(dvo_blob* b) {
    if (!b) return DVO_OK;
    cudaSetDevice(b->device);
    delete b;
    return DVO_OK;
}

}  // extern "C"
