// The C ABI's context (include/sfm_b200.h): creation and destruction, the stream, configuration, errors, pinned host
// memory and timing.  sfm_host.h lists the stage files that hold the rest of the ABI.
#include <cstdarg>

#include "sfm_host.h"
#include "sfm_misc.cuh"

using namespace sfm;
using namespace sfm_host;

thread_local std::string sfm_host::g_err;

int sfm_host::fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

// error setter for the host-only translation units (sfm_sampler.cpp)
int sfm_internal_set_error(int code, const char* message) {
    g_err = message;
    return code;
}

int sfm_version(void) { return 100; }
const char* sfm_last_error(void) { return g_err.c_str(); }

int sfm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int sfm_create(int device, sfm_ctx** out) {
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(SFM_ERR_NO_DEVICE, "no CUDA device available (%s)",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= n) return fail(SFM_ERR_ARG, "device %d out of range [0,%d)", device, n);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(SFM_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    sfm_ctx* c = new sfm_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    for (int i = 0; i < T_COUNT; ++i) {
        CU(cudaEventCreate(&c->ev0[i]));
        CU(cudaEventCreate(&c->ev1[i]));
        c->ev_used[i] = false;
    }
    if (int r = allow_fit_smem()) return r;
    *out = c;
    return 0;
}

int sfm_destroy(sfm_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    Buf* bufs[] = {&c->raw, &c->pts, &c->offsets, &c->Ks, &c->table, &c->E, &c->valid, &c->eig, &c->acc,
                   &c->count_extra, &c->S1, &c->S2, &c->err, &c->blocks, &c->best,
                   &c->invalid, &c->winnerE, &c->record, &c->merged, &c->rows, &c->blockinv, &c->mask, &c->sed, &c->poses, &c->pass, &c->X, &c->idx,
                   &c->planes, &c->hK, &c->selstate, &c->selio, &c->selpp, &c->refstate, &c->refpart, &c->reftick, &c->refrec, &c->refrep, &c->k2pts, &c->k2box, &c->k2sort,
                   &c->scan, &c->tmp, &c->gathered, &c->tailstate, &c->num, &c->winrec, &c->bout, &c->spts, &c->bounds, &c->fitflag,
                   &c->m_img, &c->m_feat, &c->m_W, &c->m_ss, &c->m_ok, &c->m_S, &c->m_out,
                   &c->h_img, &c->h_gx, &c->h_gy, &c->h_corner, &c->h_alive, &c->h_key, &c->h_idx, &c->h_small, &c->h_xy};
    for (Buf* b : bufs) b->release();
    for (int i = 0; i < T_COUNT; ++i) {
        cudaEventDestroy(c->ev0[i]);
        cudaEventDestroy(c->ev1[i]);
    }
    sfm_nccl_destroy(c);
    if (c->hpin) cudaFreeHost(c->hpin);
    cudaStreamDestroy(c->own_stream);
    delete c;
    return 0;
}

int sfm_set_stream(sfm_ctx* c, void* s) {
    if (int r = use(c)) return r;
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return 0;
}

int sfm_use_default_stream(sfm_ctx* c) {
    if (int r = use(c)) return r;
    c->stream = cudaStreamLegacy;
    return 0;
}

int sfm_synchronize(sfm_ctx* c) {
    if (int r = use(c)) return r;
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_set_refinement(sfm_ctx* c, int max_iterations) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    if (max_iterations < 0) return fail(SFM_ERR_ARG, "max_iterations must be >= 0, got %d", max_iterations);
    c->refine_iters = max_iterations;
    return 0;
}

int sfm_host_alloc(uint64_t bytes, void** out) {
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    CU(cudaMallocHost(out, bytes ? bytes : 1));
    return 0;
}
int sfm_host_free(void* p) {
    if (p) CU(cudaFreeHost(p));
    return 0;
}

// ---- measurement ----------------------------------------------------------------------------
int sfm_enable_timing(sfm_ctx* c, int on) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    c->timing = on != 0;
    for (int i = 0; i < T_COUNT; ++i) c->ev_used[i] = false;
    return 0;
}

int sfm_get_timing(sfm_ctx* c, float ms[8], int64_t* launches) {
    if (int r = use(c)) return r;
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < T_COUNT; ++i) {
        ms[i] = 0.f;
        if (c->timing && c->ev_used[i]) CU(cudaEventElapsedTime(&ms[i], c->ev0[i], c->ev1[i]));
        c->ev_used[i] = false;  // each stage is reported once
    }
    if (launches) *launches = c->launches;
    return 0;
}

int sfm_measure_fp64_peak(sfm_ctx* c, double* dfma_per_s) {
    if (int r = use(c)) return r;
    if (!dfma_per_s) return fail(SFM_ERR_ARG, "null argument");
    if (int r = c->tmp.reserve(1 << 20)) return r;
    const int blocks = c->sm_count * 8, threads = 256, iters = 4096;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CU(cudaEventRecord(a, c->stream));
        k_fp64_peak<<<blocks, threads, 0, c->stream>>>(c->tmp.as<double>(), iters, 1.0000001);
        if (int r = check_launch(c, "k_fp64_peak")) return r;
        CU(cudaEventRecord(b, c->stream));
        CU(cudaEventSynchronize(b));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, a, b));
        const double rate = (double)blocks * threads * iters * 16.0 / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *dfma_per_s = best;
    return 0;
}
