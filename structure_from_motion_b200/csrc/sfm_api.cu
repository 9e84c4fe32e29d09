// C ABI (include/sfm_b200.h) over the sm_100a kernels.  Host side: context, grow-only
// device buffers, launch geometry, and the CPython-compatible MT19937 sampler.
#include "../../include/sfm_b200.h"

#include <dlfcn.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "sfm_device.cuh"
#include "sfm_fit.cuh"
#include "sfm_linalg.cuh"
#include "sfm_score.cuh"
#include "sfm_homography.cuh"
#include "sfm_pose.cuh"
#include "sfm_tail.cuh"
#include "sfm_misc.cuh"
#include "sfm_match.cuh"
#include "sfm_harris.cuh"
#include "sfm_select.cuh"
#include "sfm_refine.cuh"

using namespace sfm;

static_assert(sizeof(Corr) == 32, "Corr must be 32 bytes");
static_assert(sizeof(PoseSet) == sizeof(sfm_poses), "PoseSet/sfm_poses layout mismatch");
static_assert(sizeof(SelectRecord) == SFM_RECORD_BYTES, "SelectRecord / SFM_RECORD_BYTES mismatch");
static_assert(sizeof(ModelScores) == sizeof(sfm_model_scores), "ModelScores / sfm_model_scores layout mismatch");
static_assert(sizeof(RefineReport) == sizeof(sfm_refinement), "RefineReport / sfm_refinement layout mismatch");

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

}  // namespace

// error setter for the host-only translation units (sfm_sampler.cpp)
int sfm_internal_set_error(int code, const char* message) {
    g_err = message;
    return code;
}

namespace {

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(SFM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                                 \
    } while (0)

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return fail(SFM_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

enum { T_UPLOAD = 0, T_SAMPLE, T_FIT, T_SCORE, T_SELECT, T_MASK, T_POSE, T_TRI, T_COUNT };

}  // namespace

struct sfm_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // data
    Buf raw, pts, offsets, Ks, table, E, valid, eig;
    Buf acc, count_extra, S1, S2, err, blocks, best, invalid, winnerE, spts, bounds, fitflag, record, merged, rows, blockinv;
    Buf m_img, m_feat, m_W, m_ss, m_ok, m_S, m_out;
    Buf h_img, h_gx, h_gy, h_corner, h_alive, h_key, h_idx, h_small, h_xy;
    Buf mask, sed, poses, pass, X, idx, scan, tmp, tailstate, num, winrec, bout;
    Buf planes, hK;  // the homography tail's HPlane and the K it was called with (the upload's K stays in Ks)
    Buf k2pts, k2box, k2sort;  // K2's copy of pts in image-B Morton order, its tile boxes, the sort's scratch
    Buf selstate, selio, selpp;  // k_score_models: self-cleaning sums; models and results; per-correspondence errors
    Buf refstate, refpart, reftick, refrec, refrep;  // refinement: LM state, chunk partials, tickets, records, reports
    long long n = 0, h = 0, npairs = 1;
    long long first_len = 0;  // batched: correspondences of the first pair (what the AUTO pilot samples)
    long long batch_max_len = 0;  // batched: correspondences of the longest pair
    long long raw_stride = 1;
    bool batched = false, has_pts = false, has_table = false, has_models = false, has_score = false;
    bool models_h = false;       // the current models are homographies (sfm_fit_homography), not essential matrices
    bool k2_ready = false;       // k2pts / k2box belong to the current upload (K-normalised records only)
    int hscore_occ = 0;          // resident blocks per SM of k_score_homography (queried once)
    bool table_pending = false;  // sfm_sample_device was called: the table is drawn by the fit kernel (or on demand)
    unsigned long long smp_seed = 0, smp_stream = 0;
    long long smp_offset = 0;
    bool acc_clean = false;  // K2's accumulators (+ tail words) are zero: the fit kernel cleared them
    size_t acc_planes_for = 0;  // hypotheses (all pairs) the cleared accumulators were laid out for
    double Kstage[9] = {0};
    double hstage[18] = {0};  // H and K of sfm_decompose_homography, K of the homography tail, staged for async copies
    std::vector<SelectModels> sstage;  // the models of sfm_score_models / sfm_batch_score_models, staged for the async copy
    std::vector<double> Kbatch;        // the cameras of the current batched upload, [P][9] (the device copy is Ks)
    const void* occ_fn[4] = {nullptr, nullptr, nullptr, nullptr};  // scoring kernels whose launch configuration is cached
    int occ_blocks[4] = {0, 0, 0, 0};
    int occ_next = 0;
    void* nccl_comm = nullptr;  // ncclComm_t of sfm_nccl_init (hypothesis-sharded runs without torch)
    int nccl_rank = 0, nccl_world = 1;
    Buf gathered;
    const unsigned long long* rescored_dev = nullptr;  // K3's rescore counter of the last scoring call
    long long winner_local = -1;  // index into E of the current winner, -1 = use winnerE
    bool winner_set = false;
    long long last_idx_offset = 0;
    double Khost[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    // config
    int variant = SFM_SCORE_AUTO, hpt = 2, group = 16;  // AUTO: a pilot on the device picks SCREEN or FULL per call
    int refine_iters = 0;          // sfm_set_refinement: 0 = off
    long long refined_pairs = 0;   // pairs whose reports the last tail call left in refrep (0: it did not refine)
    // timing
    bool timing = false;
    cudaEvent_t ev0[T_COUNT], ev1[T_COUNT];
    bool ev_used[T_COUNT];
    long long launches = 0;
    // pinned scratch for small results
    void* hpin = nullptr;
    size_t hpin_cap = 0;

    void tic(int s) {
        if (timing) { cudaEventRecord(ev0[s], stream); }
    }
    void toc(int s) {
        if (timing) { cudaEventRecord(ev1[s], stream); ev_used[s] = true; }
    }
};

namespace {

int ensure_pinned(sfm_ctx* c, size_t bytes) {
    if (bytes <= c->hpin_cap) return 0;
    if (c->hpin) cudaFreeHost(c->hpin);
    c->hpin = nullptr;
    c->hpin_cap = 0;
    CU(cudaMallocHost(&c->hpin, bytes + 4096));
    c->hpin_cap = bytes + 4096;
    return 0;
}

int use(sfm_ctx* c) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    CU(cudaSetDevice(c->device));
    return 0;
}

// Device buffer that must read as zero before its first use (self-cleaning kernel state).
int reserve_zeroed(sfm_ctx* c, Buf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (int r = b.reserve(bytes)) return r;
    CU(cudaMemsetAsync(b.p, 0, b.cap, c->stream));
    return 0;
}

int check_launch(sfm_ctx* c, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(SFM_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    c->launches += 1;
#ifdef SFM_TRACE  // debugging builds only (tools/bin/libsfm_trace.so): name every launch and wait for it
    fprintf(stderr, "[sfm] %s ...", what);
    fflush(stderr);
    e = cudaStreamSynchronize(c->stream);
    fprintf(stderr, " %s\n", e == cudaSuccess ? "ok" : cudaGetErrorString(e));
    fflush(stderr);
#endif
    return 0;
}

// Launch of a kernel of the per-estimate chain (fit -> screening copy -> score -> select -> tail): programmatic stream
// serialization lets its blocks be scheduled while the preceding kernel of the chain drains; every chain kernel starts
// with chain_enter() (griddepcontrol.wait), so the data dependence is the ordinary stream order.
inline void chain_config(sfm_ctx* c, dim3 grid, dim3 block, size_t smem, cudaLaunchConfig_t* cfg, cudaLaunchAttribute* at) {
    memset(cfg, 0, sizeof *cfg);
    cfg->gridDim = grid;
    cfg->blockDim = block;
    cfg->dynamicSmemBytes = smem;
    cfg->stream = c->stream;
    at->id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at->val.programmaticStreamSerializationAllowed = 1;
    cfg->attrs = at;
    cfg->numAttrs = 1;
}
template <typename... KArgs, typename... Args>
cudaError_t chain_launch(sfm_ctx* c, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at;
    chain_config(c, grid, block, smem, &cfg, &at);
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
inline cudaError_t chain_launch_ptr(sfm_ctx* c, const void* fn, dim3 grid, dim3 block, size_t smem, void** kargs) {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at;
    chain_config(c, grid, block, smem, &cfg, &at);
    return cudaLaunchKernelExC(&cfg, fn, kargs);
}

// K2's kernel for a variant and shape, and the dynamic shared memory it takes per warp; fn is null for a shape without
// a kernel.  fp64: 2 x 16 only.  The fp32 pre-filter: 4 x 8 (its default) and 2 x 16.  tiles: the upload holds K2's
// sorted copy and its boxes (k2_order), so SCREEN is the 9-slot body; else the 11-slot one.  AUTO holds a one-sided
// body and the two-sided one.
struct ScoreKernel {
    const void* fn;
    size_t warp_bytes;
};
template <typename K>
ScoreKernel score_kernel_of(K* kernel, size_t warp_bytes) {
    return {reinterpret_cast<const void*>(kernel), warp_bytes};
}
ScoreKernel score_kernel(int variant, int hpt, int group, bool tiles) {
    if (variant == SFM_SCORE_SCREEN32) {
        if (hpt == 4 && group == 8) return score_kernel_of(&k_score<4, 8, MODE_SCREEN32>, sizeof(ScoreWarpSmem<4>));
        if (hpt == 2 && group == 16) return score_kernel_of(&k_score<2, 16, MODE_SCREEN32>, sizeof(ScoreWarpSmem<2>));
        return {nullptr, 0};
    }
    if (hpt != 2 || group != 16) return {nullptr, 0};
    const size_t one = tiles ? sizeof(ScoreWarpSmemBox<2>) : sizeof(ScoreWarpSmem<2>), two = sizeof(ScoreWarpSmemFS<2>);
    switch (variant) {
        case SFM_SCORE_FULL: return score_kernel_of(&k_score<2, 16, MODE_FULL>, two);
        case SFM_SCORE_SCREEN:
            return tiles ? score_kernel_of(&k_score<2, 16, MODE_SCREEN>, one) : score_kernel_of(&k_score<2, 16, MODE_SCREEN11>, one);
        default:  // SFM_SCORE_AUTO
            return tiles ? score_kernel_of(&k_score_auto<2, 16, MODE_SCREEN>, one > two ? one : two)
                         : score_kernel_of(&k_score_auto<2, 16, MODE_SCREEN11>, one > two ? one : two);
    }
}

}  // namespace

extern "C" {

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
    CU(cudaFuncSetAttribute(k_fit, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(kFitThreads * kFitSmemDoubles * sizeof(double))));
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

int sfm_set_score_variant(sfm_ctx* c, int variant, int hpt, int group) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    if (variant != SFM_SCORE_SCREEN && variant != SFM_SCORE_FULL && variant != SFM_SCORE_SCREEN32 && variant != SFM_SCORE_AUTO)
        return fail(SFM_ERR_ARG, "bad variant %d", variant);
    // hyps_per_thread == 0: keep the current shape, or the variant's default when the arithmetic changes
    int nh = hpt ? hpt : c->hpt, ng = group ? group : c->group;
    if (!hpt && (variant == SFM_SCORE_SCREEN32) != (c->variant == SFM_SCORE_SCREEN32)) {
        nh = variant == SFM_SCORE_SCREEN32 ? 4 : 2;
        ng = variant == SFM_SCORE_SCREEN32 ? 8 : 16;
    }
    if (!score_kernel(variant, nh, ng, true).fn)
        return fail(SFM_ERR_ARG, "unsupported combination: hyps_per_thread %d, group %d", nh, ng);
    c->variant = variant;
    c->hpt = nh;
    c->group = ng;
    return 0;
}

int sfm_set_refinement(sfm_ctx* c, int max_iterations) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    if (max_iterations < 0) return fail(SFM_ERR_ARG, "max_iterations must be >= 0, got %d", max_iterations);
    c->refine_iters = max_iterations;
    return 0;
}

int sfm_get_refinement(sfm_ctx* c, sfm_refinement* out, int64_t P) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "null argument");
    if (c->refined_pairs == 0) return fail(SFM_ERR_STATE, "the last tail call did not refine (sfm_set_refinement)");
    if (P != c->refined_pairs) return fail(SFM_ERR_ARG, "the last call refined %lld pairs, not %lld", c->refined_pairs, (long long)P);
    CU(cudaMemcpyAsync(out, c->refrep.p, (size_t)P * sizeof(RefineReport), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
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

// ---- sampling ---------------------------------------------------------------------------
int sfm_set_table(sfm_ctx* c, const int32_t* table, int64_t h) {
    if (int r = use(c)) return r;
    if (!table || h <= 0) return fail(SFM_ERR_ARG, "bad table");
    if (!c->has_pts) return fail(SFM_ERR_STATE, "upload correspondences before the sample table");
    for (int64_t i = 0; i < 8 * h; ++i)
        if (table[i] < 0 || table[i] >= c->n) return fail(SFM_ERR_ARG, "table[%lld] = %d out of range", (long long)i, table[i]);
    if (int r = c->table.reserve((size_t)h * 32)) return r;
    CU(cudaMemcpyAsync(c->table.p, table, (size_t)h * 32, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->h = h;
    c->npairs = 1;
    c->has_table = true;
    c->table_pending = false;
    c->has_models = false;
    c->has_score = false;
    return 0;
}

// The device sampler is lazy: the call records (seed, stream, offset) and the next fit draws every row inside the fit
// kernel (one launch less per estimate); anything else that needs the table first materialises it with k_sample.
static int sample_device(sfm_ctx* c, uint64_t seed, uint64_t stream, int64_t hyp_offset, int64_t h) {
    if (h <= 0) return fail(SFM_ERR_ARG, "need h > 0");
    if (!c->has_pts) return fail(SFM_ERR_STATE, "upload correspondences before sampling");
    if (!c->batched && c->n < 8) return fail(SFM_ERR_ARG, "need at least 8 correspondences");
    if (int r = c->table.reserve((size_t)h * c->npairs * 32)) return r;
    c->smp_seed = seed;
    c->smp_stream = stream;
    c->smp_offset = hyp_offset;
    c->table_pending = true;
    c->h = h;
    c->has_table = true;
    c->has_models = false;
    c->has_score = false;
    return 0;
}

static int ensure_table(sfm_ctx* c) {
    if (!c->table_pending) return 0;
    c->tic(T_SAMPLE);
    dim3 grid((unsigned)((c->h + 127) / 128), (unsigned)c->npairs);
    k_sample<<<grid, 128, 0, c->stream>>>(c->smp_seed, c->smp_stream, c->smp_offset, c->h, c->n,
                                          c->batched ? c->offsets.as<long long>() : nullptr, c->table.as<int32_t>());
    if (int r = check_launch(c, "k_sample")) return r;
    c->toc(T_SAMPLE);
    c->table_pending = false;
    return 0;
}

int sfm_sample_device(sfm_ctx* c, uint64_t seed, uint64_t stream, int64_t hyp_offset, int64_t h) {
    if (int r = use(c)) return r;
    return sample_device(c, seed, stream, hyp_offset, h);
}

int sfm_get_table(sfm_ctx* c, int32_t* table, int64_t first, int64_t h) {
    if (int r = use(c)) return r;
    if (!c->has_table || first < 0 || h < 0 || first + h > c->h * c->npairs)
        return fail(SFM_ERR_STATE, "no table rows [%lld, %lld)", (long long)first, (long long)(first + h));
    if (int r = ensure_table(c)) return r;
    CU(cudaMemcpyAsync(table, c->table.as<int32_t>() + 8 * first, (size_t)h * 32, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- correspondences --------------------------------------------------------------------
// K2's copy of c->pts (sfm_score.cuh, K2 header): the records of a single pair stably sorted by the Morton code of
// (xb, yb) quantised to 16 bits per axis inside the pair's B bounding box, and the box of every tile of kTile records.
// Only K2 reads it; every other kernel keeps the input order, and K2's integer sums do not depend on the order.
// Single pairs of at least kK2SortMin correspondences get it, and K2 then screens in 9 slots against the tile bounds.
// The sort is paid once per upload and costs 60-75 us below 100 000 correspondences, mostly launches; K2 saves about 7 %
// of its time per estimate, so the trade depends on N x H, which the upload does not know.  Measured for one upload plus
// one estimate (tools/sort_threshold.py, profiles/tile_screen_ab.txt): at 32 768 x 16 384 the sort cost 8.7 % end to
// end and at 65 536 x 16 384 2.8 %, while 65 536 x 65 536 gained 4.3 %, 131 072 x 16 384 1.8 % and config3
// (100 000 x 65 536) 0.36 ms.  So pairs below 65 536 keep the parent's path; single estimates just above it with few
// hypotheses pay up to ~3 %, and everything with more correspondences, more hypotheses or several estimates per upload
// gains.  Batches do not get
// the sorted copy: at 512 pairs x 2 000 (bench config4) a sort of the whole batch cost 0.19 ms per 1M records at upload
// and the 9-slot body was 1.5 % slower on K2 than the 11-slot one (the boxes of 2 000-point pairs are wide).
constexpr long long kK2SortMin = 65536;
static int k2_order(sfm_ctx* c, long long n) {
    size_t cub_bytes = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr,
                                       (int*)nullptr, (int)n, 0, 32, c->stream));
    const size_t vb = ((size_t)n * 4 + 255) & ~(size_t)255;  // one array of n keys or indices
    if (int r = c->k2sort.reserve(4 * vb + 256 + cub_bytes)) return r;
    char* w = c->k2sort.as<char>();
    auto* keys = reinterpret_cast<unsigned*>(w);
    auto* keys2 = reinterpret_cast<unsigned*>(w + vb);
    int* idx = reinterpret_cast<int*>(w + 2 * vb);
    int* idx2 = reinterpret_cast<int*>(w + 3 * vb);
    auto* bb = reinterpret_cast<unsigned long long*>(w + 4 * vb);
    void* tmp = w + 4 * vb + 256;
    const long long tiles = (n + kTile - 1) / kTile;
    if (int r = c->k2pts.reserve((size_t)n * sizeof(Corr))) return r;
    if (int r = c->k2box.reserve((size_t)tiles * sizeof(double4))) return r;
    CU(cudaMemsetAsync(bb, 0, 32, c->stream));
    const unsigned grid = (unsigned)((n + 255) / 256);
    k2_order_bbox<<<grid, 256, 0, c->stream>>>(c->pts.as<Corr>(), n, bb);
    if (int r = check_launch(c, "k2_order_bbox")) return r;
    k2_order_keys<<<grid, 256, 0, c->stream>>>(c->pts.as<Corr>(), n, bb, keys, idx);
    if (int r = check_launch(c, "k2_order_keys")) return r;
    CU(cub::DeviceRadixSort::SortPairs(tmp, cub_bytes, keys, keys2, idx, idx2, (int)n, 0, 32, c->stream));
    k2_order_gather<<<(unsigned)((tiles + kOrderWarps - 1) / kOrderWarps), 32 * kOrderWarps, 0, c->stream>>>(
        c->pts.as<Corr>(), n, idx2, c->k2pts.as<Corr>(), c->k2box.as<double4>());
    if (int r = check_launch(c, "k2_order_gather")) return r;
    c->k2_ready = true;
    return 0;
}

static int normalise_from(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                          int64_t stride, int64_t n, int64_t max_len) {
    if (int r = c->pts.reserve((size_t)n * sizeof(Corr))) return r;
    if (int r = c->bounds.reserve(16)) return r;
    CU(cudaMemsetAsync(c->bounds.p, 0, 16, c->stream));
    dim3 grid((unsigned)((max_len + 255) / 256), (unsigned)c->npairs);
    k_normalise<<<grid, 256, 0, c->stream>>>(xa, ya, xb, yb, stride, n,
                                             c->batched ? c->offsets.as<long long>() : nullptr,
                                             c->Ks.as<double>(), c->pts.as<Corr>(), c->bounds.as<unsigned long long>());
    if (int r = check_launch(c, "k_normalise")) return r;
    c->k2_ready = false;
    return (!c->batched && n >= kK2SortMin) ? k2_order(c, n) : 0;
}

// Host coordinates to the device buffer d (room for 4 n doubles) in the caller's layout: four arrays (stride 1) or two
// interleaved [n][2] arrays (stride 2).  s[] = the device addresses of xa, ya, xb, yb.
static int stage_coords(sfm_ctx* c, double* d, const double* xa, const double* ya, const double* xb, const double* yb,
                        int64_t stride, int64_t n, const double* s[4]) {
    if (stride == 1) {
        const double* src[4] = {xa, ya, xb, yb};
        for (int k = 0; k < 4; ++k)
            CU(cudaMemcpyAsync(d + (size_t)k * n, src[k], (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        s[0] = d; s[1] = d + n; s[2] = d + 2 * n; s[3] = d + 3 * n;
    } else if (stride == 2 && ya == xa + 1 && yb == xb + 1) {
        CU(cudaMemcpyAsync(d, xa, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(d + 2 * n, xb, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        s[0] = d; s[1] = d + 1; s[2] = d + 2 * n; s[3] = d + 2 * n + 1;
    } else {
        return fail(SFM_ERR_ARG, "unsupported layout: stride must be 1 (four arrays) or 2 (two interleaved [n][2] arrays)");
    }
    return 0;
}

// the device addresses of xa, ya, xb, yb of the current single-pair upload in c->raw (element i at [i * raw_stride])
static void raw_coords(const sfm_ctx* c, const double* s[4]) {
    const double* d = c->raw.as<double>();
    const long long n = c->n;
    if (c->raw_stride == 1) { s[0] = d; s[1] = d + n; s[2] = d + 2 * n; s[3] = d + 3 * n; }
    else { s[0] = d; s[1] = d + 1; s[2] = d + 2 * n; s[3] = d + 2 * n + 1; }
}

// the uploaded pixel coordinates, kept on the device for the triangulation tail
static int stage_raw(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                     int64_t stride, int64_t n, const double* s[4]) {
    if (int r = c->raw.reserve((size_t)n * 4 * sizeof(double))) return r;
    if (int r = stage_coords(c, c->raw.as<double>(), xa, ya, xb, yb, stride, n, s)) return r;
    c->raw_stride = stride;
    return 0;
}

// One pair's correspondences from host memory (stride 1 or 2) or from device memory (any stride, packed to stride 1).
static int upload_pairs_impl(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                             int64_t stride, int64_t n, const double* K, bool on_device, bool sync) {
    if (int r = use(c)) return r;
    if (!xa || !ya || !xb || !yb || !K) return fail(SFM_ERR_ARG, "null argument");
    if (n <= 0 || (uint64_t)n >= kMaxPoints) return fail(SFM_ERR_ARG, "need 0 < n < 2^25 correspondences, got %lld", (long long)n);
    c->tic(T_UPLOAD);
    c->batched = false;
    c->npairs = 1;
    const double* s[4];
    if (on_device) {
        if (int r = c->raw.reserve((size_t)n * 4 * sizeof(double))) return r;
        double* d = c->raw.as<double>();
        const double* src[4] = {xa, ya, xb, yb};
        for (int k = 0; k < 4; ++k) {
            CU(cudaMemcpy2DAsync(d + (size_t)k * n, sizeof(double), src[k], (size_t)stride * sizeof(double),
                                 sizeof(double), (size_t)n, cudaMemcpyDeviceToDevice, c->stream));
            s[k] = d + (size_t)k * n;
        }
        c->raw_stride = stride = 1;
    } else if (int r = stage_raw(c, xa, ya, xb, yb, stride, n, s)) {
        return r;
    }
    if (int r = c->Ks.reserve(9 * sizeof(double))) return r;
    memcpy(c->Khost, K, sizeof c->Khost);
    CU(cudaMemcpyAsync(c->Ks.p, c->Khost, 9 * sizeof(double), cudaMemcpyHostToDevice, c->stream));  // context-owned copy of K
    c->n = n;
    if (int r = normalise_from(c, s[0], s[1], s[2], s[3], stride, n, n)) return r;
    c->toc(T_UPLOAD);
    // the coordinate copies read caller memory: finish before returning unless the caller took that on (_async)
    if (sync) CU(cudaStreamSynchronize(c->stream));
    c->has_pts = true;
    c->has_table = c->has_models = c->has_score = false;
    c->table_pending = false;
    c->winner_set = false;
    return 0;
}

int sfm_upload_pairs(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                     int64_t stride, int64_t n, const double* K) {
    return upload_pairs_impl(c, xa, ya, xb, yb, stride, n, K, false, true);
}

int sfm_upload_pairs_async(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                           int64_t stride, int64_t n, const double* K) {
    return upload_pairs_impl(c, xa, ya, xb, yb, stride, n, K, false, false);
}

int sfm_upload_pairs_d(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                       int64_t stride, int64_t n, const double* K) {
    return upload_pairs_impl(c, xa, ya, xb, yb, stride, n, K, true, true);
}

int sfm_get_normalised(sfm_ctx* c, double* out, int64_t n) {
    if (int r = use(c)) return r;
    if (!c->has_pts || n > c->n) return fail(SFM_ERR_STATE, "no correspondences of that size");
    CU(cudaMemcpyAsync(out, c->pts.p, (size_t)n * sizeof(Corr), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- fit ----------------------------------------------------------------------------------
// K2's accumulator buffer is [kAccWords][H] planes followed by this tail, cleared with them: +0 work counter,
// +8 rescore counter, +16 pilot totals, +24 pilot ticket, +32 mode, +64 K3 tickets [P]
static size_t acc_tail_bytes(long long P) { return 64 + (size_t)P * 4; }

static int fit_launch(sfm_ctx* c, bool want_eig) {
    if (!c->has_pts || !c->has_table) return fail(SFM_ERR_STATE, "fit needs correspondences and a sample table");
    const size_t H = (size_t)c->h * c->npairs;
    if (int r = c->E.reserve(H * 9 * sizeof(double))) return r;
    if (int r = c->valid.reserve(H)) return r;
    if (want_eig)
        if (int r = c->eig.reserve(H * 9 * sizeof(double))) return r;
    if (int r = reserve_zeroed(c, c->fitflag, 16)) return r;  // K3 resets it after use
    if (int r = c->rows.reserve(H * sizeof(ModelRow))) return r;
    // K2's accumulators are cleared by the fit itself
    const size_t acc_tail = acc_tail_bytes(c->npairs);
    if (int r = c->acc.reserve(H * kAccWords * 8 + acc_tail)) return r;
    if (want_eig)
        if (int r = ensure_table(c)) return r;  // the Jacobi kernel reads the table
    c->tic(T_FIT);
    const long long* off = c->batched ? c->offsets.as<long long>() : nullptr;
    dim3 grid((unsigned)((c->h + kFitThreads - 1) / kFitThreads), (unsigned)c->npairs);
    const unsigned* only = nullptr;
    if (!want_eig) {
        // fast path: Householder null vector in registers; flags the (rare) samples whose validity
        // test is too close to call, which the Y^T Y Jacobi kernel then redoes
        dim3 gq((unsigned)((c->h + kFitQrThreads - 1) / kFitQrThreads), (unsigned)c->npairs);
        CU(chain_launch(c, k_fit_qr, gq, dim3(kFitQrThreads), 0, c->pts.as<Corr>(), off, c->table.as<int32_t>(), c->h,
                        c->E.as<double>(), c->valid.as<uint8_t>(), c->fitflag.as<unsigned>(), c->rows.as<ModelRow>(),
                        c->acc.as<unsigned long long>(), kAccWords, (int)((acc_tail + 7) / 8), c->table_pending ? 1 : 0,
                        c->smp_seed, c->smp_stream, c->smp_offset, c->n));
        if (int r = check_launch(c, "k_fit_qr")) return r;
        c->table_pending = false;  // the fit kernel wrote the rows it drew
        only = c->fitflag.as<unsigned>();
        c->acc_clean = true;
        c->acc_planes_for = H;
    } else {
        c->acc_clean = false;
    }
    CU(chain_launch(c, k_fit, grid, dim3(kFitThreads), kFitThreads * kFitSmemDoubles * sizeof(double), c->pts.as<Corr>(), off,
                    c->table.as<int32_t>(), c->h, c->E.as<double>(), c->valid.as<uint8_t>(),
                    want_eig ? c->eig.as<double>() : nullptr, only, c->rows.as<ModelRow>()));
    if (int r = check_launch(c, "k_fit")) return r;
    c->toc(T_FIT);
    c->has_models = true;
    c->models_h = false;
    c->has_score = false;
    return 0;
}

int sfm_fit(sfm_ctx* c, double* E_out, uint8_t* valid_out, double* eig_out) {
    if (int r = use(c)) return r;
    if (int r = fit_launch(c, eig_out != nullptr)) return r;
    const size_t H = (size_t)c->h * c->npairs;
    if (E_out) CU(cudaMemcpyAsync(E_out, c->E.p, H * 72, cudaMemcpyDeviceToHost, c->stream));
    if (valid_out) CU(cudaMemcpyAsync(valid_out, c->valid.p, H, cudaMemcpyDeviceToHost, c->stream));
    if (eig_out) CU(cudaMemcpyAsync(eig_out, c->eig.p, H * 72, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_get_models(sfm_ctx* c, int64_t first, int64_t count, double* E_out, uint8_t* valid_out) {
    if (int r = use(c)) return r;
    const int64_t total = c->h * c->npairs;
    if (!c->has_models || first < 0 || count < 0 || first + count > total)
        return fail(SFM_ERR_STATE, "no models [%lld, %lld)", (long long)first, (long long)(first + count));
    if (E_out) CU(cudaMemcpyAsync(E_out, c->E.as<double>() + 9 * first, (size_t)count * 72, cudaMemcpyDeviceToHost, c->stream));
    if (valid_out) CU(cudaMemcpyAsync(valid_out, c->valid.as<uint8_t>() + first, (size_t)count, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_set_models(sfm_ctx* c, const double* E, const uint8_t* valid, int64_t h) {
    if (int r = use(c)) return r;
    if (!E || h <= 0) return fail(SFM_ERR_ARG, "bad models");
    if (c->batched) return fail(SFM_ERR_STATE, "set_models is a single-pair call");
    if (c->has_table && h != c->h) return fail(SFM_ERR_ARG, "model count %lld != table rows %lld", (long long)h, c->h);
    if (int r = c->E.reserve((size_t)h * 72)) return r;
    if (int r = c->valid.reserve((size_t)h)) return r;
    CU(cudaMemcpyAsync(c->E.p, E, (size_t)h * 72, cudaMemcpyHostToDevice, c->stream));
    if (valid) CU(cudaMemcpyAsync(c->valid.p, valid, (size_t)h, cudaMemcpyHostToDevice, c->stream));
    else CU(cudaMemsetAsync(c->valid.p, 1, (size_t)h, c->stream));
    if (int r = c->rows.reserve((size_t)h * sizeof(ModelRow))) return r;
    k_pad_models<<<(unsigned)((h + 255) / 256), 256, 0, c->stream>>>(c->E.as<double>(), (long long)h, c->rows.as<ModelRow>());
    if (int r = check_launch(c, "k_pad_models")) return r;
    CU(cudaStreamSynchronize(c->stream));
    c->h = h;
    c->has_models = true;
    c->models_h = false;
    c->has_score = false;
    c->acc_clean = false;
    return 0;
}

// ---- score + select ---------------------------------------------------------------------
// K3's outputs for h hypotheses in each of P pairs.  Reserved before a scoring chain's first launch: a cudaMalloc
// between chained launches would break the chain.
static int reserve_selection(sfm_ctx* c, long long h, long long P) {
    const size_t H = (size_t)h * P;
    const int fblocks = (int)((h + 255) / 256);
    if (int r = c->count_extra.reserve(H * 4)) return r;
    if (int r = c->S1.reserve(H * 8)) return r;
    if (int r = c->S2.reserve(H * 8)) return r;
    if (int r = c->err.reserve(H * 8)) return r;
    if (int r = c->blocks.reserve((size_t)fblocks * P * sizeof(Best))) return r;
    if (int r = c->best.reserve((size_t)P * sizeof(Best))) return r;
    if (int r = c->invalid.reserve((size_t)P * 16)) return r;
    return 0;
}

// Work items of a persistent scoring launch: every (hypothesis block, pair) is split along the correspondences into
// nsplit chunks of `chunk` (a multiple of the tile), aiming at target_items items in all, keeping >= min_tiles tiles per
// item, and at most kMaxItemPoints correspondences per item so that 32-bit chunk sums cannot overflow.
struct ItemSplit { long long chunk, nsplit; };
static ItemSplit split_items(long long target_items, long long hyp_items, long long max_len, long long tile) {
    const long long tiles = (max_len + tile - 1) / tile;
    long long nsplit = (target_items + hyp_items - 1) / hyp_items;
    constexpr int min_tiles = 2;  // 8 -> 2: mid-size pairs (config 2) get enough items to balance the warps (+6 %)
    const long long max_split = tiles / min_tiles > 0 ? tiles / min_tiles : 1;
    if (nsplit > max_split) nsplit = max_split;
    const long long min_split = (max_len + kMaxItemPoints - 1) / kMaxItemPoints;
    if (nsplit < min_split) nsplit = min_split;
    if (nsplit < 1) nsplit = 1;
    const long long chunk = ((tiles + nsplit - 1) / nsplit) * tile;
    nsplit = (max_len + chunk - 1) / chunk;
    if (nsplit < 1) nsplit = 1;
    return {chunk, nsplit};
}

// The fit kernels leave the accumulators cleared; a second score of the same models (or of uploaded models) clears here.
static int clear_acc(sfm_ctx* c, size_t H, long long P) {
    if (!(c->acc_clean && c->acc_planes_for == H))
        CU(cudaMemsetAsync(c->acc.p, 0, H * kAccWords * 8 + acc_tail_bytes(P), c->stream));
    c->acc_clean = false;
    return 0;
}

// K3 of a scoring call (essential matrices or homographies): finalise, rescore, select into the selection record
static int finalise_launch(sfm_ctx* c, int kind, double thr, double min_extra, int agg, int mode, bool use_table,
                           long long idx_offset, int sums, int e2, int force_rescore, unsigned long long* acc_dev) {
    const long long h = c->h, P = c->npairs;
    const size_t H = (size_t)h * P;
    const int fblocks = (int)((h + 255) / 256);
    c->tic(T_SELECT);
    FinalArgs f;
    f.pts = c->pts.as<Corr>();
    f.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    f.E = c->E.as<double>();
    f.valid = c->valid.as<uint8_t>();
    f.table = use_table ? c->table.as<int32_t>() : nullptr;
    f.h = h;
    f.n = c->n;
    f.idx_offset = idx_offset;
    f.htotal = (long long)H;
    f.acc = acc_dev;
    f.inv_scale1 = ldexp(1.0, e2 - kFixedBits);
    f.sums = sums;
    f.inv_scale2 = ldexp(1.0, 2 * e2 - kFixedBits);
    f.thr = thr;
    f.min_extra = min_extra;
    f.agg = agg;
    f.mode = mode;
    f.count_extra = c->count_extra.as<int32_t>();
    f.S1 = c->S1.as<double>();
    f.S2 = c->S2.as<double>();
    f.err = c->err.as<double>();
    f.block_out = c->blocks.as<Best>();
    if (int r = c->blockinv.reserve((size_t)fblocks * P * 16)) return r;
    f.block_inv = c->blockinv.as<long long>();
    if (int r = c->record.reserve((size_t)P * sizeof(SelectRecord))) return r;
    f.force_rescore = force_rescore;
    f.rescored = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(acc_dev + H * kAccWords) + 8);
    f.tickets = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(acc_dev + H * kAccWords) + 64);
    c->rescored_dev = f.rescored;
    f.out = c->best.as<Best>();
    f.invalid_out = c->invalid.as<long long>();
    f.record = c->record.as<SelectRecord>();
    f.fitflag = c->fitflag.as<unsigned>();
    if (kind == MODEL_H) CU(chain_launch(c, k_finalise<MODEL_H>, dim3((unsigned)fblocks, (unsigned)P), dim3(256), 0, f));
    else CU(chain_launch(c, k_finalise<MODEL_E>, dim3((unsigned)fblocks, (unsigned)P), dim3(256), 0, f));
    if (int r = check_launch(c, "k_finalise")) return r;
    c->toc(T_SELECT);
    c->has_score = true;
    c->last_idx_offset = idx_offset;
    c->winner_set = false;
    return 0;
}

static int score_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, bool use_table,
                        long long idx_offset, long long max_len, bool both_sums = false) {
    // K2 accumulates only the sum the aggregation needs (ransac.py:96-108) unless the caller wants both
    int sums = both_sums ? (SUM_S1 | SUM_S2) : ((agg == AGG_SUM || agg == AGG_MEAN) ? SUM_S1 : SUM_S2);
    if (mode == SELECT_MSAC) sums |= SUM_S1;  // the MSAC cost is built from the sum of the inlier distances
    if (!c->has_pts || !c->has_models) return fail(SFM_ERR_STATE, "score needs correspondences and fitted models");
    if (c->models_h) return fail(SFM_ERR_STATE, "the models are homographies: score them with sfm_ransac_homography");
    if (use_table && !c->has_table) return fail(SFM_ERR_STATE, "sample rule requested but no table is loaded");
    if (use_table)
        if (int r = ensure_table(c)) return r;
    if (agg < 0 || agg > 3) return fail(SFM_ERR_ARG, "bad aggregation %d", agg);
    if (mode < 0 || mode > 2) return fail(SFM_ERR_ARG, "bad selection %d", mode);
    // ransac.py accepts any float: a negative (or NaN) threshold means "no extra inliers" (score <= thr is never true),
    // +inf "every finite score".  K2's fixed-point sums cover thresholds up to 1e100; outside that range K2 is
    // skipped and K3 counts and sums every hypothesis with its exact double-double pass.
    const bool skip_k2 = !(thr >= 0.0) || thr > 1e100;
    const int force_rescore = (thr > 1e100) ? 1 : 0;
    const long long h = c->h, P = c->npairs;
    const int hpt = (c->variant == SFM_SCORE_SCREEN32 && thr > 1e6) ? 2 : c->hpt;
    const int G = (c->variant == SFM_SCORE_SCREEN32 && thr > 1e6) ? 16 : c->group;
    const long long hblocks = (h + 32ll * hpt - 1) / (32ll * hpt);  // groups of 32*hpt hypotheses (one per warp item)
    const size_t H = (size_t)h * P;
    if (int r = reserve_selection(c, h, P)) return r;
    int e2 = 0;
    if (thr > 0.0 && !skip_k2) (void)frexp(thr, &e2);  // thr = m * 2^e2, m in [0.5, 1)  =>  thr < 2^e2
    if (e2 < -400) e2 = -400;
    // rounding guard of the screening tests: relative slack + an absolute term that covers a
    // cancelling residual r at the 1-ulp level (only matters for thr -> 0)
    // the fp32 pre-filter needs s = sqrt(thr32) and 1/s inside the fp32 range: huge thresholds use the fp64 screen
    // AUTO: the one-sided screen is prepared as usual; a pilot (k_pilot, or riding on the screening-copy kernel)
    // measures its survivor rate and k_score_auto runs the one-sided or the two-sided body
    const bool autov = c->variant == SFM_SCORE_AUTO;
    int variant = autov ? SFM_SCORE_SCREEN : c->variant;
    if (variant == SFM_SCORE_SCREEN32 && thr > 1e6) variant = SFM_SCORE_SCREEN;  // with hpt 2 / group 16, see above
    const bool f32 = variant == SFM_SCORE_SCREEN32;
    const bool screen = variant != SFM_SCORE_FULL;
    // SCREEN: relative guard here, absolute guard = kappa_h inside the kernel (see sfm_score.cuh);
    // SCREEN32: thr32 = 1.0316 thr, kappa32; FULL: relative guard + an absolute term that covers a
    // cancelling residual at the 1-ulp level
    double thr_pre = f32 ? thr * kThr32Factor : (screen ? thr * kThrScreenFactor : thr * (1.0 + 1e-9) + 1e-22);
    if (f32 && thr_pre < 1e-24) thr_pre = 1e-24;  // keeps s and 1/s comfortably inside fp32; only widens the screen
    if (screen && thr_pre < 1e-280) thr_pre = 1e-280;  // keeps thr' NB+ clear of underflow; only widens the screen
    const double s_scale = sqrt(thr_pre);
    const double scale1 = ldexp(1.0, 63 - e2), scale2 = ldexp(1.0, 63 - 2 * e2);
    unsigned long long* acc_dev = nullptr;
    {
        // persistent blocks over (pair, split, hypothesis block) items
        const bool tiles = c->k2_ready;
        const ScoreKernel sk = score_kernel(autov ? SFM_SCORE_AUTO : variant, hpt, G, tiles);
        if (!sk.fn) return fail(SFM_ERR_ARG, "unsupported scoring configuration (variant %d, hpt %d, group %d)", variant, hpt, G);
        const size_t smem = (size_t)kScoreWarps * sk.warp_bytes;
        // attribute set and occupancy queried once per kernel instantiation (small cache)
        int occ = 0;
        for (int k = 0; k < 4 && !occ; ++k)
            if (c->occ_fn[k] == sk.fn) occ = c->occ_blocks[k];
        if (!occ) {
            CU(cudaFuncSetAttribute(sk.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sk.fn, kScoreThreads, smem));
            if (occ < 1) occ = 1;
            c->occ_fn[c->occ_next] = sk.fn;
            c->occ_blocks[c->occ_next] = occ;
            c->occ_next = (c->occ_next + 1) & 3;
        }
        const long long grid_blocks = (long long)c->sm_count * occ;
        constexpr int items_per_warp = 32;  // 12 -> 32 shortens the end-of-launch tail (+1 % on config 3)
        const ItemSplit sp = split_items(grid_blocks * kScoreWarps * items_per_warp, hblocks * P, max_len, kTile);
        const long long chunk = sp.chunk, nsplit = sp.nsplit;
        const long long total_items = hblocks * nsplit * P;
        if (int r = c->acc.reserve(H * kAccWords * 8 + acc_tail_bytes(P))) return r;
        const long long npts = c->n;  // total records (all pairs)
        const bool scaled = screen && !f32 && !tiles;  // the 11-slot screen streams a scaled copy
        if (f32) { if (int r = c->spts.reserve((size_t)npts * sizeof(Corr32))) return r; }
        else if (scaled) { if (int r = c->spts.reserve((size_t)npts * sizeof(Corr))) return r; }
        // only the 9-slot body streams the sorted copy; the others keep the input order (sorting by image-B position
        // clusters a hypothesis' survivors into the same batches, which the two-sided body's rounds pay for)
        const Corr* kpts = (tiles && screen && !f32) ? c->k2pts.as<Corr>() : c->pts.as<Corr>();
        ScoreArgs a;
        a.pts = kpts;
        a.spts = (f32 || scaled) ? c->spts.p : (const void*)kpts;
        a.boxes = tiles ? c->k2box.as<double4>() : nullptr;
        a.bounds = c->bounds.as<double>();
        a.s = s_scale;
        a.kappa_coef = kKappaCoef * (1.0 + thr);
        a.kappa32_coef = kKappa32Coef * (1.0 + thr);
        a.n = c->n;
        a.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
        a.E = c->E.as<double>();
        a.rows = c->rows.as<ModelRow>();  // written by the fit kernels / sfm_set_models
        a.h = h;
        a.thr = thr;
        a.thr_pre = thr_pre;
        a.scale1 = scale1;
        a.scale2 = scale2;
        a.sums = sums;
        a.chunk = chunk;
        a.hblocks = (int)hblocks;
        a.nsplit = (int)nsplit;
        a.total_items = total_items;
        a.htotal = (long long)H;
        a.acc = c->acc.as<unsigned long long>();
        a.work_counter = reinterpret_cast<unsigned*>(a.acc + H * kAccWords);
        char* tailp = reinterpret_cast<char*>(a.acc + H * kAccWords);  // see acc_tail_bytes
        a.mode_flag = autov ? reinterpret_cast<const int*>(tailp + 32) : nullptr;
        acc_dev = a.acc;
        c->tic(T_SCORE);
        if (int r = clear_acc(c, H, P)) return r;
        if (f32 && !skip_k2) {
            k_screen_pts32<<<(unsigned)((npts + 255) / 256), 256, 0, c->stream>>>(kpts, npts, 1.0 / s_scale,
                                                                                  reinterpret_cast<Corr32*>(c->spts.p));
            if (int r = check_launch(c, "k_screen_pts32")) return r;
        }
        else if ((scaled || autov) && !skip_k2) {
            PilotArgs pa;
            pa.E = c->E.as<double>();
            pa.h = h;
            pa.plen = c->batched ? c->first_len : c->n;  // batches: the pilot looks at the first pair
            pa.thr_pre = thr_pre;
            pa.bounds = a.bounds;
            pa.kappa_coef = a.kappa_coef;
            pa.boxes = a.boxes;
            pa.counters = reinterpret_cast<unsigned*>(tailp + 16);
            pa.mode_flag = autov ? reinterpret_cast<int*>(tailp + 32) : nullptr;
            const long long copy_blocks = (npts + 255) / 256;
            if (scaled) {  // the copy carries the pilot
                CU(chain_launch(c, k_screen_pts64, dim3((unsigned)copy_blocks), dim3(256), 0, kpts, npts, 1.0 / s_scale,
                                reinterpret_cast<Corr*>(c->spts.p), pa));
                if (int r = check_launch(c, "k_screen_pts64")) return r;
            } else {
                CU(chain_launch(c, k_pilot, dim3((unsigned)(copy_blocks < kPilotBlocks ? copy_blocks : kPilotBlocks)), dim3(256),
                                0, kpts, pa));
                if (int r = check_launch(c, "k_pilot")) return r;
            }
        }
        const long long want_blocks = (total_items + kScoreWarps - 1) / kScoreWarps;
        const long long launch_blocks = grid_blocks < want_blocks ? grid_blocks : want_blocks;
        if (!skip_k2 && autov) {
            ScoreArgs a2 = a;  // the two-sided body: its guard, on the unscaled records
            a2.thr_pre = thr * (1.0 + 1e-9) + 1e-22;
            a2.pts = c->pts.as<Corr>();
            a2.spts = a2.pts;
            void* kargs[] = {(void*)&a, (void*)&a2};
            CU(chain_launch_ptr(c, sk.fn, dim3((unsigned)launch_blocks), dim3(kScoreThreads), smem, kargs));
            if (int r = check_launch(c, "k_score_auto")) return r;
        } else if (!skip_k2) {
            void* kargs[] = {(void*)&a};
            CU(chain_launch_ptr(c, sk.fn, dim3((unsigned)launch_blocks), dim3(kScoreThreads), smem, kargs));
            if (int r = check_launch(c, "k_score")) return r;
        }
        c->toc(T_SCORE);
    }

    return finalise_launch(c, MODEL_E, thr, min_extra, agg, mode, use_table, idx_offset, sums, e2, force_rescore, acc_dev);
}

int sfm_score(sfm_ctx* c, double thr, double min_extra, int agg, int mode, int use_table, int64_t idx_offset,
              int32_t* count_extra, double* S1, double* S2, double* err) {
    if (int r = use(c)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "sfm_score is a single-pair call; use sfm_batch_ransac");
    if (int r = score_launch(c, thr, min_extra, agg, mode, use_table != 0, idx_offset, c->n, S1 || S2)) return r;
    const size_t H = (size_t)c->h;
    if (count_extra) CU(cudaMemcpyAsync(count_extra, c->count_extra.p, H * 4, cudaMemcpyDeviceToHost, c->stream));
    if (S1) CU(cudaMemcpyAsync(S1, c->S1.p, H * 8, cudaMemcpyDeviceToHost, c->stream));
    if (S2) CU(cudaMemcpyAsync(S2, c->S2.p, H * 8, cudaMemcpyDeviceToHost, c->stream));
    if (err) CU(cudaMemcpyAsync(err, c->err.p, H * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// a selection record as the ABI's sfm_best; without a winner (index < 0) the error reads inf
static void unpack_best(const SelectRecord& r, sfm_best* out) {
    out->err = r.best.idx >= 0 ? r.best.err : __builtin_inf();
    out->index = r.best.idx;
    out->count_extra = r.best.count;
    out->reserved = 0;
    out->num_invalid = r.num_invalid;
    out->first_invalid = r.first_invalid;
    memcpy(out->E, r.E, 72);
    memcpy(out->sample, r.sample, 32);
}

static int fetch_best(sfm_ctx* c, sfm_best* out) {
    // k_select left {best, invalid counters, winning E} in one record: one copy, one synchronisation
    if (int r = ensure_pinned(c, sizeof(SelectRecord))) return r;
    CU(cudaMemcpyAsync(c->hpin, c->record.p, sizeof(SelectRecord), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    SelectRecord r;
    memcpy(&r, c->hpin, sizeof r);
    unpack_best(r, out);
    if (r.best.idx >= 0) {
        c->winner_local = r.best.idx - c->last_idx_offset;
        c->winner_set = true;
    }
    return 0;
}

int sfm_get_best(sfm_ctx* c, sfm_best* out) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    if (!c->has_score || c->batched) return fail(SFM_ERR_STATE, "no single-pair score to read");
    return fetch_best(c, out);
}

int sfm_near_ties(sfm_ctx* c, double rel_tol, int64_t cap, int64_t* idx_out, int64_t* count) {
    if (int r = use(c)) return r;
    if (!idx_out || !count || cap <= 0 || cap > 4096) return fail(SFM_ERR_ARG, "bad near-tie arguments");
    if (!c->has_score || c->batched) return fail(SFM_ERR_STATE, "no single-pair score to read");
    if (int r = c->tmp.reserve((size_t)cap * 8 + 16)) return r;
    unsigned* cnt = c->tmp.as<unsigned>();
    long long* out = reinterpret_cast<long long*>(c->tmp.as<char>() + 16);
    CU(cudaMemsetAsync(cnt, 0, 16, c->stream));
    const int blocks = (int)((c->h + 255) / 256 < 4 * c->sm_count ? (c->h + 255) / 256 : 4 * c->sm_count);
    k_near_ties<<<blocks, 256, 0, c->stream>>>(c->err.as<double>(), c->h, c->record.as<SelectRecord>(), rel_tol, (int)cap, out, cnt);
    if (int r = check_launch(c, "k_near_ties")) return r;
    if (int r = ensure_pinned(c, (size_t)cap * 8 + 16)) return r;
    CU(cudaMemcpyAsync(c->hpin, c->tmp.p, (size_t)cap * 8 + 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    unsigned n;
    memcpy(&n, c->hpin, 4);
    *count = n;  // may exceed cap: only the first cap entries were kept
    const int64_t take = n < (unsigned)cap ? n : cap;
    memcpy(idx_out, (char*)c->hpin + 16, (size_t)take * 8);
    return 0;
}

int sfm_get_rescored(sfm_ctx* c, int64_t* count) {
    if (int r = use(c)) return r;
    if (!count) return fail(SFM_ERR_ARG, "null argument");
    if (!c->rescored_dev) return fail(SFM_ERR_STATE, "no scoring call yet");
    if (int r = ensure_pinned(c, 8)) return r;
    CU(cudaMemcpyAsync(c->hpin, c->rescored_dev, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    unsigned long long v;
    memcpy(&v, c->hpin, 8);
    *count = (int64_t)v;
    return 0;
}

int sfm_set_winner(sfm_ctx* c, int64_t local_index, const double* E) {
    if (int r = use(c)) return r;
    if (local_index >= 0) {
        if (!c->has_models || local_index >= c->h) return fail(SFM_ERR_ARG, "winner index out of range");
        c->winner_local = local_index;
    } else {
        if (!E) return fail(SFM_ERR_ARG, "need the winning model when it lives on another rank");
        if (int r = c->winnerE.reserve(72)) return r;
        CU(cudaMemcpyAsync(c->winnerE.p, E, 72, cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->winner_local = -1;
    }
    c->winner_set = true;
    return 0;
}

static const double* winner_E_dev(sfm_ctx* c) {
    return c->winner_local >= 0 ? c->E.as<double>() + 9 * c->winner_local : c->winnerE.as<double>();
}

static int mask_launch(sfm_ctx* c, double thr, const Best* best_dev, const double* E_override = nullptr) {
    if (int r = c->mask.reserve((size_t)c->n)) return r;
    if (int r = c->sed.reserve((size_t)c->n * 8)) return r;
    c->tic(T_MASK);
    // E_override: one model on the device (the merged winner of a sharded run), used as is
    const double* E = E_override ? E_override : (best_dev ? c->E.as<double>() : winner_E_dev(c));
    k_inlier_mask<<<(unsigned)((c->n + 255) / 256), 256, 0, c->stream>>>(
        c->pts.as<Corr>(), c->n, E, E_override ? nullptr : best_dev, c->last_idx_offset, 0, thr, c->mask.as<uint8_t>(),
        c->sed.as<double>());
    if (int r = check_launch(c, "k_inlier_mask")) return r;
    c->toc(T_MASK);
    return 0;
}

int sfm_inlier_mask(sfm_ctx* c, double thr, uint8_t* mask, double* sed) {
    if (int r = use(c)) return r;
    if (!c->has_pts || c->batched) return fail(SFM_ERR_STATE, "no single-pair correspondences loaded");
    if (!c->winner_set) return fail(SFM_ERR_STATE, "no winner: call sfm_get_best or sfm_set_winner first");
    if (c->models_h && c->winner_local >= 0) return fail(SFM_ERR_STATE, "the winner is a homography: use sfm_homography_mask");
    if (int r = mask_launch(c, thr, nullptr)) return r;
    if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    if (sed) CU(cudaMemcpyAsync(sed, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_ransac_essential(sfm_ctx* c, double thr, double min_extra, int agg, int mode, sfm_best* best,
                         uint8_t* mask, double* sed) {
    if (int r = use(c)) return r;
    if (!best) return fail(SFM_ERR_ARG, "best is null");
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, c->n)) return r;
    if (mask || sed) {
        if (int r = mask_launch(c, thr, c->best.as<Best>())) return r;
        if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
        if (sed) CU(cudaMemcpyAsync(sed, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    return fetch_best(c, best);
}

// ---- homography (sfm_homography.cuh) -------------------------------------------------------
// the 4-point fits of h hypotheses in each pair of the upload (a batch: device-sampler rows only)
static int fit_h_launch(sfm_ctx* c) {
    if (!c->has_pts || !c->has_table) return fail(SFM_ERR_STATE, "fit needs correspondences and a sample table");
    if (c->batched && !c->table_pending) return fail(SFM_ERR_STATE, "a batch is fitted from the device sampler's draw");
    const long long h = c->h, P = c->npairs;
    const size_t H = (size_t)h * P;
    if (int r = c->E.reserve(H * 72)) return r;
    if (int r = c->valid.reserve(H)) return r;
    const size_t acc_tail = acc_tail_bytes(P);
    if (int r = c->acc.reserve(H * kAccWords * 8 + acc_tail)) return r;
    c->tic(T_FIT);
    CU(chain_launch(c, k_fit_homography, dim3((unsigned)((h + kFitHThreads - 1) / kFitHThreads), (unsigned)P),
                    dim3(kFitHThreads), 0, c->pts.as<Corr>(), c->batched ? c->offsets.as<long long>() : nullptr,
                    c->table.as<int32_t>(), h, c->E.as<double>(), c->valid.as<uint8_t>(), c->acc.as<unsigned long long>(),
                    kAccWords, (int)((acc_tail + 7) / 8), c->table_pending ? 1 : 0, c->smp_seed, c->smp_stream,
                    c->smp_offset, c->n));
    if (int r = check_launch(c, "k_fit_homography")) return r;
    c->toc(T_FIT);
    c->table_pending = false;
    c->acc_clean = true;
    c->acc_planes_for = H;
    c->has_models = true;
    c->models_h = true;
    c->has_score = false;
    return 0;
}

// K2 + K3 of homographies over every pair of the upload; max_len = the longest pair
static int score_h_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, long long max_len) {
    if (agg < 0 || agg > 3) return fail(SFM_ERR_ARG, "bad aggregation %d", agg);
    if (mode < 0 || mode > 2) return fail(SFM_ERR_ARG, "bad selection %d", mode);
    int sums = (agg == AGG_SUM || agg == AGG_MEAN) ? SUM_S1 : SUM_S2;
    if (mode == SELECT_MSAC) sums |= SUM_S1;
    // the same threshold ranges as the E path: below 0, NaN and above 1e100 the scorer is skipped and K3 rescores
    const bool skip_k2 = !(thr >= 0.0) || thr > 1e100;
    const int force_rescore = (thr > 1e100) ? 1 : 0;
    const long long h = c->h, n = c->n, P = c->npairs;
    const size_t H = (size_t)h * P;
    // an inlier's value F/P + G/Q can exceed thr by a few ulps (the decision is division-free): the fixed-point scale
    // leaves room for that, value < thr (1 + 2^-20) < 2^e2
    int e2 = 0;
    if (thr > 0.0 && !skip_k2) (void)frexp(thr * (1.0 + 0x1p-20), &e2);
    if (e2 < -400) e2 = -400;
    if (int r = reserve_selection(c, h, P)) return r;
    if (int r = c->acc.reserve(H * kAccWords * 8 + acc_tail_bytes(P))) return r;
    unsigned long long* acc = c->acc.as<unsigned long long>();
    const size_t smem = kHScoreWarps * sizeof(HScoreWarpSmem);
    if (!c->hscore_occ) {
        int o = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_score_homography<kHScoreHpt>, kHScoreThreads, smem));
        c->hscore_occ = o > 0 ? o : 1;
    }
    // persistent warps over (pair, correspondence split, group of 32 * HPT hypotheses) items
    const long long grid_blocks = (long long)c->sm_count * c->hscore_occ;
    const long long hblocks = (h + 32ll * kHScoreHpt - 1) / (32ll * kHScoreHpt);
    const ItemSplit sp = split_items(grid_blocks * kHScoreWarps * 32, hblocks * P, max_len, kHTile);
    const long long chunk = sp.chunk, nsplit = sp.nsplit;
    HScoreArgs a;
    a.pts = c->pts.as<Corr>();
    a.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    a.H = c->E.as<double>();
    a.n = n;
    a.h = h;
    a.htotal = (long long)H;
    a.thr = thr;
    a.scale1 = ldexp(1.0, 63 - e2);
    a.scale2 = ldexp(1.0, 63 - 2 * e2);
    a.sums = sums;
    a.chunk = chunk;
    a.hblocks = (int)hblocks;
    a.nsplit = (int)nsplit;
    a.total_items = hblocks * nsplit * P;
    a.work_counter = reinterpret_cast<unsigned*>(acc + H * kAccWords);
    a.acc = acc;
    c->tic(T_SCORE);
    if (int r = clear_acc(c, H, P)) return r;
    if (!skip_k2) {
        const long long want = (a.total_items + kHScoreWarps - 1) / kHScoreWarps;
        CU(chain_launch(c, k_score_homography<kHScoreHpt>, dim3((unsigned)(grid_blocks < want ? grid_blocks : want)),
                        dim3(kHScoreThreads), smem, a));
        if (int r = check_launch(c, "k_score_homography")) return r;
    }
    c->toc(T_SCORE);
    return finalise_launch(c, MODEL_H, thr, min_extra, agg, mode, true, 0, sums, e2, force_rescore, acc);
}

static int hmask_launch(sfm_ctx* c, double thr, const double* H_dev, const Best* best_dev) {
    if (int r = c->mask.reserve((size_t)c->n)) return r;
    if (int r = c->sed.reserve((size_t)c->n * 8)) return r;
    c->tic(T_MASK);
    CU(chain_launch(c, k_homography_mask, dim3((unsigned)((c->n + 255) / 256)), dim3(256), 0, c->pts.as<Corr>(), c->n,
                    H_dev, best_dev, thr, c->mask.as<uint8_t>(), c->sed.as<double>()));
    if (int r = check_launch(c, "k_homography_mask")) return r;
    c->toc(T_MASK);
    return 0;
}

int sfm_fit_homography(sfm_ctx* c, double* H_out, uint8_t* valid_out) {
    if (int r = use(c)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "homography estimation is a single-pair call; use sfm_batch_two_view_homography");
    if (int r = fit_h_launch(c)) return r;
    if (H_out) CU(cudaMemcpyAsync(H_out, c->E.p, (size_t)c->h * 72, cudaMemcpyDeviceToHost, c->stream));
    if (valid_out) CU(cudaMemcpyAsync(valid_out, c->valid.p, (size_t)c->h, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_ransac_homography(sfm_ctx* c, double thr, double min_extra, int agg, int mode, sfm_best* best, uint8_t* mask,
                          double* err, int32_t* count_extra_h, double* err_h) {
    if (int r = use(c)) return r;
    if (!best) return fail(SFM_ERR_ARG, "best is null");
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (c->has_pts && c->n < 8) return fail(SFM_ERR_ARG, "need at least 8 correspondences, got %lld", c->n);
    if (int r = fit_h_launch(c)) return r;
    if (int r = score_h_launch(c, thr, min_extra, agg, mode, c->n)) return r;
    if (mask || err) {
        if (int r = hmask_launch(c, thr, c->E.as<double>(), c->best.as<Best>())) return r;
        if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
        if (err) CU(cudaMemcpyAsync(err, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    if (count_extra_h) CU(cudaMemcpyAsync(count_extra_h, c->count_extra.p, (size_t)c->h * 4, cudaMemcpyDeviceToHost, c->stream));
    if (err_h) CU(cudaMemcpyAsync(err_h, c->err.p, (size_t)c->h * 8, cudaMemcpyDeviceToHost, c->stream));
    return fetch_best(c, best);
}

int sfm_homography_mask(sfm_ctx* c, const double* H, double thr, uint8_t* mask, double* err) {
    if (int r = use(c)) return r;
    if (!c->has_pts || c->batched) return fail(SFM_ERR_STATE, "no single-pair correspondences loaded");
    const double* H_dev;
    if (H) {
        if (int r = c->winnerE.reserve(72)) return r;
        CU(cudaMemcpyAsync(c->winnerE.p, H, 72, cudaMemcpyHostToDevice, c->stream));
        H_dev = c->winnerE.as<double>();
    } else {
        if (!c->models_h || !c->winner_set || c->winner_local < 0)
            return fail(SFM_ERR_STATE, "no homography winner: pass H or run sfm_ransac_homography first");
        H_dev = c->E.as<double>() + 9 * c->winner_local;
    }
    if (int r = hmask_launch(c, thr, H_dev, nullptr)) return r;
    if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    if (err) CU(cudaMemcpyAsync(err, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- pose + triangulation ---------------------------------------------------------------
int sfm_decompose_essential(sfm_ctx* c, const double* E, sfm_poses* out) {
    if (int r = use(c)) return r;
    if (!E || !out) return fail(SFM_ERR_ARG, "null argument");
    if (int r = c->tmp.reserve(72)) return r;
    if (int r = c->poses.reserve(sizeof(PoseSet))) return r;
    CU(cudaMemcpyAsync(c->tmp.p, E, 72, cudaMemcpyHostToDevice, c->stream));
    k_decompose<<<1, 32, 0, c->stream>>>(c->tmp.as<double>(), nullptr, 0, c->poses.as<PoseSet>(), 1);
    if (int r = check_launch(c, "k_decompose")) return r;
    CU(cudaMemcpyAsync(out, c->poses.p, sizeof(PoseSet), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

static int recover_pose_impl(sfm_ctx* c, const double* E, const double* K9, const double* xa, const double* ya,
                             const double* xb, const double* yb, int64_t stride, int64_t m, double dist_thr,
                             sfm_poses* out, uint8_t* pass4) {
    if (int r = use(c)) return r;
    if (!E || !out) return fail(SFM_ERR_ARG, "null argument");
    if (m < 0) return fail(SFM_ERR_ARG, "negative count");
    if (int r = c->tmp.reserve(72 + 9 * 8 + (size_t)m * 4 * 8 + (size_t)m * sizeof(Corr) + 64)) return r;
    if (int r = c->poses.reserve(sizeof(PoseSet))) return r;
    if (int r = c->pass.reserve((size_t)m + 1)) return r;
    c->tic(T_POSE);
    double* dE = c->tmp.as<double>();
    double* dK = dE + 9;
    double* draw = dK + 9;
    Corr* dpts = reinterpret_cast<Corr*>(((uintptr_t)(draw + 4 * m) + 31) & ~(uintptr_t)31);
    CU(cudaMemcpyAsync(dE, E, 72, cudaMemcpyHostToDevice, c->stream));
    k_decompose<<<1, 32, 0, c->stream>>>(dE, nullptr, 0, c->poses.as<PoseSet>(), 1);
    if (int r = check_launch(c, "k_decompose")) return r;
    if (m > 0) {
        if (!xa || !ya || !xb || !yb) return fail(SFM_ERR_ARG, "null coordinates");
        // K9 == null: the inputs are already K-normalised and are packed into Corr records with an identity K;
        // otherwise k_normalise applies eight_point.py:127-133 on the device (bit-identical IEEE operations)
        const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        memcpy(c->Kstage, K9 ? K9 : I, 72);  // staged in the context: the async copy must not read caller memory later
        CU(cudaMemcpyAsync(dK, c->Kstage, 72, cudaMemcpyHostToDevice, c->stream));
        const double* s[4];
        if (int r = stage_coords(c, draw, xa, ya, xb, yb, stride, m, s)) return r;
        k_normalise<<<dim3((unsigned)((m + 255) / 256), 1), 256, 0, c->stream>>>(s[0], s[1], s[2], s[3], stride, m, nullptr, dK, dpts, nullptr);
        if (int r = check_launch(c, "k_normalise")) return r;
        k_cheirality<<<(unsigned)((4 * m + 127) / 128), 128, 0, c->stream>>>(dpts, m, nullptr, nullptr, c->poses.as<PoseSet>(),
                                                                        dist_thr, c->pass.as<uint8_t>(), nullptr);
        if (int r = check_launch(c, "k_cheirality")) return r;
    }
    k_vote<<<1, 32, 0, c->stream>>>(c->poses.as<PoseSet>());
    if (int r = check_launch(c, "k_vote")) return r;
    c->toc(T_POSE);
    CU(cudaMemcpyAsync(out, c->poses.p, sizeof(PoseSet), cudaMemcpyDeviceToHost, c->stream));
    if (pass4 && m > 0) CU(cudaMemcpyAsync(pass4, c->pass.p, (size_t)m, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_recover_pose(sfm_ctx* c, const double* E, const double* xa, const double* ya, const double* xb,
                     const double* yb, int64_t stride, int64_t m, double dist_thr, sfm_poses* out,
                     uint8_t* pass4) {
    return recover_pose_impl(c, E, nullptr, xa, ya, xb, yb, stride, m, dist_thr, out, pass4);
}

int sfm_recover_pose_pixels(sfm_ctx* c, const double* E, const double* K, const double* xa, const double* ya,
                            const double* xb, const double* yb, int64_t stride, int64_t m, double dist_thr,
                            sfm_poses* out, uint8_t* pass4) {
    if (!K) return fail(SFM_ERR_ARG, "null camera matrix");
    return recover_pose_impl(c, E, K, xa, ya, xb, yb, stride, m, dist_thr, out, pass4);
}

int sfm_triangulate(sfm_ctx* c, const double* P1, const double* P2, const double* xa, const double* ya,
                    const double* xb, const double* yb, int64_t stride, int64_t m, double* X) {
    if (int r = use(c)) return r;
    if (!P1 || !P2 || !X) return fail(SFM_ERR_ARG, "null argument");
    if (m <= 0) return m == 0 ? 0 : fail(SFM_ERR_ARG, "negative count");
    if (!xa || !ya || !xb || !yb) return fail(SFM_ERR_ARG, "null coordinates");
    if (int r = c->tmp.reserve(24 * 8 + (size_t)m * 4 * 8)) return r;
    if (int r = c->X.reserve((size_t)m * 24)) return r;
    c->tic(T_TRI);
    double* dP = c->tmp.as<double>();
    double* draw = dP + 24;
    CU(cudaMemcpyAsync(dP, P1, 96, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(dP + 12, P2, 96, cudaMemcpyHostToDevice, c->stream));
    const double* s[4];
    if (int r = stage_coords(c, draw, xa, ya, xb, yb, stride, m, s)) return r;
    k_triangulate<<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(s[0], s[1], s[2], s[3], stride, m, nullptr, dP, dP + 12,
                                                                      nullptr, nullptr, nullptr, 0, c->X.as<double>());
    if (int r = check_launch(c, "k_triangulate")) return r;
    c->toc(T_TRI);
    CU(cudaMemcpyAsync(X, c->X.p, (size_t)m * 24, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// The refinement of sfm_refine.cuh behind T1: init, refine_iters + 1 LM steps (the first evaluates the start), finish -
// all enqueued without a round trip.  *rec_out: the refined records for the rest of the tail.
static int refine_launch(sfm_ctx* c, int kind, const SelectRecord* rec_dev, long long max_len, const SelectRecord** rec_out) {
    const long long P = c->npairs;
    const long long maxch = (max_len + kRefineChunk - 1) / kRefineChunk;
    const int nv = kind == MODEL_H ? refine_nv<MODEL_H>() : refine_nv<MODEL_E>();
    if (int r = c->refstate.reserve((size_t)P * sizeof(RefineState))) return r;
    // chunk partials by total length (refine_chunk_base): n / kRefineChunk + P + 1 slots cover every pair's chunks
    if (int r = c->refpart.reserve((size_t)(c->n / kRefineChunk + P + 1) * nv * 8)) return r;
    if (int r = reserve_zeroed(c, c->reftick, (size_t)P * 4)) return r;
    if (int r = c->refrec.reserve((size_t)P * sizeof(SelectRecord))) return r;
    if (int r = c->refrep.reserve((size_t)P * sizeof(RefineReport))) return r;
    RefineArgs a;
    a.pts = c->pts.as<Corr>();
    a.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    a.rec = rec_dev;
    a.idx = c->idx.as<long long>();
    a.num = c->num.as<long long>();
    a.state = c->refstate.as<RefineState>();
    a.partial = c->refpart.as<double>();
    a.ticket = c->reftick.as<unsigned>();
    a.npairs = (int)P;
    a.max_iter = c->refine_iters;
    a.out_rec = c->refrec.as<SelectRecord>();
    a.report = c->refrep.as<RefineReport>();
    const dim3 gp((unsigned)((P + 127) / 128));
    // about 4 blocks per SM in all: a pair gets its share, at least one; blocks grid-stride over the pair's chunks, and
    // the blocks beyond a pair's own chunk count leave at once
    const long long cap = (4ll * c->sm_count + P - 1) / P;
    const dim3 gs((unsigned)(maxch < 1 ? 1 : (maxch < cap ? maxch : cap)), (unsigned)P);
    if (kind == MODEL_H) CU(chain_launch(c, k_refine_init<MODEL_H>, gp, dim3(128), 0, a));
    else CU(chain_launch(c, k_refine_init<MODEL_E>, gp, dim3(128), 0, a));
    if (int r = check_launch(c, "k_refine_init")) return r;
    for (int it = 0; it <= c->refine_iters; ++it) {
        if (kind == MODEL_H) CU(chain_launch(c, k_refine_step<MODEL_H>, gs, dim3(kRefineBlock), 0, a));
        else CU(chain_launch(c, k_refine_step<MODEL_E>, gs, dim3(kRefineBlock), 0, a));
        if (int r = check_launch(c, "k_refine_step")) return r;
    }
    if (kind == MODEL_H) CU(chain_launch(c, k_refine_finish<MODEL_H>, gp, dim3(128), 0, a));
    else CU(chain_launch(c, k_refine_finish<MODEL_E>, gp, dim3(128), 0, a));
    if (int r = check_launch(c, "k_refine_finish")) return r;
    *rec_out = a.out_rec;
    return 0;
}

// The tail of apps/sfm.py:133-186 for the winner described by rec_dev (one SelectRecord per pair on the device):
// T1 inlier mask + ordered compaction + decomposition, T2 4-pose cheirality + vote, T3 triangulation of the passing
// inliers - three launches, nothing synchronised (see sfm_tail.cuh).  max_len = the longest pair.
// kind = MODEL_H: the winners are homographies; a single pair's K is the one hpose_stage_k put in c->hK, a batch's are
// the caller's cameras in c->Ks (its records hold pixels).
static int pose_tail_launch(sfm_ctx* c, double thr, double dist_thr, const SelectRecord* rec_dev, long long max_len,
                            uint8_t* mask_host = nullptr, double* sed_host = nullptr, int kind = MODEL_E,
                            double rot_tol = 0.0) {
    const long long n = c->n, P = c->npairs;
    if (max_len < 1) max_len = 1;
    const int nblk = (int)((max_len + kTailPerBlock - 1) / kTailPerBlock);
    if (int r = c->mask.reserve((size_t)n)) return r;
    if (int r = c->sed.reserve((size_t)n * 8)) return r;
    if (int r = c->idx.reserve((size_t)n * 8)) return r;
    if (int r = c->num.reserve((size_t)P * 8)) return r;
    if (int r = c->poses.reserve((size_t)P * sizeof(PoseSet))) return r;
    if (int r = c->pass.reserve((size_t)n + 1)) return r;
    if (int r = c->X.reserve((size_t)n * 24)) return r;
    // every word of this state is zero between launches (the kernels clean up behind themselves), whatever P and nblk
    const size_t state_bytes = (size_t)P * nblk * 8 + (size_t)P * 8;
    if (int r = reserve_zeroed(c, c->tailstate, state_bytes)) return r;
    TailArgs a;
    a.pts = c->pts.as<Corr>();
    a.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    a.n = n;
    a.rec = rec_dev;
    a.thr = thr;
    a.dist_thr = dist_thr;
    a.mask = c->mask.as<uint8_t>();
    a.sed = c->sed.as<double>();
    a.idx = c->idx.as<long long>();
    a.num = c->num.as<long long>();
    a.agg = c->tailstate.as<unsigned long long>();
    a.ticket = reinterpret_cast<unsigned*>(a.agg + (size_t)P * nblk);
    a.done = a.ticket + P;
    a.poses = c->poses.as<PoseSet>();
    a.pass = c->pass.as<uint8_t>();
    const double* s[4];
    raw_coords(c, s);
    a.xa = s[0]; a.ya = s[1]; a.xb = s[2]; a.yb = s[3];
    a.stride = c->raw_stride;
    a.Ks = c->Ks.as<double>();
    a.X = c->X.as<double>();
    a.planes = nullptr;
    a.rot_tol = rot_tol;
    if (kind == MODEL_H) {
        if (int r = c->planes.reserve((size_t)P * sizeof(HPlane))) return r;
        a.planes = c->planes.as<HPlane>();
        if (!c->batched) a.Ks = c->hK.as<double>();
    }
    c->tic(T_MASK);
    if (kind == MODEL_H) CU(chain_launch(c, k_tail_mask<MODEL_H>, dim3((unsigned)nblk, (unsigned)P), dim3(kTailBlock), 0, a));
    else CU(chain_launch(c, k_tail_mask<MODEL_E>, dim3((unsigned)nblk, (unsigned)P), dim3(kTailBlock), 0, a));
    if (int r = check_launch(c, "k_tail_mask")) return r;
    c->toc(T_MASK);
    // the caller's mask is "sed <= thr" (the forced sample points live in the compacted list only)
    if (mask_host) CU(cudaMemcpyAsync(mask_host, c->mask.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    if (sed_host) CU(cudaMemcpyAsync(sed_host, c->sed.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
    c->refined_pairs = 0;
    if (c->refine_iters > 0) {
        // refine over the list T1 just compacted, then T1 again from the refined records (mask and sed stay those of
        // the RANSAC winner)
        if (int r = refine_launch(c, kind, rec_dev, max_len, &a.rec)) return r;
        a.mask = nullptr;
        a.sed = nullptr;
        if (kind == MODEL_H) CU(chain_launch(c, k_tail_mask<MODEL_H>, dim3((unsigned)nblk, (unsigned)P), dim3(kTailBlock), 0, a));
        else CU(chain_launch(c, k_tail_mask<MODEL_E>, dim3((unsigned)nblk, (unsigned)P), dim3(kTailBlock), 0, a));
        if (int r = check_launch(c, "k_tail_mask")) return r;
        c->refined_pairs = P;
    }
    c->tic(T_POSE);
    // grids sized for the machine (grid-stride inside): the number of inliers is only known on the device
    const long long cap_blocks = P >= 64 ? 8 : 2ll * c->sm_count;
    const long long g2 = (4 * max_len + 127) / 128, g3 = (max_len + 127) / 128;
    const dim3 grid2((unsigned)(g2 < cap_blocks ? g2 : cap_blocks), (unsigned)P);
    if (kind == MODEL_H) CU(chain_launch(c, k_tail_cheirality<MODEL_H>, grid2, dim3(128), 0, a));
    else CU(chain_launch(c, k_tail_cheirality<MODEL_E>, grid2, dim3(128), 0, a));
    if (int r = check_launch(c, "k_tail_cheirality")) return r;
    c->toc(T_POSE);
    c->tic(T_TRI);
    CU(chain_launch(c, k_tail_triangulate, dim3((unsigned)(g3 < cap_blocks ? g3 : cap_blocks), (unsigned)P), dim3(128), 0, a));
    if (int r = check_launch(c, "k_tail_triangulate")) return r;
    c->toc(T_TRI);
    return 0;
}

// the record of a winner the host chose (sfm_get_best / sfm_set_winner) for the tail
static int host_winner_record(sfm_ctx* c, const SelectRecord** out) {
    if (int r = c->winrec.reserve(sizeof(SelectRecord))) return r;
    if (c->has_table)
        if (int r = ensure_table(c)) return r;
    const int32_t* row = (c->has_table && c->winner_local >= 0) ? c->table.as<int32_t>() + 8 * c->winner_local : nullptr;
    k_make_record<<<1, 32, 0, c->stream>>>(winner_E_dev(c), row, c->winner_local >= 0 ? c->winner_local : 0,
                                           c->winrec.as<SelectRecord>());
    if (int r = check_launch(c, "k_make_record")) return r;
    *out = c->winrec.as<SelectRecord>();
    return 0;
}

// results of pose_tail_launch to the host: fixed-size part first (one synchronisation), then the per-inlier arrays
// A winner of the reference's selection rule (minimum error) usually has ~100 inliers: the first kSpecInliers entries of
// the per-inlier arrays ride along with the fixed-size results, so that the common case needs ONE synchronisation.
constexpr long long kSpecInliers = 2048;

// the first `take` entries of the tail's per-inlier arrays, straight from the device
static int copy_inliers(sfm_ctx* c, long long take, int64_t* inlier_idx, uint8_t* pass, double* X) {
    if (inlier_idx) CU(cudaMemcpyAsync(inlier_idx, c->idx.p, (size_t)take * 8, cudaMemcpyDeviceToHost, c->stream));
    if (pass) CU(cudaMemcpyAsync(pass, c->pass.p, (size_t)take, cudaMemcpyDeviceToHost, c->stream));
    if (X) CU(cudaMemcpyAsync(X, c->X.p, (size_t)take * 24, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

static int pose_tail_fetch(sfm_ctx* c, sfm_poses* poses, int64_t cap, int64_t* num_inliers, int64_t* inlier_idx,
                           uint8_t* pass, double* X, sfm_best* best /* may be null */, HPlane* planes = nullptr) {
    const long long* cnt_dev = c->num.as<long long>();
    const long long spec = c->n < kSpecInliers ? c->n : kSpecInliers;
    const size_t o_idx = 64 + ((sizeof(SelectRecord) + 63) / 64) * 64, o_pass = o_idx + (size_t)spec * 8,
                 o_X = ((o_pass + (size_t)spec + 63) / 64) * 64;
    if (int r = ensure_pinned(c, o_X + (size_t)spec * 24)) return r;
    char* hp = (char*)c->hpin;
    CU(cudaMemcpyAsync(hp, cnt_dev, 8, cudaMemcpyDeviceToHost, c->stream));
    if (best) CU(cudaMemcpyAsync(hp + 64, c->record.p, sizeof(SelectRecord), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(poses, c->poses.p, sizeof(PoseSet), cudaMemcpyDeviceToHost, c->stream));
    if (planes) CU(cudaMemcpyAsync(planes, c->planes.p, sizeof(HPlane), cudaMemcpyDeviceToHost, c->stream));
    if (spec > 0) {
        if (inlier_idx) CU(cudaMemcpyAsync(hp + o_idx, c->idx.p, (size_t)spec * 8, cudaMemcpyDeviceToHost, c->stream));
        if (pass) CU(cudaMemcpyAsync(hp + o_pass, c->pass.p, (size_t)spec, cudaMemcpyDeviceToHost, c->stream));
        if (X) CU(cudaMemcpyAsync(hp + o_X, c->X.p, (size_t)spec * 24, cudaMemcpyDeviceToHost, c->stream));
    }
    CU(cudaStreamSynchronize(c->stream));
    long long m;
    memcpy(&m, hp, 8);
    if (best) {
        SelectRecord r;
        memcpy(&r, hp + 64, sizeof r);
        unpack_best(r, best);
        if (r.best.idx >= 0) {
            c->winner_local = r.best.idx - c->last_idx_offset;
            c->winner_set = true;
        } else {
            m = 0;  // no model: the tail ran on an empty mask
        }
    }
    *num_inliers = m;
    const long long take = m < cap ? m : cap;
    if (take > 0 && take <= spec) {  // everything already sits in the pinned scratch
        if (inlier_idx) memcpy(inlier_idx, hp + o_idx, (size_t)take * 8);
        if (pass) memcpy(pass, hp + o_pass, (size_t)take);
        if (X) memcpy(X, hp + o_X, (size_t)take * 24);
    } else if (take > 0) {
        return copy_inliers(c, take, inlier_idx, pass, X);
    }
    return 0;
}

int sfm_pose_and_triangulate(sfm_ctx* c, double thr, double dist_thr, sfm_poses* poses, int64_t cap,
                             int64_t* num_inliers, int64_t* inlier_idx, uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (!c->has_pts || c->batched) return fail(SFM_ERR_STATE, "no single-pair correspondences loaded");
    if (!c->winner_set) return fail(SFM_ERR_STATE, "no winner: run sfm_ransac_essential / sfm_get_best first");
    if (c->models_h && c->winner_local >= 0)
        return fail(SFM_ERR_STATE, "the winner is a homography: use sfm_homography_pose_and_triangulate");
    const SelectRecord* rec = nullptr;
    if (int r = host_winner_record(c, &rec)) return r;
    if (int r = pose_tail_launch(c, thr, dist_thr, rec, c->n)) return r;
    return pose_tail_fetch(c, poses, cap, num_inliers, inlier_idx, pass, X, nullptr);
}

// ---- homography pose (sfm_hpose.cuh) -------------------------------------------------------
static void pack_hposes(const PoseSet& p, const HPlane& pl, sfm_hposes* out) {
    memcpy(out->R, p.R, sizeof out->R);
    memcpy(out->t, p.t, sizeof out->t);
    memcpy(out->n, pl.n, sizeof out->n);
    memcpy(out->d, pl.d, sizeof out->d);
    memcpy(out->sv, p.sv, sizeof out->sv);
    memcpy(out->counts, p.counts, sizeof out->counts);
    out->best = p.best;
    out->rotation_only = pl.rotation_only;
}

// pose_tail_fetch after a homography tail: the poses and the plane as one sfm_hposes
static int hpose_tail_fetch(sfm_ctx* c, sfm_hposes* poses, int64_t cap, int64_t* num_inliers, int64_t* inlier_idx,
                            uint8_t* pass, double* X, sfm_best* best /* may be null */) {
    PoseSet p;
    HPlane pl;
    if (int r = pose_tail_fetch(c, reinterpret_cast<sfm_poses*>(&p), cap, num_inliers, inlier_idx, pass, X, best, &pl))
        return r;
    pack_hposes(p, pl, poses);
    return 0;
}

// a camera matrix the homography pose and the model scores can invert
static int check_camera(const double* K) {
    if (!K) return fail(SFM_ERR_ARG, "null camera matrix");
    for (int i = 0; i < 9; ++i)
        if (!std::isfinite(K[i])) return fail(SFM_ERR_ARG, "the camera matrix is not finite");
    const double det = K[0] * (K[4] * K[8] - K[5] * K[7]) - K[1] * (K[3] * K[8] - K[5] * K[6]) +
                       K[2] * (K[3] * K[7] - K[4] * K[6]);
    if (det == 0.0 || K[0] == 0.0 || K[4] == 0.0) return fail(SFM_ERR_ARG, "the camera matrix is singular");
    return 0;
}

// The homography pose reads pixels through K^-1 in three places (the decomposition, the vote's rays, the triangulation):
// only an upper-triangular K with K[2,2] = 1 makes the vote's (x - cx - s yn) / fx the same camera as the other two.
static int hpose_args(const double* K, double rot_tol) {
    if (int r = check_camera(K)) return r;
    if (K[3] != 0.0 || K[6] != 0.0 || K[7] != 0.0 || K[8] != 1.0)
        return fail(SFM_ERR_ARG, "the camera matrix must be upper triangular with K[2,2] = 1");
    if (std::isnan(rot_tol)) return fail(SFM_ERR_ARG, "rotation_tolerance is NaN");
    return 0;
}

// the caller's K to the device (staged in the context: the async copy must not read caller memory later)
static int hpose_stage_k(sfm_ctx* c, const double* K) {
    if (int r = c->hK.reserve(72)) return r;
    memcpy(c->hstage + 9, K, 72);
    CU(cudaMemcpyAsync(c->hK.p, c->hstage + 9, 72, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

int sfm_decompose_homography(sfm_ctx* c, const double* H, const double* K, double rotation_tolerance, sfm_hposes* out) {
    if (int r = use(c)) return r;
    if (!H || !out) return fail(SFM_ERR_ARG, "null argument");
    if (int r = hpose_args(K, rotation_tolerance)) return r;
    if (int r = c->tmp.reserve(144)) return r;
    if (int r = c->poses.reserve(sizeof(PoseSet))) return r;
    if (int r = c->planes.reserve(sizeof(HPlane))) return r;
    memcpy(c->hstage, H, 72);
    memcpy(c->hstage + 9, K, 72);
    CU(cudaMemcpyAsync(c->tmp.p, c->hstage, 144, cudaMemcpyHostToDevice, c->stream));
    k_decompose_homography<<<1, 32, 0, c->stream>>>(c->tmp.as<double>(), c->tmp.as<double>() + 9, rotation_tolerance,
                                                    c->poses.as<PoseSet>(), c->planes.as<HPlane>());
    if (int r = check_launch(c, "k_decompose_homography")) return r;
    PoseSet p;
    HPlane pl;
    CU(cudaMemcpyAsync(&p, c->poses.p, sizeof p, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(&pl, c->planes.p, sizeof pl, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    pack_hposes(p, pl, out);
    return 0;
}

int sfm_homography_pose_and_triangulate(sfm_ctx* c, const double* K, double thr, double dist_thr, double rotation_tolerance,
                                        sfm_hposes* poses, int64_t cap, int64_t* num_inliers, int64_t* inlier_idx,
                                        uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (int r = hpose_args(K, rotation_tolerance)) return r;
    if (!c->has_pts || c->batched) return fail(SFM_ERR_STATE, "no single-pair correspondences loaded");
    if (!c->models_h || !c->winner_set || c->winner_local < 0)
        return fail(SFM_ERR_STATE, "no homography winner: run sfm_ransac_homography or sfm_set_winner first");
    const SelectRecord* rec = nullptr;
    if (int r = host_winner_record(c, &rec)) return r;
    if (int r = hpose_stage_k(c, K)) return r;
    if (int r = pose_tail_launch(c, thr, dist_thr, rec, c->n, nullptr, nullptr, MODEL_H, rotation_tolerance)) return r;
    return hpose_tail_fetch(c, poses, cap, num_inliers, inlier_idx, pass, X, nullptr);
}

int sfm_two_view_homography(sfm_ctx* c, const double* K, double thr, double min_extra, int agg, int mode, double dist_thr,
                            double rotation_tolerance, sfm_best* best, sfm_hposes* poses, int64_t cap, int64_t* num_inliers,
                            int64_t* inlier_idx, uint8_t* pass, double* X, uint8_t* mask, double* err) {
    if (int r = use(c)) return r;
    if (!best || !poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (int r = hpose_args(K, rotation_tolerance)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (c->has_pts && c->n < 8) return fail(SFM_ERR_ARG, "need at least 8 correspondences, got %lld", c->n);
    // K goes first: no copy between the selection and the tail, which is chained right behind it; the winner stays on
    // the device and the host synchronises once, at the fetch
    if (int r = hpose_stage_k(c, K)) return r;
    if (int r = fit_h_launch(c)) return r;
    if (int r = score_h_launch(c, thr, min_extra, agg, mode, c->n)) return r;
    // T1's mask / err are those of sfm_homography_mask for the winner
    if (int r = pose_tail_launch(c, thr, dist_thr, c->record.as<SelectRecord>(), c->n, mask, err, MODEL_H, rotation_tolerance))
        return r;
    return hpose_tail_fetch(c, poses, cap, num_inliers, inlier_idx, pass, X, best);
}

// ---- essential matrix or homography (sfm_select.cuh) --------------------------------------------
// k_score_models over the P pairs of the upload with the models staged in c->sstage; out[P], per_point [n][4] or null.
// selstate: the kernel's sums and tickets [P][kSelectStateWords], zero between launches (only the kernel writes it);
// selio: the models [P], then the results [P].
static int score_models_launch(sfm_ctx* c, double sigma, double homography_ratio, long long max_len,
                               sfm_model_scores* out, double* per_point) {
    const long long P = c->npairs;
    const size_t o_out = (size_t)P * sizeof(SelectModels);
    if (int r = reserve_zeroed(c, c->selstate, (size_t)P * kSelectStateWords * 8)) return r;
    if (int r = c->selio.reserve(o_out + (size_t)P * sizeof(ModelScores))) return r;
    if (per_point)
        if (int r = c->selpp.reserve((size_t)c->n * 32)) return r;
    char* base = c->selio.as<char>();
    CU(cudaMemcpyAsync(base, c->sstage.data(), (size_t)P * sizeof(SelectModels), cudaMemcpyHostToDevice, c->stream));
    SelectArgs a;
    const double* s[4];
    raw_coords(c, s);
    a.xa = s[0]; a.ya = s[1]; a.xb = s[2]; a.yb = s[3];
    a.stride = c->raw_stride;
    a.n = c->n;
    a.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    a.models = reinterpret_cast<const SelectModels*>(base);
    a.sigma = sigma;
    a.ratio = homography_ratio;
    a.state = c->selstate.as<unsigned long long>();
    a.out = reinterpret_cast<ModelScores*>(base + o_out);
    a.per_point = per_point ? c->selpp.as<double>() : nullptr;
    // about 4 blocks per SM in all: a pair gets its share of them, at least one
    const long long blocks = (max_len + kSelectBlock - 1) / kSelectBlock, cap = (4ll * c->sm_count + P - 1) / P;
    const long long gx = blocks < cap ? blocks : cap;
    c->tic(T_SCORE);
    k_score_models<<<dim3((unsigned)(gx > 0 ? gx : 1), (unsigned)P), kSelectBlock, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_score_models")) return r;
    c->toc(T_SCORE);
    CU(cudaMemcpyAsync(out, a.out, (size_t)P * sizeof(ModelScores), cudaMemcpyDeviceToHost, c->stream));
    if (per_point) CU(cudaMemcpyAsync(per_point, c->selpp.p, (size_t)c->n * 32, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// the checks of sigma and the ratio shared by both scoring calls
static int score_models_args(double sigma, double homography_ratio) {
    if (!(sigma > 0.0) || !std::isfinite(sigma)) return fail(SFM_ERR_ARG, "sigma must be finite and > 0");
    if (!std::isfinite(homography_ratio)) return fail(SFM_ERR_ARG, "homography_ratio is not finite");
    return 0;
}

static int models_finite(const double* E, const double* H, const char* pair) {
    for (int i = 0; i < 9; ++i) {
        if (E && !std::isfinite(E[i])) return fail(SFM_ERR_ARG, "E%s is not finite", pair);
        if (H && !std::isfinite(H[i])) return fail(SFM_ERR_ARG, "H%s is not finite", pair);
    }
    return 0;
}

// one pair's models into the staging record; E / H null = not given
static void stage_models(SelectModels& m, const double* E, const double* H, const double* K) {
    memset(&m, 0, sizeof m);
    if (E) memcpy(m.E, E, 72);
    if (H) memcpy(m.H, H, 72);
    memcpy(m.K, K, 72);
    m.have_e = E ? 1 : 0;
    m.have_h = H ? 1 : 0;
}

int sfm_score_models(sfm_ctx* c, const double* E, const double* H, const double* K, double sigma, double homography_ratio,
                     sfm_model_scores* out, double* per_point) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    if (!E && !H) return fail(SFM_ERR_ARG, "give E, H or both");
    if (int r = models_finite(E, H, "")) return r;
    if (int r = check_camera(K)) return r;
    if (int r = score_models_args(sigma, homography_ratio)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (!c->has_pts) return fail(SFM_ERR_STATE, "no correspondences loaded");
    c->sstage.resize(1);
    stage_models(c->sstage[0], E, H, K);
    return score_models_launch(c, sigma, homography_ratio, c->n, out, per_point);
}

int sfm_batch_score_models(sfm_ctx* c, const double* E, const uint8_t* have_e, const double* H, const uint8_t* have_h,
                           double sigma, double homography_ratio, sfm_model_scores* out, double* per_point) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    if (!E && !H) return fail(SFM_ERR_ARG, "give E, H or both");
    if (int r = score_models_args(sigma, homography_ratio)) return r;
    if (!c->batched || !c->has_pts) return fail(SFM_ERR_STATE, "no batched upload: run a batch call first");
    const long long P = c->npairs;
    c->sstage.resize((size_t)P);
    for (long long p = 0; p < P; ++p) {
        char which[48];
        snprintf(which, sizeof which, " of pair %lld", p);
        const double* K = c->Kbatch.data() + 9 * p;
        const double* Ep = (E && (!have_e || have_e[p])) ? E + 9 * p : nullptr;
        const double* Hp = (H && (!have_h || have_h[p])) ? H + 9 * p : nullptr;
        if (int r = models_finite(Ep, Hp, which)) return r;
        if (int r = check_camera(K)) {
            const std::string why = g_err;
            return fail(r, "pair %lld: %s", p, why.c_str());
        }
        stage_models(c->sstage[(size_t)p], Ep, Hp, K);
    }
    return score_models_launch(c, sigma, homography_ratio, c->batch_max_len, out, per_point);
}

int sfm_two_view_async(sfm_ctx* c, double thr, double min_extra, int agg, int mode, double dist_thr, uint8_t* mask,
                       double* sed) {
    if (int r = use(c)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, c->n)) return r;
    // the winner stays on the device: mask, compaction, decomposition, vote and triangulation are enqueued right
    // behind the selection, and the host synchronises once for all fixed-size results (sfm_two_view_fetch)
    return pose_tail_launch(c, thr, dist_thr, c->record.as<SelectRecord>(), c->n, mask, sed);
}

int sfm_two_view_fetch(sfm_ctx* c, sfm_best* best, sfm_poses* poses, int64_t cap, int64_t* num_inliers,
                       int64_t* inlier_idx, uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!best || !poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (!c->has_score || c->batched) return fail(SFM_ERR_STATE, "sfm_two_view_async first");
    return pose_tail_fetch(c, poses, cap, num_inliers, inlier_idx, pass, X, best);
}

int sfm_two_view(sfm_ctx* c, double thr, double min_extra, int agg, int mode, double dist_thr, sfm_best* best,
                 sfm_poses* poses, int64_t cap, int64_t* num_inliers, int64_t* inlier_idx, uint8_t* pass, double* X,
                 uint8_t* mask, double* sed) {
    if (!best || !poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (int r = sfm_two_view_async(c, thr, min_extra, agg, mode, dist_thr, mask, sed)) return r;
    return sfm_two_view_fetch(c, best, poses, cap, num_inliers, inlier_idx, pass, X);
}

// ---- hypothesis-sharded runs without a host round trip (SURVEY.md 8(e)) -----------------------
int sfm_score_async(sfm_ctx* c, double thr, double min_extra, int agg, int mode, void** record_dev) {
    if (int r = use(c)) return r;
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, c->n)) return r;
    if (record_dev) *record_dev = c->record.p;  // SFM_RECORD_BYTES bytes, valid once the stream reaches this point
    return 0;
}

int sfm_sharded_tail(sfm_ctx* c, const void* gathered_records_dev, int world, int rank, int64_t hyps_per_rank, int mode,
                     double thr, double dist_thr) {
    if (int r = use(c)) return r;
    if (!gathered_records_dev || world < 1 || rank < 0 || rank >= world) return fail(SFM_ERR_ARG, "bad gather arguments");
    if (!c->has_score) return fail(SFM_ERR_STATE, "sfm_score_async first");
    if (c->refine_iters > 0) return fail(SFM_ERR_STATE, "refinement is not supported on hypothesis-sharded runs");
    if (mode < 0 || mode > 2) return fail(SFM_ERR_ARG, "bad selection %d", mode);
    if (int r = c->winnerE.reserve(72)) return r;
    if (int r = c->merged.reserve(sizeof(SelectRecord) + sizeof(Best) + 16)) return r;
    SelectRecord* merged = c->merged.as<SelectRecord>();
    Best* local_best = reinterpret_cast<Best*>(merged + 1);
    int* owner = reinterpret_cast<int*>(local_best + 1);
    k_merge_records<<<1, 32, 0, c->stream>>>(reinterpret_cast<const SelectRecord*>(gathered_records_dev), world, rank,
                                             (long long)hyps_per_rank, mode, merged, owner, c->winnerE.as<double>(), local_best);
    if (int r = check_launch(c, "k_merge_records")) return r;
    return pose_tail_launch(c, thr, dist_thr, merged, c->n);
}

int sfm_sharded_fetch(sfm_ctx* c, sfm_best* best, int32_t* owner, sfm_poses* poses, int64_t cap, int64_t* num_inliers,
                      int64_t* inlier_idx, uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!best || !owner || !poses || !num_inliers) return fail(SFM_ERR_ARG, "null argument");
    if (!c->merged.p) return fail(SFM_ERR_STATE, "sfm_sharded_tail first");
    const long long* cnt_dev = c->num.as<long long>();
    const size_t mbytes = sizeof(SelectRecord) + sizeof(Best) + 16;
    if (int r = ensure_pinned(c, 64 + mbytes)) return r;
    CU(cudaMemcpyAsync(c->hpin, cnt_dev, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync((char*)c->hpin + 64, c->merged.p, mbytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(poses, c->poses.p, sizeof(PoseSet), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    long long m;
    memcpy(&m, c->hpin, 8);
    SelectRecord r;
    Best lb;
    int own;
    memcpy(&r, (char*)c->hpin + 64, sizeof r);
    memcpy(&lb, (char*)c->hpin + 64 + sizeof r, sizeof lb);
    memcpy(&own, (char*)c->hpin + 64 + sizeof r + sizeof lb, sizeof own);
    unpack_best(r, best);  // index: the GLOBAL hypothesis index
    *owner = own;
    c->winner_local = lb.idx >= 0 ? lb.idx : -1;  // -1: the model lives in winnerE
    c->winner_set = r.best.idx >= 0;
    if (r.best.idx < 0) m = 0;
    *num_inliers = m;
    const long long take = m < cap ? m : cap;
    if (take > 0) return copy_inliers(c, take, inlier_idx, pass, X);
    return 0;
}

}  // extern "C"

// ---- NCCL behind the C ABI (SURVEY.md 8(b): sfm_nccl_init / sharded estimate without torch) ---------------------
// libnccl is resolved at run time (dlopen): the library a host process already loaded (torch bundles one) is reused,
// otherwise the system's libnccl.so.2.  Only four entry points are needed; their prototypes are restated here so that
// the build does not depend on nccl.h.
struct NcclId { char internal[128]; };  // ncclUniqueId, passed BY VALUE to ncclCommInitRank
static_assert(sizeof(NcclId) == SFM_NCCL_ID_BYTES, "ncclUniqueId is 128 bytes");
namespace {
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

int nccl_load() {
    if (g_nccl.lib) return 0;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // already in the process (torch)?
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(SFM_ERR_STATE, "libnccl.so.2 not found: %s", dlerror());
    g_nccl.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclGetUniqueId"));
    g_nccl.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(h, "ncclCommInitRank"));
    g_nccl.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(h, "ncclAllGather"));
    g_nccl.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
    g_nccl.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy)
        return fail(SFM_ERR_STATE, "libnccl.so.2 lacks a required symbol");
    g_nccl.lib = h;
    return 0;
}
#define NC(call)                                                                                          \
    do {                                                                                                  \
        int e_ = (call);                                                                                  \
        if (e_ != 0)                                                                                      \
            return fail(SFM_ERR_CUDA, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(e_) : "?"); \
    } while (0)
}  // namespace

extern "C" {

int sfm_nccl_unique_id(void* id_out) {
    if (!id_out) return fail(SFM_ERR_ARG, "null argument");
    if (int r = nccl_load()) return r;
    NC(g_nccl.GetUniqueId(id_out));
    return 0;
}

int sfm_nccl_init(sfm_ctx* c, int rank, int nranks, const void* unique_id) {
    if (int r = use(c)) return r;
    if (!unique_id || nranks < 1 || rank < 0 || rank >= nranks) return fail(SFM_ERR_ARG, "bad communicator arguments");
    if (int r = nccl_load()) return r;
    if (c->nccl_comm) { g_nccl.CommDestroy(c->nccl_comm); c->nccl_comm = nullptr; }
    NcclId id;
    memcpy(&id, unique_id, sizeof id);
    NC(g_nccl.CommInitRank(&c->nccl_comm, nranks, id, rank));
    c->nccl_rank = rank;
    c->nccl_world = nranks;
    return 0;
}

int sfm_nccl_destroy(sfm_ctx* c) {
    if (!c) return 0;
    if (c->nccl_comm && g_nccl.lib) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        g_nccl.CommDestroy(c->nccl_comm);
    }
    c->nccl_comm = nullptr;
    c->nccl_world = 1;
    c->nccl_rank = 0;
    return 0;
}

// One complete hypothesis-sharded estimate on the communicator of sfm_nccl_init, nothing synchronised: this rank's
// hypotheses [rank * hyps_per_rank, (rank + 1) * hyps_per_rank) of the device sampler -> fit -> score -> select, ONE
// ncclAllGather of the SFM_RECORD_BYTES selection records on the context's stream (the path's only collective), merge
// kernel, tail.  Results through sfm_sharded_fetch.
int sfm_two_view_sharded(sfm_ctx* c, uint64_t seed, int64_t hyps_per_rank, double thr, double min_extra, int agg,
                         int mode, double dist_thr) {
    if (int r = use(c)) return r;
    if (!c->nccl_comm) return fail(SFM_ERR_STATE, "sfm_nccl_init first");
    if (c->refine_iters > 0) return fail(SFM_ERR_STATE, "refinement is not supported on hypothesis-sharded runs");
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (int r = sample_device(c, seed, 0, (int64_t)c->nccl_rank * hyps_per_rank, hyps_per_rank)) return r;
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, c->n)) return r;
    if (int r = c->gathered.reserve((size_t)c->nccl_world * sizeof(SelectRecord))) return r;
    NC(g_nccl.AllGather(c->record.p, c->gathered.p, sizeof(SelectRecord), /* ncclUint8 */ 1, c->nccl_comm, c->stream));
    return sfm_sharded_tail(c, c->gathered.p, c->nccl_world, c->nccl_rank, hyps_per_rank, mode, thr, dist_thr);
}

}  // extern "C"

extern "C" {

// ---- batched pairs ------------------------------------------------------------------------
// The upload of P independent pairs: offsets, the caller's cameras (c->Ks, and c->Kbatch on the host) and the raw
// coordinates (c->raw), from which the records are built - K-normalised with each pair's K for essential matrices, in
// pixels (an identity camera) for homographies.  Nothing synchronised.
static int batch_upload(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                        int64_t stride, const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h, bool pixels,
                        long long* max_len_out) {
    if (!xa || !ya || !xb || !yb || !offsets || !Ks) return fail(SFM_ERR_ARG, "null argument");
    if (npairs <= 0 || npairs > 65535) return fail(SFM_ERR_ARG, "need 1 <= npairs <= 65535 per call");
    if (h <= 0) return fail(SFM_ERR_ARG, "need h > 0");
    const long long n = offsets[npairs];
    if (offsets[0] != 0 || n <= 0 || (uint64_t)n >= kMaxPoints) return fail(SFM_ERR_ARG, "bad offsets (total %lld)", n);
    long long max_len = 0;
    for (int64_t p = 0; p < npairs; ++p) {
        const long long len = offsets[p + 1] - offsets[p];
        if (len < 0) return fail(SFM_ERR_ARG, "offsets must be non-decreasing");
        if (len > max_len) max_len = len;
    }
    c->tic(T_UPLOAD);
    c->batched = true;
    c->npairs = npairs;
    c->n = n;
    c->first_len = offsets[1] - offsets[0];
    if (int r = c->offsets.reserve((size_t)(npairs + 1) * 8)) return r;
    if (int r = c->Ks.reserve((size_t)npairs * 72)) return r;
    CU(cudaMemcpyAsync(c->offsets.p, offsets, (size_t)(npairs + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->Ks.p, Ks, (size_t)npairs * 72, cudaMemcpyHostToDevice, c->stream));
    c->Kbatch.assign(Ks, Ks + 9 * npairs);
    c->batch_max_len = max_len;
    const double* s[4];
    if (int r = stage_raw(c, xa, ya, xb, yb, stride, n, s)) return r;
    if (pixels) {  // one identity camera for all records: x / 1 = x
        const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        if (int r = hpose_stage_k(c, I)) return r;
        if (int r = c->pts.reserve((size_t)n * sizeof(Corr))) return r;
        k_normalise<<<dim3((unsigned)((n + 255) / 256), 1), 256, 0, c->stream>>>(s[0], s[1], s[2], s[3], stride, n, nullptr,
                                                                                c->hK.as<double>(), c->pts.as<Corr>(), nullptr);
        if (int r = check_launch(c, "k_normalise")) return r;
        c->k2_ready = false;  // pixel records: the essential-matrix scorer does not run on them
    } else if (int r = normalise_from(c, s[0], s[1], s[2], s[3], stride, n, max_len)) {
        return r;
    }
    c->toc(T_UPLOAD);
    c->has_pts = true;
    c->has_table = c->has_models = c->has_score = false;
    c->table_pending = false;
    c->winner_set = false;
    *max_len_out = max_len;
    return 0;
}

// upload -> device sampler -> fit -> score + select of P independent pairs (nothing synchronised)
static int batch_core(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb, int64_t stride,
                      const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h, uint64_t seed, uint64_t pair_id0,
                      double thr, double min_extra, int agg, int mode, long long* max_len_out) {
    long long max_len = 0;
    if (int r = batch_upload(c, xa, ya, xb, yb, stride, offsets, npairs, Ks, h, false, &max_len)) return r;
    if (int r = sample_device(c, seed, pair_id0, 0, h)) return r;
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, max_len)) return r;
    *max_len_out = max_len;
    return 0;
}

// per-pair winners of the last batch score -> host arrays (the selection records hold everything)
static int batch_fetch_winners(sfm_ctx* c, int64_t npairs, size_t extra_pinned, char** extra) {
    const size_t rbytes = (size_t)npairs * sizeof(SelectRecord);
    if (int r = ensure_pinned(c, rbytes + extra_pinned + 64)) return r;
    char* hp = (char*)c->hpin;
    CU(cudaMemcpyAsync(hp, c->record.p, rbytes, cudaMemcpyDeviceToHost, c->stream));
    if (extra) *extra = hp + ((rbytes + 63) / 64) * 64;
    return 0;
}

static void batch_unpack_winners(const char* hp, int64_t npairs, double* E, int64_t* best_index, double* best_err,
                                 int32_t* count_extra, int64_t* num_invalid) {
    const SelectRecord* hr = reinterpret_cast<const SelectRecord*>(hp);
    for (int64_t p = 0; p < npairs; ++p) {
        const bool ok = hr[p].best.idx >= 0;
        if (best_index) best_index[p] = hr[p].best.idx;
        if (best_err) best_err[p] = ok ? hr[p].best.err : __builtin_inf();
        if (count_extra) count_extra[p] = ok ? hr[p].best.count : -1;
        if (num_invalid) num_invalid[p] = hr[p].num_invalid;
        if (E) memcpy(E + 9 * p, hr[p].E, 72);
    }
}

int sfm_batch_ransac(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                     int64_t stride, const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h,
                     uint64_t seed, uint64_t pair_id0, double thr, double min_extra, int agg, int mode, double* E,
                     int64_t* best_index, double* best_err, int32_t* count_extra, int64_t* num_invalid) {
    if (int r = use(c)) return r;
    long long max_len = 0;
    if (int r = batch_core(c, xa, ya, xb, yb, stride, offsets, npairs, Ks, h, seed, pair_id0, thr, min_extra, agg, mode,
                           &max_len)) return r;
    if (int r = batch_fetch_winners(c, npairs, 0, nullptr)) return r;
    CU(cudaStreamSynchronize(c->stream));
    batch_unpack_winners((const char*)c->hpin, npairs, E, best_index, best_err, count_extra, num_invalid);
    c->has_score = false;  // per-hypothesis single-pair getters do not apply to batches
    c->winner_set = false;
    return 0;
}

// After a batch tail: dense packing of the per-pair inlier segments, then winners, poses (and planes) and offsets with
// one synchronisation, the packed per-inlier arrays with a second one.
static int batch_tail_fetch(sfm_ctx* c, int64_t npairs, long long max_len, double* E, int64_t* best_index,
                            double* best_err, int32_t* count_extra, int64_t* num_invalid, PoseSet* poses, HPlane* planes,
                            int64_t* inlier_offsets, int64_t cap, int32_t* inlier_idx, uint8_t* pass, double* X) {
    const long long n = c->n;
    const size_t o_off = 0, o_idx = ((size_t)(npairs + 1) * 8 + 63) / 64 * 64, o_pass = o_idx + ((size_t)n * 4 + 63) / 64 * 64,
                 o_X = o_pass + ((size_t)n + 63) / 64 * 64;
    if (int r = c->bout.reserve(o_X + (size_t)n * 24)) return r;
    char* bo = c->bout.as<char>();
    long long* d_off = reinterpret_cast<long long*>(bo + o_off);
    k_batch_offsets<<<1, 1024, 0, c->stream>>>(c->num.as<long long>(), (int)npairs, d_off);
    if (int r = check_launch(c, "k_batch_offsets")) return r;
    const unsigned gx = (unsigned)((max_len + 255) / 256 > 0 ? (max_len + 255) / 256 : 1);
    k_batch_pack<<<dim3(gx, (unsigned)npairs), 256, 0, c->stream>>>(
        c->offsets.as<long long>(), c->num.as<long long>(), d_off, c->idx.as<long long>(), c->pass.as<uint8_t>(),
        c->X.as<double>(), reinterpret_cast<int32_t*>(bo + o_idx), reinterpret_cast<uint8_t*>(bo + o_pass),
        reinterpret_cast<double*>(bo + o_X));
    if (int r = check_launch(c, "k_batch_pack")) return r;
    char* extra = nullptr;
    const size_t pose_bytes = (size_t)npairs * sizeof(PoseSet);
    if (int r = batch_fetch_winners(c, npairs, pose_bytes, &extra)) return r;
    CU(cudaMemcpyAsync(poses, c->poses.p, pose_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (planes)
        CU(cudaMemcpyAsync(planes, c->planes.p, (size_t)npairs * sizeof(HPlane), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(inlier_offsets, d_off, (size_t)(npairs + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    batch_unpack_winners((const char*)c->hpin, npairs, E, best_index, best_err, count_extra, num_invalid);
    const long long total = inlier_offsets[npairs];
    const long long take = total < cap ? total : cap;
    if (take > 0) {
        if (inlier_idx) CU(cudaMemcpyAsync(inlier_idx, bo + o_idx, (size_t)take * 4, cudaMemcpyDeviceToHost, c->stream));
        if (pass) CU(cudaMemcpyAsync(pass, bo + o_pass, (size_t)take, cudaMemcpyDeviceToHost, c->stream));
        if (X) CU(cudaMemcpyAsync(X, bo + o_X, (size_t)take * 24, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    c->has_score = false;
    c->winner_set = false;
    return 0;
}

// The whole path per pair (apps/sfm.py:110-186 for every pair of the batch): RANSAC E, then for each pair's winner the
// inlier list, the 4-pose cheirality vote and the triangulation of the passing inliers - the same three tail kernels as
// the single-pair call, with the pair as blockIdx.y.  Per-inlier results come back densely packed:
// inlier_offsets[p] .. inlier_offsets[p+1] index inlier_idx (pair-relative, ascending), pass and X.
int sfm_batch_two_view(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                       int64_t stride, const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h,
                       uint64_t seed, uint64_t pair_id0, double thr, double min_extra, int agg, int mode,
                       double dist_thr, double* E, int64_t* best_index, double* best_err, int32_t* count_extra,
                       int64_t* num_invalid, sfm_poses* poses, int64_t* inlier_offsets, int64_t cap,
                       int32_t* inlier_idx, uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!poses || !inlier_offsets) return fail(SFM_ERR_ARG, "null argument");
    long long max_len = 0;
    if (int r = batch_core(c, xa, ya, xb, yb, stride, offsets, npairs, Ks, h, seed, pair_id0, thr, min_extra, agg, mode,
                           &max_len)) return r;
    if (int r = pose_tail_launch(c, thr, dist_thr, c->record.as<SelectRecord>(), max_len)) return r;
    return batch_tail_fetch(c, npairs, max_len, E, best_index, best_err, count_extra, num_invalid,
                            reinterpret_cast<PoseSet*>(poses), nullptr, inlier_offsets, cap, inlier_idx, pass, X);
}

// sfm_batch_two_view for homographies: the pixel records of every pair, the device sampler's rows (columns 0-3), the 4-point
// fits, K2 and K3 over (pair, split, group) items, then the homography tail of every pair's winner with that pair's K.
int sfm_batch_two_view_homography(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
                                  int64_t stride, const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h,
                                  uint64_t seed, uint64_t pair_id0, double thr, double min_extra, int agg, int mode,
                                  double dist_thr, double rotation_tolerance, double* H, int64_t* best_index,
                                  double* best_err, int32_t* count_extra, int64_t* num_invalid, sfm_hposes* poses,
                                  int64_t* inlier_offsets, int64_t cap, int32_t* inlier_idx, uint8_t* pass, double* X) {
    if (int r = use(c)) return r;
    if (!poses || !inlier_offsets || !Ks) return fail(SFM_ERR_ARG, "null argument");
    if (npairs <= 0 || npairs > 65535) return fail(SFM_ERR_ARG, "need 1 <= npairs <= 65535 per call");
    for (int64_t p = 0; p < npairs; ++p)
        if (int r = hpose_args(Ks + 9 * p, rotation_tolerance)) {
            const std::string why = g_err;
            return fail(r, "pair %lld: %s", (long long)p, why.c_str());
        }
    long long max_len = 0;
    if (int r = batch_upload(c, xa, ya, xb, yb, stride, offsets, npairs, Ks, h, true, &max_len)) return r;
    if (int r = sample_device(c, seed, pair_id0, 0, h)) return r;
    if (int r = fit_h_launch(c)) return r;
    if (int r = score_h_launch(c, thr, min_extra, agg, mode, max_len)) return r;
    if (int r = pose_tail_launch(c, thr, dist_thr, c->record.as<SelectRecord>(), max_len, nullptr, nullptr, MODEL_H,
                                 rotation_tolerance))
        return r;
    std::vector<PoseSet> ps((size_t)npairs);
    std::vector<HPlane> pl((size_t)npairs);
    if (int r = batch_tail_fetch(c, npairs, max_len, H, best_index, best_err, count_extra, num_invalid, ps.data(), pl.data(),
                                 inlier_offsets, cap, inlier_idx, pass, X))
        return r;
    for (int64_t p = 0; p < npairs; ++p) pack_hposes(ps[(size_t)p], pl[(size_t)p], poses + p);
    return 0;
}

// ---- N1: brute-force matcher (the stage in front of the hot path) ---------------------------
// Selection + validations on the device score matrix c->m_S (na x nb), results to the host.
static int match_finish(sfm_ctx* c, int64_t na, int64_t nb, int validation, double ratio_threshold, int32_t* best_b,
                        double* best_score, uint8_t* keep) {
    // outputs: best_b int32[na] | pad | best_s double[na] | heap1 double[na] | keep u8[na] | key u64[nb] | first int[nb]
    const size_t o_bs = ((size_t)na * 4 + 7) / 8 * 8, o_h1 = o_bs + (size_t)na * 8, o_keep = o_h1 + (size_t)na * 8;
    const size_t o_key = (o_keep + (size_t)na + 7) / 8 * 8, o_first = o_key + (size_t)nb * 8;
    if (int r = c->m_out.reserve(o_first + (size_t)nb * 4)) return r;
    char* out = c->m_out.as<char>();
    int32_t* d_bb = reinterpret_cast<int32_t*>(out);
    double* d_bs = reinterpret_cast<double*>(out + o_bs);
    double* d_h1 = reinterpret_cast<double*>(out + o_h1);
    uint8_t* d_keep = reinterpret_cast<uint8_t*>(out + o_keep);
    unsigned long long* d_key = reinterpret_cast<unsigned long long*>(out + o_key);
    int* d_first = reinterpret_cast<int*>(out + o_first);
    k_match_select<<<(unsigned)((na * 32 + 127) / 128), 128, 0, c->stream>>>(c->m_S.as<double>(), na, nb, validation,
                                                                            ratio_threshold, d_bb, d_bs, d_h1, d_keep);
    if (int r = check_launch(c, "k_match_select")) return r;
    if (validation & VALIDATE_CROSSCHECK) {
        CU(cudaMemsetAsync(d_key, 0xff, (size_t)nb * 8, c->stream));
        CU(cudaMemsetAsync(d_first, 0x7f, (size_t)nb * 4, c->stream));
        const unsigned gb = (unsigned)((na + 255) / 256);
        k_cross_min_score<<<gb, 256, 0, c->stream>>>(d_bb, d_bs, d_keep, na, d_key);
        if (int r = check_launch(c, "k_cross_min_score")) return r;
        k_cross_min_index<<<gb, 256, 0, c->stream>>>(d_bb, d_bs, d_keep, na, d_key, d_first);
        if (int r = check_launch(c, "k_cross_min_index")) return r;
        k_cross_filter<<<gb, 256, 0, c->stream>>>(d_bb, na, d_first, d_keep);
        if (int r = check_launch(c, "k_cross_filter")) return r;
    }
    CU(cudaMemcpyAsync(best_b, d_bb, (size_t)na * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(best_score, d_bs, (size_t)na * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(keep, d_keep, (size_t)na, cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

static int match_check_counts(int64_t na, int64_t nb, const void* best_b, const void* best_score, const void* keep) {
    if (na < 0 || nb < 0) return fail(SFM_ERR_ARG, "negative feature count");
    if (na > 0 && nb == 0) return fail(SFM_ERR_ARG, "features_b is empty (the reference raises IndexError, matching.py:79)");
    if (nb > 0x7fffffffLL || na > 0x7fffffffLL) return fail(SFM_ERR_ARG, "too many features");
    if (na > 0 && (!best_b || !best_score || !keep)) return fail(SFM_ERR_ARG, "null output");
    return 0;
}

int sfm_match_brute_force(sfm_ctx* c, const void* image_a, const void* image_b, int image_dtype, int64_t rows,
                          int64_t cols, const double* feats_a, int64_t na, const double* feats_b, int64_t nb,
                          int score_kind, int window, int validation, double ratio_threshold, int32_t* best_b,
                          double* best_score, uint8_t* keep, double* scores) {
    if (int r = use(c)) return r;
    if (!image_a || !image_b || rows <= 0 || cols <= 0) return fail(SFM_ERR_ARG, "bad images");
    if (image_dtype != IMG_U8 && image_dtype != IMG_F64) return fail(SFM_ERR_ARG, "image dtype must be 0 (uint8) or 1 (float64)");
    if (score_kind != SCORE_NCC && score_kind != SCORE_SSD) return fail(SFM_ERR_ARG, "score kind must be 0 (ncc) or 1 (ssd)");
    if (window < 1 || window > kMaxWindow) return fail(SFM_ERR_ARG, "window size must be in [1, %d]", kMaxWindow);
    window = 2 * (window / 2) + 1;  // util.py:21-27 cuts [c - int(w/2), c + int(w/2)]: an even w yields w + 1 pixels
    if (int r = match_check_counts(na, nb, best_b, best_score, keep)) return r;
    if ((na > 0 && !feats_a) || (nb > 0 && !feats_b)) return fail(SFM_ERR_ARG, "bad feature arrays");
    if (na == 0) return 0;
    const size_t px = (size_t)rows * cols, pxb = px * (image_dtype == IMG_U8 ? 1 : 8);
    const int ww = window * window;
    const size_t n = (size_t)(na + nb);
    const size_t img_b_off = (pxb + 15) / 16 * 16;  // second image, 16-byte aligned
    if (int r = c->m_img.reserve(img_b_off + pxb)) return r;
    if (int r = c->m_feat.reserve(n * 16)) return r;
    if (int r = c->m_W.reserve(n * ww * 8)) return r;
    if (int r = c->m_ss.reserve(n * 8)) return r;
    if (int r = c->m_ok.reserve(n)) return r;
    if (int r = c->m_S.reserve((size_t)na * nb * 8)) return r;
    char* img = c->m_img.as<char>();
    CU(cudaMemcpyAsync(img, image_a, pxb, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(img + img_b_off, image_b, pxb, cudaMemcpyHostToDevice, c->stream));
    double* feat = c->m_feat.as<double>();
    CU(cudaMemcpyAsync(feat, feats_a, (size_t)na * 16, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(feat + 2 * na, feats_b, (size_t)nb * 16, cudaMemcpyHostToDevice, c->stream));
    double* W = c->m_W.as<double>();
    double* ss = c->m_ss.as<double>();
    uint8_t* ok = c->m_ok.as<uint8_t>();
    k_patch_prepare<<<(unsigned)((na + 127) / 128), 128, 0, c->stream>>>(img, image_dtype, rows, cols, feat, na, window,
                                                                        score_kind, W, ss, ok);
    if (int r = check_launch(c, "k_patch_prepare")) return r;
    k_patch_prepare<<<(unsigned)((nb + 127) / 128), 128, 0, c->stream>>>(img + img_b_off, image_dtype, rows, cols,
                                                                        feat + 2 * na, nb, window, score_kind,
                                                                        W + (size_t)na * ww, ss + na, ok + na);
    if (int r = check_launch(c, "k_patch_prepare")) return r;
    dim3 grid((unsigned)((nb + kScoreTile - 1) / kScoreTile), (unsigned)((na + kScoreTile - 1) / kScoreTile));
    k_patch_scores<<<grid, kScoreTile * kScoreTile, 0, c->stream>>>(W, ss, ok, na, W + (size_t)na * ww, ss + na, ok + na,
                                                                   nb, ww, score_kind, image_dtype, c->m_S.as<double>());
    if (int r = check_launch(c, "k_patch_scores")) return r;
    if (int r = match_finish(c, na, nb, validation, ratio_threshold, best_b, best_score, keep)) return r;
    if (scores) CU(cudaMemcpyAsync(scores, c->m_S.p, (size_t)na * nb * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_match_from_scores(sfm_ctx* c, const double* scores, int64_t na, int64_t nb, int validation,
                          double ratio_threshold, int32_t* best_b, double* best_score, uint8_t* keep) {
    if (int r = use(c)) return r;
    if (int r = match_check_counts(na, nb, best_b, best_score, keep)) return r;
    if (na == 0) return 0;
    if (!scores) return fail(SFM_ERR_ARG, "null score matrix");
    if (int r = c->m_S.reserve((size_t)na * nb * 8)) return r;
    CU(cudaMemcpyAsync(c->m_S.p, scores, (size_t)na * nb * 8, cudaMemcpyHostToDevice, c->stream));
    if (int r = match_finish(c, na, nb, validation, ratio_threshold, best_b, best_score, keep)) return r;
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- N2: Harris corner detector (the first stage of apps/sfm.py) ------------------------------
static int harris_check_image(const void* image, int image_dtype, int64_t rows, int64_t cols) {
    if (!image || rows <= 0 || cols <= 0) return fail(SFM_ERR_ARG, "bad image");
    if (image_dtype != IMG_U8 && image_dtype != IMG_F64) return fail(SFM_ERR_ARG, "image dtype must be 0 (uint8) or 1 (float64)");
    if (rows * cols > 0x7fffffffLL) return fail(SFM_ERR_ARG, "image too large");
    return 0;
}

int sfm_cross_correlate(sfm_ctx* c, const void* image, int image_dtype, int64_t rows, int64_t cols,
                        const double* kernel, int ksize, double* out) {
    if (int r = use(c)) return r;
    if (int r = harris_check_image(image, image_dtype, rows, cols)) return r;
    if (!kernel || !out) return fail(SFM_ERR_ARG, "null kernel or output");
    if (ksize < 1 || (ksize % 2) == 0) return fail(SFM_ERR_ARG, "only odd-sized square kernels are supported");  // correlate.py:18-19
    if (rows < ksize || cols < ksize) return fail(SFM_ERR_ARG, "kernel cannot be larger than image");           // correlate.py:21-22
    const size_t px = (size_t)rows * cols, pxb = px * (image_dtype == IMG_U8 ? 1 : 8);
    if (int r = c->h_img.reserve(pxb)) return r;
    if (int r = c->h_gx.reserve(px * 8)) return r;
    if (int r = c->h_small.reserve((size_t)ksize * ksize * 8 + 64)) return r;
    CU(cudaMemcpyAsync(c->h_img.p, image, pxb, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->h_small.p, kernel, (size_t)ksize * ksize * 8, cudaMemcpyHostToDevice, c->stream));
    k_cross_correlate<<<(unsigned)((px + 255) / 256), 256, 0, c->stream>>>(c->h_img.p, image_dtype, (int)rows, (int)cols,
                                                                          c->h_small.as<double>(), ksize,
                                                                          c->h_gx.as<double>());
    if (int r = check_launch(c, "k_cross_correlate")) return r;
    CU(cudaMemcpyAsync(out, c->h_gx.p, px * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_harris_output_shape(int64_t rows, int64_t cols, int block_size, int64_t* out_rows, int64_t* out_cols) {
    if (block_size < 1 || !out_rows || !out_cols) return fail(SFM_ERR_ARG, "bad block size or null output");
    // int(np.around(block_size / 2)): round half to even (harris_detector.py:66-72)
    const int half = block_size / 2;
    const int shrink = (block_size % 2 == 0) ? half : ((half % 2 == 0) ? half : half + 1);
    *out_rows = rows - shrink;
    *out_cols = cols - shrink;
    return 0;
}

int sfm_harris_corners(sfm_ctx* c, const void* image, int image_dtype, int64_t rows, int64_t cols,
                       int64_t num_corners, int block_size, double k, double* xy, double* score, int64_t* num_found,
                       double* cornerness, int32_t* nms_sweeps) {
    if (int r = use(c)) return r;
    if (int r = harris_check_image(image, image_dtype, rows, cols)) return r;
    if (num_corners <= 0) return fail(SFM_ERR_ARG, "num_corners needs to be at least 1");  // harris_detector.py:24-25
    if (block_size < 1 || block_size > 64) return fail(SFM_ERR_ARG, "block_size must be in [1, 64]");
    if (rows < 3 || cols < 3) return fail(SFM_ERR_ARG, "kernel cannot be larger than image");  // correlate.py:21-22 (Sobel)
    if (!xy || !score || !num_found) return fail(SFM_ERR_ARG, "null output");
    int64_t orows = 0, ocols = 0;
    sfm_harris_output_shape(rows, cols, block_size, &orows, &ocols);
    if (orows <= 0 || ocols <= 0) return fail(SFM_ERR_ARG, "block_size too large for this image");
    const size_t px = (size_t)rows * cols, pxb = px * (image_dtype == IMG_U8 ? 1 : 8);
    const size_t opx = (size_t)orows * ocols;
    size_t padded = kSortTile;
    while (padded < opx) padded <<= 1;
    if (int r = c->h_img.reserve(pxb)) return r;
    if (int r = c->h_gx.reserve(px * 8)) return r;
    if (int r = c->h_gy.reserve(px * 8)) return r;
    if (int r = c->h_corner.reserve(opx * 8)) return r;
    if (int r = c->h_alive.reserve(2 * opx)) return r;
    if (int r = c->h_small.reserve(64)) return r;
    const int64_t nout = num_corners < (int64_t)opx ? num_corners : (int64_t)opx;
    if (int r = c->h_xy.reserve((size_t)nout * 24)) return r;
    CU(cudaMemcpyAsync(c->h_img.p, image, pxb, cudaMemcpyHostToDevice, c->stream));
    const unsigned gpx = (unsigned)((px + 255) / 256), gopx = (unsigned)((opx + 255) / 256);
    k_sobel_pair<<<gpx, 256, 0, c->stream>>>(c->h_img.p, image_dtype, (int)rows, (int)cols, c->h_gx.as<double>(),
                                             c->h_gy.as<double>());
    if (int r = check_launch(c, "k_sobel_pair")) return r;
    double* corner = c->h_corner.as<double>();
    k_cornerness<<<gopx, 256, 0, c->stream>>>(c->h_gx.as<double>(), c->h_gy.as<double>(), (int)rows, (int)cols, block_size,
                                              k, (int)orows, (int)ocols, corner);
    if (int r = check_launch(c, "k_cornerness")) return r;
    // non-maximum suppression: sweeps in batches of 8, one "changed" flag per sweep; a sweep that changes
    // nothing has reached the fixed point, so only the last flag of a batch needs to be looked at
    uint8_t* alive[2] = {c->h_alive.as<uint8_t>(), c->h_alive.as<uint8_t>() + opx};
    int* d_changed = c->h_small.as<int>();            // [8]
    unsigned* d_count = reinterpret_cast<unsigned*>(d_changed + 8);
    CU(cudaMemsetAsync(alive[0], 1, opx, c->stream));
    int cur = 0, sweeps = 0;
    for (;;) {
        CU(cudaMemsetAsync(d_changed, 0, 32, c->stream));
        for (int it = 0; it < 8; ++it) {
            k_nms_sweep<<<gopx, 256, 0, c->stream>>>(corner, (int)orows, (int)ocols, alive[cur], alive[cur ^ 1], d_changed + it);
            if (int r = check_launch(c, "k_nms_sweep")) return r;
            cur ^= 1;
        }
        sweeps += 8;
        int changed[8] = {0};
        CU(cudaMemcpyAsync(changed, d_changed, 32, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (!changed[7]) break;
        if ((size_t)sweeps > opx + 16) return fail(SFM_ERR_CUDA, "non-maximum suppression did not converge");
    }
    k_nms_apply<<<gopx, 256, 0, c->stream>>>(corner, (long long)opx, alive[cur]);
    if (int r = check_launch(c, "k_nms_apply")) return r;
    // candidates -> sort -> first num_corners
    CU(cudaMemsetAsync(d_count, 0, 4, c->stream));
    if (int r = c->h_key.reserve(padded * 8)) return r;
    if (int r = c->h_idx.reserve(padded * 4)) return r;
    unsigned long long* key = c->h_key.as<unsigned long long>();
    unsigned* idx = c->h_idx.as<unsigned>();
    k_corner_compact<<<gopx, 256, 0, c->stream>>>(corner, (long long)opx, key, idx, d_count);
    if (int r = check_launch(c, "k_corner_compact")) return r;
    unsigned count = 0;
    CU(cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    size_t n = kSortTile;
    while (n < count) n <<= 1;
    k_corner_pad<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(key, idx, d_count, (unsigned)n);
    if (int r = check_launch(c, "k_corner_pad")) return r;
    const unsigned tiles = (unsigned)(n / kSortTile);
    k_bitonic_local<<<tiles, kSortTile / 2, 0, c->stream>>>(key, idx, 0u, 0);
    if (int r = check_launch(c, "k_bitonic_local")) return r;
    for (size_t ks = 2 * (size_t)kSortTile; ks <= n; ks <<= 1) {
        for (size_t j = ks >> 1; j >= (size_t)kSortTile; j >>= 1) {
            k_bitonic_global<<<(unsigned)((n / 2 + 255) / 256), 256, 0, c->stream>>>(key, idx, (unsigned)n, (unsigned)ks, (unsigned)j);
            if (int r = check_launch(c, "k_bitonic_global")) return r;
        }
        k_bitonic_local<<<tiles, kSortTile / 2, 0, c->stream>>>(key, idx, (unsigned)ks, 1);
        if (int r = check_launch(c, "k_bitonic_local")) return r;
    }
    const int64_t found = (int64_t)count < num_corners ? (int64_t)count : num_corners;
    *num_found = found;
    if (found > 0) {
        double* d_xy = c->h_xy.as<double>();
        double* d_score = d_xy + 2 * nout;
        k_corner_emit<<<(unsigned)((found + 255) / 256), 256, 0, c->stream>>>(key, idx, d_count, found, (int)ocols,
                                                                             (double)block_size / 2.0, corner, d_xy, d_score);
        if (int r = check_launch(c, "k_corner_emit")) return r;
        CU(cudaMemcpyAsync(xy, d_xy, (size_t)found * 16, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(score, d_score, (size_t)found * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    if (cornerness) CU(cudaMemcpyAsync(cornerness, corner, opx * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (nms_sweeps) *nms_sweeps = sweeps;
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

}  // extern "C"
