// Host side shared by the translation units of the C ABI: the context, device buffers, error reporting, launch helpers
// and the few internal functions one stage calls in another.  Each stage file owns its kernel headers:
//   sfm_api.cu          context lifecycle, stream, errors, timing               sfm_misc.cuh
//   sfm_ransac.cu       upload, sampler, E and H fit, K2 and its shape, K3,     sfm_fit.cuh, sfm_score.cuh, sfm_homography.cuh
//                       masks, batches, hypothesis-sharded scoring
//   sfm_two_view.cu     pose/triangulation list API, tail, refinement           sfm_pose.cuh, sfm_hpose.cuh, sfm_tail.cuh,
//                                                                               sfm_refine.cuh
//   sfm_model_select.cu essential matrix or homography                          sfm_select.cuh
//   sfm_front_end.cu    matcher, cross-correlation, Harris                      sfm_match.cuh, sfm_harris.cuh
//   sfm_nccl.cpp, sfm_sampler.cpp: host only, compiled by the host compiler
// include/sfm_b200.h declares every sfm_* entry point extern "C"; their definitions in the stage files take that linkage.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sfm_b200.h"
#include "sfm_types.h"

namespace sfm {
struct Corr;
}

namespace sfm_host {

extern thread_local std::string g_err;

int fail(int code, const char* fmt, ...);

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

}  // namespace sfm_host

struct sfm_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // data
    sfm_host::Buf raw, pts, offsets, Ks, table, E, valid, eig;
    sfm_host::Buf acc, count_extra, S1, S2, err, blocks, best, invalid, winnerE, spts, bounds, fitflag, record, merged, rows, blockinv;
    sfm_host::Buf m_img, m_feat, m_W, m_ss, m_ok, m_S, m_out;
    sfm_host::Buf h_img, h_gx, h_gy, h_corner, h_alive, h_key, h_idx, h_small, h_xy;
    sfm_host::Buf mask, sed, poses, pass, X, idx, scan, tmp, tailstate, num, winrec, bout;
    sfm_host::Buf planes, hK;  // the homography tail's HPlane and the K it was called with (the upload's K stays in Ks)
    sfm_host::Buf k2pts, k2box, k2sort;  // K2's copy of pts in image-B Morton order, its tile boxes, the sort's scratch
    sfm_host::Buf selstate, selio, selpp;  // k_score_models: self-cleaning sums; models and results; per-correspondence errors
    sfm_host::Buf refstate, refpart, reftick, refrec, refrep;  // refinement: LM state, chunk partials, tickets, records, reports
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
    double Estage[9] = {0};   // caller's E (stand-alone decomposition / pose), prescaled
    double Pstage[24] = {0};  // caller's P1, P2 (stand-alone triangulation), prescaled
    double hstage[18] = {0};  // H and K of sfm_decompose_homography, K of the homography tail, staged for async copies
    std::vector<sfm::SelectModels> sstage;  // the models of sfm_score_models / sfm_batch_score_models, staged for the async copy
    std::vector<double> Kbatch;        // the cameras of the current batched upload, [P][9] (the device copy is Ks)
    const void* occ_fn[4] = {nullptr, nullptr, nullptr, nullptr};  // scoring kernels whose launch configuration is cached
    int occ_blocks[4] = {0, 0, 0, 0};
    int occ_next = 0;
    void* nccl_comm = nullptr;  // ncclComm_t of sfm_nccl_init (hypothesis-sharded runs without torch)
    int nccl_rank = 0, nccl_world = 1;
    sfm_host::Buf gathered;
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
    cudaEvent_t ev0[sfm_host::T_COUNT], ev1[sfm_host::T_COUNT];
    bool ev_used[sfm_host::T_COUNT];
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

namespace sfm_host {

inline int ensure_pinned(sfm_ctx* c, size_t bytes) {
    if (bytes <= c->hpin_cap) return 0;
    if (c->hpin) cudaFreeHost(c->hpin);
    c->hpin = nullptr;
    c->hpin_cap = 0;
    CU(cudaMallocHost(&c->hpin, bytes + 4096));
    c->hpin_cap = bytes + 4096;
    return 0;
}

inline int use(sfm_ctx* c) {
    if (!c) return fail(SFM_ERR_ARG, "null context");
    CU(cudaSetDevice(c->device));
    return 0;
}

// Device buffer that must read as zero before its first use (self-cleaning kernel state).
inline int reserve_zeroed(sfm_ctx* c, Buf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (int r = b.reserve(bytes)) return r;
    CU(cudaMemsetAsync(b.p, 0, b.cap, c->stream));
    return 0;
}

inline int check_launch(sfm_ctx* c, const char* what) {
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

// ---- sfm_ransac.cu ------------------------------------------------------------------------
int allow_fit_smem();
int sample_device(sfm_ctx* c, uint64_t seed, uint64_t stream, int64_t hyp_offset, int64_t h);
int ensure_table(sfm_ctx* c);
int stage_coords(sfm_ctx* c, double* d, const double* xa, const double* ya, const double* xb, const double* yb,
                 int64_t stride, int64_t n, const double* s[4]);
void raw_coords(const sfm_ctx* c, const double* s[4]);
int normalise_launch(sfm_ctx* c, const double* const s[4], int64_t stride, int64_t m, const double* K_dev, sfm::Corr* out);
int batch_upload(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb, int64_t stride,
                 const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h, bool pixels, long long* max_len_out);
int batch_core(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb, int64_t stride,
               const int64_t* offsets, int64_t npairs, const double* Ks, int64_t h, uint64_t seed, uint64_t pair_id0,
               double thr, double min_extra, int agg, int mode, long long* max_len_out);
int fit_launch(sfm_ctx* c, bool want_eig);
int score_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, bool use_table, long long idx_offset,
                 long long max_len, bool both_sums = false);
int fit_h_launch(sfm_ctx* c);
int score_h_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, long long max_len);
void unpack_best(const sfm::SelectRecord& r, sfm_best* out);
const double* winner_E_dev(sfm_ctx* c);
int batch_fetch_winners(sfm_ctx* c, int64_t npairs, size_t extra_pinned, char** extra);
void batch_unpack_winners(const char* hp, int64_t npairs, double* E, int64_t* best_index, double* best_err,
                          int32_t* count_extra, int64_t* num_invalid);

// ---- sfm_two_view.cu ----------------------------------------------------------------------
int pose_tail_launch(sfm_ctx* c, double thr, double dist_thr, const sfm::SelectRecord* rec_dev, long long max_len,
                     uint8_t* mask_host = nullptr, double* sed_host = nullptr, int kind = sfm::MODEL_E,
                     double rot_tol = 0.0);
int copy_inliers(sfm_ctx* c, long long take, int64_t* inlier_idx, uint8_t* pass, double* X);
int check_camera(const double* K);
int hpose_stage_k(sfm_ctx* c, const double* K);

}  // namespace sfm_host
