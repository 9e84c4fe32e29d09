// The C ABI's RANSAC stages: correspondence upload and K2's sorted copy, the sample table, the essential-matrix,
// homography and absolute-pose fits (K1), scoring (K2), finalise + select (K3), inlier masks, the batched estimate and
// the hypothesis-sharded score, merge and fetch.
#include <cmath>

#include <cub/device/device_radix_sort.cuh>

#include "sfm_host.h"
#include "sfm_fit.cuh"
#include "sfm_score.cuh"
#include "sfm_homography.cuh"
#include "sfm_pnp.cuh"

using namespace sfm;
using namespace sfm_host;

static_assert(sizeof(Corr) == 32, "Corr must be 32 bytes");
static_assert(sizeof(SelectRecord) == SFM_RECORD_BYTES, "SelectRecord / SFM_RECORD_BYTES mismatch");

namespace {

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

// ---- sampling ---------------------------------------------------------------------------
int sfm_set_table(sfm_ctx* c, const int32_t* table, int64_t h) {
    if (int r = use(c)) return r;
    if (!table || h <= 0) return fail(SFM_ERR_ARG, "bad table");
    if (!c->has_pts && !c->has_pnp) return fail(SFM_ERR_STATE, "upload correspondences before the sample table");
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
int sfm_host::sample_device(sfm_ctx* c, uint64_t seed, uint64_t stream, int64_t hyp_offset, int64_t h) {
    if (h <= 0) return fail(SFM_ERR_ARG, "need h > 0");
    if (!c->has_pts && !c->has_pnp) return fail(SFM_ERR_STATE, "upload correspondences before sampling");
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

int sfm_host::ensure_table(sfm_ctx* c) {
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

// m correspondences of one pair at s[] (stride as in stage_coords) to records normalised with the K at K_dev
int sfm_host::normalise_launch(sfm_ctx* c, const double* const s[4], int64_t stride, int64_t m, const double* K_dev, Corr* out) {
    k_normalise<<<dim3((unsigned)((m + 255) / 256), 1), 256, 0, c->stream>>>(s[0], s[1], s[2], s[3], stride, m, nullptr, K_dev, out,
                                                                            nullptr);
    return check_launch(c, "k_normalise");
}

// Host coordinates to the device buffer d (room for 4 n doubles) in the caller's layout: four arrays (stride 1) or two
// interleaved [n][2] arrays (stride 2).  s[] = the device addresses of xa, ya, xb, yb.
int sfm_host::stage_coords(sfm_ctx* c, double* d, const double* xa, const double* ya, const double* xb, const double* yb,
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
void sfm_host::raw_coords(const sfm_ctx* c, const double* s[4]) {
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
    c->has_pnp = c->pnp_models = false;
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
// k_fit's dynamic shared memory is above the default limit: raised once, when a context is created
int sfm_host::allow_fit_smem() {
    CU(cudaFuncSetAttribute(k_fit, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(kFitThreads * kFitSmemDoubles * sizeof(double))));
    return 0;
}

// K2's accumulator buffer is [kAccWords][H] planes followed by this tail, cleared with them: +0 work counter,
// +8 rescore counter, +16 pilot totals, +24 pilot ticket, +32 mode, +64 K3 tickets [P]
static size_t acc_tail_bytes(long long P) { return 64 + (size_t)P * 4; }

int sfm_host::fit_launch(sfm_ctx* c, bool want_eig) {
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
    f.pts = kind == MODEL_P ? c->ppts.p : c->pts.p;
    f.offsets = c->batched ? c->offsets.as<long long>() : nullptr;
    f.E = kind == MODEL_P ? c->pmodels.as<double>() : c->E.as<double>();
    f.K = c->pK.as<double>();
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
    else if (kind == MODEL_P) CU(chain_launch(c, k_finalise<MODEL_P>, dim3((unsigned)fblocks, (unsigned)P), dim3(256), 0, f));
    else CU(chain_launch(c, k_finalise<MODEL_E>, dim3((unsigned)fblocks, (unsigned)P), dim3(256), 0, f));
    if (int r = check_launch(c, "k_finalise")) return r;
    c->toc(T_SELECT);
    c->has_score = true;
    c->last_idx_offset = idx_offset;
    c->winner_set = false;
    return 0;
}

int sfm_host::score_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, bool use_table,
                        long long idx_offset, long long max_len, bool both_sums) {
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
void sfm_host::unpack_best(const SelectRecord& r, sfm_best* out) {
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
        // the decomposition of the refinement's start and the tail square E's entries: a power of two keeps them in
        // range whatever the caller's scale, and every result is the same as for 2^k E
        double Es[9];
        prescaled(E, 9, prescale_exponent(E, 9), Es);
        CU(cudaMemcpyAsync(c->winnerE.p, Es, 72, cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->winner_local = -1;
    }
    c->winner_set = true;
    return 0;
}

const double* sfm_host::winner_E_dev(sfm_ctx* c) {
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
int sfm_host::fit_h_launch(sfm_ctx* c) {
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
int sfm_host::score_h_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode, long long max_len) {
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

// ---- absolute pose (sfm_pnp.cuh) --------------------------------------------------------------
int sfm_upload_pnp(sfm_ctx* c, const double* X, const double* x, int64_t n, const double* K) {
    if (int r = use(c)) return r;
    if (!X || !x) return fail(SFM_ERR_ARG, "null argument");
    if (n <= 0 || (uint64_t)n >= kMaxPoints) return fail(SFM_ERR_ARG, "need 0 < n < 2^25 records, got %lld", (long long)n);
    if (int r = check_camera(K)) return r;
    if (K[3] != 0.0 || K[6] != 0.0 || K[7] != 0.0 || K[8] != 1.0)
        return fail(SFM_ERR_ARG, "the camera matrix must be upper triangular with K[2,2] = 1");
    std::vector<PnpRec> rec((size_t)n);
    for (int64_t i = 0; i < n; ++i)
        rec[(size_t)i] = PnpRec{X[3 * i], X[3 * i + 1], X[3 * i + 2], x[2 * i], x[2 * i + 1], 0.0};
    if (int r = c->ppts.reserve((size_t)n * sizeof(PnpRec))) return r;
    if (int r = c->pK.reserve(72)) return r;
    c->tic(T_UPLOAD);
    CU(cudaMemcpyAsync(c->ppts.p, rec.data(), (size_t)n * sizeof(PnpRec), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->pK.p, K, 72, cudaMemcpyHostToDevice, c->stream));
    c->toc(T_UPLOAD);
    CU(cudaStreamSynchronize(c->stream));  // the copies read host memory
    c->n = n;
    c->batched = false;
    c->npairs = 1;
    c->has_pts = false;  // c->pts no longer describes the upload: the E and H calls refuse
    c->has_pnp = true;
    c->pnp_models = false;
    c->has_table = c->has_models = c->has_score = false;
    c->table_pending = false;
    c->winner_set = false;
    return 0;
}

// the P3P fits of the h rows of the table or the device draw; clears K2's accumulators as the other fits do
static int fit_p_launch(sfm_ctx* c) {
    if (!c->has_pnp || !c->has_table) return fail(SFM_ERR_STATE, "fit needs PnP records and a sample table");
    const long long h = c->h;
    if (int r = c->pmodels.reserve((size_t)h * 96)) return r;
    if (int r = c->valid.reserve((size_t)h)) return r;
    const size_t acc_tail = acc_tail_bytes(1);
    if (int r = c->acc.reserve((size_t)h * kAccWords * 8 + acc_tail)) return r;
    c->tic(T_FIT);
    CU(chain_launch(c, k_fit_pnp, dim3((unsigned)((h + kFitPThreads - 1) / kFitPThreads)), dim3(kFitPThreads), 0,
                    c->ppts.as<PnpRec>(), c->pK.as<double>(), c->table.as<int32_t>(), h, c->pmodels.as<double>(),
                    c->valid.as<uint8_t>(), c->acc.as<unsigned long long>(), kAccWords, (int)((acc_tail + 7) / 8),
                    c->table_pending ? 1 : 0, c->smp_seed, c->smp_stream, c->smp_offset, c->n));
    if (int r = check_launch(c, "k_fit_pnp")) return r;
    c->toc(T_FIT);
    c->table_pending = false;
    c->acc_clean = true;
    c->acc_planes_for = (size_t)h;
    c->pnp_models = true;
    c->has_score = false;
    return 0;
}

// K2 + K3 of the poses of the last fit
static int score_p_launch(sfm_ctx* c, double thr, double min_extra, int agg, int mode) {
    if (agg < 0 || agg > 3) return fail(SFM_ERR_ARG, "bad aggregation %d", agg);
    if (mode < 0 || mode > 2) return fail(SFM_ERR_ARG, "bad selection %d", mode);
    int sums = (agg == AGG_SUM || agg == AGG_MEAN) ? SUM_S1 : SUM_S2;
    if (mode == SELECT_MSAC) sums |= SUM_S1;
    // the threshold ranges of the E and H paths: below 0, NaN and above 1e100 the scorer is skipped and K3 rescores
    const bool skip_k2 = !(thr >= 0.0) || thr > 1e100;
    const int force_rescore = (thr > 1e100) ? 1 : 0;
    const long long h = c->h, n = c->n;
    // an inlier's value F / W can exceed thr by a few ulps (the decision is division-free), as on the H path
    int e2 = 0;
    if (thr > 0.0 && !skip_k2) (void)frexp(thr * (1.0 + 0x1p-20), &e2);
    if (e2 < -400) e2 = -400;
    if (int r = reserve_selection(c, h, 1)) return r;
    if (int r = c->acc.reserve((size_t)h * kAccWords * 8 + acc_tail_bytes(1))) return r;
    unsigned long long* acc = c->acc.as<unsigned long long>();
    const size_t smem = kPScoreWarps * sizeof(PScoreWarpSmem);
    if (!c->pscore_occ) {
        int o = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_score_pnp<kPScoreHpt>, kPScoreThreads, smem));
        c->pscore_occ = o > 0 ? o : 1;
    }
    const long long grid_blocks = (long long)c->sm_count * c->pscore_occ;
    const long long hblocks = (h + 32ll * kPScoreHpt - 1) / (32ll * kPScoreHpt);
    const ItemSplit sp = split_items(grid_blocks * kPScoreWarps * 32, hblocks, n, kPTile);
    PScoreArgs a;
    a.pts = c->ppts.as<PnpRec>();
    a.K = c->pK.as<double>();
    a.Rt = c->pmodels.as<double>();
    a.n = n;
    a.h = h;
    a.thr = thr;
    a.scale1 = ldexp(1.0, 63 - e2);
    a.scale2 = ldexp(1.0, 63 - 2 * e2);
    a.sums = sums;
    a.chunk = sp.chunk;
    a.hblocks = (int)hblocks;
    a.nsplit = (int)sp.nsplit;
    a.total_items = hblocks * sp.nsplit;
    a.work_counter = reinterpret_cast<unsigned*>(acc + (size_t)h * kAccWords);
    a.acc = acc;
    c->tic(T_SCORE);
    if (int r = clear_acc(c, (size_t)h, 1)) return r;
    if (!skip_k2) {
        const long long want = (a.total_items + kPScoreWarps - 1) / kPScoreWarps;
        CU(chain_launch(c, k_score_pnp<kPScoreHpt>, dim3((unsigned)(grid_blocks < want ? grid_blocks : want)),
                        dim3(kPScoreThreads), smem, a));
        if (int r = check_launch(c, "k_score_pnp")) return r;
    }
    c->toc(T_SCORE);
    return finalise_launch(c, MODEL_P, thr, min_extra, agg, mode, true, 0, sums, e2, force_rescore, acc);
}

// decision and value of every record under the pose at Rt_dev[12 * best->idx] (best != null) or at Rt_dev
int sfm_host::pmask_launch(sfm_ctx* c, double thr, const double* Rt_dev, const Best* best_dev, double* winner_out) {
    if (int r = c->mask.reserve((size_t)c->n)) return r;
    if (int r = c->sed.reserve((size_t)c->n * 8)) return r;
    c->tic(T_MASK);
    CU(chain_launch(c, k_pnp_mask, dim3((unsigned)((c->n + 255) / 256)), dim3(256), 0, c->ppts.as<PnpRec>(), c->n,
                    c->pK.as<double>(), Rt_dev, best_dev, thr, c->mask.as<uint8_t>(), c->sed.as<double>(), winner_out));
    if (int r = check_launch(c, "k_pnp_mask")) return r;
    c->toc(T_MASK);
    return 0;
}

int sfm_fit_pnp(sfm_ctx* c, double* Rt_out, uint8_t* valid_out) {
    if (int r = use(c)) return r;
    if (int r = fit_p_launch(c)) return r;
    if (Rt_out) CU(cudaMemcpyAsync(Rt_out, c->pmodels.p, (size_t)c->h * 96, cudaMemcpyDeviceToHost, c->stream));
    if (valid_out) CU(cudaMemcpyAsync(valid_out, c->valid.p, (size_t)c->h, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_get_pnp_models(sfm_ctx* c, int64_t first, int64_t count, double* Rt_out, uint8_t* valid_out) {
    if (int r = use(c)) return r;
    if (!c->has_pnp || !c->pnp_models || first < 0 || count < 0 || first + count > c->h)
        return fail(SFM_ERR_STATE, "no poses [%lld, %lld)", (long long)first, (long long)(first + count));
    if (Rt_out) CU(cudaMemcpyAsync(Rt_out, c->pmodels.as<double>() + 12 * first, (size_t)count * 96, cudaMemcpyDeviceToHost, c->stream));
    if (valid_out) CU(cudaMemcpyAsync(valid_out, c->valid.as<uint8_t>() + first, (size_t)count, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int sfm_ransac_pnp(sfm_ctx* c, double thr, double min_extra, int agg, int mode, sfm_best* best, double* Rt,
                   uint8_t* mask, double* err, int32_t* count_extra_h, double* err_h) {
    if (int r = use(c)) return r;
    if (!best) return fail(SFM_ERR_ARG, "best is null");
    if (c->has_pnp && c->n < 8) return fail(SFM_ERR_ARG, "need at least 8 records, got %lld", c->n);
    if (int r = c->pwin.reserve(96)) return r;
    if (int r = fit_p_launch(c)) return r;
    if (int r = score_p_launch(c, thr, min_extra, agg, mode)) return r;
    // the mask kernel also copies the winner out of the poses (K3's record has no room for 12 doubles)
    if (int r = pmask_launch(c, thr, c->pmodels.as<double>(), c->best.as<Best>(), c->pwin.as<double>())) return r;
    if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    if (err) CU(cudaMemcpyAsync(err, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    if (Rt) CU(cudaMemcpyAsync(Rt, c->pwin.p, 96, cudaMemcpyDeviceToHost, c->stream));
    if (count_extra_h) CU(cudaMemcpyAsync(count_extra_h, c->count_extra.p, (size_t)c->h * 4, cudaMemcpyDeviceToHost, c->stream));
    if (err_h) CU(cudaMemcpyAsync(err_h, c->err.p, (size_t)c->h * 8, cudaMemcpyDeviceToHost, c->stream));
    return fetch_best(c, best);
}

int sfm_pnp_mask(sfm_ctx* c, const double* Rt, double thr, uint8_t* mask, double* err) {
    if (int r = use(c)) return r;
    if (!c->has_pnp) return fail(SFM_ERR_STATE, "no PnP records loaded");
    const double* Rt_dev;
    if (Rt) {
        if (int r = c->pwin.reserve(96)) return r;
        CU(cudaMemcpyAsync(c->pwin.p, Rt, 96, cudaMemcpyHostToDevice, c->stream));
        Rt_dev = c->pwin.as<double>();
    } else {
        if (!c->pnp_models || !c->has_score || !c->winner_set || c->winner_local < 0)
            return fail(SFM_ERR_STATE, "no pose winner: pass Rt or run sfm_ransac_pnp first");
        Rt_dev = c->pmodels.as<double>() + 12 * c->winner_local;
    }
    if (int r = pmask_launch(c, thr, Rt_dev, nullptr, nullptr)) return r;
    if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    if (err) CU(cudaMemcpyAsync(err, c->sed.p, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
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

// ---- batched pairs ------------------------------------------------------------------------
// The upload of P independent pairs: offsets, the caller's cameras (c->Ks, and c->Kbatch on the host) and the raw
// coordinates (c->raw), from which the records are built - K-normalised with each pair's K for essential matrices, in
// pixels (an identity camera) for homographies.  Nothing synchronised.
int sfm_host::batch_upload(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb,
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
        if (int r = normalise_launch(c, s, stride, n, c->hK.as<double>(), c->pts.as<Corr>())) return r;
        c->k2_ready = false;  // pixel records: the essential-matrix scorer does not run on them
    } else if (int r = normalise_from(c, s[0], s[1], s[2], s[3], stride, n, max_len)) {
        return r;
    }
    c->toc(T_UPLOAD);
    c->has_pts = true;
    c->has_pnp = c->pnp_models = false;
    c->has_table = c->has_models = c->has_score = false;
    c->table_pending = false;
    c->winner_set = false;
    *max_len_out = max_len;
    return 0;
}

// upload -> device sampler -> fit -> score + select of P independent pairs (nothing synchronised)
int sfm_host::batch_core(sfm_ctx* c, const double* xa, const double* ya, const double* xb, const double* yb, int64_t stride,
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
int sfm_host::batch_fetch_winners(sfm_ctx* c, int64_t npairs, size_t extra_pinned, char** extra) {
    const size_t rbytes = (size_t)npairs * sizeof(SelectRecord);
    if (int r = ensure_pinned(c, rbytes + extra_pinned + 64)) return r;
    char* hp = (char*)c->hpin;
    CU(cudaMemcpyAsync(hp, c->record.p, rbytes, cudaMemcpyDeviceToHost, c->stream));
    if (extra) *extra = hp + ((rbytes + 63) / 64) * 64;
    return 0;
}

void sfm_host::batch_unpack_winners(const char* hp, int64_t npairs, double* E, int64_t* best_index, double* best_err,
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
