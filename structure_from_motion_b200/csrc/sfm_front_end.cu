// The C ABI's front end, the stages in front of the hot path: brute-force matching and Harris corners.
#include "sfm_host.h"
#include "sfm_match.cuh"
#include "sfm_harris.cuh"

using namespace sfm;
using namespace sfm_host;

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
