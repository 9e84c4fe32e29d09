// The C ABI's multi-view triangulation of tracks (sfm_tracks.cuh): argument checks, the item offsets of the pair search,
// the three launches and the copies back.
#include <cmath>

#include "sfm_host.h"
#include "sfm_tracks.cuh"

using namespace sfm;
using namespace sfm_host;

static_assert(sizeof(TrackRefineReport) == sizeof(sfm_track_refinement), "TrackRefineReport / sfm_track_refinement layout mismatch");
static_assert(SFM_TRACK_MAX_OBSERVATIONS == kMaxTrack, "the header's track length limit is the kernel's");

int sfm_triangulate_tracks(sfm_ctx* c, const double* K, const double* Rt, int32_t V, const int64_t* offsets, int64_t T,
                           const int32_t* view, const double* x, double threshold, double min_angle_deg,
                           int32_t min_views, int32_t refine_iterations, double* X, int32_t* status,
                           int32_t* num_inliers, double* angle, uint8_t* mask, double* err,
                           sfm_track_refinement* refine_report) {
    if (int r = use(c)) return r;
    if (V < 1) return fail(SFM_ERR_ARG, "at least one view is needed, got %d", V);
    if (T < 0) return fail(SFM_ERR_ARG, "negative track count");
    if (!K || !Rt || !offsets) return fail(SFM_ERR_ARG, "null argument");
    if (!std::isfinite(threshold)) return fail(SFM_ERR_ARG, "the threshold must be finite");
    if (!std::isfinite(min_angle_deg)) return fail(SFM_ERR_ARG, "min_angle_deg must be finite");
    if (min_views < 2) return fail(SFM_ERR_ARG, "min_views must be >= 2, got %d", min_views);
    if (refine_iterations < 0) return fail(SFM_ERR_ARG, "refine_iterations must be >= 0, got %d", refine_iterations);
    for (int v = 0; v < V; ++v) {
        const double* Kv = K + 9 * (size_t)v;
        if (int r = check_camera(Kv)) {
            const std::string why = g_err;
            return fail(r, "camera %d: %s", v, why.c_str());
        }
        if (Kv[3] != 0.0 || Kv[6] != 0.0 || Kv[7] != 0.0 || Kv[8] != 1.0)
            return fail(SFM_ERR_ARG, "camera %d: the camera matrix must be upper triangular with K[2,2] = 1", v);
        for (int k = 0; k < 12; ++k)
            if (!std::isfinite(Rt[12 * (size_t)v + k])) return fail(SFM_ERR_ARG, "pose %d is not finite", v);
    }
    if (offsets[0] != 0) return fail(SFM_ERR_ARG, "offsets[0] must be 0, got %lld", (long long)offsets[0]);
    // the pair search's item offsets: a track of n_t >= 3 observations owns n_t (n_t - 1) / 2 items from pbase[t]; a
    // track of 2 is its own single item in k_track_solve
    std::vector<long long> pbase((size_t)T + 1);
    pbase[0] = 0;
    for (int64_t t = 0; t < T; ++t) {
        const int64_t n = offsets[t + 1] - offsets[t];
        if (n < 0) return fail(SFM_ERR_ARG, "offsets decrease at track %lld", (long long)t);
        if (n > kMaxTrack)
            return fail(SFM_ERR_ARG, "track %lld has %lld observations, more than %d", (long long)t, (long long)n, kMaxTrack);
        pbase[t + 1] = pbase[t] + (n > 2 ? n * (n - 1) / 2 : 0);
    }
    const long long M = offsets[T], items = pbase[T];
    if (M > 0 && (!view || !x)) return fail(SFM_ERR_ARG, "null observations");
    for (long long i = 0; i < M; ++i)
        if (view[i] < 0 || view[i] >= V) return fail(SFM_ERR_ARG, "observation %lld: view %d outside [0, %d)", i, view[i], V);
    if (T == 0) return 0;
    // inputs: K, Rt, views, frame, offsets, pbase, view, x (each 16-byte aligned); outputs in trkout
    auto up = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const size_t bK = up((size_t)V * 72), bRt = up((size_t)V * 96), bV = up((size_t)V * sizeof(TrackView)), bF = 16,
                 bO = up(((size_t)T + 1) * 8), bview = up((size_t)M * 4), bx = up((size_t)M * 16);
    if (int r = c->trkin.reserve(bK + bRt + bV + bF + 2 * bO + bview + bx)) return r;
    if (int r = c->trkpairs.reserve((size_t)(items > 0 ? items : 1) * sizeof(TrackPair))) return r;
    const size_t oX = up((size_t)T * 24), oS = up((size_t)T * 4), oA = up((size_t)T * 8), oM = up((size_t)M),
                 oE = up((size_t)M * 8), oR = refine_iterations > 0 ? up((size_t)T * sizeof(TrackRefineReport)) : 0;
    if (int r = c->trkout.reserve(oX + 2 * oS + oA + oM + oE + oR)) return r;
    char* in = c->trkin.as<char>();
    char* out = c->trkout.as<char>();
    TrackArgs a;
    memset(&a, 0, sizeof a);
    a.K = reinterpret_cast<const double*>(in);
    a.Rt = reinterpret_cast<const double*>(in + bK);
    a.V = V;
    a.views = reinterpret_cast<TrackView*>(in + bK + bRt);
    a.frame = reinterpret_cast<int*>(in + bK + bRt + bV);
    a.offsets = reinterpret_cast<const long long*>(in + bK + bRt + bV + bF);
    a.pbase = reinterpret_cast<const long long*>(in + bK + bRt + bV + bF + bO);
    a.view = reinterpret_cast<const int*>(in + bK + bRt + bV + bF + 2 * bO);
    a.x = reinterpret_cast<const double2*>(in + bK + bRt + bV + bF + 2 * bO + bview);
    a.T = T;
    a.items = items;
    a.pairs = c->trkpairs.as<TrackPair>();
    a.thr = threshold;
    a.min_angle = min_angle_deg * (M_PI / 180.0);
    a.min_views = min_views;
    a.max_iter = refine_iterations;
    a.X = reinterpret_cast<double*>(out);
    a.status = reinterpret_cast<int*>(out + oX);
    a.num_inliers = reinterpret_cast<int*>(out + oX + oS);
    a.angle = reinterpret_cast<double*>(out + oX + 2 * oS);
    a.mask = reinterpret_cast<unsigned char*>(out + oX + 2 * oS + oA);
    a.err = reinterpret_cast<double*>(out + oX + 2 * oS + oA + oM);
    a.report = refine_iterations > 0 ? reinterpret_cast<TrackRefineReport*>(out + oX + 2 * oS + oA + oM + oE) : nullptr;
    // the copies read caller memory synchronously (pageable) or before the synchronisation below
    CU(cudaMemcpyAsync((void*)a.K, K, (size_t)V * 72, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.Rt, Rt, (size_t)V * 96, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.offsets, offsets, ((size_t)T + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.pbase, pbase.data(), ((size_t)T + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    if (M > 0) {
        CU(cudaMemcpyAsync((void*)a.view, view, (size_t)M * 4, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync((void*)a.x, x, (size_t)M * 16, cudaMemcpyHostToDevice, c->stream));
    }
    k_track_views<<<1, 256, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_track_views")) return r;
    if (items > 0) {
        k_track_pairs<<<(unsigned)((items + kTrackBlock - 1) / kTrackBlock), kTrackBlock, 0, c->stream>>>(a);
        if (int r = check_launch(c, "k_track_pairs")) return r;
    }
    k_track_solve<<<(unsigned)((T + kTrackBlock - 1) / kTrackBlock), kTrackBlock, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_track_solve")) return r;
    if (X) CU(cudaMemcpyAsync(X, a.X, (size_t)T * 24, cudaMemcpyDeviceToHost, c->stream));
    if (status) CU(cudaMemcpyAsync(status, a.status, (size_t)T * 4, cudaMemcpyDeviceToHost, c->stream));
    if (num_inliers) CU(cudaMemcpyAsync(num_inliers, a.num_inliers, (size_t)T * 4, cudaMemcpyDeviceToHost, c->stream));
    if (angle) CU(cudaMemcpyAsync(angle, a.angle, (size_t)T * 8, cudaMemcpyDeviceToHost, c->stream));
    if (mask && M > 0) CU(cudaMemcpyAsync(mask, a.mask, (size_t)M, cudaMemcpyDeviceToHost, c->stream));
    if (err && M > 0) CU(cudaMemcpyAsync(err, a.err, (size_t)M * 8, cudaMemcpyDeviceToHost, c->stream));
    if (refine_report && a.report)
        CU(cudaMemcpyAsync(refine_report, a.report, (size_t)T * sizeof(TrackRefineReport), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}
