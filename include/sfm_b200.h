/* sfm_b200 — C ABI of the B200-native two-view geometry hot path.
 *
 * Drop-in acceleration boundary for Bazs/structure_from_motion's
 *   RANSAC essential-matrix estimation -> cheirality vote -> linear triangulation.
 * The reference is pure Python and has no FFI of its own; the boundary it exposes is the
 * set of Python callables in lib/ransac/ransac.py and lib/epipolar/*.py.  Each entry point
 * below names the reference callable (file:line) whose work it replaces; the Python
 * mirror in structure_from_motion_b200/ (re-exported under the reference's import paths
 * in lib/) binds these with ctypes — see INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; all pointers are HOST memory unless the parameter name ends in _d
 *   - every function returns 0 on success, a negative sfm_status otherwise;
 *     sfm_last_error() gives the message for the calling thread
 *   - a context owns one CUDA device, one stream and grow-only device buffers; calls on
 *     one context are serialised by the caller (the reference is single-threaded)
 *   - "correspondence" = one matched feature pair (xa, ya) <-> (xb, yb) in pixel
 *     coordinates; "hypothesis" = one RANSAC iteration (one minimal sample of 8
 *     correspondences and the essential matrix fitted to it)
 */
#ifndef SFM_B200_H
#define SFM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sfm_ctx sfm_ctx;

enum sfm_status {
    SFM_OK = 0,
    SFM_ERR_ARG = -1,      /* bad argument                                  */
    SFM_ERR_CUDA = -2,     /* CUDA runtime error (see sfm_last_error)        */
    SFM_ERR_STATE = -3,    /* call order violated (e.g. score before fit)   */
    SFM_ERR_NO_DEVICE = -4 /* no usable CUDA device                         */
};

/* lib/ransac/ransac.py:12-16  ErrorAggregationMethod */
enum sfm_aggregation { SFM_AGG_SUM = 0, SFM_AGG_SQUARE = 1, SFM_AGG_MEAN = 2, SFM_AGG_RMS = 3 };
/* lib/ransac/ransac.py:83 selects by minimum aggregated error (default).  Extras behind non-default values
 * (SURVEY.md 8(f) N4): max-inliers; MSAC = minimum of sum_i min(sed_i, threshold) over all correspondences
 * (best.err / err[] then hold that cost). */
enum sfm_selection { SFM_SELECT_MIN_ERROR = 0, SFM_SELECT_MAX_INLIERS = 1, SFM_SELECT_MSAC = 2 };
/* scoring kernel variant — all of them give bit-identical results (every inlier decision and
 * every summed value comes from the exact fp64 scorer):
 *   AUTO      (default) a pilot on the device measures the survivor rate of the one-sided screen and the
 *             scoring kernel takes SCREEN below 9 % survivors, FULL above
 *   SCREEN    fp64 one-sided screen (11 FP64 slots per evaluation) + exact re-check of survivors
 *   FULL      fp64 two-sided division-free decision (21 slots) + exact re-check
 *   SCREEN32  the screen evaluated in fp32 as a pre-filter (rigorous guard band, ~2 % more
 *             survivors) + exact fp64 re-check; reported separately from the fp64 headline */
enum sfm_score_variant { SFM_SCORE_SCREEN = 0, SFM_SCORE_FULL = 1, SFM_SCORE_SCREEN32 = 2, SFM_SCORE_AUTO = 3 };

/* ---- context ------------------------------------------------------------------------ */
int sfm_version(void);
const char *sfm_last_error(void);
int sfm_device_count(void);
int sfm_create(int device, sfm_ctx **out);
int sfm_destroy(sfm_ctx *ctx);
/* Use an externally owned cudaStream_t (e.g. torch's current stream); NULL restores the
 * context's own (non-blocking) stream. */
int sfm_set_stream(sfm_ctx *ctx, void *cuda_stream);
/* Use the legacy default stream (cudaStreamLegacy) - what a framework's "default stream" handle 0 means; needed
 * when the context's work has to be ordered with that stream's work (NCCL collectives, timing events). */
int sfm_use_default_stream(sfm_ctx *ctx);
int sfm_synchronize(sfm_ctx *ctx);
/* hyps_per_thread: essential matrices per thread; group: correspondences per vote.  The shapes
 * (hyps_per_thread x group) with a kernel are 2 x 16 for the fp64 variants, and 4 x 8 (the default)
 * and 2 x 16 for SCREEN32; any other shape fails with SFM_ERR_ARG.  hyps_per_thread 0 keeps the
 * current shape, or selects the variant's default when switching to/from SCREEN32. */
int sfm_set_score_variant(sfm_ctx *ctx, int variant, int hyps_per_thread, int group);
/* Pinned host memory for the caller's buffers (so that H2D/D2H copies are true async DMA). */
int sfm_host_alloc(uint64_t bytes, void **out);
int sfm_host_free(void *p);

/* ---- sampling ----------------------------------------------------------------------- */
/* lib/ransac/ransac.py:62-63 — `random.shuffle(data); data[:8]`, cumulative over iterations,
 * restated for CPython's MT19937 + Fisher-Yates (random.py shuffle/_randbelow_with_getrandbits).
 * state: the 625 words of random.getstate()[1] (624 MT words + position), updated in place so
 * the caller can random.setstate() it back.  table: int32[h][8].  If perm_at >= 0,
 * perm_out[n] receives the full permutation after iteration perm_at (the reference returns
 * the inliers in that order, ransac.py:70-76).  Host-only; needs no context. */
int sfm_mt_shuffle_table(uint32_t *state625, int64_t n, int64_t h, int32_t *table, int64_t perm_at,
                         int32_t *perm_out);
/* The same iterations continued from a caller-held permutation (perm_inout[n], updated in place; table may be NULL):
 * lets the caller keep (state, permutation) snapshots every few iterations and replay only a short stretch to
 * recover the permutation of the winning iteration. */
int sfm_mt_shuffle_resume(uint32_t *state625, int64_t n, int64_t h, int32_t *table, int32_t *perm_inout);
/* sfm_mt_shuffle_table from the identity permutation that also records, before every iteration k * stride, the
 * generator state (snap_states[k][625]) and the permutation (snap_perms[k][n]) - so that the permutation or the state
 * after ANY iteration is recovered by replaying at most `stride` iterations (sfm_mt_shuffle_resume) instead of the
 * whole run: the reference returns the inliers in that iteration's permutation order (ransac.py:70-76) and, when a
 * degenerate sample aborts the run, leaves the generator where that iteration left it. */
int sfm_mt_shuffle_snapshots(uint32_t *state625, int64_t n, int64_t h, int32_t *table, int64_t stride,
                             uint32_t *snap_states, int32_t *snap_perms);
/* Upload a sample table (h x 8 indices into the correspondences). */
int sfm_set_table(sfm_ctx *ctx, const int32_t *table, int64_t h);
/* Device sampler (Philox4x32-10 keyed by seed/stream/global hypothesis index): 8 distinct
 * uniform indices per hypothesis; hyp_offset shifts the global index for hypothesis-sharded
 * runs so that the union over ranks equals the single-GPU table. */
int sfm_sample_device(sfm_ctx *ctx, uint64_t seed, uint64_t stream, int64_t hyp_offset, int64_t h);
/* Read back rows [first, first + h) of the current table. */
int sfm_get_table(sfm_ctx *ctx, int32_t *table, int64_t first, int64_t h);

/* ---- correspondences ---------------------------------------------------------------- */
/* lib/epipolar/eight_point.py:127-133 (to_normalized_image_coords), applied once on the
 * device.  xa/ya/xb/yb: pixel coordinates, element i at ptr[i*stride] (stride 1 = four
 * separate arrays; stride 2 = two interleaved [n][2] arrays with ya = xa + 1).
 * K: row-major 3x3; only fx, fy, cx, cy are used, as in the reference. */
int sfm_upload_pairs(sfm_ctx *ctx, const double *xa, const double *ya, const double *xb,
                     const double *yb, int64_t stride, int64_t n, const double *K);
/* The same without the trailing synchronisation: the copies out of the caller's arrays are only ENQUEUED, so the
 * arrays must stay valid and unchanged until the next synchronising call on this context (sfm_two_view_fetch,
 * sfm_synchronize, ...).  Lets the upload of one estimate overlap the kernels of another context. */
int sfm_upload_pairs_async(sfm_ctx *ctx, const double *xa, const double *ya, const double *xb,
                           const double *yb, int64_t stride, int64_t n, const double *K);
/* Same, inputs already in device memory. */
int sfm_upload_pairs_d(sfm_ctx *ctx, const double *xa_d, const double *ya_d, const double *xb_d,
                       const double *yb_d, int64_t stride, int64_t n, const double *K);
/* Read back the K-normalised records: out[n][4] = (xa, ya, xb, yb). */
int sfm_get_normalised(sfm_ctx *ctx, double *out, int64_t n);

/* ---- model fitting ------------------------------------------------------------------- */
/* lib/epipolar/epipolar_ransac.py:28-42 (eight_point_model_fitter) ->
 * lib/epipolar/eight_point.py:99-170 for every row of the current sample table.
 * E_out: double[h][9] or NULL; valid_out: uint8[h] or NULL (0 = the reference would raise
 * EightPointCalculationError, eight_point.py:414-421); eig_out: double[h][9] or NULL
 * (eigenvalues of Y^T Y, diagnostics). */
int sfm_fit(sfm_ctx *ctx, double *E_out, uint8_t *valid_out, double *eig_out);
/* The fitted (or uploaded) models [first, first+count) back to the host: E_out double[count][9], valid_out uint8[count]
 * (either may be NULL). */
int sfm_get_models(sfm_ctx *ctx, int64_t first, int64_t count, double *E_out, uint8_t *valid_out);
/* Replace the fitted models by caller-supplied ones (scorer-only parity tests). */
int sfm_set_models(sfm_ctx *ctx, const double *E, const uint8_t *valid /* or NULL */, int64_t h);

/* ---- scoring + selection ------------------------------------------------------------- */
/* lib/ransac/ransac.py:66-86 + :96-108 with lib/epipolar/epipolar_ransac.py:18-25 /
 * lib/epipolar/sed.py:7-30 as the scorer.  use_table != 0 applies the sample rule of
 * ransac.py:63-64,76 with the current table.  Outputs (each may be NULL):
 * count_extra int32[h] (-1 for invalid hypotheses), S1/S2 double[h] (sum of sed / sed^2 over
 * samples + extra inliers), err double[h] (+inf when not a candidate). */
int sfm_score(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection,
              int use_table, int64_t idx_offset, int32_t *count_extra, double *S1, double *S2,
              double *err);

typedef struct sfm_best {
    double err;            /* aggregated error of the winner                          */
    int64_t index;         /* global hypothesis index, -1 if no candidate              */
    int32_t count_extra;   /* inliers beyond the 8 samples                             */
    int32_t reserved;
    int64_t num_invalid;   /* hypotheses the reference would have raised on           */
    int64_t first_invalid; /* lowest such index, -1 if none                            */
    double E[9];           /* the winning model (row-major), E[8] == 1                 */
    int32_t sample[8];     /* the winner's minimal sample (ransac.py:63), -1 without a table or a winner */
} sfm_best;
/* Winner of the last sfm_score (ransac.py:83: minimum error, earliest iteration on ties). */
int sfm_get_best(sfm_ctx *ctx, sfm_best *out);
/* Tell the context which hypothesis won (hypothesis-sharded runs: after the cross-rank
 * merge).  local_index < 0 = the winner lives on another rank; E then supplies the model, at any scale: an E whose
 * largest finite entry lies outside [2^-100, 2^100] is brought to [0.5, 1) by a power of two, so the tail and the
 * refinement of 2^k E equal those of E bit for bit.  Such an E is stored scaled: a refinement report that falls back
 * to the unrefined model (nonfinite) returns it as 2^j E, the same model. */
int sfm_set_winner(sfm_ctx *ctx, int64_t local_index, const double *E);
/* SURVEY.md H1 (ransac.py:83,96-108: strict < on errors summed in LIST order): the local indices of the hypotheses
 * of the last score whose error is <= best * (1 + rel_tol), unordered, at most cap of them; *count is their total
 * number.  The Python mirror re-evaluates such near-ties in the reference's own summation order. */
int sfm_near_ties(sfm_ctx *ctx, double rel_tol, int64_t cap, int64_t *idx_out, int64_t *count);
/* How many hypotheses of the last score went through K3's exact double-double rescore (their inliers were more than
 * 2^31 times tighter than the threshold, so the 84-bit fixed-point sums of K2 would have lost precision). */
int sfm_get_rescored(sfm_ctx *ctx, int64_t *count);
/* Inlier mask (sed <= threshold) and SED value of every correspondence under the current
 * winner.  mask uint8[n], sed double[n]; either may be NULL. */
int sfm_inlier_mask(sfm_ctx *ctx, double threshold, uint8_t *mask, double *sed);

/* One call for the whole estimate (lib/epipolar/epipolar_ransac.py:45-70): fit -> score ->
 * select -> mask of the winner, no host round trip in between. */
int sfm_ransac_essential(sfm_ctx *ctx, double threshold, double min_extra, int aggregation,
                         int selection, sfm_best *best, uint8_t *mask, double *sed);

/* ---- homography (planar scenes, rotation-only pairs) ----------------------------------
 * H (row-major, H[8] == 1) maps image-A pixels to image-B pixels.  Upload the correspondences with K = I (pixel
 * coordinates), then a sample table or the device sampler: each row's columns 0-3 are the minimal sample.  The error
 * is the symmetric transfer error in px^2 (|x_b - pi(H x_a)|^2 + |x_a - pi(adj(H) x_b)|^2); a correspondence is an
 * inlier iff the division-free test F Q + G P <= thr P Q holds with p2 != 0 and q2 != 0 (csrc/sfm_homography.cuh
 * pins the evaluation order).  A sample with three collinear points in either image, or an H[2,2] that is 0 or not
 * finite, is invalid: it is never a candidate and is counted in sfm_best.num_invalid / first_invalid. */
/* The exact 4-point solve for every row of the current table or device draw.  H_out: double[h][9] (zeros for an
 * invalid sample) or NULL; valid_out: uint8[h] or NULL. */
int sfm_fit_homography(sfm_ctx *ctx, double *H_out, uint8_t *valid_out);
/* RANSAC homography in one call: fit -> score -> select (fit_with_ransac with 4-point samples: samples never counted,
 * always in the error; the aggregation and selection rules of sfm_score) -> mask of the winner.  Needs n >= 8
 * correspondences (the sampler draws 8 distinct indices per row).  best->E carries H, best->sample[4..7] = -1.
 * Optional (NULL = not wanted): mask uint8[n] / err double[n] = decision / transfer error under the winner;
 * count_extra_h int32[h] (-1 = invalid), err_h double[h] (+inf = not a candidate).  sfm_near_ties works afterwards. */
int sfm_ransac_homography(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection,
                          sfm_best *best, uint8_t *mask, double *err, int32_t *count_extra_h, double *err_h);
/* Decision and transfer error of every correspondence under H (double[9], row-major), or under the winner of the
 * last sfm_ransac_homography when H is NULL.  mask uint8[n], err double[n]; either may be NULL. */
int sfm_homography_mask(sfm_ctx *ctx, const double *H, double threshold, uint8_t *mask, double *err);

/* ---- absolute pose of a new view (PnP) ---------------------------------------------------
 * Records: n world points X (double[n][3]) and their observed pixels x (double[n][2]) in the new image, with its K
 * (double[9], row-major): finite, non-singular, upper triangular with K[2,2] = 1, else SFM_ERR_ARG.  The model is
 * [R | t] (double[12], row-major 3 x 4, x_cam = R X + t); P = K [R | t] and p = P (X, 1) are formed in the pinned order
 * of csrc/sfm_pnp.cuh.  A record is an inlier iff p2 >= 2^-537 && F < inf && F <= thr p2^2 with
 * F = (p0 - u p2)^2 + (p1 - v p2)^2; its value is the squared reprojection error F / p2^2 in px^2 (always finite for an
 * inlier).  The minimal solver is P3P (Lambda Twist) on columns 0-2
 * of a sample, with column 3 choosing among the solutions (smallest error at point 3).  A sample with a non-finite
 * coordinate, three collinear world points, no solution with three positive depths and an R orthonormal to 1e-6, or a
 * non-finite pose is invalid:
 * never a candidate, counted in sfm_best.num_invalid / first_invalid. */
/* Replace the context's records with PnP records: the essential-matrix and homography calls refuse until the next
 * sfm_upload_pairs.  Then load a sample table or call the device sampler (columns 0-3 are the sample). */
int sfm_upload_pnp(sfm_ctx *ctx, const double *X, const double *x, int64_t n, const double *K);
/* The P3P fit of every row of the current table or device draw.  Rt_out double[h][12] (zeros for an invalid sample)
 * or NULL; valid_out uint8[h] or NULL. */
int sfm_fit_pnp(sfm_ctx *ctx, double *Rt_out, uint8_t *valid_out);
/* RANSAC absolute pose in one call: fit -> score -> select (fit_with_ransac with 4-point samples: samples never counted,
 * always in the error; the aggregation and selection rules of sfm_score) -> mask of the winner.  Needs n >= 8.
 * best->E is unused (zeros); Rt (double[12], may be NULL) receives the winner, zeros without one.  Optional (NULL =
 * not wanted): mask uint8[n] / err double[n] = decision / reprojection error under the winner; count_extra_h
 * int32[h] (-1 = invalid), err_h double[h] (+inf = not a candidate).  sfm_near_ties works afterwards. */
int sfm_ransac_pnp(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection, sfm_best *best,
                   double *Rt, uint8_t *mask, double *err, int32_t *count_extra_h, double *err_h);
/* Decision and reprojection error of every record under Rt (double[12]), or under the winner of the last
 * sfm_ransac_pnp when Rt is NULL.  mask uint8[n], err double[n]; either may be NULL. */
int sfm_pnp_mask(sfm_ctx *ctx, const double *Rt, double threshold, uint8_t *mask, double *err);
/* Poses [first, first + count) of the last PnP fit: Rt_out double[count][12], valid_out uint8[count]; either may be NULL. */
int sfm_get_pnp_models(sfm_ctx *ctx, int64_t first, int64_t count, double *Rt_out, uint8_t *valid_out);

/* ---- pose + triangulation ------------------------------------------------------------ */
typedef struct sfm_poses {
    double R[4][9];      /* (R1,t) (R1,-t) (R2,t) (R2,-t)  — eight_point.py:210-212 order */
    double t[4][3];
    double sv[3];        /* singular values of E, descending                             */
    int64_t counts[4];   /* cheirality votes (index-0 quirk of eight_point.py:228-230)   */
    int32_t best;        /* np.argmax(counts) (eight_point.py:237), -1 before the vote    */
    int32_t reserved;
} sfm_poses;
/* lib/epipolar/eight_point.py:245-280 (_recover_all_r_t) on the device. */
int sfm_decompose_essential(sfm_ctx *ctx, const double *E, sfm_poses *out);
/* lib/epipolar/eight_point.py:181-242 (_recover_r_t): decomposition + 4-pose cheirality vote
 * (eight_point.py:449-488) over m correspondences given in K-NORMALISED coordinates
 * (element i at ptr[i*stride]).  pass4: uint8[m], bit p set = passes pose p. */
int sfm_recover_pose(sfm_ctx *ctx, const double *E, const double *xa, const double *ya,
                     const double *xb, const double *yb, int64_t stride, int64_t m,
                     double distance_threshold, sfm_poses *out, uint8_t *pass4);
/* The same with PIXEL coordinates: to_normalized_image_coords (eight_point.py:127-133) is applied on the device with
 * K (double[9], row-major) first — recover_r_t_from_e (eight_point.py:65-96). */
int sfm_recover_pose_pixels(sfm_ctx *ctx, const double *E, const double *K, const double *xa, const double *ya,
                            const double *xb, const double *yb, int64_t stride, int64_t m,
                            double distance_threshold, sfm_poses *out, uint8_t *pass4);
/* lib/epipolar/triangulation.py:9-62: DLT triangulation of m correspondences (pixel
 * coordinates) with 3x4 row-major camera matrices P1, P2.  X: double[m][3]. */
int sfm_triangulate(sfm_ctx *ctx, const double *P1, const double *P2, const double *xa,
                    const double *ya, const double *xb, const double *yb, int64_t stride, int64_t m,
                    double *X);
/* Fused tail of the pipeline for the current winner (apps/sfm.py:110-186): inliers of the
 * winner -> decomposition -> cheirality vote -> triangulation of the passing inliers with
 * P1 = K[I|0], P2 = K[R|t], all on the device.  inlier_idx int64[cap] receives the indices
 * (ascending) of the winner's inliers, pass uint8[cap] the vote result per inlier, X
 * double[cap][3] the points (NaN rows where pass == 0).  SFM_ERR_STATE when the winner is a homography
 * (sfm_homography_pose_and_triangulate decomposes those). */
int sfm_pose_and_triangulate(sfm_ctx *ctx, double threshold, double distance_threshold,
                             sfm_poses *poses, int64_t cap, int64_t *num_inliers,
                             int64_t *inlier_idx, uint8_t *pass, double *X);
/* sfm_ransac_essential + sfm_pose_and_triangulate in one call (apps/sfm.py:110-186): the winner never leaves the
 * device between selection and the tail, the host synchronises once for the fixed-size results.  mask / sed
 * (optional) are "sed <= threshold" / the distances under the winner, as sfm_ransac_essential returns them. */
int sfm_two_view(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection,
                 double distance_threshold, sfm_best *best, sfm_poses *poses, int64_t cap, int64_t *num_inliers,
                 int64_t *inlier_idx, uint8_t *pass, double *X, uint8_t *mask, double *sed);
/* sfm_two_view in two halves: _async enqueues everything (device sampler or uploaded table -> fit -> score -> select ->
 * tail, plus the copies of mask / sed into the caller's arrays when given) and returns at once; _fetch synchronises
 * and returns the results.  With two contexts on one GPU the host buffers of estimate s+1 upload while estimate s is
 * being scored (structure_from_motion_b200.two_view.TwoViewStream). */
int sfm_two_view_async(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection,
                       double distance_threshold, uint8_t *mask, double *sed);
int sfm_two_view_fetch(sfm_ctx *ctx, sfm_best *best, sfm_poses *poses, int64_t cap, int64_t *num_inliers,
                       int64_t *inlier_idx, uint8_t *pass, double *X);

/* ---- pose + triangulation from a homography (planar scenes, rotation-only pairs) ------------
 * Hn = K^-1 H K (one K for both images), divided by its middle singular value and negated when det(Hn) < 0 (both
 * camera centres on the same side of the plane).  Candidates: the SVD construction of Ma, Soatto, Kosecka & Sastry,
 * "An Invitation to 3-D Vision", Alg. 5.2, in the order (R+, T+, N+), (R+, -T+, -N+), (R-, T-, N-), (R-, -T-, -N-);
 * t = T / |T|, n = N, d = 1 / |T|.  The order of the four depends on eigenvector signs: compare candidate sets.
 * Rotation-only (sv[0] - sv[2] < rotation_tolerance, 1e-2 ~ 0.6 degrees of plane-induced parallax): all four slots hold
 * the rotation nearest to Hn with t = 0, n = NaN, d = inf; no vote, best = -1.
 * Camera: every step reads pixels through the same K^-1 - the decomposition (K^-1 H K), the vote's rays
 * (yn = (y - cy) / fy, xn = (x - cx - s yn) / fx with the skew s = K[0,1]) and the triangulation (P = K[R|t]).  K must
 * therefore be upper triangular with K[2,2] = 1: the three calls below refuse any other K (a scaled one included) with
 * SFM_ERR_ARG, as they refuse a singular or non-finite K.  The E path's (x - cx) / fx normalisation is unchanged. */
typedef struct sfm_hposes {
    double R[4][9];
    double t[4][3];      /* unit; 0 when rotation_only                                    */
    double n[4][3];      /* plane n^T X = d in camera-1 coordinates, units of the baseline */
    double d[4];
    double sv[3];        /* singular values of K^-1 H K scaled so that sv[1] == 1          */
    int64_t counts[4];   /* cheirality votes: every passing inlier counts                  */
    int32_t best;        /* voted candidate (first maximum); -1 no vote (rotation only); -2 no model */
    int32_t rotation_only;
} sfm_hposes;
/* The decomposition of one homography H (double[9], pixel coordinates) with K (double[9]). */
int sfm_decompose_homography(sfm_ctx *ctx, const double *H, const double *K, double rotation_tolerance,
                             sfm_hposes *out);
/* The tail of the current homography winner (sfm_ransac_homography / sfm_set_winner on homography models): the
 * winner's inliers (decision under H plus its 4 sample points) -> decomposition -> cheirality vote (the test of
 * sfm_pose_and_triangulate on K-normalised coordinates, P1 = [I|0], P2 = [R|t]) -> DLT of the inliers passing the
 * voted candidate in pixel coordinates (P1 = K[I|0], P2 = K[R|t]).  inlier_idx, pass, X and cap as in
 * sfm_pose_and_triangulate; a rotation-only pair has no passing inlier and NaN points. */
int sfm_homography_pose_and_triangulate(sfm_ctx *ctx, const double *K, double threshold, double distance_threshold,
                                        double rotation_tolerance, sfm_hposes *poses, int64_t cap,
                                        int64_t *num_inliers, int64_t *inlier_idx, uint8_t *pass, double *X);
/* sfm_ransac_homography + sfm_homography_pose_and_triangulate in one call: the winner never leaves the device between
 * selection and the tail, the host synchronises once for the fixed-size results.  mask / err (optional) are those of
 * sfm_ransac_homography. */
int sfm_two_view_homography(sfm_ctx *ctx, const double *K, double threshold, double min_extra, int aggregation,
                            int selection, double distance_threshold, double rotation_tolerance, sfm_best *best,
                            sfm_hposes *poses, int64_t cap, int64_t *num_inliers, int64_t *inlier_idx, uint8_t *pass,
                            double *X, uint8_t *mask, double *err);

/* ---- essential matrix or homography for one pair ---------------------------------------
 * The score ratio of ORB-SLAM (Mur-Artal, Montiel & Tardos, 2015, section IV) over the pixel correspondences of the
 * current single-pair upload, whatever K that upload used.  E becomes F = Kd^-T E Kd^-1 (b^T E a = 0 as the SED uses
 * it) with Kd = [[fx, 0, cx], [0, fy, cy], [0, 0, 1]] of K: the camera of the E path, whose (x - cx) / fx, (y - cy) / fy
 * normalisation ignores the skew and the bottom row of K, so an E it estimated is scored in the coordinates it was
 * fitted in.  H is scored in pixels and does not use K.
 * One-way errors in px^2 per correspondence and image: for E the squared distance to the epipolar line (F a in image B,
 * F^T b in image A), for H the transfer terms of the homography scorer (|x_b - pi(H x_a)|^2 and |x_a - pi(adj(H) x_b)|^2).
 * rho(d2) = 5.99 - d2/sigma^2 when d2/sigma^2 < T (T_E = 3.84, T_H = 5.99), else 0 (also for NaN / inf errors); each rho is
 * rounded to a multiple of 2^-32 and summed exactly: fixed_* are those sums, score_* = fixed_* * 2^-32.
 * ratio_h = score_h / (score_h + score_e) (0 when both are 0); model = 1 (H) iff ratio_h > homography_ratio, and when only
 * one of E and H is given (the other may be NULL) that one is chosen.  count_* = correspondences whose two errors both
 * pass T (a diagnostic).  per_point (optional) double[n][4] = (d2_A,E, d2_B,E, d2_A,H, d2_B,H), NaN for a model not
 * given.  SFM_ERR_ARG: E and H both NULL, a non-finite E or H, a singular or non-finite K, sigma not finite and > 0, a
 * non-finite homography_ratio.  SFM_ERR_STATE: a batched context or no correspondences. */
typedef struct sfm_model_scores {
    double score_e, score_h, ratio_h;
    uint64_t fixed_e, fixed_h;
    int64_t count_e, count_h;
    int32_t model;       /* 0 = E, 1 = H, -1 = neither given (sfm_batch_score_models only) */
    int32_t reserved;
} sfm_model_scores;
int sfm_score_models(sfm_ctx *ctx, const double *E, const double *H, const double *K, double sigma,
                     double homography_ratio, sfm_model_scores *out, double *per_point);

/* ---- batched image pairs (pair-sharded workloads) ------------------------------------ */
/* P independent pairs; pair p owns correspondences [offsets[p], offsets[p+1]) of the
 * concatenated arrays, its own K (Ks[p][9]) and h hypotheses drawn by the device sampler
 * (stream = pair_id0 + p).  Outputs per pair: E[p][9], best_index[p] (-1 = none),
 * best_err[p], count_extra[p], num_invalid[p].  Degenerate samples are skipped. */
int sfm_batch_ransac(sfm_ctx *ctx, const double *xa, const double *ya, const double *xb,
                     const double *yb, int64_t stride, const int64_t *offsets, int64_t npairs,
                     const double *Ks, int64_t h, uint64_t seed, uint64_t pair_id0, double threshold,
                     double min_extra, int aggregation, int selection, double *E, int64_t *best_index,
                     double *best_err, int32_t *count_extra, int64_t *num_invalid);

/* The same batch carried through the rest of the path (apps/sfm.py:118-186 per pair): for every pair's winner the
 * inlier list (sed <= threshold plus the 8 sample points, ransac.py:70-76, ascending pair-relative indices), the four
 * candidate poses with the cheirality vote (lib/epipolar/eight_point.py:65-96, 181-280, 449-488; poses[p].best = the
 * voted candidate, -2 = the pair has no model) and the triangulated points of the inliers that pass the voted pose
 * (lib/epipolar/triangulation.py:42-62, pixel coordinates with the pair's K; NaN for the others).  Per-inlier results
 * are packed densely: pair p owns [inlier_offsets[p], inlier_offsets[p+1]) of inlier_idx int32[cap], pass uint8[cap]
 * (bit q = passes candidate q) and X double[cap][3]; cap >= offsets[npairs] always suffices. */
int sfm_batch_two_view(sfm_ctx *ctx, const double *xa, const double *ya, const double *xb, const double *yb,
                       int64_t stride, const int64_t *offsets, int64_t npairs, const double *Ks, int64_t h,
                       uint64_t seed, uint64_t pair_id0, double threshold, double min_extra, int aggregation,
                       int selection, double distance_threshold, double *E, int64_t *best_index, double *best_err,
                       int32_t *count_extra, int64_t *num_invalid, sfm_poses *poses, int64_t *inlier_offsets,
                       int64_t cap, int32_t *inlier_idx, uint8_t *pass, double *X);

/* sfm_batch_two_view for homographies: per pair, RANSAC H over the device sampler's rows (columns 0-3; stream =
 * pair_id0 + p) in pixel coordinates, then the homography tail of sfm_two_view_homography with that pair's K (the
 * decomposition of K^-1 H K, the vote, the triangulation).  Every Ks[p] must pass the checks of sfm_two_view_homography
 * (finite, non-singular, upper triangular, K[2,2] = 1), else SFM_ERR_ARG naming the pair; rotation_tolerance must not be
 * NaN.  Per pair, bit for bit what sfm_two_view_homography returns on that pair alone (uploaded with K = I, sampled with
 * stream pair_id0 + p): H[p][9] (zeros without a model), best_index / best_err / count_extra / num_invalid as
 * sfm_batch_two_view, poses[p] (best = -2: no model, -1: rotation-only), and the inlier list (the transfer decision plus
 * the 4 sample points), pass bits and points packed as sfm_batch_two_view packs them.  A pair of fewer than 8
 * correspondences has no model and an empty segment.  One synchronisation for the fixed-size results, one for the
 * packed arrays. */
int sfm_batch_two_view_homography(sfm_ctx *ctx, const double *xa, const double *ya, const double *xb, const double *yb,
                                  int64_t stride, const int64_t *offsets, int64_t npairs, const double *Ks, int64_t h,
                                  uint64_t seed, uint64_t pair_id0, double threshold, double min_extra, int aggregation,
                                  int selection, double distance_threshold, double rotation_tolerance, double *H,
                                  int64_t *best_index, double *best_err, int32_t *count_extra, int64_t *num_invalid,
                                  sfm_hposes *poses, int64_t *inlier_offsets, int64_t cap, int32_t *inlier_idx,
                                  uint8_t *pass, double *X);

/* sfm_score_models for every pair of the current batched upload (sfm_batch_ransac, sfm_batch_two_view or
 * sfm_batch_two_view_homography: all keep the pixel coordinates): E[p][9] / H[p][9], given for pair p when have_e[p] /
 * have_h[p] is non-zero (a NULL flag array = all given, a NULL model array = none given), scored with the pair's own
 * Ks[p] of the upload as K_d.  out[P] is bit for bit what sfm_score_models returns on that pair alone; a pair with
 * neither model reports model = -1 and zero scores.  per_point (optional) double[n_total][4].  SFM_ERR_ARG: E and H both
 * NULL, a given model not finite, an upload K that is singular or not finite, sigma or homography_ratio as for
 * sfm_score_models.  SFM_ERR_STATE: no batched upload.  One synchronisation. */
int sfm_batch_score_models(sfm_ctx *ctx, const double *E, const uint8_t *have_e, const double *H,
                           const uint8_t *have_h, double sigma, double homography_ratio, sfm_model_scores *out,
                           double *per_point);

/* ---- least-squares refinement of the winner (opt-in; csrc/sfm_refine.cuh) ---------------
 * With max_iterations > 0 (0 = off, the default; a context setting like sfm_set_score_variant) the calls that run a
 * pose tail - sfm_two_view, sfm_two_view_async / _fetch, sfm_pose_and_triangulate, sfm_two_view_homography,
 * sfm_homography_pose_and_triangulate, sfm_batch_two_view, sfm_batch_two_view_homography - refine every pair's winner
 * between the selection and the pose:
 *   data   the winner's inlier list as the tail compacts it (E: sed <= threshold plus the 8 samples; H: the transfer
 *          decision plus the 4 samples), fixed during the refinement;
 *   cost   the sum over that list of the error RANSAC scored: E the symmetric epipolar distance in K-normalised
 *          coordinates, H the symmetric transfer error in px^2 (4 residuals per correspondence);
 *   model  E = [t]x R (R <- R exp([w]x), unit t moved in its tangent plane: 5 parameters), started from candidate 0 of
 *          the decomposition of the RANSAC E (its projection onto the essential manifold); H: h0..h7 with H[2,2] = 1;
 *   solver Levenberg-Marquardt with Marquardt's diagonal damping: lambda starts at 1e-3, / 10 on an accepted step
 *          (cost strictly lower), * 10 on a rejected one; converged when an accepted step lowers the cost by a relative
 *          1e-12 or less, when the cost is at most 1e-24 times the sum of the squared coordinates of the list
 *          (rounding noise), or when the scaled step |diag(J^T J)^1/2 d| <= 1e-9 sqrt(cost); stalled
 *          when lambda exceeds 1e16; max_iterations evaluated proposals at most.  The final cost never exceeds the start's.
 * The RANSAC result is untouched (best, mask, sed / err, the E / H arrays of the batch calls).  The tail then runs on
 * the refined model as on a caller-supplied one: inliers = the decision under the refined model with no forced samples
 * (the E vote's index-0 rule applies to list position 0, as after sfm_set_winner(ctx, -1, E)), vote, triangulation.
 * A pair without a winner, or whose start is not finite, keeps the RANSAC model and its tail.  An empty list (a
 * caller's E that explains no correspondence) reports converged at iteration 0 with cost 0, and its model is the start:
 * the caller's E projected onto the essential manifold.  The refined bits depend on
 * the pair's inlier list only (fixed-order sums): pair p of a batch equals the single-pair call on that pair.
 * sfm_two_view_sharded and sfm_sharded_tail refuse with SFM_ERR_STATE while refinement is on. */
enum sfm_refine_status {
    SFM_REFINE_CONVERGED = 0,
    SFM_REFINE_MAX_ITERATIONS = 1,
    SFM_REFINE_STALLED = 2,      /* lambda reached its cap */
    SFM_REFINE_NO_MODEL = 3,     /* no winner: nothing refined */
    SFM_REFINE_NONFINITE = 4     /* the start (model or cost) is not finite: the RANSAC model is kept */
};
typedef struct sfm_refinement {
    double model[9];       /* refined E or H (row-major, model[8] == 1); the RANSAC model when not refined */
    double cost_ransac;    /* cost of the RANSAC model over the inlier list                              */
    double cost_start;     /* cost at the start point (E: the projection onto the manifold)              */
    double cost_final;     /* cost of the refined model, <= cost_start                                   */
    int64_t num;           /* correspondences in the inlier list                                         */
    int32_t iterations;    /* proposals evaluated                                                         */
    int32_t status;        /* sfm_refine_status                                                           */
    int32_t rejected;      /* of those, proposals rejected (cost not strictly lower)                     */
    int32_t reserved;
} sfm_refinement;
int sfm_set_refinement(sfm_ctx *ctx, int max_iterations);
/* The reports of the last tail call, one per pair (P = 1 for the single-pair calls); SFM_ERR_STATE when that call did
 * not refine, SFM_ERR_ARG when P is not its number of pairs. */
int sfm_get_refinement(sfm_ctx *ctx, sfm_refinement *out, int64_t P);

/* ---- hypothesis-sharded estimates without a host round trip (SURVEY.md 8(e)) ---------- */
/* One rank of a run whose hypotheses are split over `world` GPUs (correspondences replicated):
 *   1. sfm_score_async  : fit + score + select of this rank's hypotheses, nothing synchronised; *record_dev is the
 *                         DEVICE address of this rank's SFM_RECORD_BYTES-byte selection record;
 *   2. the caller all-gathers the records of all ranks into one device buffer on the context's stream
 *      (ncclAllGather / torch.distributed.all_gather_into_tensor - the path's only collective, SFM_RECORD_BYTES per rank);
 *      a record = {err f64, index i64, count i32, pad, num_invalid i64, first_invalid i64, E f64[9], sample i32[8]}:
 *      the winner's model AND its minimal sample travel with it, so every rank finishes with identical results;
 *   3. sfm_sharded_tail : merges the records on the device with the reference's rule (ransac.py:83: smallest error,
 *                         earliest GLOBAL iteration = rank * hyps_per_rank + local index on ties) and enqueues the
 *                         inlier mask, pose vote and triangulation of the global winner;
 *   4. sfm_sharded_fetch: the single synchronisation; best->index is the global index, *owner the rank that fitted
 *                         the winner (-1: no model anywhere). */
#define SFM_RECORD_BYTES 144
int sfm_score_async(sfm_ctx *ctx, double threshold, double min_extra, int aggregation, int selection,
                    void **record_dev);
int sfm_sharded_tail(sfm_ctx *ctx, const void *gathered_records_dev, int world, int rank, int64_t hyps_per_rank,
                     int selection, double threshold, double distance_threshold);
int sfm_sharded_fetch(sfm_ctx *ctx, sfm_best *best, int32_t *owner, sfm_poses *poses, int64_t cap,
                      int64_t *num_inliers, int64_t *inlier_idx, uint8_t *pass, double *X);

/* The same without any host framework: the collective behind the C ABI (SURVEY.md 8(b) sfm_nccl_init /
 * sfm_ransac_E_sharded).  libnccl.so.2 is resolved at run time (the copy already loaded in the process, else the
 * system's).  Rank 0 calls sfm_nccl_unique_id and ships the SFM_NCCL_ID_BYTES bytes to its peers by any means; every
 * rank calls sfm_nccl_init (collective).  sfm_two_view_sharded then enqueues one complete estimate - this rank's
 * hypotheses [rank * hyps_per_rank, (rank+1) * hyps_per_rank) of the device sampler, ONE ncclAllGather of the
 * selection records on the context's stream, merge kernel, tail - and sfm_sharded_fetch returns, on every rank, what
 * one GPU returns for the union of the hypotheses (ransac.py:83 applied across ranks). */
#define SFM_NCCL_ID_BYTES 128
int sfm_nccl_unique_id(void *id_out);
int sfm_nccl_init(sfm_ctx *ctx, int rank, int nranks, const void *unique_id);
int sfm_nccl_destroy(sfm_ctx *ctx);
int sfm_two_view_sharded(sfm_ctx *ctx, uint64_t seed, int64_t hyps_per_rank, double threshold, double min_extra,
                         int aggregation, int selection, double distance_threshold);

/* ---- the stage in front of the hot path: brute-force matcher (SURVEY.md 8(f) N1) ------ */
/* lib/feature_matching/matching.py:36-118 match_brute_force with ncc.py:7-54 (score_kind 0, score
 * in [0,2], 2.0 when a window leaves the image) or ssd.py:7-36 (score_kind 1, +inf outside) as the
 * score function.  window <= 15; like util.py:21-27 the patch spans center +- int(window/2), so an even
 * window covers window + 1 pixels.  Images: row-major rows x cols, image_dtype 0 = uint8 (numpy's uint8 arithmetic
 * of ssd.py is reproduced), 1 = float64.  feats_*: double[n][2] = (x, y) (lib/common/feature.py).
 * validation: bit 0 RATIO_TEST (heap[0]/heap[1] <= ratio_threshold, matching.py:84-97 - heap[1] of
 * the reference's heapq, not the second smallest score), bit 1 CROSSCHECK (matching.py:100-118).
 * Outputs per feature of image A: best_b int32[na], best_score double[na], keep uint8[na] (1 = the
 * match survives the validations; the reference returns exactly those, in order); scores (optional)
 * double[na][nb] = the full score matrix. */
int sfm_match_brute_force(sfm_ctx *ctx, const void *image_a, const void *image_b, int image_dtype,
                          int64_t rows, int64_t cols, const double *feats_a, int64_t na,
                          const double *feats_b, int64_t nb, int score_kind, int window, int validation,
                          double ratio_threshold, int32_t *best_b, double *best_score, uint8_t *keep,
                          double *scores);

/* The same selection + validations on a caller-supplied score matrix double[na][nb] (the scores of
 * an arbitrary Python score_function, matching.py:55-65). */
int sfm_match_from_scores(sfm_ctx *ctx, const double *scores, int64_t na, int64_t nb, int validation,
                          double ratio_threshold, int32_t *best_b, double *best_score, uint8_t *keep);

/* ---- the first stage of apps/sfm.py: Harris corners (SURVEY.md 8(f) N2) -------------------- */
/* lib/common/correlate.py:4-39 cross_correlate: zero "same" border, odd square kernel double[ksize][ksize],
 * out double[rows][cols].  image_dtype as above. */
int sfm_cross_correlate(sfm_ctx *ctx, const void *image, int image_dtype, int64_t rows, int64_t cols,
                        const double *kernel, int ksize, double *out);
/* Shape of the cornerness image: rows/cols - int(np.around(block_size / 2)) (harris_detector.py:66-72). */
int sfm_harris_output_shape(int64_t rows, int64_t cols, int block_size, int64_t *out_rows, int64_t *out_cols);
/* lib/harris/harris_detector.py:11-55 detect_harris_corners: Sobel responses, block sums, det - k trace^2,
 * negatives clamped to 0, the reference's in-place (scan-order dependent) 3x3 non-maximum suppression, the
 * num_corners highest non-zero values in descending order (exact ties: descending flat index).
 * xy double[num_corners][2] = (x, y) = (col, row) + block_size/2; score double[num_corners];
 * *num_found <= num_corners; cornerness (optional) double[out_rows][out_cols] after suppression;
 * nms_sweeps (optional) = parallel sweeps the suppression needed. */
int sfm_harris_corners(sfm_ctx *ctx, const void *image, int image_dtype, int64_t rows, int64_t cols,
                       int64_t num_corners, int block_size, double k, double *xy, double *score,
                       int64_t *num_found, double *cornerness, int32_t *nms_sweeps);

/* ---- measurement --------------------------------------------------------------------- */
/* Per-stage device times (CUDA events on the context's stream) of the most recent
 * pipeline call: ms[0]=upload+normalise ms[1]=sample ms[2]=fit ms[3]=score ms[4]=finalise+select
 * ms[5]=mask ms[6]=pose ms[7]=triangulate (a stage is reported once, then reads 0 until it runs
 * again).  launches = kernels launched by this library since the context was created. */
int sfm_enable_timing(sfm_ctx *ctx, int on);
int sfm_get_timing(sfm_ctx *ctx, float ms[8], int64_t *launches);
/* FP64 FMA throughput microbenchmark (denominator of the FP64 roofline): returns achieved
 * DFMA/s over the whole device. */
int sfm_measure_fp64_peak(sfm_ctx *ctx, double *dfma_per_s);

#ifdef __cplusplus
}
#endif
#endif /* SFM_B200_H */
