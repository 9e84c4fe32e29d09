// The C ABI's two-view stages after the selection: decomposition, pose recovery and triangulation of caller-given
// data, the pose tail of a winner (inlier list, cheirality vote, triangulation) with its optional refinement, the
// homography pose, and the single-pair and batched two-view entry points.
#include <cmath>

#include "sfm_host.h"
#include "sfm_pose.cuh"
#include "sfm_hpose.cuh"
#include "sfm_tail.cuh"
#include "sfm_refine.cuh"

using namespace sfm;
using namespace sfm_host;

static_assert(sizeof(PoseSet) == sizeof(sfm_poses), "PoseSet/sfm_poses layout mismatch");
static_assert(sizeof(RefineReport) == sizeof(sfm_refinement), "RefineReport / sfm_refinement layout mismatch");
static_assert(sizeof(PnpRefineReport) == sizeof(sfm_pnp_refinement), "PnpRefineReport / sfm_pnp_refinement layout mismatch");

int sfm_get_refinement(sfm_ctx* c, sfm_refinement* out, int64_t P) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "null argument");
    if (c->refined_pairs == 0) return fail(SFM_ERR_STATE, "the last tail call did not refine (sfm_set_refinement)");
    if (P != c->refined_pairs) return fail(SFM_ERR_ARG, "the last call refined %lld pairs, not %lld", c->refined_pairs, (long long)P);
    CU(cudaMemcpyAsync(out, c->refrep.p, (size_t)P * sizeof(RefineReport), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- pose + triangulation ---------------------------------------------------------------
// Caller-supplied E (sfm_set_winner too), P1 and P2 may have any scale, but the decomposition and the DLT square their entries (twice, in
// the cross products of svd3_rank2_frames) and leave the double range from about 2^+-250 on.  Their answers do not
// depend on the scale: the frames of E and 2^k E are the same, as is the null vector of 2^k A.  So the stand-alone
// calls bring an input whose largest finite magnitude lies outside [2^-100, 2^100] to [0.5, 1) by a power of two - exact,
// and no bit changes inside that range - and undo it on the singular values.  Returns the exponent applied (0 = none).
int sfm_host::prescale_exponent(const double* a, int n) {
    double big = 0.0;
    for (int i = 0; i < n; ++i)
        if (std::isfinite(a[i])) big = std::fmax(big, std::fabs(a[i]));
    if (big == 0.0 || (big >= 0x1p-100 && big <= 0x1p100)) return 0;
    int e = 0;
    std::frexp(big, &e);  // big = f 2^e, f in [0.5, 1)
    return -e;
}

void sfm_host::prescaled(const double* a, int n, int k, double* out) {
    for (int i = 0; i < n; ++i) out[i] = std::ldexp(a[i], k);
}

int sfm_decompose_essential(sfm_ctx* c, const double* E, sfm_poses* out) {
    if (int r = use(c)) return r;
    if (!E || !out) return fail(SFM_ERR_ARG, "null argument");
    if (int r = c->tmp.reserve(72)) return r;
    if (int r = c->poses.reserve(sizeof(PoseSet))) return r;
    const int k = prescale_exponent(E, 9);
    prescaled(E, 9, k, c->Estage);  // staged in the context: the async copy must not read caller memory later
    CU(cudaMemcpyAsync(c->tmp.p, c->Estage, 72, cudaMemcpyHostToDevice, c->stream));
    k_decompose<<<1, 32, 0, c->stream>>>(c->tmp.as<double>(), nullptr, 0, c->poses.as<PoseSet>(), 1);
    if (int r = check_launch(c, "k_decompose")) return r;
    CU(cudaMemcpyAsync(out, c->poses.p, sizeof(PoseSet), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 3; ++i) out->sv[i] = std::ldexp(out->sv[i], -k);
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
    const int k = prescale_exponent(E, 9);
    prescaled(E, 9, k, c->Estage);
    CU(cudaMemcpyAsync(dE, c->Estage, 72, cudaMemcpyHostToDevice, c->stream));
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
        if (int r = normalise_launch(c, s, stride, m, dK, dpts)) return r;
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
    for (int i = 0; i < 3; ++i) out->sv[i] = std::ldexp(out->sv[i], -k);
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
    // one power of two for both cameras: the DLT system scales as a whole and its null vector does not change
    double* Ps = c->Pstage;
    memcpy(Ps, P1, 96);
    memcpy(Ps + 12, P2, 96);
    prescaled(Ps, 24, prescale_exponent(Ps, 24), Ps);
    CU(cudaMemcpyAsync(dP, Ps, 192, cudaMemcpyHostToDevice, c->stream));
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

// Least-squares refinement of a pose over its inlier list (sfm_refine.cuh, MODEL_P): list, init, max_iterations + 1
// LM steps, finish and, when wanted, the mask under the reported pose - enqueued back to back, one synchronisation.
int sfm_refine_pnp(sfm_ctx* c, const double* Rt, const int32_t* sample, double thr, int max_iterations,
                   sfm_pnp_refinement* out, uint8_t* mask, double* err) {
    if (int r = use(c)) return r;
    if (!out) return fail(SFM_ERR_ARG, "out is null");
    if (!c->has_pnp) return fail(SFM_ERR_STATE, "no PnP records loaded");
    if (max_iterations < 1) return fail(SFM_ERR_ARG, "max_iterations must be >= 1, got %d", max_iterations);
    if (!std::isfinite(thr)) return fail(SFM_ERR_ARG, "the threshold must be finite");
    if (sample)
        for (int k = 0; k < 4; ++k)
            if (sample[k] < 0 || sample[k] >= c->n) return fail(SFM_ERR_ARG, "sample index %d outside [0, %lld)", sample[k], c->n);
    if (!Rt && (!c->pnp_models || !c->has_score || !c->winner_set || c->winner_local < 0))
        return fail(SFM_ERR_STATE, "no pose winner: pass Rt or run sfm_ransac_pnp first");
    const long long n = c->n;
    const int nv = refine_nv<MODEL_P>();
    const long long nblk = (n + kListPerBlock - 1) / kListPerBlock;
    if (int r = c->prstate.reserve(sizeof(RefineState))) return r;
    if (int r = c->prpart.reserve((size_t)(n / kRefineChunk + 2) * nv * 8)) return r;
    if (int r = c->pridx.reserve((size_t)n * 8 + 8)) return r;
    // tickets of the step (1) and of the list (2), then the list's look-back words: zero between calls
    if (int r = reserve_zeroed(c, c->przero, 16 + (size_t)nblk * 8)) return r;
    if (int r = c->prio.reserve(96 + 96 + 16 + sizeof(PnpRefineReport))) return r;
    double* d_start = c->prio.as<double>();
    double* d_pose = d_start + 12;
    int32_t* d_forced = reinterpret_cast<int32_t*>(d_pose + 12);
    PnpRefineReport* d_rep = reinterpret_cast<PnpRefineReport*>(d_pose + 14);
    PnpRefineArgs a;
    memset(&a, 0, sizeof a);
    if (Rt) {
        memcpy(c->prstage, Rt, 96);  // staged in the context: the async copy must not read caller memory later
        CU(cudaMemcpyAsync(d_start, c->prstage, 96, cudaMemcpyHostToDevice, c->stream));
        a.start = d_start;
        if (sample) {
            memcpy(c->prforced, sample, 16);
            CU(cudaMemcpyAsync(d_forced, c->prforced, 16, cudaMemcpyHostToDevice, c->stream));
            a.forced = d_forced;
        }
    } else {  // the winner of the last sfm_ransac_pnp and its sample row (K3's record)
        a.start = c->pmodels.as<double>() + 12 * c->winner_local;
        a.forced = c->record.as<SelectRecord>()->sample;
    }
    a.list_out = c->pridx.as<long long>();
    a.idx = a.list_out;
    a.num = a.list_out + n;
    a.state = c->prstate.as<RefineState>();
    a.partial = c->prpart.as<double>();
    a.ticket = c->przero.as<unsigned>();
    a.list_ticket = a.ticket + 2;
    a.list_agg = c->przero.as<unsigned long long>() + 2;
    a.npairs = 1;
    a.max_iter = max_iterations;
    a.ppts = c->ppts.as<PnpRec>();
    a.n = n;
    a.K = c->pK.as<double>();
    a.thr = thr;
    a.pose_out = d_pose;
    a.preport = d_rep;
    const long long maxch = (n + kRefineChunk - 1) / kRefineChunk;  // the list is at most n long
    const dim3 gs((unsigned)(maxch < 4ll * c->sm_count ? maxch : 4ll * c->sm_count));
    CU(chain_launch(c, k_refine_list<MODEL_P>, dim3((unsigned)nblk), dim3(kListBlock), 0, a));
    if (int r = check_launch(c, "k_refine_list")) return r;
    CU(chain_launch(c, k_refine_init<MODEL_P>, dim3(1), dim3(128), 0, a));
    if (int r = check_launch(c, "k_refine_init")) return r;
    for (int it = 0; it <= max_iterations; ++it) {
        CU(chain_launch(c, k_refine_step<MODEL_P>, gs, dim3(kRefineBlock), 0, a));
        if (int r = check_launch(c, "k_refine_step")) return r;
    }
    CU(chain_launch(c, k_refine_finish<MODEL_P>, dim3(1), dim3(128), 0, a));
    if (int r = check_launch(c, "k_refine_finish")) return r;
    if (mask || err) {
        if (int r = pmask_launch(c, thr, d_pose, nullptr, nullptr)) return r;
        if (mask) CU(cudaMemcpyAsync(mask, c->mask.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
        if (err) CU(cudaMemcpyAsync(err, c->sed.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    CU(cudaMemcpyAsync(out, d_rep, sizeof(PnpRefineReport), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// The tail of apps/sfm.py:133-186 for the winner described by rec_dev (one SelectRecord per pair on the device):
// T1 inlier mask + ordered compaction + decomposition, T2 4-pose cheirality + vote, T3 triangulation of the passing
// inliers - three launches, nothing synchronised (see sfm_tail.cuh).  max_len = the longest pair.
// kind = MODEL_H: the winners are homographies; a single pair's K is the one hpose_stage_k put in c->hK, a batch's are
// the caller's cameras in c->Ks (its records hold pixels).
int sfm_host::pose_tail_launch(sfm_ctx* c, double thr, double dist_thr, const SelectRecord* rec_dev, long long max_len,
                            uint8_t* mask_host, double* sed_host, int kind, double rot_tol) {
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
int sfm_host::copy_inliers(sfm_ctx* c, long long take, int64_t* inlier_idx, uint8_t* pass, double* X) {
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
int sfm_host::check_camera(const double* K) {
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
int sfm_host::hpose_stage_k(sfm_ctx* c, const double* K) {
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
