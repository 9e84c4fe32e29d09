// The C ABI's bundle adjustment (sfm_bundle.cuh): argument checks, the structure of the reduced camera system (the
// view-major observation order, the S blocks and their observation pairs), buffers, the chained rounds and the copies.
#include <cmath>

#include "sfm_bundle.cuh"
#include "sfm_host.h"

using namespace sfm;
using namespace sfm_host;

static_assert(sizeof(BaReport) == sizeof(sfm_bundle_report), "BaReport / sfm_bundle_report layout mismatch");
static_assert(SFM_BA_MAX_VIEWS == kBaMaxViews, "the header's view limit is the kernel's");
static_assert(SFM_TRACK_MAX_OBSERVATIONS == kBaMaxTrack, "the header's track length limit is the kernel's");

namespace {

size_t up16(size_t b) { return (b + 15) & ~(size_t)15; }

// carves 16-byte aligned pieces out of one device buffer
struct Carve {
    char* base;
    size_t off = 0;
    template <class T>
    T* take(size_t count) {
        T* p = reinterpret_cast<T*>(base + off);
        off += up16(count * sizeof(T));
        return p;
    }
};

// the launches of one LM round
int ba_round(sfm_ctx* c, const BaArgs& a, long long nptch, long long nvch_blocks, long long schur_threads, long long nsum) {
    CU(chain_launch(c, k_ba_eval, dim3((unsigned)nptch), dim3(kBaBlock), 0, a));
    CU(chain_launch(c, k_ba_views, dim3((unsigned)nvch_blocks), dim3(kBaBlock), 0, a));
    CU(chain_launch(c, k_ba_views_sum, dim3((unsigned)((27LL * a.F + kBaBlock / 32 - 1) / (kBaBlock / 32) + 1)),
                    dim3(kBaBlock), 0, a));
    CU(chain_launch(c, k_ba_schur_pts, dim3((unsigned)nptch), dim3(kBaBlock), 0, a));
    if (a.M > 0) CU(chain_launch(c, k_ba_schur_obs, dim3((unsigned)((a.M + kBaBlock - 1) / kBaBlock)), dim3(kBaBlock), 0, a));
    if (a.npad > 0) {
        if (schur_threads > 0)
            CU(chain_launch(c, k_ba_schur, dim3((unsigned)((schur_threads + kBaBlock - 1) / kBaBlock)), dim3(kBaBlock), 0, a));
        CU(chain_launch(c, k_ba_schur_sum, dim3((unsigned)((nsum + 255) / 256)), dim3(256), 0, a));
        const int nt = a.npad / kBaTile;
        for (int j = 0; j < nt; ++j) CU(chain_launch(c, k_ba_chol, dim3((unsigned)(nt + 1 - j)), dim3(kBaCholThreads), 0, a, j));
        CU(chain_launch(c, k_ba_backsolve, dim3(1), dim3(kBaTile * kBaSolveSlices), 0, a));
    }
    CU(chain_launch(c, k_ba_points, dim3((unsigned)nptch), dim3(kBaBlock), 0, a));
    return check_launch(c, "bundle round");
}

}  // namespace

int sfm_bundle_adjust(sfm_ctx* c, const double* K, const double* Rt, int32_t V, const uint8_t* fixed, int32_t scale_view,
                      const int64_t* offsets, int64_t T, const int32_t* view, const double* x, const double* X,
                      double threshold, int32_t max_iterations, double* Rt_out, double* X_out,
                      sfm_bundle_report* report, uint8_t* mask, double* err) {
    if (int r = use(c)) return r;
    if (V < 1 || V > SFM_BA_MAX_VIEWS) return fail(SFM_ERR_ARG, "V must be in [1, %d], got %d", SFM_BA_MAX_VIEWS, V);
    if (T < 0) return fail(SFM_ERR_ARG, "negative track count");
    if (!K || !Rt || !fixed || !offsets || (T > 0 && !X)) return fail(SFM_ERR_ARG, "null argument");
    if (!std::isfinite(threshold)) return fail(SFM_ERR_ARG, "the threshold must be finite");
    if (max_iterations < 1) return fail(SFM_ERR_ARG, "max_iterations must be >= 1, got %d", max_iterations);
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
    std::vector<int> fidx(V);
    int F = 0;
    for (int v = 0; v < V; ++v) fidx[v] = fixed[v] ? -1 : F++;
    if (F == V) return fail(SFM_ERR_ARG, "at least one view must be fixed");
    int anchor_comp = 0;
    if (scale_view != -1) {
        if (scale_view < 0 || scale_view >= V) return fail(SFM_ERR_ARG, "scale_view %d outside [-1, %d)", scale_view, V);
        if (fixed[scale_view]) return fail(SFM_ERR_ARG, "scale_view %d is a fixed view", scale_view);
        const double* t = Rt + 12 * (size_t)scale_view;
        for (int k = 1; k < 3; ++k)
            if (std::fabs(t[4 * k + 3]) > std::fabs(t[4 * anchor_comp + 3])) anchor_comp = k;
    }
    if (offsets[0] != 0) return fail(SFM_ERR_ARG, "offsets[0] must be 0, got %lld", (long long)offsets[0]);
    for (int64_t t = 0; t < T; ++t) {
        const int64_t n = offsets[t + 1] - offsets[t];
        if (n < 0) return fail(SFM_ERR_ARG, "offsets decrease at track %lld", (long long)t);
        if (n > kBaMaxTrack)
            return fail(SFM_ERR_ARG, "track %lld has %lld observations, more than %d", (long long)t, (long long)n, kBaMaxTrack);
    }
    const long long M = offsets[T];
    if (M > 0x7fffffffLL || T > 0x7fffffffLL) return fail(SFM_ERR_ARG, "more than 2^31 - 1 observations or tracks");
    if (M > 0 && (!view || !x)) return fail(SFM_ERR_ARG, "null observations");
    for (long long i = 0; i < M; ++i)
        if (view[i] < 0 || view[i] >= V) return fail(SFM_ERR_ARG, "observation %lld: view %d outside [0, %d)", i, view[i], V);

    // structure: the observations of the free views by view (ascending within a view) in chunks, and the observation
    // pairs (i, j) of one track with free(view i) >= free(view j), by S block, then track, i and j, in chunks
    std::vector<int> otrack((size_t)M);
    for (int64_t t = 0; t < T; ++t)
        for (int64_t i = offsets[t]; i < offsets[t + 1]; ++i) otrack[(size_t)i] = (int)t;
    std::vector<long long> vcount(F + 1, 0);
    for (long long i = 0; i < M; ++i)
        if (fidx[view[i]] >= 0) ++vcount[fidx[view[i]] + 1];
    std::vector<long long> vstart(F + 1, 0);
    for (int f = 0; f < F; ++f) vstart[f + 1] = vstart[f] + vcount[f + 1];
    std::vector<int> vperm((size_t)vstart[F]);
    {
        std::vector<long long> fill(vstart.begin(), vstart.end() - 1);
        for (long long i = 0; i < M; ++i)
            if (fidx[view[i]] >= 0) vperm[fill[fidx[view[i]]]++] = (int)i;
    }
    std::vector<long long> vfirst(F + 1, 0), vch_begin;
    for (int f = 0; f < F; ++f) {
        vfirst[f] = (long long)vch_begin.size();
        for (long long b = vstart[f]; b < vstart[f + 1]; b += kBaObsChunk) vch_begin.push_back(b);
    }
    vfirst[F] = (long long)vch_begin.size();
    const long long nvch = (long long)vch_begin.size();
    vch_begin.push_back(vstart[F]);
    std::vector<long long> bcount((size_t)F * F, 0);
    for (int64_t t = 0; t < T; ++t)
        for (int64_t i = offsets[t]; i < offsets[t + 1]; ++i) {
            const int fi = fidx[view[i]];
            if (fi < 0) continue;
            for (int64_t j = offsets[t]; j < offsets[t + 1]; ++j) {
                const int fj = fidx[view[j]];
                if (fj >= 0 && fi >= fj) ++bcount[(size_t)fi * F + fj];
            }
        }
    std::vector<int> blk_id((size_t)F * F, -1);
    std::vector<int2> blk_ac;
    std::vector<long long> bstart(1, 0), bfirst, tch_begin;
    for (size_t key = 0; key < bcount.size(); ++key)
        if (bcount[key] > 0) {
            blk_id[key] = (int)(bstart.size() - 1);
            blk_ac.push_back(make_int2((int)(key / F), (int)(key % F)));
            bstart.push_back(bstart.back() + bcount[key]);
        }
    const long long ntrip = bstart.back();
    std::vector<int2> triples((size_t)ntrip);
    {
        std::vector<long long> fill(bstart.begin(), bstart.end() - 1);
        for (int64_t t = 0; t < T; ++t)
            for (int64_t i = offsets[t]; i < offsets[t + 1]; ++i) {
                const int fi = fidx[view[i]];
                if (fi < 0) continue;
                for (int64_t j = offsets[t]; j < offsets[t + 1]; ++j) {
                    const int fj = fidx[view[j]];
                    if (fj >= 0 && fi >= fj) triples[fill[blk_id[(size_t)fi * F + fj]]++] = make_int2((int)i, (int)j);
                }
            }
    }
    const size_t nblk = bstart.size() - 1;
    for (size_t b = 0; b < nblk; ++b) {
        bfirst.push_back((long long)tch_begin.size());
        for (long long k = bstart[b]; k < bstart[b + 1]; k += kBaTripleChunk) tch_begin.push_back(k);
    }
    bfirst.push_back((long long)tch_begin.size());
    const long long ntch = (long long)tch_begin.size();
    tch_begin.push_back(ntrip);

    const int n6 = 6 * F, npad = (n6 + kBaTile - 1) / kBaTile * kBaTile;
    const long long nptch = T > 0 ? (T + kBaBlock - 1) / kBaBlock : 1;
    const long long nvblocks = nvch > 0 ? nvch : 1;
    const long long Tn = T > 0 ? T : 1, Mn = M > 0 ? M : 1;

    // inputs and structure
    const size_t in_bytes = up16((size_t)V * 72) + up16((size_t)V * 96) + up16((size_t)V * 4) + up16(((size_t)T + 1) * 8) +
                            up16((size_t)Mn * 4) + up16((size_t)Mn * 16) + up16((size_t)Tn * 24) + up16((size_t)Mn * 4) + up16(vperm.size() * 4 + 4) +
                            up16(vch_begin.size() * 8) + up16(vfirst.size() * 8) + up16(triples.size() * 8 + 8) +
                            up16(tch_begin.size() * 8) + up16(bfirst.size() * 8) + up16(blk_id.size() * 4 + 4) + up16(blk_ac.size() * 8 + 8);
    if (int r = c->bain.reserve(in_bytes)) return r;
    Carve ci{c->bain.as<char>()};
    BaArgs a;
    memset(&a, 0, sizeof a);
    a.K = ci.take<double>((size_t)V * 9);
    a.Rt = ci.take<double>((size_t)V * 12);
    a.fidx = ci.take<int>(V);
    a.offsets = ci.take<long long>((size_t)T + 1);
    a.view = ci.take<int>(Mn);
    a.x = ci.take<double2>(Mn);
    a.X0 = ci.take<double>((size_t)Tn * 3);
    a.otrack = ci.take<int>(Mn);
    a.vperm = ci.take<int>(vperm.size() + 1);
    a.vch_begin = ci.take<long long>(vch_begin.size());
    a.vfirst = ci.take<long long>(vfirst.size());
    a.triples = ci.take<int2>(triples.size() + 1);
    a.tch_begin = ci.take<long long>(tch_begin.size());
    a.bfirst = ci.take<long long>(bfirst.size());
    a.blk_id = ci.take<int>(blk_id.size() + 1);
    a.blk_ac = ci.take<int2>(blk_ac.size() + 1);
    a.nblk = (long long)nblk;
    a.V = V;
    a.F = F;
    a.anchor = scale_view;
    a.anchor_comp = anchor_comp;
    a.npad = npad;
    a.max_iter = max_iterations;
    a.T = T;
    a.M = M;
    a.thr = threshold;
    a.nvch = nvch;
    a.ntch = ntch;
    a.nptch = nptch;

    // state, equations, partials, S and outputs
    Carve cw{nullptr};
    auto layout = [&](Carve& w) {
        a.st = w.take<BaState>(1);
        a.inlist = w.take<unsigned char>(Mn);
        a.param = w.take<unsigned char>(Tn);
        a.pose = w.take<double>((size_t)2 * V * 12);
        a.Pprop = w.take<double>((size_t)V * 12);
        a.Xp = w.take<double>((size_t)2 * Tn * 3);
        a.oeq = w.take<BaObsEq>((size_t)2 * Mn);
        a.peq = w.take<BaPtEq>((size_t)2 * Tn);
        a.veq = w.take<BaViewEq>((size_t)2 * (F > 0 ? F : 1));
        a.osch = w.take<BaObsSchur>(Mn);
        a.psol = w.take<BaPtSolve>(Tn);
        a.part_pt = w.take<double>(nptch);
        a.part_v = w.take<double>((size_t)nvblocks * 27);
        a.part_t = w.take<double>((size_t)(ntch > 0 ? ntch : 1) * 36);
        a.part_r = w.take<double>((size_t)nvblocks * 6);
        a.S = w.take<double>((size_t)(npad + kBaTile) * (npad > 0 ? npad : 1));
        a.y = w.take<double>(npad > 0 ? npad : 1);
        a.Ldiag = w.take<double>((size_t)(npad > 0 ? npad : 1) * kBaTile);
        a.Rt_out = w.take<double>((size_t)V * 12);
        a.Prep = w.take<double>((size_t)V * 12);
        a.X_out = w.take<double>((size_t)Tn * 3);
        a.mask = w.take<unsigned char>(Mn);
        a.err = w.take<double>(Mn);
        a.report = w.take<BaReport>(1);
    };
    layout(cw);  // sizes only
    if (int r = c->bawork.reserve(cw.off)) return r;
    Carve cw2{c->bawork.as<char>()};
    layout(cw2);
    if (int r = reserve_zeroed(c, c->batick, 64)) return r;
    a.ticket = c->batick.as<unsigned>();

    // the copies read caller memory synchronously (pageable) or before the synchronisation below
    CU(cudaMemcpyAsync((void*)a.K, K, (size_t)V * 72, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.Rt, Rt, (size_t)V * 96, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.fidx, fidx.data(), (size_t)V * 4, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.offsets, offsets, ((size_t)T + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    if (M > 0) {
        CU(cudaMemcpyAsync((void*)a.view, view, (size_t)M * 4, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync((void*)a.x, x, (size_t)M * 16, cudaMemcpyHostToDevice, c->stream));
    }
    if (T > 0) CU(cudaMemcpyAsync((void*)a.X0, X, (size_t)T * 24, cudaMemcpyHostToDevice, c->stream));
    if (M > 0) CU(cudaMemcpyAsync((void*)a.otrack, otrack.data(), (size_t)M * 4, cudaMemcpyHostToDevice, c->stream));
    if (!vperm.empty())
        CU(cudaMemcpyAsync((void*)a.vperm, vperm.data(), vperm.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.vch_begin, vch_begin.data(), vch_begin.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.vfirst, vfirst.data(), vfirst.size() * 8, cudaMemcpyHostToDevice, c->stream));
    if (!triples.empty())
        CU(cudaMemcpyAsync((void*)a.triples, triples.data(), triples.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.tch_begin, tch_begin.data(), tch_begin.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync((void*)a.bfirst, bfirst.data(), bfirst.size() * 8, cudaMemcpyHostToDevice, c->stream));
    if (!blk_id.empty())
        CU(cudaMemcpyAsync((void*)a.blk_id, blk_id.data(), blk_id.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (!blk_ac.empty())
        CU(cudaMemcpyAsync((void*)a.blk_ac, blk_ac.data(), blk_ac.size() * 8, cudaMemcpyHostToDevice, c->stream));
    // rows npad + 1 .. of the right-hand side tile stay zero
    CU(cudaMemsetAsync(a.S, 0, (size_t)(npad + kBaTile) * (npad > 0 ? npad : 1) * 8, c->stream));

    CU(chain_launch(c, k_ba_init, dim3(1), dim3(256), 0, a));
    CU(chain_launch(c, k_ba_list, dim3((unsigned)nptch), dim3(kBaBlock), 0, a));
    if (int r = check_launch(c, "k_ba_list")) return r;
    const long long schur_threads = ntch + nvch;
    // one thread per entry outside the blocks (rounded up to whole warps), then a warp per block entry and rhs entry
    const long long nsum = ((long long)npad * (npad + 1) / 2 + npad + 31) / 32 * 32 + 32LL * ((long long)nblk * 36 + 6 * F);
    if (int r = ensure_pinned(c, sizeof(BaState))) return r;
    BaState* hs = reinterpret_cast<BaState*>(c->hpin);
    // max_iter + 1 rounds finish every problem whose damped systems are positive definite; each re-solve after one
    // that is not takes one more round, so the host enqueues more until the state says done (one check per batch).
    // Every round evaluates a proposal (at most max_iter + 1 of them) or re-solves after a system that is not positive
    // definite, multiplying a positive lambda by 10.  lambda falls (/ 10) only on the at most max_iter accepts, it is
    // stalled once above kRefineLambdaCap (19 decades above kRefineLambda0) or at 0, and rounding among subnormals
    // loses at most 16 more decades: at most max_iter + 36 re-solves, so at most 20 batches even for max_iter = 1.
    // kBaMaxBatches bounds the loop with a margin, so that a defect cannot keep a GPU busy.
    for (int batch = 0;; ++batch) {
        if (batch == kBaMaxBatches) return fail(SFM_ERR_STATE, "bundle adjustment did not finish in %d rounds",
                                                 kBaMaxBatches * (max_iterations + 1));
        for (int k = 0; k <= max_iterations; ++k)
            if (int r = ba_round(c, a, nptch, nvblocks, schur_threads, nsum)) return r;
        CU(chain_launch(c, k_ba_finish, dim3(1), dim3(256), 0, a));
        CU(chain_launch(c, k_ba_mask, dim3((unsigned)nptch), dim3(kBaBlock), 0, a));
        if (int r = check_launch(c, "k_ba_mask")) return r;
        CU(cudaMemcpyAsync(hs, a.st, sizeof(BaState), cudaMemcpyDeviceToHost, c->stream));
        if (Rt_out) CU(cudaMemcpyAsync(Rt_out, a.Rt_out, (size_t)V * 96, cudaMemcpyDeviceToHost, c->stream));
        if (X_out && T > 0) CU(cudaMemcpyAsync(X_out, a.X_out, (size_t)T * 24, cudaMemcpyDeviceToHost, c->stream));
        if (mask && M > 0) CU(cudaMemcpyAsync(mask, a.mask, (size_t)M, cudaMemcpyDeviceToHost, c->stream));
        if (err && M > 0) CU(cudaMemcpyAsync(err, a.err, (size_t)M * 8, cudaMemcpyDeviceToHost, c->stream));
        if (report) CU(cudaMemcpyAsync(report, a.report, sizeof(BaReport), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (hs->done) break;
    }
    return 0;
}
