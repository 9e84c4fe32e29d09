// The C ABI's model selection: the essential matrix or a homography for one pair or every pair of a batch.
#include <cmath>

#include "sfm_host.h"
#include "sfm_select.cuh"

using namespace sfm;
using namespace sfm_host;

static_assert(sizeof(ModelScores) == sizeof(sfm_model_scores), "ModelScores / sfm_model_scores layout mismatch");

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
