// The C ABI's track building from pairwise matches (sfm_track_build.cuh): argument checks, the pair table, the
// union-find launches, the select / sort / scan of the track order and the copies back.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <climits>

#include "sfm_host.h"
#include "sfm_track_build.cuh"

using namespace sfm;
using namespace sfm_host;

static_assert(SFM_TRACK_MAX_OBSERVATIONS == kTbMaxObservations, "the header's track length limit is the kernel's");
static_assert((int)SFM_BUILT_TRACK_OK == TB_OK && (int)SFM_BUILT_TRACK_CONFLICT == TB_CONFLICT &&
                  (int)SFM_BUILT_TRACK_LONG == TB_LONG,
              "sfm_built_track_status is the kernel's");

static unsigned tb_grid(long long n) { return (unsigned)std::max(1LL, std::min((n + kTbBlock - 1) / kTbBlock, 1LL << 20)); }
static size_t up(size_t b) { return (b + 255) & ~(size_t)255; }

int sfm_build_tracks(sfm_ctx* c, int32_t V, const int64_t* feature_offsets, int64_t P, const int32_t* pair_views,
                     const int64_t* match_offsets, const int32_t* matches, int64_t* T_out, int64_t* M_out, int64_t* offsets,
                     int32_t* status, int32_t* view, int32_t* feature, int32_t* track) {
    if (int r = use(c)) return r;
    if (V < 1) return fail(SFM_ERR_ARG, "at least one view is needed, got %d", V);
    if (P < 0) return fail(SFM_ERR_ARG, "negative pair count");
    if (!feature_offsets) return fail(SFM_ERR_ARG, "null feature_offsets");
    if (feature_offsets[0] != 0)
        return fail(SFM_ERR_ARG, "feature_offsets[0] must be 0, got %lld", (long long)feature_offsets[0]);
    for (int v = 0; v < V; ++v)
        if (feature_offsets[v + 1] < feature_offsets[v]) return fail(SFM_ERR_ARG, "feature_offsets decrease at view %d", v);
    const long long N = feature_offsets[V];
    if (N > INT32_MAX) return fail(SFM_ERR_ARG, "%lld features, more than INT32_MAX", N);
    if (P > 0 && (!pair_views || !match_offsets)) return fail(SFM_ERR_ARG, "null pair_views or match_offsets");
    if (match_offsets && match_offsets[0] != 0)
        return fail(SFM_ERR_ARG, "match_offsets[0] must be 0, got %lld", (long long)match_offsets[0]);
    std::vector<TbPair> ptab((size_t)P);
    for (long long p = 0; p < P; ++p) {
        const int a = pair_views[2 * p], b = pair_views[2 * p + 1];
        if (a < 0 || a >= V || b < 0 || b >= V) return fail(SFM_ERR_ARG, "pair %lld: view outside [0, %d)", p, V);
        if (a == b) return fail(SFM_ERR_ARG, "pair %lld: both views are %d", p, a);
        if (match_offsets[p + 1] < match_offsets[p]) return fail(SFM_ERR_ARG, "match_offsets decrease at pair %lld", p);
        ptab[p] = {(int)feature_offsets[a], (int)feature_offsets[b]};
    }
    const long long E = P > 0 ? match_offsets[P] : 0;
    if (E > 0 && !matches) return fail(SFM_ERR_ARG, "null matches");
    for (long long p = 0; p < P; ++p) {
        const int a = pair_views[2 * p], b = pair_views[2 * p + 1];
        const long long na = feature_offsets[a + 1] - feature_offsets[a], nb = feature_offsets[b + 1] - feature_offsets[b];
        for (long long e = match_offsets[p]; e < match_offsets[p + 1]; ++e)
            if (matches[2 * e] < 0 || matches[2 * e] >= na || matches[2 * e + 1] < 0 || matches[2 * e + 1] >= nb)
                return fail(SFM_ERR_ARG, "match %lld of pair %lld: (%d, %d) outside the views' %lld x %lld features", e, p,
                            matches[2 * e], matches[2 * e + 1], na, nb);
    }
    if (N == 0) {  // no feature, no track
        if (T_out) *T_out = 0;
        if (M_out) *M_out = 0;
        if (offsets) offsets[0] = 0;
        return 0;
    }
    // inputs: feature offsets, match offsets, the pair table, the matches
    const size_t bF = up(((size_t)V + 1) * 8), bMo = up(((size_t)P + 1) * 8), bP = up((size_t)P * sizeof(TbPair)),
                 bE = up((size_t)E * 8);
    if (int r = c->tbin.reserve(bF + bMo + bP + bE)) return r;
    // the union-find over N features and the selection's scan (into size, dead after k_tb_flag)
    size_t scan_bytes = 0;
    CU(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int*)nullptr, (int*)nullptr, (int)N, c->stream));
    const size_t bN = up((size_t)N * 4);
    if (int r = c->tbwork.reserve(5 * bN + scan_bytes)) return r;
    char* in = c->tbin.as<char>();
    char* w = c->tbwork.as<char>();
    TbArgs a;
    memset(&a, 0, sizeof a);
    a.N = (int)N;
    a.V = V;
    a.E = E;
    a.P = P;
    a.foff = reinterpret_cast<const long long*>(in);
    a.moff = reinterpret_cast<const long long*>(in + bF);
    a.pairs = reinterpret_cast<const TbPair*>(in + bF + bMo);
    a.matches = reinterpret_cast<const int2*>(in + bF + bMo + bP);
    a.parent = reinterpret_cast<int*>(w);
    a.size = reinterpret_cast<int*>(w + bN);
    a.track = reinterpret_cast<int*>(w + 2 * bN);
    a.flag = reinterpret_cast<int*>(w + 3 * bN);
    a.label = reinterpret_cast<int*>(w + 4 * bN);
    int* pos = a.size;
    void* scan_tmp = w + 5 * bN;
    // the copies read caller memory synchronously (pageable) or before the synchronisation below
    CU(cudaMemcpyAsync((void*)a.foff, feature_offsets, ((size_t)V + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    if (P > 0) {
        CU(cudaMemcpyAsync((void*)a.moff, match_offsets, ((size_t)P + 1) * 8, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync((void*)a.pairs, ptab.data(), (size_t)P * sizeof(TbPair), cudaMemcpyHostToDevice, c->stream));
    }
    if (E > 0) CU(cudaMemcpyAsync((void*)a.matches, matches, (size_t)E * 8, cudaMemcpyHostToDevice, c->stream));
    k_tb_init<<<tb_grid(N), kTbBlock, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_tb_init")) return r;
    if (E > 0) {
        k_tb_hook<<<tb_grid(E), kTbBlock, 0, c->stream>>>(a);
        if (int r = check_launch(c, "k_tb_hook")) return r;
    }
    k_tb_compress<<<tb_grid(N), kTbBlock, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_tb_compress")) return r;
    k_tb_flag<<<tb_grid(N), kTbBlock, 0, c->stream>>>(a);
    if (int r = check_launch(c, "k_tb_flag")) return r;
    CU(cub::DeviceScan::InclusiveSum(scan_tmp, scan_bytes, a.flag, pos, (int)N, c->stream));
    int M = 0;
    CU(cudaMemcpyAsync(&M, pos + (N - 1), 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (M == 0) {
        if (T_out) *T_out = 0;
        if (M_out) *M_out = 0;
        if (offsets) offsets[0] = 0;
        if (track) CU(cudaMemcpyAsync(track, a.track, (size_t)N * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return 0;
    }
    // the track order over the M selected features: sort by label (stable: ids stay ascending), runs, per observation
    int bits = 1;
    while (bits < 32 && ((N - 1) >> bits) != 0) ++bits;
    size_t sort_bytes = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (unsigned*)nullptr, (unsigned*)nullptr, (unsigned*)nullptr,
                                       (unsigned*)nullptr, M, 0, bits, c->stream));
    CU(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int*)nullptr, (int*)nullptr, M, c->stream));
    const long long Tcap = M / 2;  // every track has at least two observations
    const size_t bM = up((size_t)M * 4), bO = up(((size_t)Tcap + 1) * 8), bS = up((size_t)Tcap * 4);
    if (int r = c->tbsort.reserve(7 * bM + bO + bS + 256 + std::max(sort_bytes, scan_bytes))) return r;
    char* s = c->tbsort.as<char>();
    unsigned* key = reinterpret_cast<unsigned*>(s);
    unsigned* key2 = reinterpret_cast<unsigned*>(s + bM);
    unsigned* id = reinterpret_cast<unsigned*>(s + 2 * bM);
    unsigned* id2 = reinterpret_cast<unsigned*>(s + 3 * bM);
    int* tix = reinterpret_cast<int*>(s + 4 * bM);
    int* view_d = reinterpret_cast<int*>(s + 5 * bM);
    int* feature_d = reinterpret_cast<int*>(s + 6 * bM);
    long long* offsets_d = reinterpret_cast<long long*>(s + 7 * bM);
    int* status_d = reinterpret_cast<int*>(s + 7 * bM + bO);
    int* T_d = reinterpret_cast<int*>(s + 7 * bM + bO + bS);
    void* tmp = s + 7 * bM + bO + bS + 256;
    int* head = reinterpret_cast<int*>(key);  // the unsorted keys are dead after the sort
    k_tb_select<<<tb_grid(N), kTbBlock, 0, c->stream>>>(a, pos, key, id);
    if (int r = check_launch(c, "k_tb_select")) return r;
    CU(cub::DeviceRadixSort::SortPairs(tmp, sort_bytes, key, key2, id, id2, M, 0, bits, c->stream));
    k_tb_heads<<<tb_grid(M), kTbBlock, 0, c->stream>>>(key2, M, head);
    if (int r = check_launch(c, "k_tb_heads")) return r;
    CU(cub::DeviceScan::InclusiveSum(tmp, scan_bytes, head, tix, M, c->stream));
    CU(cudaMemsetAsync(status_d, 0, (size_t)Tcap * 4, c->stream));
    k_tb_obs<<<tb_grid(M), kTbBlock, 0, c->stream>>>(a.foff, V, id2, tix, M, offsets_d, status_d, view_d, feature_d,
                                                     a.track, T_d);
    if (int r = check_launch(c, "k_tb_obs")) return r;
    int T = 0;
    CU(cudaMemcpyAsync(&T, T_d, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    k_tb_status<<<tb_grid(T), kTbBlock, 0, c->stream>>>(offsets_d, T, status_d);
    if (int r = check_launch(c, "k_tb_status")) return r;
    if (T_out) *T_out = T;
    if (M_out) *M_out = M;
    if (offsets) CU(cudaMemcpyAsync(offsets, offsets_d, ((size_t)T + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
    if (status) CU(cudaMemcpyAsync(status, status_d, (size_t)T * 4, cudaMemcpyDeviceToHost, c->stream));
    if (view) CU(cudaMemcpyAsync(view, view_d, (size_t)M * 4, cudaMemcpyDeviceToHost, c->stream));
    if (feature) CU(cudaMemcpyAsync(feature, feature_d, (size_t)M * 4, cudaMemcpyDeviceToHost, c->stream));
    if (track) CU(cudaMemcpyAsync(track, a.track, (size_t)N * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}
