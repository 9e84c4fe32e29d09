// Choosing between the essential matrix and a homography for each image pair: the score ratio of ORB-SLAM (Mur-Artal,
// Montiel & Tardos, 2015, section IV) over the uploaded pixel correspondences, in one launch for one pair or a batch.
//
// E is turned into the pixel fundamental matrix F = Kd^-T E Kd^-1 (the convention b^T E a = 0 of sed_exact), Kd = K
// without its skew and with (0, 0, 1) as the bottom row: the camera E was fitted in.  Per
// correspondence and image, one-way errors in px^2:
//   E: r = b^T F a,  d2_B = r^2 / ((F a)_0^2 + (F a)_1^2),  d2_A = r^2 / ((F^T b)_0^2 + (F^T b)_1^2)
//   H: d2_B = F/P, d2_A = G/Q of transfer_terms (sfm_device.cuh)
// score rho_M(d2) = Gamma - d2/sigma^2 when d2/sigma^2 < T_M, else 0 (NaN and inf fail the compare), Gamma = 5.99,
// T_E = 3.84, T_H = 5.99.  Every rho is rounded to a multiple of 2^-32 and summed exactly in a uint64 (a term is
// below 2^35, n < 2^25, so a sum stays below 2^61): the scores and the choice do not depend on the block schedule, and
// oracle/select_exact.c reproduces them bit for bit.  Every operation below is one IEEE operation or one explicit
// __fma_rn; the oracle evaluates the same order with fma() under -ffp-contract=off.
#pragma once
#include "sfm_device.cuh"
#include "sfm_types.h"

namespace sfm {

constexpr int kSelectBlock = 256;
constexpr double kSelectGamma = 5.99;  // chi^2 95 % quantile, 2 degrees of freedom
constexpr double kSelectTE = 3.84;     // chi^2 95 % quantile, 1 degree of freedom (a point-to-line distance)
constexpr double kSelectTH = 5.99;     // 2 degrees of freedom (a point-to-point distance)
constexpr double kSelectFixed = 4294967296.0;  // 2^32

// include/sfm_b200.h sfm_model_scores
struct ModelScores {
    double score_e, score_h, ratio_h;
    unsigned long long fixed_e, fixed_h;
    long long count_e, count_h;
    int model, reserved;
};

constexpr int kSelectStateWords = 8;  // per pair: fixed_e, fixed_h, count_e, count_h, ticket, 3 unused

struct SelectArgs {
    const double* xa; const double* ya; const double* xb; const double* yb;  // pixel coordinates, element i at [i*stride]
    long long stride, n;
    const long long* offsets;    // [P+1] or null (one pair of n)
    const SelectModels* models;  // [P]
    double sigma, ratio;
    unsigned long long* state;   // [P][kSelectStateWords], zero on entry and on exit
    ModelScores* out;            // [P]
    double* per_point;           // [n_total][4] (d2_A,E, d2_B,E, d2_A,H, d2_B,H) or null
};

// F = Kd^-T E Kd^-1 with Kd^-1 = adj(Kd) / det(Kd), Kd = [[fx, 0, cx], [0, fy, cy], [0, 0, 1]]: the camera of the
// E path, whose (x - cx) / fx, (y - cy) / fy normalisation ignores the skew and the bottom row of K.  One thread.
__device__ __forceinline__ void fundamental_from_essential(const double* E, const double* K, double (&F)[9]) {
    const double k[9] = {K[0], 0.0, K[2], 0.0, K[4], K[5], 0.0, 0.0, 1.0};
    double adj[9], ki[9], m[9];
    homography_adj(k, adj);
    const double det = __fma_rn(k[0], adj[0], __fma_rn(k[1], adj[3], __dmul_rn(k[2], adj[6])));
#pragma unroll
    for (int i = 0; i < 9; ++i) ki[i] = __ddiv_rn(adj[i], det);
#pragma unroll
    for (int i = 0; i < 3; ++i)  // m = E K^-1
#pragma unroll
        for (int j = 0; j < 3; ++j)
            m[3 * i + j] = __fma_rn(E[3 * i + 2], ki[6 + j], __fma_rn(E[3 * i + 1], ki[3 + j], __dmul_rn(E[3 * i], ki[j])));
#pragma unroll
    for (int i = 0; i < 3; ++i)  // F = K^-T m
#pragma unroll
        for (int j = 0; j < 3; ++j)
            F[3 * i + j] = __fma_rn(ki[6 + i], m[6 + j], __fma_rn(ki[3 + i], m[3 + j], __dmul_rn(ki[i], m[j])));
}

// rho of one error, as a multiple of 2^-32; *pass = the error is below T
__device__ __forceinline__ unsigned long long select_rho(double d2, double s2, double T, bool& pass) {
    const double x = __ddiv_rn(d2, s2);
    pass = x < T;
    return pass ? __double2ull_rn(__dmul_rn(__dsub_rn(kSelectGamma, x), kSelectFixed)) : 0ull;
}

// Grid (blocks, P): blockIdx.y = image pair; the blocks of a pair stride over its records and the last of them to
// finish writes the pair's result.
__global__ void __launch_bounds__(kSelectBlock) k_score_models(const SelectArgs a) {
    __shared__ double s_f[9], s_h[9], s_adj[9];
    __shared__ unsigned long long s_part[kSelectBlock / 32][4];
    __shared__ unsigned s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pair = blockIdx.y;
    const SelectModels& m = a.models[pair];
    const int have_e = m.have_e, have_h = m.have_h;
    if (tid == 0) {  // the same operations in every block: every block sees the same F and adj(H)
        double f[9], h[9], adj[9];
        if (have_e) fundamental_from_essential(m.E, m.K, f);
#pragma unroll
        for (int i = 0; i < 9; ++i) h[i] = m.H[i];
        homography_adj(h, adj);
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            s_f[i] = have_e ? f[i] : 0.0;
            s_h[i] = h[i];
            s_adj[i] = adj[i];
        }
    }
    __syncthreads();
    double f[9], h[9], adj[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        f[i] = s_f[i];
        h[i] = s_h[i];
        adj[i] = s_adj[i];
    }
    const double s2 = __dmul_rn(a.sigma, a.sigma);
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    unsigned long long se = 0, sh = 0, ce = 0, ch = 0;
    const long long pbase = a.offsets ? a.offsets[pair] : 0;
    const long long pend = a.offsets ? a.offsets[pair + 1] : a.n;
    for (long long i = pbase + blockIdx.x * (long long)blockDim.x + tid; i < pend; i += (long long)gridDim.x * blockDim.x) {
        const long long g = i * a.stride;
        const double xa = a.xa[g], ya = a.ya[g], xb = a.xb[g], yb = a.yb[g];
        double dae = nan, dbe = nan, dah = nan, dbh = nan;
        if (have_e) {
            const double la0 = __fma_rn(f[0], xa, __fma_rn(f[1], ya, f[2]));
            const double la1 = __fma_rn(f[3], xa, __fma_rn(f[4], ya, f[5]));
            const double la2 = __fma_rn(f[6], xa, __fma_rn(f[7], ya, f[8]));
            const double lb0 = __fma_rn(f[0], xb, __fma_rn(f[3], yb, f[6]));
            const double lb1 = __fma_rn(f[1], xb, __fma_rn(f[4], yb, f[7]));
            const double r = __fma_rn(xb, la0, __fma_rn(yb, la1, la2));
            const double r2 = __dmul_rn(r, r);
            dbe = __ddiv_rn(r2, __fma_rn(la0, la0, __dmul_rn(la1, la1)));
            dae = __ddiv_rn(r2, __fma_rn(lb0, lb0, __dmul_rn(lb1, lb1)));
            bool pa, pb;
            se += select_rho(dae, s2, kSelectTE, pa) + select_rho(dbe, s2, kSelectTE, pb);
            ce += (pa && pb) ? 1ull : 0ull;
        }
        if (have_h) {
            const TransferTerms t = transfer_terms(h, adj, xa, ya, xb, yb);
            dbh = __ddiv_rn(t.F, t.P);
            dah = __ddiv_rn(t.G, t.Q);
            bool pa, pb;
            sh += select_rho(dah, s2, kSelectTH, pa) + select_rho(dbh, s2, kSelectTH, pb);
            ch += (pa && pb) ? 1ull : 0ull;
        }
        if (a.per_point) {
            double* o = a.per_point + 4 * i;
            o[0] = dae; o[1] = dbe; o[2] = dah; o[3] = dbh;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        se += __shfl_xor_sync(0xffffffffu, se, d);
        sh += __shfl_xor_sync(0xffffffffu, sh, d);
        ce += __shfl_xor_sync(0xffffffffu, ce, d);
        ch += __shfl_xor_sync(0xffffffffu, ch, d);
    }
    if (lane == 0) {
        s_part[warp][0] = se; s_part[warp][1] = sh; s_part[warp][2] = ce; s_part[warp][3] = ch;
    }
    __syncthreads();
    unsigned long long* state = a.state + (long long)pair * kSelectStateWords;
    if (tid < 4) {  // integer sums: the order of the blocks' atomics does not matter
        unsigned long long v = 0;
        for (int w = 0; w < kSelectBlock / 32; ++w) v += s_part[w][tid];
        if (v) atomicAdd(&state[tid], v);
    }
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(&state[4], 1ull) == (unsigned long long)(gridDim.x - 1)) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last || tid != 0) return;
    // the pair's last block: its other blocks' sums are visible; write the result and leave the state zero for the next
    // call
    __threadfence();
    volatile unsigned long long* st = state;
    const unsigned long long fe = st[0], fh = st[1], ne = st[2], nh = st[3];
    st[0] = 0; st[1] = 0; st[2] = 0; st[3] = 0; st[4] = 0;
    ModelScores r;
    r.fixed_e = fe;
    r.fixed_h = fh;
    r.count_e = (long long)ne;
    r.count_h = (long long)nh;
    r.score_e = __dmul_rn(__ull2double_rn(fe), 1.0 / kSelectFixed);
    r.score_h = __dmul_rn(__ull2double_rn(fh), 1.0 / kSelectFixed);
    const double tot = __dadd_rn(r.score_h, r.score_e);
    r.ratio_h = tot > 0.0 ? __ddiv_rn(r.score_h, tot) : 0.0;
    r.model = !have_e ? (have_h ? 1 : -1) : (!have_h ? 0 : (r.ratio_h > a.ratio ? 1 : 0));
    r.reserved = 0;
    a.out[pair] = r;
}

}  // namespace sfm
