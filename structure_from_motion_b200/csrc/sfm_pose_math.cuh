// Device functions of K5 that the tail and the refinement share: the decomposition of E into its four pose candidates
// and the DLT triangulation of one correspondence.
#pragma once
#include "sfm_device.cuh"
#include "sfm_fastsvd.cuh"
#include "sfm_linalg.cuh"
#include "sfm_types.h"

namespace sfm {

// _recover_all_r_t (lib/epipolar/eight_point.py:245-280): SVD of E, proper U and V,
// R1 = U W^T V^T, R2 = U W V^T, t from U Z U^T.  One-sided Jacobi SVD; U and V are made
// proper by construction (third columns are cross products), which is what the
// reference's sign fixes (:263-266) achieve.  The LAPACK sign convention is not
// reproducible, so (R1,R2) may come out swapped and t negated relative to numpy — the
// candidate *set* is identical (the reference's own test accepts exactly this ambiguity,
// lib/epipolar/tests/test_epipolar.py:205-229).
__device__ inline void decompose_essential(const double (&E)[9], PoseSet& out) {
    double u0[3], u1[3], u2[3], v0[3], v1[3], v2[3], s0, s1, s2;
    double Uf[9], Vf[9], svf[3];
    if (svd3_rank2_frames(E, Uf, Vf, svf)) {
        // closed form (sfm_fastsvd.cuh): E is rank 2 after the fit's projection, so its null vectors are cross
        // products and the rest is one 2x2 rotation - the same frames the Jacobi SVD below converges to
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            u0[i] = Uf[3 * i]; u1[i] = Uf[3 * i + 1]; u2[i] = Uf[3 * i + 2];
            v0[i] = Vf[3 * i]; v1[i] = Vf[3 * i + 1]; v2[i] = Vf[3 * i + 2];
        }
        s0 = svf[0]; s1 = svf[1]; s2 = svf[2];
    } else {
        double g[9], v[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) g[i] = E[i];
        jacobi_svd_onesided<3, 3>(g, v, 30);
        double s[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) s[j] = sqrt(fma(g[6 + j], g[6 + j], fma(g[3 + j], g[3 + j], g[j] * g[j])));
        // order columns by descending singular value
        int o0 = 0, o1 = 1, o2 = 2;
        if (s[o0] < s[o1]) { int t = o0; o0 = o1; o1 = t; }
        if (s[o1] < s[o2]) { int t = o1; o1 = o2; o2 = t; }
        if (s[o0] < s[o1]) { int t = o0; o0 = o1; o1 = t; }
        auto col = [&](const double (&m)[9], int j, double (&c)[3]) {
#pragma unroll
            for (int i = 0; i < 3; ++i) c[i] = (j == 0) ? m[i * 3] : ((j == 1) ? m[i * 3 + 1] : m[i * 3 + 2]);
        };
        col(g, o0, u0); col(g, o1, u1); col(v, o0, v0); col(v, o1, v1);
        s0 = (o0 == 0) ? s[0] : ((o0 == 1) ? s[1] : s[2]);
        s1 = (o1 == 0) ? s[0] : ((o1 == 1) ? s[1] : s[2]);
        s2 = (o2 == 0) ? s[0] : ((o2 == 1) ? s[1] : s[2]);
#pragma unroll
        for (int i = 0; i < 3; ++i) { u0[i] /= s0; u1[i] /= s1; }
        // proper U and V by construction: third columns are cross products
        u2[0] = u0[1] * u1[2] - u0[2] * u1[1];
        u2[1] = u0[2] * u1[0] - u0[0] * u1[2];
        u2[2] = u0[0] * u1[1] - u0[1] * u1[0];
        v2[0] = v0[1] * v1[2] - v0[2] * v1[1];
        v2[1] = v0[2] * v1[0] - v0[0] * v1[2];
        v2[2] = v0[0] * v1[1] - v0[1] * v1[0];
    }
    const double U[9] = {u0[0], u1[0], u2[0], u0[1], u1[1], u2[1], u0[2], u1[2], u2[2]};
    const double Vh[9] = {v0[0], v0[1], v0[2], v1[0], v1[1], v1[2], v2[0], v2[1], v2[2]};
    const double W[9] = {0, -1, 0, 1, 0, 0, 0, 0, 1};   // :273
    const double Wt[9] = {0, 1, 0, -1, 0, 0, 0, 0, 1};
    const double Z[9] = {0, 1, 0, -1, 0, 0, 0, 0, 0};   // :274
    double Ut[9], tmp[9], tx[9], R1[9], R2[9];
    mat3_transpose(U, Ut);
    mat3_mul(U, Z, tmp);
    mat3_mul(tmp, Ut, tx);                               // :275
    const double t1[3] = {-tx[5], tx[2], -tx[1]};        // :276
    mat3_mul(U, Wt, tmp);
    mat3_mul(tmp, Vh, R1);                               // :277
    mat3_mul(U, W, tmp);
    mat3_mul(tmp, Vh, R2);                               // :278
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        out.R[0][i] = R1[i]; out.R[1][i] = R1[i]; out.R[2][i] = R2[i]; out.R[3][i] = R2[i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        out.t[0][i] = t1[i]; out.t[1][i] = -t1[i]; out.t[2][i] = t1[i]; out.t[3][i] = -t1[i];
    }
    out.sv[0] = s0; out.sv[1] = s1; out.sv[2] = s2;
#pragma unroll
    for (int i = 0; i < 4; ++i) out.counts[i] = 0;
    out.best = -1;
    out.pad = 0;
}

// triangulate_point_correspondence (lib/epipolar/triangulation.py:9-39): 4x4 DLT system,
// right singular vector of the smallest singular value, dehomogenise.  P1, P2 are 3x4
// row-major (only rows 0-2 of the reference's 4x4 Tmat are used, :24-31).
// One copy per kernel (noinline): T2 calls it for the cheirality test and again for the short triangulation, and the
// second use finds the code in the instruction cache.  inline for the linkage only: two translation units include it.
__device__ __noinline__ inline void dlt_triangulate(double xa, double ya, double xb, double yb,
                                             const double* __restrict__ P1,
                                             const double* __restrict__ P2, double (&X)[3]) {
    double g[16], v[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        g[0 + j] = __dsub_rn(__dmul_rn(ya, P1[8 + j]), P1[4 + j]);   // ya * P1[2,:] - P1[1,:]
        g[4 + j] = __dsub_rn(P1[j], __dmul_rn(xa, P1[8 + j]));       // P1[0,:] - xa * P1[2,:]
        g[8 + j] = __dsub_rn(__dmul_rn(yb, P2[8 + j]), P2[4 + j]);
        g[12 + j] = __dsub_rn(P2[j], __dmul_rn(xb, P2[8 + j]));
    }
    double xf[4];
    if (null_vector4_fast(g, xf)) {  // QR + checked inverse iteration (sfm_fastsvd.cuh); inliers always take this route
        X[0] = xf[0] / xf[3];
        X[1] = xf[1] / xf[3];
        X[2] = xf[2] / xf[3];
        return;
    }
    jacobi_svd_onesided<4, 4>(g, v, 20);
    double nrm[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        nrm[j] = fma(g[12 + j], g[12 + j], fma(g[8 + j], g[8 + j], fma(g[4 + j], g[4 + j], g[j] * g[j])));
    int m = 0;
#pragma unroll
    for (int j = 1; j < 4; ++j) {
        const double cur = (m == 0) ? nrm[0] : ((m == 1) ? nrm[1] : ((m == 2) ? nrm[2] : nrm[3]));
        if (nrm[j] < cur) m = j;
    }
    double x[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        x[i] = (m == 0) ? v[i * 4] : ((m == 1) ? v[i * 4 + 1] : ((m == 2) ? v[i * 4 + 2] : v[i * 4 + 3]));
    X[0] = x[0] / x[3];
    X[1] = x[1] / x[3];
    X[2] = x[2] / x[3];
}

// The point of a 4-column DLT system given as a row-major 4x4 g (sfm_tracks.cuh: the triangular factor of an N-view
// system): the null vector of dlt_triangulate - null_vector4_fast, else the Jacobi SVD's column of the smallest singular
// value - dehomogenised.  dlt_triangulate keeps its own inline copy: calling this from it changes the code of its kernels.
__device__ __forceinline__ void dlt_null_point(double (&g)[16], double (&X)[3]) {
    double xf[4];
    if (null_vector4_fast(g, xf)) {  // QR + checked inverse iteration (sfm_fastsvd.cuh); inliers always take this route
        X[0] = xf[0] / xf[3];
        X[1] = xf[1] / xf[3];
        X[2] = xf[2] / xf[3];
        return;
    }
    double v[16];
    jacobi_svd_onesided<4, 4>(g, v, 20);
    double nrm[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        nrm[j] = fma(g[12 + j], g[12 + j], fma(g[8 + j], g[8 + j], fma(g[4 + j], g[4 + j], g[j] * g[j])));
    int m = 0;
#pragma unroll
    for (int j = 1; j < 4; ++j) {
        const double cur = (m == 0) ? nrm[0] : ((m == 1) ? nrm[1] : ((m == 2) ? nrm[2] : nrm[3]));
        if (nrm[j] < cur) m = j;
    }
    double x[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        x[i] = (m == 0) ? v[i * 4] : ((m == 1) ? v[i * 4 + 1] : ((m == 2) ? v[i * 4 + 2] : v[i * 4 + 3]));
    X[0] = x[0] / x[3];
    X[1] = x[1] / x[3];
    X[2] = x[2] / x[3];
}

}  // namespace sfm
