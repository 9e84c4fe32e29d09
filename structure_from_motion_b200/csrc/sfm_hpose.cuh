// Relative pose and plane of a homography: the decomposition that k_tail_mask<MODEL_H> runs on its rider thread and
// k_decompose_homography runs for the per-function API.
//
// Hn = K^-1 H K (one K for both images), divided by its middle singular value and negated when det(Hn) < 0 - the sign
// for which both camera centres lie on the same side of the plane (1 + n^T R^T t / d > 0), i.e. any plane both
// cameras see from the same face.  Candidates: the SVD construction of Ma, Soatto, Kosecka & Sastry, "An Invitation to
// 3-D Vision", Algorithm 5.2, with v1, v2, v3 the right singular vectors of Hn (eigenvectors of Hn^T Hn, eigenvalues
// s1^2 >= 1 >= s3^2):
//   u+- = (sqrt(1 - s3^2) v1 +- sqrt(s1^2 - 1) v3) / sqrt(s1^2 - s3^2)
//   U = [v2, u, v2 x u],  W = [Hn v2, Hn u, Hn v2 x Hn u],  R = W U^T,  N = v2 x u,  T = (Hn - R) N
// in the order (R+, T+, N+), (R+, -T+, -N+), (R-, T-, N-), (R-, -T-, -N-).  Both square-root arguments are clamped at
// 0: with t parallel to n one of them comes out as -eps.  Reported: t = T / |T| (unit, as on the E path), n = N and
// d = 1 / |T| - the plane n^T X = d in camera-1 coordinates, in units of the baseline.
// Rotation-only (s1 - s3 < rotation tolerance; s1 - s3 is about the plane-induced parallax in radians): R = the
// rotation nearest to Hn, t = 0, n = NaN, d = inf in all four slots, and no vote.
#pragma once
#include "sfm_device.cuh"
#include "sfm_linalg.cuh"
#include "sfm_types.h"

namespace sfm {

// The plane part of a homography's candidates; R, t, the votes and the voted index live in the PoseSet beside it.
struct HPlane {
    double n[4][3];
    double d[4];
    int rotation_only;
    int pad;
};

// Hn = K^-1 H K (K^-1 = adj(K) / det(K))
__device__ inline void homography_normalise_k(const double (&H)[9], const double* __restrict__ Kp, double (&Hn)[9]) {
    double K[9], Ka[9], tmp[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) K[i] = Kp[i];
    homography_adj(K, Ka);
    const double det = fma(K[0], Ka[0], fma(K[1], Ka[3], K[2] * Ka[6]));
#pragma unroll
    for (int i = 0; i < 9; ++i) Ka[i] /= det;
    mat3_mul(Ka, H, tmp);
    mat3_mul(tmp, K, Hn);
}

__device__ __forceinline__ void cross3(const double (&a)[3], const double (&b)[3], double (&c)[3]) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}

__device__ __forceinline__ void mat3_vec(const double (&m)[9], const double (&x)[3], double (&y)[3]) {
#pragma unroll
    for (int i = 0; i < 3; ++i) y[i] = fma(m[3 * i], x[0], fma(m[3 * i + 1], x[1], m[3 * i + 2] * x[2]));
}

__device__ __noinline__ void decompose_homography(const double (&Hn)[9], double rotation_tolerance, PoseSet& out,
                                                  HPlane& pl) {
    double g[9], v[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) g[i] = Hn[i];
    jacobi_svd_onesided<3, 3>(g, v, 30);
    double s[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) s[j] = sqrt(fma(g[6 + j], g[6 + j], fma(g[3 + j], g[3 + j], g[j] * g[j])));
    int o[3] = {0, 1, 2};  // columns by descending singular value
    if (s[o[0]] < s[o[1]]) { int t = o[0]; o[0] = o[1]; o[1] = t; }
    if (s[o[1]] < s[o[2]]) { int t = o[1]; o[1] = o[2]; o[2] = t; }
    if (s[o[0]] < s[o[1]]) { int t = o[0]; o[0] = o[1]; o[1] = t; }
    double vc[3][3], sv[3];
    for (int k = 0; k < 3; ++k) {
        sv[k] = s[o[k]];
        for (int i = 0; i < 3; ++i) vc[k][i] = v[3 * i + o[k]];
    }
    const double det = fma(Hn[0], fma(Hn[4], Hn[8], -Hn[5] * Hn[7]),
                           fma(-Hn[1], fma(Hn[3], Hn[8], -Hn[5] * Hn[6]), Hn[2] * fma(Hn[3], Hn[7], -Hn[4] * Hn[6])));
    const double sc = (det < 0.0 ? -1.0 : 1.0) / sv[1];
    double h[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) h[i] = Hn[i] * sc;
    const double s1 = sv[0] / sv[1], s3 = sv[2] / sv[1];
    out.sv[0] = s1; out.sv[1] = 1.0; out.sv[2] = s3;
#pragma unroll
    for (int q = 0; q < 4; ++q) out.counts[q] = 0;
    out.best = -1;
    out.pad = 0;
    pl.pad = 0;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (!(s1 - s3 >= rotation_tolerance) || !(s1 > s3)) {
        // nearest rotation U diag(1, 1, det(U V^T)) V^T = u1 v1^T + u2 v2^T + (u1 x u2)(v1 x v2)^T, u_k = h v_k / |h v_k|
        double u1[3], u2[3], u3[3], w3[3];
        mat3_vec(h, vc[0], u1);
        mat3_vec(h, vc[1], u2);
        const double r1 = 1.0 / sqrt(fma(u1[0], u1[0], fma(u1[1], u1[1], u1[2] * u1[2])));
        const double r2 = 1.0 / sqrt(fma(u2[0], u2[0], fma(u2[1], u2[1], u2[2] * u2[2])));
#pragma unroll
        for (int i = 0; i < 3; ++i) { u1[i] *= r1; u2[i] *= r2; }
        cross3(u1, u2, u3);
        cross3(vc[0], vc[1], w3);
        for (int q = 0; q < 4; ++q) {
            for (int i = 0; i < 3; ++i) {
                for (int j = 0; j < 3; ++j)
                    out.R[q][3 * i + j] = fma(u1[i], vc[0][j], fma(u2[i], vc[1][j], u3[i] * w3[j]));
                out.t[q][i] = 0.0;
                pl.n[q][i] = nan;
            }
            pl.d[q] = __longlong_as_double(0x7ff0000000000000LL);
        }
        pl.rotation_only = 1;
        return;
    }
    pl.rotation_only = 0;
    const double q1 = s1 * s1, q3 = s3 * s3;
    const double ca = sqrt(fmax(1.0 - q3, 0.0)), cb = sqrt(fmax(q1 - 1.0, 0.0)), den = 1.0 / sqrt(q1 - q3);
    double hv2[3];
    mat3_vec(h, vc[1], hv2);
    for (int k = 0; k < 2; ++k) {
        const double sg = k ? -1.0 : 1.0;
        double u[3], hu[3], w3[3], N[3], R[9], T[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) u[i] = fma(ca, vc[0][i], sg * cb * vc[2][i]) * den;
        mat3_vec(h, u, hu);
        cross3(hv2, hu, w3);
        cross3(vc[1], u, N);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) R[3 * i + j] = fma(hv2[i], vc[1][j], fma(hu[i], u[j], w3[i] * N[j]));
        double D[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) D[i] = h[i] - R[i];
        mat3_vec(D, N, T);
        const double nt = sqrt(fma(T[0], T[0], fma(T[1], T[1], T[2] * T[2])));
        for (int c = 0; c < 2; ++c) {
            const int q = 2 * k + c;
            const double sd = c ? -1.0 : 1.0;
#pragma unroll
            for (int i = 0; i < 9; ++i) out.R[q][i] = R[i];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                out.t[q][i] = sd * T[i] / nt;
                pl.n[q][i] = sd * N[i];
            }
            pl.d[q] = 1.0 / nt;
        }
    }
}

// The pose set of "no model" (the tail of an estimate that found none): best = -2, nothing voted.
__device__ __forceinline__ void homography_no_model(PoseSet& out, HPlane& pl) {
#pragma unroll
    for (int q = 0; q < 4; ++q) out.counts[q] = 0;
    out.best = -2;
    out.pad = 0;
    pl.rotation_only = 0;
    pl.pad = 0;
}

// Per-function API: one homography (pixel coordinates) and its K.
__global__ void k_decompose_homography(const double* __restrict__ H, const double* __restrict__ K, double rotation_tolerance,
                                       PoseSet* __restrict__ out, HPlane* __restrict__ pl) {
    if (threadIdx.x || blockIdx.x) return;
    double h[9], hn[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) h[i] = H[i];
    homography_normalise_k(h, K, hn);
    decompose_homography(hn, rotation_tolerance, *out, *pl);
}

}  // namespace sfm
