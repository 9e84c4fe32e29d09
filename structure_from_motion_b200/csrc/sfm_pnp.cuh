// Absolute pose of a new view (PnP): the P3P fitter, the reprojection-error scorer and the mask of one pose.  The record
// and the pinned evaluation of one record (pnp_projection, pnp_terms, pnp_exact) are in sfm_pnp_model.cuh.
//
// Input.  n records, each a world point X = (X, Y, Z) and its observed pixel (u, v) in the new image, and K: upper
// triangular, K[2,2] = 1, finite and non-singular (checked on the host).  The world frame is the frame of the points;
// for points from the essential-matrix tail that is camera 1 with the baseline |t| = 1.
//
// Model.  [R | t] as 12 doubles, row-major 3 x 4, x_cam = R X + t.  Every consumer (scorer, K3, mask, the fitter's
// fourth-point rule and oracle/reproj_exact.c) forms P = K [R | t] with pnp_projection's pinned order,
//   P[r][c] = fma(K[r][0], M[0][c], fma(K[r][1], M[1][c], K[r][2] * M[2][c])),
// once per model load, and then p = P (X, Y, Z, 1) with pnp_terms' pinned order.
//
// Error.  With d0 = p0 - u p2, d1 = p1 - v p2 (one fma each), F = d0^2 + d1^2 and W = p2^2:
//   inlier   <=>  p2 >= 2^-537 && F < inf && F <= thr W   (every evaluation; division-free; NaN fails)
//   value     =   F / W, the squared reprojection error in px^2   (inliers only; summed)
// A point on or behind the camera plane is never an inlier.  thr is in px^2 and the test is "<=" (ransac.py:73).
// The two range terms keep every inlier's value finite: without them a finite record some 1e154 units or pixels out
// has F = W = inf and would pass with the value NaN, and a record with 0 < p2 < 2^-537 (W = 0) and F = 0 with 0 / 0.
// A finite record with W = inf but F finite (on its ray, ~1e154 out) passes and is scored 0: its true squared error is
// somewhere below 1 px^2, so with thr < 1 such a record can be admitted wrongly; its value stays finite.
// Both are integer tests on the high words and use no FP64 slot; k_score_pnp still measured 2.3 % slower with them
// on one B200 (DESIGN.md 7f).
//
// FP64 issue slots of one evaluation (the scorer's hot loop, counted from the source, one per DFMA/DMUL):
//   p 9, the two differences 2, F 2, W 1, thr W 1, the compare 1                              = 16
// Pipe floor at the measured 18.35e12 DFMA/s per B200 (sfm_homography.cuh): 1.15e12 evaluations/s.  An inlier adds
// one division and the fixed-point conversion on top.
//
// Minimal solver.  Lambda Twist (Persson & Nordberg, ECCV 2018) on sample columns 0-2: the cubic of the degenerate
// conic D1 + g D2, its closed-form eigen step, the two planes of the degenerate conic, a quadratic per plane, and a
// Gauss-Newton polish of the three depths.  Column 3 chooses among the (up to four) solutions with positive depth at
// all three points: the smallest F / W of point 3, the first in the solver's root order on a tie (OpenCV's 4-point
// P3P rule).  Root order: one root of the cubic (see p3p_lambda_twist), the plane of +s before the plane of -s, and
// within a plane the smaller root of the quadratic first.  A sample is invalid (never a candidate, counted in num_invalid /
// first_invalid) when a coordinate is not finite, when the three world points are collinear
// (|w1 x w2|^2 <= kPnpCollinear^2 |w1|^2 |w2|^2, w1 = X0 - X1, w2 = X0 - X2), when no real solution has three
// positive depths, or when the chosen [R | t] is not finite or its R is not orthonormal to kPnpOrthonormal
// (max |R R^T - I|).  The last rule is for near-collinear world points (sine below ~1e-2): the rotation about their
// line rests on the last bits of the depths, and float64 Lambda Twist then returns solutions that are wrong, not merely
// imprecise (up to ~1 in R at sine 1e-5), and visibly non-orthonormal.  Such a sample is invalid rather than wrong;
// well-spread samples, narrow cameras included, stay below 3e-7.
// Range.  The solver runs on the world points scaled by a power of two taken from their largest coordinate difference
// and scales t back, so it is exactly equivariant under world x 2^k and works at any world scale whose coordinate
// differences and pose are finite.  A pixel's bearing takes a power-of-two-scaled norm when xn^2 + yn^2 overflows
// (more than ~1e154 focal lengths off axis), so every finite pixel has a unit bearing.
//
// RANSAC semantics: fit_with_ransac(data, 4, ...) (lib/ransac/ransac.py:19-93) exactly as the homography path applies
// it: columns 0-3 of the shared int32[H][8] table, samples never extra inliers and always in the error, K3
// (k_finalise<MODEL_P>) with the same aggregations and selection rules.
#pragma once
#include "sfm_device.cuh"
#include "sfm_fit.cuh"
#include "sfm_score.cuh"
#include "sfm_pnp_model.cuh"

namespace sfm {

// ---- Lambda Twist -------------------------------------------------------------------------------------------------
__device__ __forceinline__ double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ double det3c(const double* c0, const double* c1, const double* c2) {
    double x[3];
    cross3(c1, c2, x);
    return dot3(c0, x);
}

// the real roots of k3 g^3 + k2 g^2 + k1 g + k0 (k3 != 0), each polished by Newton steps that reduce |f|
__device__ __forceinline__ int cubic_roots(double k3, double k2, double k1, double k0, double (&g)[3]) {
    const double p = k2 / k3, q = k1 / k3, r = k0 / k3;
    const double P = q - p * p / 3.0, Q = 2.0 * p * p * p / 27.0 - p * q / 3.0 + r;
    const double disc = 0.25 * Q * Q + P * P * P / 27.0;
    int nr;
    if (disc > 0.0) {
        const double sq = sqrt(disc);
        g[0] = cbrt(-0.5 * Q + sq) + cbrt(-0.5 * Q - sq) - p / 3.0;
        nr = 1;
    } else {
        const double m = 2.0 * sqrt(-P / 3.0);
        double arg = P < 0.0 ? (3.0 * Q / (P * m)) : 0.0;
        arg = arg > 1.0 ? 1.0 : (arg < -1.0 ? -1.0 : arg);
        const double th = acos(arg) / 3.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) g[k] = m * cos(th - 2.0943951023931957 * k) - p / 3.0;
        nr = 3;
    }
    for (int k = 0; k < nr; ++k) {
        double x = g[k], f = ((x + p) * x + q) * x + r;
#pragma unroll
        for (int it = 0; it < 3; ++it) {
            const double df = (3.0 * x + 2.0 * p) * x + q;
            if (df == 0.0) break;
            const double xn = x - f / df, fn = ((xn + p) * xn + q) * xn + r;
            if (!(fabs(fn) < fabs(f))) break;
            x = xn;
            f = fn;
        }
        g[k] = x;
    }
    return nr;
}

// unit eigenvector of the symmetric A for eigenvalue s: the largest cross product of two rows of A - s I
__device__ __forceinline__ void eigvec3(const double (&A)[9], double s, double (&e)[3]) {
    const double r0[3] = {A[0] - s, A[1], A[2]}, r1[3] = {A[3], A[4] - s, A[5]}, r2[3] = {A[6], A[7], A[8] - s};
    double c0[3], c1[3], c2[3];
    cross3(r0, r1, c0);
    cross3(r0, r2, c1);
    cross3(r1, r2, c2);
    const double n0 = dot3(c0, c0), n1 = dot3(c1, c1), n2 = dot3(c2, c2);
    const double* c = c0;
    double nn = n0;
    if (n1 > nn) { c = c1; nn = n1; }
    if (n2 > nn) { c = c2; nn = n2; }
    const double inv = 1.0 / sqrt(nn);
    e[0] = c[0] * inv; e[1] = c[1] * inv; e[2] = c[2] * inv;
}

// Gauss-Newton polish of the depths on the three distance equations (a step is kept only when it lowers the residual)
__device__ __forceinline__ void p3p_refine(double (&l)[3], double a01, double a02, double a12, double b01, double b02,
                                           double b12) {
    auto res = [&](const double (&x)[3], double (&r)[3]) {
        r[0] = x[0] * x[0] + x[1] * x[1] - 2.0 * b01 * x[0] * x[1] - a01;
        r[1] = x[0] * x[0] + x[2] * x[2] - 2.0 * b02 * x[0] * x[2] - a02;
        r[2] = x[1] * x[1] + x[2] * x[2] - 2.0 * b12 * x[1] * x[2] - a12;
    };
    double r[3];
    res(l, r);
    double e = dot3(r, r);
#pragma unroll 1
    for (int it = 0; it < 5; ++it) {
        // J columns
        const double j0[3] = {2.0 * (l[0] - b01 * l[1]), 2.0 * (l[0] - b02 * l[2]), 0.0};
        const double j1[3] = {2.0 * (l[1] - b01 * l[0]), 0.0, 2.0 * (l[1] - b12 * l[2])};
        const double j2[3] = {0.0, 2.0 * (l[2] - b02 * l[0]), 2.0 * (l[2] - b12 * l[1])};
        const double d = det3c(j0, j1, j2);
        if (!(d != 0.0)) break;
        double x[3] = {l[0] - det3c(r, j1, j2) / d, l[1] - det3c(j0, r, j2) / d, l[2] - det3c(j0, j1, r) / d};
        double rn[3];
        res(x, rn);
        const double en = dot3(rn, rn);
        if (!(en < e)) break;
        l[0] = x[0]; l[1] = x[1]; l[2] = x[2];
        r[0] = rn[0]; r[1] = rn[1]; r[2] = rn[2];
        e = en;
    }
}

// The solutions [R | t] (row-major 3 x 4) with three positive depths of the unit bearings y[i] of world points x[i].
// Of the cubic's real roots the one whose degenerate conic has the most negative product of its two non-zero
// eigenvalues is used (an indefinite conic: two real planes through the origin hold every solution).
__device__ __forceinline__ int p3p_lambda_twist(const double (&y)[3][3], const double (&x)[3][3], double (&M)[4][12]) {
    double w1[3], w2[3], w3[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { w1[k] = x[0][k] - x[1][k]; w2[k] = x[0][k] - x[2][k]; }
    const double w12[3] = {x[1][0] - x[2][0], x[1][1] - x[2][1], x[1][2] - x[2][2]};
    const double a01 = dot3(w1, w1), a02 = dot3(w2, w2), a12 = dot3(w12, w12);
    const double b01 = dot3(y[0], y[1]), b02 = dot3(y[0], y[2]), b12 = dot3(y[1], y[2]);
    // D1 = a12 M01 - a01 M12, D2 = a12 M02 - a02 M12 (symmetric: rows are columns)
    const double D1[9] = {a12, -a12 * b01, 0.0, -a12 * b01, a12 - a01, a01 * b12, 0.0, a01 * b12, -a01};
    const double D2[9] = {a12, 0.0, -a12 * b02, 0.0, -a02, a02 * b12, -a12 * b02, a02 * b12, a12 - a02};
    const double* A0 = D1; const double* A1 = D1 + 3; const double* A2 = D1 + 6;
    const double* B0 = D2; const double* B1 = D2 + 3; const double* B2 = D2 + 6;
    const double k3 = det3c(B0, B1, B2);
    const double k2 = det3c(A0, B1, B2) + det3c(B0, A1, B2) + det3c(B0, B1, A2);
    const double k1 = det3c(A0, A1, B2) + det3c(A0, B1, A2) + det3c(B0, A1, A2);
    const double k0 = det3c(A0, A1, A2);
    if (!(k3 != 0.0) || !isfinite(k3) || !isfinite(k2) || !isfinite(k1) || !isfinite(k0)) return 0;
    double g[3];
    const int ng = cubic_roots(k3, k2, k1, k0, g);
    double D0[9], mbest = 0.0;
    bool have = false;
    for (int k = 0; k < ng; ++k) {
        double D[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) D[i] = D1[i] + g[k] * D2[i];
        const double m = D[0] * D[4] - D[1] * D[1] + D[0] * D[8] - D[2] * D[2] + D[4] * D[8] - D[5] * D[5];
        if (m < 0.0 && (!have || m < mbest)) {
            have = true;
            mbest = m;
#pragma unroll
            for (int i = 0; i < 9; ++i) D0[i] = D[i];
        }
    }
    if (!have) return 0;
    const double tr = D0[0] + D0[4] + D0[8];
    const double hs = sqrt(0.25 * tr * tr - mbest);
    const double s1 = 0.5 * tr + hs, s2 = 0.5 * tr - hs;  // s1 > 0 > s2
    double e1[3], e2[3];
    eigvec3(D0, s1, e1);
    eigvec3(D0, s2, e2);
    const double s = sqrt(-s2 / s1);
    // the scale comes from the equation of the longest world distance
    const int ref = (a01 >= a02 && a01 >= a12) ? 0 : (a02 >= a12 ? 1 : 2);
    const double aref = ref == 0 ? a01 : (ref == 1 ? a02 : a12);
    const double bref = ref == 0 ? b01 : (ref == 1 ? b02 : b12);
    const int ri = ref == 2 ? 1 : 0, rj = ref == 0 ? 1 : 2;
    double W[9];  // [w1 w2 w1 x w2] as columns; inverse by adjugate
    cross3(w1, w2, w3);
    const double Wc[3][3] = {{w1[0], w2[0], w3[0]}, {w1[1], w2[1], w3[1]}, {w1[2], w2[2], w3[2]}};
    {
        double h[9] = {Wc[0][0], Wc[0][1], Wc[0][2], Wc[1][0], Wc[1][1], Wc[1][2], Wc[2][0], Wc[2][1], Wc[2][2]};
        double adj[9];
        homography_adj(h, adj);
        const double det = h[0] * adj[0] + h[1] * adj[3] + h[2] * adj[6];
#pragma unroll
        for (int i = 0; i < 9; ++i) W[i] = adj[i] / det;
    }
    int nsol = 0;
#pragma unroll 1
    for (int sg = 0; sg < 2; ++sg) {
        const double sgn = sg == 0 ? 1.0 : -1.0;
        const double u[3] = {e1[0] - sgn * s * e2[0], e1[1] - sgn * s * e2[1], e1[2] - sgn * s * e2[2]};
        const int kk = (fabs(u[0]) >= fabs(u[1]) && fabs(u[0]) >= fabs(u[2])) ? 0 : (fabs(u[1]) >= fabs(u[2]) ? 1 : 2);
        const int ii = kk == 0 ? 1 : 0, jj = kk == 2 ? 1 : 2;
        if (!(u[kk] != 0.0)) continue;
        // v(tau) = tau p + q on the plane u . v = 0: v_ii = tau, v_jj = 1, v_kk = -(u_ii tau + u_jj) / u_kk
        double p[3] = {0.0, 0.0, 0.0}, q[3] = {0.0, 0.0, 0.0};
        p[ii] = 1.0; p[kk] = -u[ii] / u[kk];
        q[jj] = 1.0; q[kk] = -u[jj] / u[kk];
        double Dp[3], Dq[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            Dp[i] = D2[3 * i] * p[0] + D2[3 * i + 1] * p[1] + D2[3 * i + 2] * p[2];
            Dq[i] = D2[3 * i] * q[0] + D2[3 * i + 1] * q[1] + D2[3 * i + 2] * q[2];
        }
        const double qa = dot3(p, Dp), qb = 2.0 * dot3(p, Dq), qc = dot3(q, Dq);
        double tau[2];
        int nt = 0;
        if (qa == 0.0) {
            if (qb != 0.0) tau[nt++] = -qc / qb;
        } else {
            const double disc = qb * qb - 4.0 * qa * qc;
            if (disc >= 0.0) {
                const double sq = sqrt(disc);
                const double t1 = (-qb - (qb >= 0.0 ? sq : -sq)) / (2.0 * qa);
                const double t2 = t1 != 0.0 ? qc / (qa * t1) : (-qb + (qb >= 0.0 ? sq : -sq)) / (2.0 * qa);
                tau[0] = t1 < t2 ? t1 : t2;
                tau[1] = t1 < t2 ? t2 : t1;
                nt = 2;
            }
        }
        for (int it = 0; it < nt; ++it) {
            if (!(tau[it] > 0.0)) continue;
            const double v[3] = {tau[it] * p[0] + q[0], tau[it] * p[1] + q[1], tau[it] * p[2] + q[2]};
            if (!(v[0] > 0.0 && v[1] > 0.0 && v[2] > 0.0)) continue;
            const double den = v[ri] * v[ri] + v[rj] * v[rj] - 2.0 * bref * v[ri] * v[rj];
            if (!(den > 0.0)) continue;
            const double sc = sqrt(aref / den);
            double l[3] = {sc * v[0], sc * v[1], sc * v[2]};
            p3p_refine(l, a01, a02, a12, b01, b02, b12);
            if (!(l[0] > 0.0 && l[1] > 0.0 && l[2] > 0.0)) continue;
            // camera points c_i = l_i y_i; R = [c0-c1, c0-c2, (c0-c1) x (c0-c2)] [w1, w2, w1 x w2]^-1, t = c0 - R x0
            double c0[3], d1[3], d2[3], d3[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                c0[k] = l[0] * y[0][k];
                d1[k] = c0[k] - l[1] * y[1][k];
                d2[k] = c0[k] - l[2] * y[2][k];
            }
            cross3(d1, d2, d3);
            double* Mo = M[nsol];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int cI = 0; cI < 3; ++cI)
                    Mo[4 * r + cI] = d1[r] * W[cI] + d2[r] * W[3 + cI] + d3[r] * W[6 + cI];
                Mo[4 * r + 3] = c0[r] - (Mo[4 * r] * x[0][0] + Mo[4 * r + 1] * x[0][1] + Mo[4 * r + 2] * x[0][2]);
            }
            ++nsol;
        }
    }
    return nsol;
}

// The 4-point fit of one sample: bearings of columns 0-2 through K^-1 (y first, then x minus the skew's share, as the
// homography tail normalises pixels), the P3P solutions, the fourth-point choice.  Returns validity.
__device__ __forceinline__ bool pnp_fit4(const PnpRec (&c)[4], const double* K, double (&Rt)[12]) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        ok = ok && isfinite(c[i].X) && isfinite(c[i].Y) && isfinite(c[i].Z) && isfinite(c[i].u) && isfinite(c[i].v);
    if (!ok) return false;
    double x[3][3], y[3][3];
    const double fx = K[0], sk = K[1], cx = K[2], fy = K[4], cy = K[5];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double yn = __ddiv_rn(__dsub_rn(c[i].v, cy), fy);
        const double xn = __ddiv_rn(__dsub_rn(__dsub_rn(c[i].u, cx), __dmul_rn(sk, yn)), fx);
        const double n2 = xn * xn + yn * yn + 1.0;
        if (isfinite(n2)) {
            const double inv = 1.0 / sqrt(n2);
            y[i][0] = xn * inv; y[i][1] = yn * inv; y[i][2] = inv;
        } else {  // a pixel ~1e154 focal lengths off axis: (xn, yn, 1) scaled by a power of two before its norm
            int e;
            (void)frexp(fmax(fabs(xn), fabs(yn)), &e);
            const double bx = ldexp(xn, -e), by = ldexp(yn, -e), bz = ldexp(1.0, -e);
            const double inv = 1.0 / sqrt(bx * bx + by * by + bz * bz);
            y[i][0] = bx * inv; y[i][1] = by * inv; y[i][2] = bz * inv;
        }
    }
    // The solver sees the world points scaled by 2^-we, 2^we the power of two just above the largest coordinate
    // difference, so that its degree-8 terms (eigvec3) and degree-6 terms (the cubic) neither overflow nor underflow;
    // t is scaled back.  Every step is homogeneous in the world scale, so this changes no bit where the unscaled
    // solve stayed in range.
#pragma unroll
    for (int i = 0; i < 3; ++i) { x[i][0] = c[i].X; x[i][1] = c[i].Y; x[i][2] = c[i].Z; }
    int we = 0;
    {
        double m = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k)
            m = fmax(m, fmax(fabs(x[0][k] - x[1][k]), fmax(fabs(x[0][k] - x[2][k]), fabs(x[1][k] - x[2][k]))));
        if (!isfinite(m)) return false;
        (void)frexp(m, &we);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) x[i][k] = ldexp(x[i][k], -we);
    {
        double w1[3], w2[3], w3[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { w1[k] = x[0][k] - x[1][k]; w2[k] = x[0][k] - x[2][k]; }
        cross3(w1, w2, w3);
        const double lhs = dot3(w3, w3), rhs = kPnpCollinear * kPnpCollinear * (dot3(w1, w1) * dot3(w2, w2));
        if (!(lhs > rhs)) return false;
    }
    double M[4][12];
    const int ns = p3p_lambda_twist(y, x, M);
    int best = -1;
    double be = 0.0;
    for (int s = 0; s < ns; ++s) {
#pragma unroll
        for (int r = 0; r < 3; ++r) M[s][4 * r + 3] = ldexp(M[s][4 * r + 3], we);
        double P[12];
        pnp_projection(K, M[s], P);
        const PnpTerms t = pnp_terms(P, c[3].X, c[3].Y, c[3].Z, c[3].u, c[3].v);
        const double e = pnp_value(t);
        if (e == e && (best < 0 || e < be)) { best = s; be = e; }
    }
    if (best < 0) return false;
    {
        // near-collinear world points leave the rotation about their line to the last bits of the depths: the chosen
        // solution then comes out visibly non-orthonormal and is wrong, not merely imprecise, so the sample is invalid
        double dev = 0.0;
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = a; b < 3; ++b)
                dev = fmax(dev, fabs(M[best][4 * a] * M[best][4 * b] + M[best][4 * a + 1] * M[best][4 * b + 1] +
                                     M[best][4 * a + 2] * M[best][4 * b + 2] - (a == b ? 1.0 : 0.0)));
        if (!(dev <= kPnpOrthonormal)) return false;
    }
#pragma unroll
    for (int k = 0; k < 12; ++k) {
        Rt[k] = M[best][k];
        ok = ok && isfinite(Rt[k]);
    }
    return ok;
}

// K1 for PnP, one thread per hypothesis (the shape of k_fit_homography, one pair): clears this hypothesis's
// accumulator column (and, thread 0, the tail words), reads its table row or draws it with the device sampler
// (recording all 8 columns), fits columns 0-3.
constexpr int kFitPThreads = 64;
__global__ void __launch_bounds__(kFitPThreads)
k_fit_pnp(const PnpRec* __restrict__ pts, const double* __restrict__ K, const int32_t* __restrict__ table, long long h,
          double* __restrict__ Rt_out, uint8_t* __restrict__ valid_out, unsigned long long* __restrict__ acc, int acc_planes,
          int acc_tail_words, int draw, unsigned long long seed, unsigned long long stream0, long long hyp_offset, long long n) {
    chain_enter();
    const long long i = blockIdx.x * (long long)kFitPThreads + threadIdx.x;
    if (i >= h) return;
    for (int k = 0; k < acc_planes; ++k) acc[(long long)k * h + i] = 0ull;
    if (i == 0)
        for (int k = 0; k < acc_tail_words; ++k) acc[(long long)acc_planes * h + k] = 0ull;
    int idx[4];
    if (draw) {
        int32_t row[8];
        philox_sample8(seed, stream0, (unsigned long long)(hyp_offset + i), (unsigned)n, row);
        int4* t = reinterpret_cast<int4*>(const_cast<int32_t*>(table) + 8 * i);
        t[0] = make_int4(row[0], row[1], row[2], row[3]);
        t[1] = make_int4(row[4], row[5], row[6], row[7]);
#pragma unroll
        for (int k = 0; k < 4; ++k) idx[k] = row[k];
    } else {
        const int4 t0 = reinterpret_cast<const int4*>(table + 8 * i)[0];
        idx[0] = t0.x; idx[1] = t0.y; idx[2] = t0.z; idx[3] = t0.w;
    }
    PnpRec c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = pts[idx[k]];
    double Rt[12];
    const bool ok = pnp_fit4(c, K, Rt);
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt_out[12 * i + k] = ok ? Rt[k] : 0.0;
    valid_out[i] = ok ? FIT_VALID : FIT_INVALID;
}

// ------------------------------------------------------------------------------------
// K2 for PnP - count and fixed-point sums of the reprojection error of every inlier, per hypothesis.  The mapping of
// k_score_homography: persistent warps claim (correspondence split x group of 32*HPT hypotheses) items from an atomic
// counter, each warp streams its records through its own ring of bulk-async tiles, lane = hypothesis, every lane
// reads the same record (broadcast).  A lane forms P = K [R | t] of its hypotheses once per item.  Integer sums in
// the same 84-bit fixed point as the E and H paths: counts and sums do not depend on the schedule.
// ------------------------------------------------------------------------------------
constexpr int kPScoreThreads = 128;
constexpr int kPScoreWarps = kPScoreThreads / 32;
constexpr int kPTile = 64;
constexpr int kPStages = 3;
constexpr int kPScoreHpt = 2;

struct PScoreArgs {
    const PnpRec* pts;
    const double* K;          // [9]
    const double* Rt;         // [h][12]
    long long n, h;
    double thr;
    double scale1, scale2;    // 2^(63-e), 2^(63-2e): every inlier's value < 2^e
    int sums;                 // SUM_S1 | SUM_S2
    long long chunk;          // records per split (multiple of kPTile, <= kMaxItemPoints)
    int hblocks, nsplit;
    long long total_items;
    unsigned* work_counter;
    unsigned long long* acc;  // [kAccWords][h], cleared by k_fit_pnp
};

struct alignas(128) PScoreWarpSmem {
    PnpRec tile[kPStages][kPTile];
    unsigned long long full_bar[kPStages];
};

template <int HPT>
__global__ void __launch_bounds__(kPScoreThreads, 3) k_score_pnp(const PScoreArgs a) {
    chain_enter();
    extern __shared__ __align__(128) unsigned char pscore_smem[];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(full, (int)(threadIdx.x >> 5), 0);
    PScoreWarpSmem& ws = reinterpret_cast<PScoreWarpSmem*>(pscore_smem)[warp];
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kPStages; ++s) mbar_init(&ws.full_bar[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    double K[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) K[k] = a.K[k];
    unsigned gt = 0;  // tiles consumed so far by this warp (stage + parity)
    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(a.work_counter, 1u);
        item = __shfl_sync(full, item, 0);
        if (item >= a.total_items) break;
        const int hw = (int)(item % (unsigned)a.hblocks);
        const int split = (int)(item / (unsigned)a.hblocks);
        long long begin = (long long)split * a.chunk;
        if (begin > a.n) begin = a.n;
        const long long end = (begin + a.chunk < a.n) ? begin + a.chunk : a.n;
        const int ntiles = (int)((end - begin + kPTile - 1) / kPTile);
        auto issue = [&](int t) {  // lane 0 only
            const int s = (int)((gt + (unsigned)t) % kPStages);
            const long long first = begin + (long long)t * kPTile;
            const long long rem = end - first;
            const uint32_t bytes = (uint32_t)((rem < kPTile ? rem : kPTile) * sizeof(PnpRec));
            mbar_expect_tx(&ws.full_bar[s], bytes);
            bulk_g2s(&ws.tile[s][0], a.pts + first, bytes, &ws.full_bar[s]);
        };
        if (lane == 0)
            for (int t = 0; t < kPStages && t < ntiles; ++t) issue(t);

        // this lane's hypotheses hyp_w + 32 j + lane; padding lanes hold P = 0 (p2 = 0: never an inlier)
        const long long hyp_w = (long long)hw * (32 * HPT);
        double pm[HPT][12];
        unsigned cw[HPT][kAccWords];
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = hyp_w + 32 * j + lane;
            double m[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) m[k] = hyp < a.h ? a.Rt[12 * hyp + k] : 0.0;
            pnp_projection(K, m, pm[j]);
#pragma unroll
            for (int k = 0; k < kAccWords; ++k) cw[j][k] = 0u;
        }

        for (int t = 0; t < ntiles; ++t) {
            const unsigned gti = gt + (unsigned)t;
            const int s = (int)(gti % kPStages);
            mbar_wait(&ws.full_bar[s], (gti / kPStages) & 1u);
            const long long first = begin + (long long)t * kPTile;
            const int np = (int)((end - first < kPTile) ? (end - first) : kPTile);
            const PnpRec* tp = &ws.tile[s][0];
            for (int p = 0; p < np; ++p) {
                const double X = tp[p].X, Y = tp[p].Y, Z = tp[p].Z, u = tp[p].u, v = tp[p].v;
#pragma unroll
                for (int j = 0; j < HPT; ++j) {
                    const PnpTerms r = pnp_terms(pm[j], X, Y, Z, u, v);
                    if (pnp_inlier(r, a.thr)) {
                        const double val = pnp_value(r);
                        unsigned ch[kChunks];
                        cw[j][0] += 1u;
                        if (a.sums & SUM_S1) {
                            chunks21(val, a.scale1, ch);
#pragma unroll
                            for (int kk = 0; kk < kChunks; ++kk) cw[j][1 + kk] += ch[kk];
                        }
                        if (a.sums & SUM_S2) {
                            chunks21(__dmul_rn(val, val), a.scale2, ch);
#pragma unroll
                            for (int kk = 0; kk < kChunks; ++kk) cw[j][1 + kChunks + kk] += ch[kk];
                        }
                    }
                }
            }
            __syncwarp();  // every lane is done with the stage: refill it
            if (lane == 0 && t + kPStages < ntiles) issue(t + kPStages);
        }
        gt += (unsigned)ntiles;
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = hyp_w + 32 * j + lane;
            if (cw[j][0]) {  // only real hypotheses can have inliers
#pragma unroll
                for (int k = 0; k < kAccWords; ++k)
                    if (cw[j][k]) atomicAdd(a.acc + (long long)k * a.h + hyp, (unsigned long long)cw[j][k]);
            }
        }
    }
}

// K3's view of a PnP hypothesis: P formed once per load
template <> struct ExactModel<MODEL_P> {
    using Rec = PnpRec;
    static constexpr int kSample = 4;
    static constexpr int kStride = 12;
    double P[12];
    __device__ __forceinline__ void load(const double* m, const double* K) { pnp_projection(K, m, P); }
    __device__ __forceinline__ bool eval(const PnpRec& c, double thr, double& v) const { return pnp_exact(P, c, thr, v); }
};

// K4 for PnP: the pinned decision and value of every record under one [R | t] - the winner of the last estimate
// (best != null: taken straight from K3's output, and copied to winner_out by thread 0) or a caller-supplied pose.
__global__ void k_pnp_mask(const PnpRec* __restrict__ pts, long long n, const double* __restrict__ K,
                           const double* __restrict__ Rt, const Best* __restrict__ best, double thr,
                           uint8_t* __restrict__ mask, double* __restrict__ err, double* __restrict__ winner_out) {
    chain_enter();
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long local = best ? best->idx : 0;
    if (winner_out && i == 0)
        for (int k = 0; k < 12; ++k) winner_out[k] = local >= 0 ? Rt[12 * local + k] : 0.0;
    if (i >= n) return;
    if (local < 0) {
        mask[i] = 0;
        err[i] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    double P[12];
    pnp_projection(K, Rt + 12 * local, P);
    double v;
    mask[i] = pnp_exact(P, pts[i], thr, v) ? 1 : 0;
    err[i] = v;
}

}  // namespace sfm
