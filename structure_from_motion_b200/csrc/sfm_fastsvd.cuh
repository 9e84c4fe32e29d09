// Short-latency replacements for two small SVDs of the tail.  Both run in one thread, in registers, with a handful
// of dependent sqrt/divide steps instead of the ~40 rotations of a Jacobi sweep sequence (each rotation is a chain
// of divide, sqrt, divide, rsqrt): the tail of a config-3 estimate handles ~100 inliers, so its kernels are pure
// latency and the SVD chain WAS that latency (36 + 30 + 9 us per estimate).
//
//   null_vector4_fast   right singular vector of the smallest singular value of a 4x4 matrix (the DLT system of
//                       lib/epipolar/triangulation.py:34-35): Householder QR, then inverse iteration on R^T R through
//                       the triangular factor (never forming A^T A: backward stable like an SVD, but the absolute stop
//                       below adds up to ~8e-13 q / (1 - q), q = (sigma4 / sigma3)^4, to the eps * sigma1 / gap of one).
//                       Convergence is checked; the caller falls back to the Jacobi SVD when 40 steps do not suffice
//                       (sigma4 close to sigma3: a correspondence whose rays do not meet - never an inlier).
//   svd3_rank2_frames   U, V of a 3x3 matrix with a (numerically) zero third singular value - what
//                       _recover_all_r_t (lib/epipolar/eight_point.py:245-280) takes from np.linalg.svd(E): the null
//                       vectors are cross products, the remaining 2x2 symmetric eigenproblem is one closed-form rotation.
//
// Host-callable too (plain fma/sqrt), so that tools/fastsvd_check.cu can compare them with LAPACK-grade references
// on the CPU.
#pragma once
#include <cmath>
#include <cuda_runtime.h>

namespace sfm {

__host__ __device__ __forceinline__ double inv_sqrt(double x) {
#ifdef __CUDA_ARCH__
    return rsqrt(x);
#else
    return 1.0 / std::sqrt(x);
#endif
}

// g: row-major 4x4.  On success x holds the unit null-ish vector (sign arbitrary but fixed) and true is returned;
// false = not converged within the iteration budget (use the SVD).
__host__ __device__ inline bool null_vector4_fast(const double (&g)[16], double (&x)[4]) {
    double r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = g[i];
    // Householder QR, columns 0..2 (only R is kept)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double s = 0.0;
#pragma unroll
        for (int i = k; i < 4; ++i) s = fma(r[i * 4 + k], r[i * 4 + k], s);
        const double nrm = sqrt(s);
        const double akk = r[k * 4 + k];
        const double alpha = (akk > 0.0) ? -nrm : nrm;
        const double v0 = akk - alpha;                  // no cancellation: same sign
        const double vn = fma(-akk, alpha, s);          // v.v / 2 = s + |akk| nrm
        const double beta = (vn > 0.0) ? 1.0 / vn : 0.0;
#pragma unroll
        for (int j = k + 1; j < 4; ++j) {
            double dot = v0 * r[k * 4 + j];
#pragma unroll
            for (int i = k + 1; i < 4; ++i) dot = fma(r[i * 4 + k], r[i * 4 + j], dot);
            const double w = dot * beta;
            r[k * 4 + j] = fma(-w, v0, r[k * 4 + j]);
#pragma unroll
            for (int i = k + 1; i < 4; ++i) r[i * 4 + j] = fma(-w, r[i * 4 + k], r[i * 4 + j]);
        }
        r[k * 4 + k] = alpha;
    }
    // reciprocal diagonal; an exactly (or numerically) singular R - noise-free data - gets a pivot at rounding level
    double big = fmax(fmax(fabs(r[0]), fabs(r[5])), fmax(fabs(r[10]), fabs(r[15])));
    if (!(big > 0.0) || !(big < 1e150)) return false;
    const double tiny = 1e-15 * big;
    double rinv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double d = r[i * 5];
        if (fabs(d) < tiny) d = (d < 0.0) ? -tiny : tiny;
        rinv[i] = 1.0 / d;
    }
    auto solve = [&](double (&v)[4]) {  // v <- R^-1 R^-T v
        double z0 = v[0] * rinv[0];
        double z1 = fma(-r[1], z0, v[1]) * rinv[1];
        double z2 = fma(-r[6], z1, fma(-r[2], z0, v[2])) * rinv[2];
        double z3 = fma(-r[11], z2, fma(-r[7], z1, fma(-r[3], z0, v[3]))) * rinv[3];
        const double y3 = z3 * rinv[3];
        const double y2 = fma(-r[11], y3, z2) * rinv[2];
        const double y1 = fma(-r[7], y3, fma(-r[6], y2, z1)) * rinv[1];
        const double y0 = fma(-r[3], y3, fma(-r[2], y2, fma(-r[1], y1, z0))) * rinv[0];
        v[0] = y0; v[1] = y1; v[2] = y2; v[3] = y3;
    };
    auto normalise = [&](double (&v)[4]) {
        const double n2 = fma(v[3], v[3], fma(v[2], v[2], fma(v[1], v[1], v[0] * v[0])));
        const double s = inv_sqrt(n2);
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] *= s;
    };
    double v[4] = {0.41, 0.27, 0.73, 1.0};
    // inverse iteration, convergence checked after step 4 and then every second step.  A real loop on purpose (not
    // unrolled): the tail kernels run this once per launch on ~100 inliers, where every straight-line instruction is a
    // cold instruction-cache miss - one copy of the step body executed a few times beats several copies executed once.
    // Inliers converge in 4-6 steps (error factor (sigma4 / sigma3)^2 per step); the candidate poses that put the point
    // near infinity (rays almost parallel: sigma3 small too) need more, and kMaxSteps of ~280 cycles each are still far
    // cheaper than the ~30 k cycles of the Jacobi SVD the caller falls back to.
    constexpr int kMaxSteps = 40;
    double prev[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
    for (int step = 1; step <= kMaxSteps; ++step) {
        const bool check = step >= 4 && (step & 1) == 0;
        if (check) {
#pragma unroll
            for (int i = 0; i < 4; ++i) prev[i] = v[i];
        }
        solve(v);
        normalise(v);
        if (check) {
            double diff = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) diff = fmax(diff, fabs(v[i] - prev[i]));
            if (diff <= 1e-13) {
#pragma unroll
                for (int i = 0; i < 4; ++i) x[i] = v[i];
                return true;
            }
        }
    }
    return false;
}

// A: row-major 3x3 with sigma3 ~ 0 (an essential matrix after the rank-2 projection of the fit).  Produces proper
// orthonormal U, V (det +1, third columns = the left / right null vectors) with A ~ U diag(s0, s1, 0) V^T, s0 >= s1.
// Returns false when the matrix is too far from rank 2 for the construction (the caller uses the Jacobi SVD).
__host__ __device__ inline bool svd3_rank2_frames(const double (&A)[9], double (&U)[9], double (&V)[9], double (&sv)[3]) {
    auto cross = [](const double* a, const double* b, double* c) {
        c[0] = fma(a[1], b[2], -a[2] * b[1]);
        c[1] = fma(a[2], b[0], -a[0] * b[2]);
        c[2] = fma(a[0], b[1], -a[1] * b[0]);
    };
    auto dot3 = [](const double* a, const double* b) { return fma(a[2], b[2], fma(a[1], b[1], a[0] * b[0])); };
    // right null vector: the largest of the three cross products of rows
    const double* r0 = A; const double* r1 = A + 3; const double* r2 = A + 6;
    double c01[3], c02[3], c12[3];
    cross(r0, r1, c01); cross(r0, r2, c02); cross(r1, r2, c12);
    const double n01 = dot3(c01, c01), n02 = dot3(c02, c02), n12 = dot3(c12, c12);
    const double* cb = c01;
    double nb = n01;
    if (n02 > nb) { cb = c02; nb = n02; }
    if (n12 > nb) { cb = c12; nb = n12; }
    if (!(nb > 0.0)) return false;
    double v2[3];
    {
        const double s = inv_sqrt(nb);
        v2[0] = cb[0] * s; v2[1] = cb[1] * s; v2[2] = cb[2] * s;
    }
    // an orthonormal basis (p, q) of the plane orthogonal to v2
    double p[3], q[3];
    {
        const double ax = fabs(v2[0]), ay = fabs(v2[1]), az = fabs(v2[2]);
        double e[3] = {0.0, 0.0, 0.0};
        if (ax <= ay && ax <= az) e[0] = 1.0; else if (ay <= az) e[1] = 1.0; else e[2] = 1.0;
        cross(v2, e, p);
        const double s = inv_sqrt(dot3(p, p));
        p[0] *= s; p[1] *= s; p[2] *= s;
        cross(v2, p, q);
    }
    // B = [A p, A q] (3x2); its Gram matrix is 2x2 symmetric: one closed-form rotation diagonalises it
    double ap[3], aq[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { ap[i] = dot3(A + 3 * i, p); aq[i] = dot3(A + 3 * i, q); }
    const double gpp = dot3(ap, ap), gqq = dot3(aq, aq), gpq = dot3(ap, aq);
    double cs = 1.0, sn = 0.0;
    if (gpq != 0.0) {
        const double d = gqq - gpp;
        const double t = (2.0 * gpq) * ((d >= 0.0) ? 1.0 : -1.0) / (fabs(d) + sqrt(fma(d, d, 4.0 * gpq * gpq)));
        cs = inv_sqrt(fma(t, t, 1.0));
        sn = t * cs;
    }
    // rotated pair: a = cs ap - sn aq, b = sn ap + cs aq  (orthogonal), v likewise
    double a[3], b[3], va[3], vb[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        a[i] = fma(cs, ap[i], -sn * aq[i]); b[i] = fma(sn, ap[i], cs * aq[i]);
        va[i] = fma(cs, p[i], -sn * q[i]); vb[i] = fma(sn, p[i], cs * q[i]);
    }
    double na = dot3(a, a), nbb = dot3(b, b);
    if (na < nbb) {  // descending singular values: swap the pair (keeps the handedness with a sign flip below)
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double t1 = a[i]; a[i] = b[i]; b[i] = t1;
            double t2 = va[i]; va[i] = vb[i]; vb[i] = t2;
        }
        const double t3 = na; na = nbb; nbb = t3;
    }
    if (!(nbb > 0.0)) return false;  // rank 1: no unique frame
    const double s0 = sqrt(na), s1 = sqrt(nbb);
    double u0[3], u1[3], u2[3];
    {
        const double i0 = 1.0 / s0;
        u0[0] = a[0] * i0; u0[1] = a[1] * i0; u0[2] = a[2] * i0;
        // u1: b orthogonalised against u0 (they are orthogonal up to rounding), normalised
        const double pr = dot3(b, u0);
        double w[3] = {fma(-pr, u0[0], b[0]), fma(-pr, u0[1], b[1]), fma(-pr, u0[2], b[2])};
        const double i1 = inv_sqrt(dot3(w, w));
        u1[0] = w[0] * i1; u1[1] = w[1] * i1; u1[2] = w[2] * i1;
        cross(u0, u1, u2);
    }
    // proper V: third column = va x vb (= +-v2)
    double v3[3];
    cross(va, vb, v3);
    // the neglected third singular value: |A v3| must be at rounding level relative to s0 for this route
    double av3[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) av3[i] = dot3(A + 3 * i, v3);
    const double s2 = sqrt(dot3(av3, av3));
    if (!(s2 <= 1e-8 * s0)) return false;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        U[3 * i] = u0[i]; U[3 * i + 1] = u1[i]; U[3 * i + 2] = u2[i];
        V[3 * i] = va[i]; V[3 * i + 1] = vb[i]; V[3 * i + 2] = v3[i];
    }
    // the reported sigma3: |A v3| is the null vector's residual of two rows only - for A of rank 3 it overstates
    // sigma3 by up to sqrt(3) (|A v3| = |det A| / |r_i x r_j| with |r_i x r_j| >= s0 s1 / sqrt(3)).  Its component
    // along u2, normal to A p and A q, is |det A| / |A p x A q| = sigma3 to rounding (|A p x A q| = s0 s1 up to
    // O(sigma3^2)), which is what the caller's absolute test against 1e-8 needs
    sv[0] = s0; sv[1] = s1; sv[2] = fabs(dot3(u2, av3));
    return true;
}

}  // namespace sfm
