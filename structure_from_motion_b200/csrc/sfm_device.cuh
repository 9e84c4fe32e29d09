// Device-side building blocks of the two-view geometry hot path (sm_100a).
//
// Every routine restates a piece of Bazs/structure_from_motion (citations are
// reference-repo paths); nothing here is translated from it — the reference is pure
// numpy/LAPACK, these are hand-written fp64 CUDA routines.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sfm {

// Programmatic dependent launch (sm_90+): the kernels of one estimate form a chain on one stream, each launched with
// cudaLaunchAttributeProgrammaticStreamSerialization.  chain_enter() is the first statement of every chain kernel:
// wait until the preceding grid has completed and its memory is visible (a no-op for an ordinary launch), then let
// the NEXT kernel of the chain be launched - its blocks become resident as resources free up and sit in their own
// wait, so the launch latency of a kernel overlaps the execution of its predecessor.
__device__ __forceinline__ void chain_enter() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
}


constexpr double kVerySmall = 1e-10;            // lib/epipolar/eight_point.py:415
constexpr double kCheiralityTolerance = 1e-8;   // lib/epipolar/eight_point.py:477

// One correspondence in K-normalised coordinates, 32 B, the unit staged through
// shared memory by the scoring kernel.
struct __align__(32) Corr {
    double xa, ya, xb, yb;
};

// One model padded to 96 bytes = three 32-byte sectors: the survivor path gathers a candidate's row with three
// 256-bit loads (one sector each) instead of nine 8-byte loads that straddle 3-4 sectors - the gather was the
// L1TEX-bound part of the drain (ncu at a 7 % inlier rate: l1tex 76 % busy).
struct __align__(32) ModelRow {
    double4 a, b, c;  // e0..e3 | e4..e7 | e8, pad
};
static_assert(sizeof(ModelRow) == 96, "ModelRow must be three sectors");

__device__ __forceinline__ void store_model_row(ModelRow* rows, long long i, const double (&e)[9], bool ok) {
    ModelRow r;
    r.a = ok ? make_double4(e[0], e[1], e[2], e[3]) : make_double4(0.0, 0.0, 0.0, 0.0);
    r.b = ok ? make_double4(e[4], e[5], e[6], e[7]) : make_double4(0.0, 0.0, 0.0, 0.0);
    r.c = make_double4(ok ? e[8] : 0.0, 0.0, 0.0, 0.0);
    rows[i] = r;
}

// ------------------------------------------------------------------------------------
// Symmetric epipolar distance — lib/epipolar/sed.py:7-30
// ------------------------------------------------------------------------------------
// Exact form: the evaluation order numpy+OpenBLAS use for sed.py:21-29 (SURVEY.md
// Appendix B), pinned with explicit intrinsics so that no call site is re-contracted by
// the compiler.  e is row-major E.  Used for every inlier decision and every error term.
__device__ __forceinline__ double sed_exact(const double (&e)[9], double xa, double ya, double xb,
                                            double yb) {
    const double lb0 = __dadd_rn(__fma_rn(yb, e[3], __dmul_rn(xb, e[0])), e[6]);
    const double lb1 = __dadd_rn(__fma_rn(yb, e[4], __dmul_rn(xb, e[1])), e[7]);
    const double lb2 = __dadd_rn(__fma_rn(yb, e[5], __dmul_rn(xb, e[2])), e[8]);
    const double la0 = __dadd_rn(__fma_rn(e[0], xa, __dmul_rn(e[1], ya)), e[2]);
    const double la1 = __dadd_rn(__fma_rn(e[3], xa, __dmul_rn(e[4], ya)), e[5]);
    const double r = __dadd_rn(__fma_rn(lb1, ya, __dmul_rn(lb0, xa)), lb2);
    const double na = __dadd_rn(__dmul_rn(la0, la0), __dmul_rn(la1, la1));
    const double nb = __dadd_rn(__dmul_rn(lb0, lb0), __dmul_rn(lb1, lb1));
    // __drcp_rn is the correctly rounded reciprocal: bit-identical to the IEEE division 1.0 / x
    return __dmul_rn(__dadd_rn(__drcp_rn(na), __drcp_rn(nb)), __dmul_rn(r, r));
}

// Full division-free decision, 21 FP64 issue slots: d = r^2 (na+nb) - thr_pre na nb.
__device__ __forceinline__ double sed_full_decision(const double (&e)[9], double xa, double ya,
                                                    double xb, double yb, double thr_pre) {
    const double lb0 = fma(xb, e[0], fma(yb, e[3], e[6]));
    const double lb1 = fma(xb, e[1], fma(yb, e[4], e[7]));
    const double lb2 = fma(xb, e[2], fma(yb, e[5], e[8]));
    const double la0 = fma(e[0], xa, fma(e[1], ya, e[2]));
    const double la1 = fma(e[3], xa, fma(e[4], ya, e[5]));
    const double r = fma(xa, lb0, fma(ya, lb1, lb2));
    const double na = fma(la0, la0, la1 * la1);
    const double nb = fma(lb0, lb0, lb1 * lb1);
    const double t = thr_pre * (na * nb);
    return fma(r * r, na + nb, -t);
}

// ------------------------------------------------------------------------------------
// Homography transfer error (sfm_homography.cuh; oracle: oracle_transfer_exact in oracle/transfer_exact.c)
// ------------------------------------------------------------------------------------
// adj(H) maps image-B points back to image A without a division.  Pinned order: every model consumer (fit, scorer,
// K3, mask) recomputes it from H with these nine fma's, so all of them see the same bits.
__device__ __forceinline__ void homography_adj(const double (&h)[9], double (&a)[9]) {
    a[0] = __fma_rn(h[4], h[8], -__dmul_rn(h[5], h[7]));
    a[1] = __fma_rn(h[2], h[7], -__dmul_rn(h[1], h[8]));
    a[2] = __fma_rn(h[1], h[5], -__dmul_rn(h[2], h[4]));
    a[3] = __fma_rn(h[5], h[6], -__dmul_rn(h[3], h[8]));
    a[4] = __fma_rn(h[0], h[8], -__dmul_rn(h[2], h[6]));
    a[5] = __fma_rn(h[2], h[3], -__dmul_rn(h[0], h[5]));
    a[6] = __fma_rn(h[3], h[7], -__dmul_rn(h[4], h[6]));
    a[7] = __fma_rn(h[1], h[6], -__dmul_rn(h[0], h[7]));
    a[8] = __fma_rn(h[0], h[4], -__dmul_rn(h[1], h[3]));
}

// The four squared terms of the symmetric transfer error of one correspondence (pixel coordinates):
// p = H (xa, ya, 1), q = adj(H) (xb, yb, 1), F = (p0 - xb p2)^2 + (p1 - yb p2)^2, G = (q0 - xa q2)^2 + (q1 - ya q2)^2,
// P = p2^2, Q = q2^2.  22 FP64 issue slots.
struct TransferTerms {
    double F, G, P, Q;
    bool finite_w;  // p2 != 0 && q2 != 0 (tested on the bit patterns: integer pipe, same truth table)
};
__device__ __forceinline__ TransferTerms transfer_terms(const double (&h)[9], const double (&a)[9], double xa, double ya,
                                                        double xb, double yb) {
    const double p0 = __fma_rn(h[0], xa, __fma_rn(h[1], ya, h[2]));
    const double p1 = __fma_rn(h[3], xa, __fma_rn(h[4], ya, h[5]));
    const double p2 = __fma_rn(h[6], xa, __fma_rn(h[7], ya, h[8]));
    const double q0 = __fma_rn(a[0], xb, __fma_rn(a[1], yb, a[2]));
    const double q1 = __fma_rn(a[3], xb, __fma_rn(a[4], yb, a[5]));
    const double q2 = __fma_rn(a[6], xb, __fma_rn(a[7], yb, a[8]));
    const double u = __fma_rn(-xb, p2, p0), v = __fma_rn(-yb, p2, p1);
    const double s = __fma_rn(-xa, q2, q0), t = __fma_rn(-ya, q2, q1);
    TransferTerms r;
    r.F = __fma_rn(u, u, __dmul_rn(v, v));
    r.G = __fma_rn(s, s, __dmul_rn(t, t));
    r.P = __dmul_rn(p2, p2);
    r.Q = __dmul_rn(q2, q2);
    r.finite_w = ((__double_as_longlong(p2) << 1) != 0) && ((__double_as_longlong(q2) << 1) != 0);
    return r;
}
// inlier decision, division-free: F Q + G P <= (thr P) Q  (+4 slots: 26 in all, plus the compare)
__device__ __forceinline__ bool transfer_inlier(const TransferTerms& r, double thr) {
    return r.finite_w && (__fma_rn(r.F, r.Q, __dmul_rn(r.G, r.P)) <= __dmul_rn(__dmul_rn(thr, r.P), r.Q));
}
// the error in px^2: F / P + G / Q
__device__ __forceinline__ double transfer_value(const TransferTerms& r) {
    return __dadd_rn(__ddiv_rn(r.F, r.P), __ddiv_rn(r.G, r.Q));
}
// decision and value together (K3's sample rule and rescore, the mask kernel)
__device__ __forceinline__ bool transfer_exact(const double (&h)[9], const double (&a)[9], double xa, double ya, double xb,
                                               double yb, double thr, double& value) {
    const TransferTerms r = transfer_terms(h, a, xa, ya, xb, yb);
    value = transfer_value(r);
    return transfer_inlier(r, thr);
}

// ------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) — counter-based generator for the device sampler
// ------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                       uint32_t c3, uint32_t k0, uint32_t k1,
                                                       uint32_t (&out)[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 8 distinct indices uniform in [0, n): draw-and-reject, the same distribution as the first
// 8 entries of a uniform permutation (what lib/ransac/ransac.py:62-63 samples).
__host__ __device__ inline void philox_sample8(uint64_t seed, uint64_t stream, uint64_t hyp,
                                               uint32_t n, int32_t (&idx)[8]) {
    uint32_t draw = 0;
    int got = 0;
    while (got < 8) {
        uint32_t o[4];
        philox4x32_10((uint32_t)hyp, (uint32_t)(hyp >> 32), draw++, (uint32_t)stream,
                      (uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(stream >> 32), o);
#pragma unroll
        for (int w = 0; w < 2 && got < 8; ++w) {
            const uint64_t r64 = ((uint64_t)o[2 * w] << 32) | o[2 * w + 1];
#if defined(__CUDA_ARCH__)
            const uint32_t cand = (uint32_t)__umul64hi(r64, (uint64_t)n);
#else
            const uint32_t cand = (uint32_t)(((unsigned __int128)r64 * n) >> 64);
#endif
            bool dup = false;
            for (int j = 0; j < got; ++j) dup |= (idx[j] == (int32_t)cand);
            if (!dup) idx[got++] = (int32_t)cand;
        }
    }
}

}  // namespace sfm
