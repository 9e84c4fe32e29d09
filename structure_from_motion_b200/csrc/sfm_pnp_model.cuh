// The PnP model's evaluation, shared by the RANSAC kernels (sfm_pnp.cuh) and the refinement (sfm_refine.cuh): the
// record, P = K [R | t] and the pinned decision and value of one record (see sfm_pnp.cuh for the rule).  No kernels, so
// any translation unit may include it.
#pragma once
#include <cuda_runtime.h>

namespace sfm {

// One PnP record, 48 B (16-byte aligned for the bulk-async tile copies)
struct __align__(16) PnpRec {
    double X, Y, Z, u, v, pad;
};
static_assert(sizeof(PnpRec) == 48, "PnpRec must be 48 bytes");

constexpr double kPnpCollinear = 1e-6;  // sine of the angle at X0 below which three world points are collinear
constexpr double kPnpOrthonormal = 1e-6;  // largest |R R^T - I| entry of a valid sample's chosen R
constexpr int kPnpMinDepthHi = 0x1e600000;  // high word of 2^-537, the smallest p2 whose square W is not 0

// P = K [R | t] in the pinned order (see the header)
__device__ __forceinline__ void pnp_projection(const double* K, const double* m, double (&P)[12]) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c)
            P[4 * r + c] = __fma_rn(K[3 * r + 0], m[c], __fma_rn(K[3 * r + 1], m[4 + c], __dmul_rn(K[3 * r + 2], m[8 + c])));
}

struct PnpTerms {
    double F, W, p2;
};
__device__ __forceinline__ PnpTerms pnp_terms(const double (&P)[12], double X, double Y, double Z, double u, double v) {
    const double p0 = __fma_rn(P[0], X, __fma_rn(P[1], Y, __fma_rn(P[2], Z, P[3])));
    const double p1 = __fma_rn(P[4], X, __fma_rn(P[5], Y, __fma_rn(P[6], Z, P[7])));
    const double p2 = __fma_rn(P[8], X, __fma_rn(P[9], Y, __fma_rn(P[10], Z, P[11])));
    const double d0 = __fma_rn(-u, p2, p0), d1 = __fma_rn(-v, p2, p1);
    PnpTerms r;
    r.F = __fma_rn(d0, d0, __dmul_rn(d1, d1));
    r.W = __dmul_rn(p2, p2);
    r.p2 = p2;
    return r;
}
// p2 >= 2^-537 and F < inf are tested on the high words, as integers: no FP64 issue slot
__device__ __forceinline__ bool pnp_inlier(const PnpTerms& r, double thr) {
    return __double2hiint(r.p2) >= kPnpMinDepthHi && __double2hiint(r.F) < 0x7ff00000 && r.F <= __dmul_rn(thr, r.W);
}
__device__ __forceinline__ double pnp_value(const PnpTerms& r) { return __ddiv_rn(r.F, r.W); }
__device__ __forceinline__ bool pnp_exact(const double (&P)[12], const PnpRec& c, double thr, double& value) {
    const PnpTerms r = pnp_terms(P, c.X, c.Y, c.Z, c.u, c.v);
    value = pnp_value(r);
    return pnp_inlier(r, thr);
}

}  // namespace sfm
