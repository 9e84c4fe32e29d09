// Host build of refine_p_residuals (csrc/sfm_refine.cuh), for tests/test_pnp_refine_oracle.py.  P = K [R | t] in
// pnp_projection's order (std::fma on the host rounds as __fma_rn does on the device).
#include <cmath>

#include "../structure_from_motion_b200/csrc/sfm_refine.cuh"
extern "C" void p_projection(const double* K, const double* Rt, double* P) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c)
            P[4 * r + c] = std::fma(K[3 * r + 0], Rt[c], std::fma(K[3 * r + 1], Rt[4 + c], K[3 * r + 2] * Rt[8 + c]));
}
extern "C" double p_residuals(const double* P, const double* K, const double* rec, double* r, double* J) {
    double rr[2], JJ[2][6];
    const double p2 = sfm::refine_p_residuals(P, K, rec[0], rec[1], rec[2], rec[3], rec[4], rr, JJ);
    for (int i = 0; i < 2; ++i) {
        r[i] = rr[i];
        for (int k = 0; k < 6; ++k) J[6 * i + k] = JJ[i][k];
    }
    return p2;
}
