// Host build of the __host__ __device__ helpers of csrc/sfm_refine.cuh, for tests/test_refine_exact_oracle.py.
#include "../structure_from_motion_b200/csrc/sfm_refine.cuh"
extern "C" void e_model(const double* R, const double* t, double* E, double* M) { double e[9], m[45]; sfm::refine_e_model(R, t, e, m); for (int i = 0; i < 9; ++i) E[i] = e[i]; for (int i = 0; i < 45; ++i) M[i] = m[i]; }
extern "C" double e_residual(const double* E, const double* c, double* g) { double gE[9]; const double r = sfm::refine_e_residual(E, c[0], c[1], c[2], c[3], gE); for (int i = 0; i < 9; ++i) g[i] = gE[i]; return r; }
extern "C" void h_residuals(const double* h, const double* c, double* r, double* J) { double rr[4], JJ[4][8]; sfm::refine_h_residuals(h, c[0], c[1], c[2], c[3], rr, JJ); for (int i = 0; i < 4; ++i) { r[i] = rr[i]; for (int k = 0; k < 8; ++k) J[8 * i + k] = JJ[i][k]; } }
extern "C" void rotate(const double* R, const double* w, double* out) { sfm::refine_rotate(R, w, out); }
extern "C" void tangent_basis(const double* t, double* b1, double* b2) { sfm::refine_tangent_basis(t, b1, b2); }
