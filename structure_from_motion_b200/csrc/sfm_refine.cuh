// Opt-in least-squares refinement of a RANSAC winner over its inliers (Levenberg-Marquardt, FP64), between the
// selection and the pose tail.  One image pair per blockIdx.y, as in the tail.
//
// Data.  The fixed inlier list T1 (k_tail_mask) compacted for the winner: E: sed <= thr plus the 8 samples, H: the
// transfer decision plus the 4 samples.  The list does not change during the refinement.
//
// Cost.  The sum over that list of the per-correspondence error RANSAC scored:
//   E: the symmetric epipolar distance (K-normalised records), residual r = (b^T E a) sqrt(1/na + 1/nb), r^2 = sed;
//   H: the symmetric transfer error in px^2 (pixel records), four residuals pi(H a) - b and pi(adj(H) b) - a,
//      whose squares sum to F/P + G/Q of transfer_terms.
// Both are invariant to the scale of the model.
//
// Parameters.  E = [t]x R on the essential manifold: R <- R exp([w]x), the unit t moves by (b1, b2) in its tangent
// plane (b1 = t x e_k / |t x e_k|, e_k the axis of t's smallest component, b2 = t x b1), then is renormalised: 5
// parameters.  The start is candidate 0 of decompose_essential of the RANSAC E (its projection onto the manifold).
// Which rotation of the twisted pair is candidate 0 matters: [t]x R1 = -[t]x R2, but the tangent moves of t are taken
// against R, so the two charts give different steps (oracle/refine_exact.py replays from the device's candidate).
// H: h0..h7 with h8 = 1 held fixed: 8 parameters.
//
// Solver (fixed control).  The normal equations J^T J, J^T r of the last accepted point are kept per pair.  A step
// solves (J^T J + lambda diag(J^T J)) d = -J^T r (Marquardt's damping: invariant to the scale of every parameter, so
// pixel-sized H entries need no conditioning) by Cholesky of the unit-diagonal scaled system.  lambda starts at
// kRefineLambda0; an evaluated proposal whose cost is strictly lower is accepted and lambda /= 10, else it is rejected
// and lambda *= 10 (the next step is re-solved from the stored equations).  Stops: converged when an accepted step
// lowers the cost by a relative kRefineFtol or less, when the cost is at most kRefineCostFloor times the sum of the
// squared coordinates of the list (an RMS residual below 1e-12 of the data's scale: rounding noise, e.g. a homography
// through its own 4 samples), or when the scaled step |D d| (D = the square
// roots of diag(J^T J): the first-order change of the residual vector) is at most kRefineXtol sqrt(cost); stalled when
// lambda exceeds kRefineLambdaCap; iteration cap after `max_iter` evaluated proposals.  The final cost is the cost of the
// last accepted point, never above the start's.  An empty list has cost 0 at the floor 0: converged at iteration 0,
// the start (E: the projected RANSAC or caller E) reported as the refined model.
//
// Determinism.  Each launch sums per-correspondence terms over fixed chunks of kRefineChunk list entries (thread t
// takes entries t and t + 128 of the chunk, in that order; warps reduce with a fixed butterfly and the four warp sums
// are added in warp order), blocks grid-stride over chunks, and the pair's last block adds the chunk partials in chunk
// order.  The bits depend on the inlier list alone: not on the grid, the number of pairs or the run.
//
// Kernels: k_refine_init (start point, per-pair state), k_refine_step (one LM iteration per launch: evaluate the
// proposal, then the last block accepts or rejects it and writes the next one; a finished pair makes every later
// launch exit at once), k_refine_finish (the refined selection record - the winner's index, sample row -1 - and the
// per-pair report).  All are chain kernels (programmatic dependent launch); the host enqueues max_iter + 1 steps
// without a round trip.
//
// MODEL_P, the absolute pose [R | t] of a new view (sfm_refine_pnp; one pose, npairs = 1, PnpRec records):
//   list   k_refine_list compacts, in ascending record order, the records whose pnp_exact decision passes under the
//          start pose at thr, plus up to 4 forced indices (the RANSAC winner's sample, or a caller's); decoupled
//          look-back as in k_tail_mask, so the list - and with it every sum - does not depend on the grid.
//   cost   the sum over the list of the squared reprojection error, two residuals per record: r0 = p0 / p2 - u,
//          r1 = p1 / p2 - v, p = P (X, 1), P = K [R | t] formed by pnp_projection and p by pnp_terms' FMA order
//          (refine_p_residuals).  Cheirality guard: a proposal under which a list record has p2 < 2^-537 (the scorer's
//          depth rule) or a non-finite residual costs +inf and is rejected; at the start point that is `nonfinite`
//          and the start pose is kept.  cost_ransac is the scorer's F / W summed under the unprojected start.
//   model  R <- R exp([w]x) (refine_rotate), t <- t + dt: 6 parameters.  The start is the nearest rotation to the given
//          R (one-sided Jacobi SVD, U's smallest column replaced so that det = +1) with the given t.  The cost floor
//          is kRefineCostFloor times the sum of u^2 + v^2 over the list.
//   report PnpRefineReport: the refined [R | t] (the unprojected start when not refined), the costs, the list length,
//          iterations, status, rejected.  An empty list is converged at iteration 0 with cost 0 and the projected
//          start.  The control is refine_control unchanged.
// Scaling the world by 2^k (t with it) or the pixels and K's first two rows by 2^k changes every sum by an exact power
// of two, and Marquardt's scaling cancels it: the report is bit-identical after exact rescaling while p2 stays above
// 2^-537 and no sum overflows.
#pragma once
#include "sfm_device.cuh"
#include "sfm_pnp_model.cuh"
#include "sfm_pose_math.cuh"
#include "sfm_types.h"

namespace sfm {

constexpr int kRefineBlock = 128;
constexpr int kRefineChunk = 2 * kRefineBlock;  // inlier-list entries per chunk partial
constexpr double kRefineLambda0 = 1e-3;
constexpr double kRefineLambdaFactor = 10.0;
constexpr double kRefineLambdaCap = 1e16;
constexpr double kRefineFtol = 1e-12;
constexpr double kRefineXtol = 1e-9;
constexpr double kRefineCostFloor = 1e-24;

enum { REFINE_CONVERGED = 0, REFINE_MAX_ITER = 1, REFINE_STALLED = 2, REFINE_NO_MODEL = 3, REFINE_NONFINITE = 4,
       REFINE_RUNNING = -1 };

template <int KIND> struct RefineDims;
template <> struct RefineDims<MODEL_E> { static constexpr int NP = 5; };
template <> struct RefineDims<MODEL_H> { static constexpr int NP = 8; };
template <> struct RefineDims<MODEL_P> { static constexpr int NP = 6; };
template <> struct RefineDims<MODEL_X> { static constexpr int NP = 3; };  // X of a track (sfm_tracks.cuh)
// partial sums: cost, cost of the RANSAC model (first evaluation only), sum of squared coordinates, J^T J upper triangle
// (row-major), J^T r
template <int KIND> __host__ __device__ constexpr int refine_nv() { return 3 + RefineDims<KIND>::NP * (RefineDims<KIND>::NP + 1) / 2 + RefineDims<KIND>::NP; }

struct RefineState {
    double x[12], px[12];   // accepted point, proposal: E and P: R[9], t[3]; H: h0..h7
    double A[64], g[8];     // J^T J (full, row-major NP x NP) and J^T r at the accepted point
    double cost, lambda, cost_ransac, cost_start;
    long long num;
    int iter, status, done, evals, rejected, pad;
};

// layout of sfm_refinement (include/sfm_b200.h)
struct RefineReport {
    double model[9];
    double cost_ransac, cost_start, cost_final;
    long long num;
    int iterations, status;
    int rejected, reserved;
};

// layout of sfm_pnp_refinement (include/sfm_b200.h)
struct PnpRefineReport {
    double Rt[12];
    double cost_ransac, cost_start, cost_final;
    long long num;
    int iterations, status;
    int rejected, reserved;
};

struct RefineArgs {
    const Corr* pts;              // E: K-normalised, H: pixel records
    const long long* offsets;     // [P+1] or null
    const SelectRecord* rec;      // [P] the RANSAC winners
    const long long* idx;         // T1's compacted inlier lists
    const long long* num;         // [P]
    RefineState* state;           // [P]
    double* partial;              // [n_total / kRefineChunk + P + 1][NV]: pair p's chunks from refine_chunk_base
    unsigned* ticket;             // [P] zero on entry and on exit
    int npairs, max_iter;
    SelectRecord* out_rec;        // [P]
    RefineReport* report;         // [P]
};

// MODEL_P's arguments: one pose (npairs 1; pts, offsets, rec, out_rec and report unused).  A type of its own, so that
// the E and H kernels keep their parameter block.
struct PnpRefineArgs : RefineArgs {
    const PnpRec* ppts;           // [n] the records
    long long n;
    const double* K;              // [9]
    const double* start;          // [12] the RANSAC winner or the caller's pose, row-major [R | t]
    const int32_t* forced;        // [4] list entries whatever their decision (-1 = none), or null
    double thr;
    unsigned long long* list_agg; // [ceil(n / kListPerBlock)] look-back state of k_refine_list, zero on entry and exit
    unsigned* list_ticket;        // [2] zero on entry and on exit
    long long* list_out;          // [n + 1] k_refine_list's list, then its length (what idx and num point at)
    double* pose_out;             // [12] the reported pose (k_pnp_mask's input)
    PnpRefineReport* preport;
};

template <int KIND> struct RefineArgsOf { using type = RefineArgs; };
template <> struct RefineArgsOf<MODEL_P> { using type = PnpRefineArgs; };

// ---- small 3x3 helpers (row-major) ----
__host__ __device__ __forceinline__ void refine_skew(const double* v, double (&S)[9]) {
    S[0] = 0.0;   S[1] = -v[2]; S[2] = v[1];
    S[3] = v[2];  S[4] = 0.0;   S[5] = -v[0];
    S[6] = -v[1]; S[7] = v[0];  S[8] = 0.0;
}
__host__ __device__ __forceinline__ void refine_mul3(const double* A, const double* B, double* C) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) C[3 * i + j] = fma(A[3 * i + 2], B[6 + j], fma(A[3 * i + 1], B[3 + j], A[3 * i] * B[j]));
}
__host__ __device__ __forceinline__ void refine_cross(const double* a, const double* b, double* c) {
    c[0] = fma(a[1], b[2], -a[2] * b[1]);
    c[1] = fma(a[2], b[0], -a[0] * b[2]);
    c[2] = fma(a[0], b[1], -a[1] * b[0]);
}

// orthonormal basis (b1, b2) of the tangent plane of the unit vector t
__host__ __device__ __forceinline__ void refine_tangent_basis(const double* t, double* b1, double* b2) {
    int k = 0;
    if (fabs(t[1]) < fabs(t[k])) k = 1;
    if (fabs(t[2]) < fabs(t[k])) k = 2;
    const double e[3] = {k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0};
    refine_cross(t, e, b1);
    const double s = 1.0 / sqrt(fma(b1[0], b1[0], fma(b1[1], b1[1], b1[2] * b1[2])));
    b1[0] *= s; b1[1] *= s; b1[2] *= s;
    refine_cross(t, b1, b2);
}

// E = [t]x R and its derivatives M[9][5] (row-major 9 x 5) with respect to (w0, w1, w2, beta1, beta2)
__host__ __device__ inline void refine_e_model(const double* R, const double* t, double (&E)[9], double (&M)[45]) {
    double T[9], G[9], D[9];
    refine_skew(t, T);
    refine_mul3(T, R, E);
    for (int k = 0; k < 3; ++k) {  // d/dw_k: [t]x R [e_k]x
        const double ek[3] = {k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0};
        refine_skew(ek, G);
        refine_mul3(E, G, D);
        for (int j = 0; j < 9; ++j) M[5 * j + k] = D[j];
    }
    double b1[3], b2[3];
    refine_tangent_basis(t, b1, b2);
    refine_skew(b1, G);
    refine_mul3(G, R, D);
    for (int j = 0; j < 9; ++j) M[5 * j + 3] = D[j];
    refine_skew(b2, G);
    refine_mul3(G, R, D);
    for (int j = 0; j < 9; ++j) M[5 * j + 4] = D[j];
}

// residual of one correspondence under E and its gradient with respect to the 9 entries of E
__host__ __device__ __forceinline__ double refine_e_residual(const double* E, double xa, double ya, double xb, double yb,
                                                             double (&gE)[9]) {
    const double a[3] = {xa, ya, 1.0}, b[3] = {xb, yb, 1.0};
    double la[3], lb[3];
    for (int j = 0; j < 3; ++j) {
        la[j] = fma(E[3 * j], xa, fma(E[3 * j + 1], ya, E[3 * j + 2]));  // (E a)_j
        lb[j] = fma(E[j], xb, fma(E[3 + j], yb, E[6 + j]));              // (E^T b)_j
    }
    const double s = fma(lb[0], xa, fma(lb[1], ya, lb[2]));
    const double na = fma(la[0], la[0], la[1] * la[1]), nb = fma(lb[0], lb[0], lb[1] * lb[1]);
    const double ia = 1.0 / na, ib = 1.0 / nb;
    const double w = sqrt(ia + ib);
    const double sw = s / w, ca = sw * ia * ia, cb = sw * ib * ib;
    for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k) {
            double v = w * b[j] * a[k];
            if (j < 2) v = fma(-ca * la[j], a[k], v);
            if (k < 2) v = fma(-cb * lb[k], b[j], v);
            gE[3 * j + k] = v;
        }
    return s * w;
}

// the four residuals of one correspondence under H (h[8] == 1) and their rows of the Jacobian over h0..h7
__host__ __device__ __forceinline__ void refine_h_residuals(const double* h, double xa, double ya, double xb, double yb,
                                                            double (&r)[4], double (&J)[4][8]) {
    const double p0 = fma(h[0], xa, fma(h[1], ya, h[2]));
    const double p1 = fma(h[3], xa, fma(h[4], ya, h[5]));
    const double p2 = fma(h[6], xa, fma(h[7], ya, h[8]));
    double ad[9];  // adj(H)
    ad[0] = fma(h[4], h[8], -h[5] * h[7]);
    ad[1] = fma(h[2], h[7], -h[1] * h[8]);
    ad[2] = fma(h[1], h[5], -h[2] * h[4]);
    ad[3] = fma(h[5], h[6], -h[3] * h[8]);
    ad[4] = fma(h[0], h[8], -h[2] * h[6]);
    ad[5] = fma(h[2], h[3], -h[0] * h[5]);
    ad[6] = fma(h[3], h[7], -h[4] * h[6]);
    ad[7] = fma(h[1], h[6], -h[0] * h[7]);
    ad[8] = fma(h[0], h[4], -h[1] * h[3]);
    const double q0 = fma(ad[0], xb, fma(ad[1], yb, ad[2]));
    const double q1 = fma(ad[3], xb, fma(ad[4], yb, ad[5]));
    const double q2 = fma(ad[6], xb, fma(ad[7], yb, ad[8]));
    const double ip = 1.0 / p2, iq = 1.0 / q2;
    const double u0 = p0 * ip, u1 = p1 * ip, v0 = q0 * iq, v1 = q1 * iq;
    r[0] = u0 - xb; r[1] = u1 - yb; r[2] = v0 - xa; r[3] = v1 - ya;
    // forward: d(p_i / p2)
    const double fa = xa * ip, fb = ya * ip;
    J[0][0] = fa;  J[0][1] = fb;  J[0][2] = ip;  J[0][3] = 0.0; J[0][4] = 0.0; J[0][5] = 0.0; J[0][6] = -u0 * fa; J[0][7] = -u0 * fb;
    J[1][0] = 0.0; J[1][1] = 0.0; J[1][2] = 0.0; J[1][3] = fa;  J[1][4] = fb;  J[1][5] = ip;  J[1][6] = -u1 * fa; J[1][7] = -u1 * fb;
    // backward: q = adj(H) b is quadratic in h; its derivatives over h0..h7 (h8 fixed)
    const double h8 = h[8];
    const double dq0[8] = {0.0, fma(-h8, yb, h[5]), fma(h[7], yb, -h[4]), 0.0, fma(h8, xb, -h[2]), fma(-h[7], xb, h[1]), 0.0,
                           fma(-h[5], xb, h[2] * yb)};
    const double dq1[8] = {fma(h8, yb, -h[5]), 0.0, fma(-h[6], yb, h[3]), fma(-h8, xb, h[2]), 0.0, fma(h[6], xb, -h[0]),
                           fma(h[5], xb, -h[2] * yb), 0.0};
    const double dq2[8] = {fma(-h[7], yb, h[4]), fma(h[6], yb, -h[3]), 0.0, fma(h[7], xb, -h[1]), fma(-h[6], xb, h[0]), 0.0,
                           fma(-h[4], xb, h[1] * yb), fma(h[3], xb, -h[0] * yb)};
    for (int k = 0; k < 8; ++k) {
        J[2][k] = fma(-v0, dq2[k], dq0[k]) * iq;
        J[3][k] = fma(-v1, dq2[k], dq1[k]) * iq;
    }
}

// R exp([w]x) (Rodrigues)
__host__ __device__ inline void refine_rotate(const double* R, const double* w, double* out) {
    const double th2 = fma(w[0], w[0], fma(w[1], w[1], w[2] * w[2]));
    const double th = sqrt(th2);
    double A, B;
    if (th < 1e-4) {
        A = 1.0 - th2 / 6.0;
        B = 0.5 - th2 / 24.0;
    } else {
        A = sin(th) / th;
        B = (1.0 - cos(th)) / th2;
    }
    double W[9], W2[9], X[9];
    refine_skew(w, W);
    refine_mul3(W, W, W2);
    for (int j = 0; j < 9; ++j) X[j] = fma(B, W2[j], A * W[j]) + ((j % 4) == 0 ? 1.0 : 0.0);
    refine_mul3(R, X, out);
}

// The two reprojection residuals of one PnP record under P = K [R | t] (pnp_projection) and their rows of the Jacobian
// over (w0, w1, w2, t0, t1, t2) of R <- R exp([w]x), t <- t + dt.  p = P (X, 1) in pnp_terms' FMA order; dp/dw_k =
// K R (e_k x X), and K R is P's left 3 x 3 block; dp/dt_k = K e_k.  Then d(p_i / p2) = (dp_i - (p_i / p2) dp2) / p2.
// Returns p2 (the cheirality guard tests it).
__host__ __device__ __forceinline__ double refine_p_residuals(const double* P, const double* K, double X, double Y,
                                                              double Z, double u, double v, double (&r)[2],
                                                              double (&J)[2][6]) {
    const double p0 = fma(P[0], X, fma(P[1], Y, fma(P[2], Z, P[3])));
    const double p1 = fma(P[4], X, fma(P[5], Y, fma(P[6], Z, P[7])));
    const double p2 = fma(P[8], X, fma(P[9], Y, fma(P[10], Z, P[11])));
    const double ip = 1.0 / p2;
    const double u0 = p0 * ip, u1 = p1 * ip;
    r[0] = u0 - u;
    r[1] = u1 - v;
    double dp[3][6];
    for (int i = 0; i < 3; ++i) {
        const double* Pi = P + 4 * i;
        dp[i][0] = fma(Pi[2], Y, -Pi[1] * Z);  // e_0 x X = (0, -Z, Y)
        dp[i][1] = fma(Pi[0], Z, -Pi[2] * X);  // e_1 x X = (Z, 0, -X)
        dp[i][2] = fma(Pi[1], X, -Pi[0] * Y);  // e_2 x X = (-Y, X, 0)
        dp[i][3] = K[3 * i];
        dp[i][4] = K[3 * i + 1];
        dp[i][5] = K[3 * i + 2];
    }
    for (int k = 0; k < 6; ++k) {
        J[0][k] = fma(-u0, dp[2][k], dp[0][k]) * ip;
        J[1][k] = fma(-u1, dp[2][k], dp[1][k]) * ip;
    }
    return p2;
}

// The rotation nearest to M (3 x 3 row-major) in the Frobenius norm: M = U S V^T by one-sided Jacobi (M V = U S), the
// columns of U normalised, the one of the smallest singular value replaced by the cross product of the other two (so
// det U = +1 = det V and a reflection is projected onto a rotation), R = U V^T.
__device__ inline void refine_nearest_rotation(const double* M, double* R) {
    double g[9], V[9];
    for (int k = 0; k < 9; ++k) g[k] = M[k];
    jacobi_svd_onesided<3, 3>(g, V, 30);
    double sv[3];
    for (int c = 0; c < 3; ++c) sv[c] = sqrt(fma(g[c], g[c], fma(g[3 + c], g[3 + c], g[6 + c] * g[6 + c])));
    int m = 0;
    if (sv[1] < sv[m]) m = 1;
    if (sv[2] < sv[m]) m = 2;
    const int a = (m + 1) % 3, b = (m + 2) % 3;  // (a, b, m) cyclic: u_m = u_a x u_b
    double ua[3], ub[3], um[3];
    for (int k = 0; k < 3; ++k) {
        ua[k] = g[3 * k + a] / sv[a];
        ub[k] = g[3 * k + b] / sv[b];
    }
    refine_cross(ua, ub, um);
    double U[9];
    for (int k = 0; k < 3; ++k) {
        U[3 * k + a] = ua[k];
        U[3 * k + b] = ub[k];
        U[3 * k + m] = um[k];
    }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[3 * i + j] = fma(U[3 * i + 2], V[3 * j + 2], fma(U[3 * i + 1], V[3 * j + 1], U[3 * i] * V[3 * j]));
}

// First chunk partial of the pair whose records start at pbase: pair q owns at most ceil(len_q / kRefineChunk) chunks,
// so floor(pbase / kRefineChunk) + pair never overlaps the previous pair's and the buffer grows with the total length,
// not with the number of pairs times the longest one.
__device__ __forceinline__ long long refine_chunk_base(long long pbase, int pair) { return pbase / kRefineChunk + pair; }

template <int KIND>
__device__ __forceinline__ void refine_load_proposal(const RefineState* s, double* x) {
#pragma unroll
    for (int k = 0; k < 12; ++k) x[k] = __ldcg(s->px + k);
}

// ---- MODEL_P: the inlier list of the start pose, ascending (T1's decoupled look-back over PnpRec records) ----
constexpr int kListBlock = 256;
constexpr int kListPerBlock = 4 * kListBlock;  // records per block

template <int KIND, class Args = typename RefineArgsOf<KIND>::type>
__global__ void __launch_bounds__(kListBlock) k_refine_list(const Args a) {
    static_assert(KIND == MODEL_P, "the E and H lists are T1's (k_tail_mask)");
    chain_enter();
    __shared__ unsigned s_bid;
    __shared__ int warp_cnt[4][kListBlock / 32];
    __shared__ long long s_prefix;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nblk = gridDim.x;
    if (tid == 0) s_bid = atomicAdd(&a.list_ticket[0], 1u);  // ticket order = start order: predecessors are running
    __syncthreads();
    const int bid = (int)s_bid;
    double P[12];
    pnp_projection(a.K, a.start, P);
    long long forced[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) forced[q] = a.forced ? a.forced[q] : -1;
    const long long base = (long long)bid * kListPerBlock;
    bool f[4];
    unsigned b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long i = base + k * kListBlock + tid;
        f[k] = false;
        if (i < a.n) {
            double v;
            bool in = pnp_exact(P, a.ppts[i], a.thr, v);
#pragma unroll
            for (int q = 0; q < 4; ++q) in |= forced[q] == i;
            f[k] = in;
        }
        b[k] = __ballot_sync(0xffffffffu, f[k]);
        if (lane == 0) warp_cnt[k][warp] = __popc(b[k]);
    }
    __syncthreads();
    int total = 0;
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            for (int w = 0; w < kListBlock / 32; ++w) total += warp_cnt[k][w];
        atomicExch(&a.list_agg[bid], (unsigned long long)total | (1ull << 62));  // value and flag in one word
    }
    if (warp == 0) {
        long long sum = 0;
        for (int j0 = 0; j0 < bid; j0 += 32) {
            const int j = j0 + lane;
            long long v = 0;
            if (j < bid) {
                unsigned long long w;
                do { w = *reinterpret_cast<volatile unsigned long long*>(a.list_agg + j); } while (!(w & (1ull << 62)));
                v = (long long)(w & ~(1ull << 62));
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
            sum += v;
        }
        if (lane == 0) s_prefix = sum;
    }
    __syncthreads();
    long long off = s_prefix;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        long long o = off;
        for (int w = 0; w < kListBlock / 32; ++w) {
            if (w < warp) o += warp_cnt[k][w];
            off += warp_cnt[k][w];
        }
        if (f[k]) a.list_out[o + __popc(b[k] & ((1u << lane) - 1u))] = base + k * kListBlock + tid;
    }
    if (bid == nblk - 1 && tid == 0) a.list_out[a.n] = s_prefix + total;
    // the last block past the look-back clears the state for the next call
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(&a.list_ticket[1], 1u) == (unsigned)(nblk - 1)) {
            for (int j = 0; j < nblk; ++j) a.list_agg[j] = 0;
            a.list_ticket[0] = 0;
            a.list_ticket[1] = 0;
        }
    }
}

// ---- start point and per-pair state ----
template <int KIND, class Args = typename RefineArgsOf<KIND>::type>
__global__ void __launch_bounds__(128) k_refine_init(const Args a) {
    chain_enter();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.npairs) return;
    RefineState& s = a.state[p];
    if constexpr (KIND == MODEL_P) {  // the nearest rotation to the start's R, and its t
        s.num = a.num[0];
        s.iter = 0;
        s.evals = 0;
        s.rejected = 0;
        s.pad = 0;
        s.lambda = kRefineLambda0;
        s.cost = s.cost_ransac = s.cost_start = __longlong_as_double(0x7ff8000000000000LL);
        s.status = REFINE_RUNNING;
        s.done = 0;
        double m[12];
        bool finite = true;
        for (int k = 0; k < 12; ++k) {
            m[k] = a.start[k];
            finite = finite && isfinite(m[k]);
            s.px[k] = s.x[k] = 0.0;
        }
        if (finite) {
            const double M[9] = {m[0], m[1], m[2], m[4], m[5], m[6], m[8], m[9], m[10]};
            double R[9];
            refine_nearest_rotation(M, R);
            for (int k = 0; k < 9; ++k) {
                s.px[k] = R[k];
                finite = finite && isfinite(R[k]);
            }
            for (int k = 0; k < 3; ++k) s.px[9 + k] = m[4 * k + 3];
        }
        if (!finite) {
            s.status = REFINE_NONFINITE;
            s.done = 1;
        }
        return;
    }
    const SelectRecord& rec = a.rec[p];
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    s.num = a.num[p];
    s.iter = 0;
    s.evals = 0;
    s.rejected = 0;
    s.pad = 0;
    s.lambda = kRefineLambda0;
    s.cost = s.cost_ransac = s.cost_start = nan;
    s.status = REFINE_RUNNING;
    s.done = 0;
    for (int k = 0; k < 12; ++k) s.px[k] = s.x[k] = 0.0;
    if (rec.best.idx < 0) {
        s.status = REFINE_NO_MODEL;
        s.done = 1;
        s.num = 0;
        return;
    }
    double e[9];
    bool finite = true;
    for (int k = 0; k < 9; ++k) {
        e[k] = rec.E[k];
        finite = finite && isfinite(e[k]);
    }
    if (finite) {
        if constexpr (KIND == MODEL_E) {
            PoseSet ps;
            decompose_essential(e, ps);
            for (int k = 0; k < 9; ++k) s.px[k] = ps.R[0][k];
            for (int k = 0; k < 3; ++k) s.px[9 + k] = ps.t[0][k];
        } else {
            for (int k = 0; k < 8; ++k) s.px[k] = e[k] / e[8];
        }
        for (int k = 0; k < 12; ++k) finite = finite && isfinite(s.px[k]);
    }
    if (!finite) {
        s.status = REFINE_NONFINITE;
        s.done = 1;
    }
}

// Cholesky solve of (A_hat + lambda I) y = -g_hat, A_hat = D^-1 A D^-1 (unit diagonal), g_hat = D^-1 g; false when the
// damped matrix is not numerically positive definite
template <int NP>
__device__ bool refine_solve(const double* A, const double* g, const double* D, double lambda, double (&y)[NP]) {
    double L[NP][NP];
    for (int i = 0; i < NP; ++i)
        for (int j = 0; j <= i; ++j) {
            double v = A[NP * i + j] / (D[i] * D[j]) + (i == j ? lambda : 0.0);
            for (int k = 0; k < j; ++k) v = fma(-L[i][k], L[j][k], v);
            if (i == j) {
                if (!(v > 0.0) || !isfinite(v)) return false;
                L[i][i] = sqrt(v);
            } else {
                L[i][j] = v / L[j][j];
            }
        }
    double z[NP];
    for (int i = 0; i < NP; ++i) {
        double v = -g[i] / D[i];
        for (int k = 0; k < i; ++k) v = fma(-L[i][k], z[k], v);
        z[i] = v / L[i][i];
    }
    for (int i = NP - 1; i >= 0; --i) {
        double v = z[i];
        for (int k = i + 1; k < NP; ++k) v = fma(-L[k][i], y[k], v);
        y[i] = v / L[i][i];
    }
    for (int i = 0; i < NP; ++i)
        if (!isfinite(y[i])) return false;
    return true;
}

// the LM control of one pair, given the totals of the proposal just evaluated (one thread; its own function, so that the
// evaluation loop's register allocation does not carry it)
template <int KIND>
__device__ __noinline__ void refine_control(RefineState& s, const double* tot, int max_iter) {
    constexpr int NP = RefineDims<KIND>::NP;
    const double c = tot[0];
    bool accept;
    if (s.evals == 0) {  // the start point
        s.cost_start = c;
        s.cost_ransac = (KIND == MODEL_E || KIND == MODEL_P) ? tot[1] : c;
        if (!isfinite(c)) {
            s.status = REFINE_NONFINITE;
            s.done = 1;
            return;
        }
        accept = true;
    } else {
        s.iter += 1;
        accept = c < s.cost;
    }
    s.evals += 1;
    if (accept) {
        const double before = s.cost;
        for (int k = 0; k < 12; ++k) s.x[k] = s.px[k];
        int q = 3;
        for (int i = 0; i < NP; ++i)
            for (int j = i; j < NP; ++j) {
                s.A[NP * i + j] = tot[q];
                s.A[NP * j + i] = tot[q];
                ++q;
            }
        for (int i = 0; i < NP; ++i) s.g[i] = tot[q + i];
        s.cost = c;
        if (s.iter > 0) {
            s.lambda /= kRefineLambdaFactor;
            if (before - c <= kRefineFtol * before) {
                s.status = REFINE_CONVERGED;
                s.done = 1;
                return;
            }
        }
        if (c <= kRefineCostFloor * tot[2]) {
            s.status = REFINE_CONVERGED;
            s.done = 1;
            return;
        }
    } else {
        s.lambda *= kRefineLambdaFactor;
        s.rejected += 1;
    }
    if (s.iter >= max_iter) {
        s.status = REFINE_MAX_ITER;
        s.done = 1;
        return;
    }
    double D[NP];
    for (int i = 0; i < NP; ++i) {
        const double d = s.A[NP * i + i];
        D[i] = (d > 0.0 && isfinite(d)) ? sqrt(d) : 1.0;
    }
    double y[NP];
    for (;;) {
        if (!(s.lambda <= kRefineLambdaCap)) {
            s.status = REFINE_STALLED;
            s.done = 1;
            return;
        }
        if (refine_solve<NP>(s.A, s.g, D, s.lambda, y)) break;
        s.lambda *= kRefineLambdaFactor;
    }
    double n2 = 0.0;
    for (int i = 0; i < NP; ++i) n2 = fma(y[i], y[i], n2);
    if (sqrt(n2) <= kRefineXtol * sqrt(s.cost)) {
        s.status = REFINE_CONVERGED;
        s.done = 1;
        return;
    }
    double d[NP];
    for (int i = 0; i < NP; ++i) d[i] = y[i] / D[i];
    if constexpr (KIND == MODEL_E) {
        refine_rotate(s.x, d, s.px);
        double b1[3], b2[3], t[3];
        refine_tangent_basis(s.x + 9, b1, b2);
        for (int k = 0; k < 3; ++k) t[k] = fma(d[3], b1[k], fma(d[4], b2[k], s.x[9 + k]));
        const double inv = 1.0 / sqrt(fma(t[0], t[0], fma(t[1], t[1], t[2] * t[2])));
        for (int k = 0; k < 3; ++k) s.px[9 + k] = t[k] * inv;
    } else if constexpr (KIND == MODEL_H) {
        for (int k = 0; k < 8; ++k) s.px[k] = s.x[k] + d[k];
    } else if constexpr (KIND == MODEL_P) {
        refine_rotate(s.x, d, s.px);
        for (int k = 0; k < 3; ++k) s.px[9 + k] = s.x[9 + k] + d[3 + k];
    } else {
        for (int k = 0; k < 3; ++k) s.px[k] = s.x[k] + d[k];
    }
}

// ---- one LM iteration: evaluate the pair's proposal over its inlier list, then the last block steps ----
template <int KIND, class Args = typename RefineArgsOf<KIND>::type>
__global__ void __launch_bounds__(kRefineBlock) k_refine_step(const Args a) {
    chain_enter();
    constexpr int NP = RefineDims<KIND>::NP;
    constexpr int NV = refine_nv<KIND>();
    constexpr int NW = kRefineBlock / 32;
    __shared__ double s_model[KIND == MODEL_P ? 12 : 9];   // P: K [R | t] of the proposal
    __shared__ double s_M[45];                             // E: dE / dtheta; P: K
    __shared__ double s_ransac[KIND == MODEL_P ? 12 : 9];  // the RANSAC model (E) or K [R | t] of the unprojected
                                                           // start (P), read by the first evaluation only
    __shared__ double s_warp[NW][NV];
    __shared__ double s_tot[NV];
    __shared__ int s_last;
    const int pair = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    RefineState* st = a.state + pair;
    if (__ldcg(&st->done)) return;
    const long long num = __ldcg(&st->num);
    const long long nch = (num + kRefineChunk - 1) / kRefineChunk;
    // only the blocks that own a chunk take part (block 0 always, so that an empty list still gets its step): the rest
    // of a grid sized for the longest pair leaves at once
    const long long nblk = nch < gridDim.x ? (nch > 0 ? nch : 1) : gridDim.x;
    if (blockIdx.x >= nblk) return;
    const bool first = __ldcg(&st->evals) == 0;
    const long long pbase = a.offsets ? a.offsets[pair] : 0;
    if (tid == 0) {
        double x[12];
        refine_load_proposal<KIND>(st, x);
        if constexpr (KIND == MODEL_E) {
            double E[9], M[45];
            refine_e_model(x, x + 9, E, M);
            for (int k = 0; k < 9; ++k) s_model[k] = E[k];
            for (int k = 0; k < 45; ++k) s_M[k] = M[k];
            for (int k = 0; k < 9; ++k) s_ransac[k] = a.rec[pair].E[k];
        } else if constexpr (KIND == MODEL_H) {
            for (int k = 0; k < 8; ++k) s_model[k] = x[k];
            s_model[8] = 1.0;
        } else {
            const double m[12] = {x[0], x[1], x[2], x[9], x[3], x[4], x[5], x[10], x[6], x[7], x[8], x[11]};
            double P[12];
            pnp_projection(a.K, m, P);
            for (int k = 0; k < 12; ++k) s_model[k] = P[k];
            for (int k = 0; k < 9; ++k) s_M[k] = a.K[k];
            pnp_projection(a.K, a.start, P);
            for (int k = 0; k < 12; ++k) s_ransac[k] = P[k];
        }
    }
    __syncthreads();
    double* part = a.partial + refine_chunk_base(pbase, pair) * NV;
    for (long long ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        double acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = 0.0;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const long long i = ch * kRefineChunk + half * kRefineBlock + tid;
            if constexpr (KIND == MODEL_P) {
                if (i < num) {
                    const PnpRec c = a.ppts[a.idx[i]];
                    acc[2] += fma(c.u, c.u, c.v * c.v);
                    double r[2], J[2][6];
                    const double p2 = refine_p_residuals(s_model, s_M, c.X, c.Y, c.Z, c.u, c.v, r, J);
                    if (first) {
                        double pm[12];
#pragma unroll
                        for (int k = 0; k < 12; ++k) pm[k] = s_ransac[k];
                        acc[1] += pnp_value(pnp_terms(pm, c.X, c.Y, c.Z, c.u, c.v));
                    }
                    // cheirality guard: the scorer's depth rule and finite residuals, else the proposal costs +inf
                    if (!(p2 >= 0x1p-537) || !isfinite(r[0]) || !isfinite(r[1])) {
                        acc[0] = __longlong_as_double(0x7ff0000000000000LL);
                    } else {
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            acc[0] = fma(r[k], r[k], acc[0]);
                            int q = 3;
#pragma unroll
                            for (int p = 0; p < 6; ++p)
#pragma unroll
                                for (int m = p; m < 6; ++m, ++q) acc[q] = fma(J[k][p], J[k][m], acc[q]);
#pragma unroll
                            for (int p = 0; p < 6; ++p) acc[q + p] = fma(J[k][p], r[k], acc[q + p]);
                        }
                    }
                }
            } else if (i < num) {
                const Corr c = a.pts[pbase + a.idx[pbase + i]];
                acc[2] += fma(c.xa, c.xa, fma(c.ya, c.ya, fma(c.xb, c.xb, c.yb * c.yb)));
                if constexpr (KIND == MODEL_E) {
                    double gE[9];
                    const double r = refine_e_residual(s_model, c.xa, c.ya, c.xb, c.yb, gE);
                    double J[5];
#pragma unroll
                    for (int p = 0; p < 5; ++p) {
                        double v = 0.0;
#pragma unroll
                        for (int j = 0; j < 9; ++j) v = fma(gE[j], s_M[5 * j + p], v);
                        J[p] = v;
                    }
                    acc[0] = fma(r, r, acc[0]);
                    if (first) {
                        double em[9];
#pragma unroll
                        for (int k = 0; k < 9; ++k) em[k] = s_ransac[k];
                        acc[1] += sed_exact(em, c.xa, c.ya, c.xb, c.yb);
                    }
                    int q = 3;
#pragma unroll
                    for (int p = 0; p < 5; ++p)
#pragma unroll
                        for (int m = p; m < 5; ++m, ++q) acc[q] = fma(J[p], J[m], acc[q]);
#pragma unroll
                    for (int p = 0; p < 5; ++p) acc[q + p] = fma(J[p], r, acc[q + p]);
                } else {
                    double r[4], J[4][8];
                    refine_h_residuals(s_model, c.xa, c.ya, c.xb, c.yb, r, J);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        acc[0] = fma(r[k], r[k], acc[0]);
                        int q = 3;
#pragma unroll
                        for (int p = 0; p < 8; ++p)
#pragma unroll
                            for (int m = p; m < 8; ++m, ++q) acc[q] = fma(J[k][p], J[k][m], acc[q]);
#pragma unroll
                        for (int p = 0; p < 8; ++p) acc[q + p] = fma(J[k][p], r[k], acc[q + p]);
                    }
                }
            }
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            double x = acc[v];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
            if (lane == 0) s_warp[warp][v] = x;
        }
        __syncthreads();
        if (tid < NV) {
            double x = s_warp[0][tid];
#pragma unroll
            for (int w = 1; w < NW; ++w) x += s_warp[w][tid];
            part[ch * NV + tid] = x;
        }
        __syncthreads();
    }
    // the pair's last block to finish sums the chunk partials in chunk order and takes the step
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(&a.ticket[pair], 1u) == (unsigned)(nblk - 1)) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (tid < NV) {
        double x = 0.0;
        for (long long ch = 0; ch < nch; ++ch) x += __ldcg(part + ch * NV + tid);
        s_tot[tid] = x;
    }
    __syncthreads();
    if (tid == 0) {
        a.ticket[pair] = 0;
        refine_control<KIND>(*st, s_tot, a.max_iter);
    }
}

// ---- the refined record and the report ----
template <int KIND, class Args = typename RefineArgsOf<KIND>::type>
__global__ void __launch_bounds__(128) k_refine_finish(const Args a) {
    chain_enter();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.npairs) return;
    const RefineState& s = a.state[p];
    if constexpr (KIND == MODEL_P) {  // the report and the pose k_pnp_mask reads
        PnpRefineReport rep;
        rep.cost_ransac = s.cost_ransac;
        rep.cost_start = s.cost_start;
        rep.cost_final = s.cost;
        rep.num = s.num;
        rep.iterations = s.iter;
        rep.rejected = s.rejected;
        rep.reserved = 0;
        rep.status = s.status;
        if (s.status == REFINE_NONFINITE) {
            for (int k = 0; k < 12; ++k) rep.Rt[k] = a.start[k];
            rep.cost_final = rep.cost_start;
        } else {
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) rep.Rt[4 * r + c] = s.x[3 * r + c];
                rep.Rt[4 * r + 3] = s.x[9 + r];
            }
        }
        for (int k = 0; k < 12; ++k) a.pose_out[k] = rep.Rt[k];
        *a.preport = rep;
        return;
    }
    const SelectRecord& rec = a.rec[p];
    SelectRecord out = rec;
    RefineReport rep;
    rep.cost_ransac = s.cost_ransac;
    rep.cost_start = s.cost_start;
    rep.cost_final = s.cost;
    rep.num = s.num;
    rep.iterations = s.iter;
    rep.rejected = s.rejected;
    rep.reserved = 0;
    int status = s.status;
    double m[9];
    bool refined = status != REFINE_NO_MODEL && status != REFINE_NONFINITE;
    if (refined) {
        if constexpr (KIND == MODEL_E) {
            double E[9], M[45];
            refine_e_model(s.x, s.x + 9, E, M);
            const double e8 = E[8];
            for (int k = 0; k < 9; ++k) m[k] = E[k] / e8;
            m[8] = 1.0;
        } else {
            for (int k = 0; k < 8; ++k) m[k] = s.x[k];
            m[8] = 1.0;
        }
        for (int k = 0; k < 9; ++k) refined = refined && isfinite(m[k]);
        if (!refined) status = REFINE_NONFINITE;  // E[2,2] of the refined pose is 0: not representable with E[8] == 1
    }
    if (refined) {
        for (int k = 0; k < 9; ++k) out.E[k] = m[k];
        for (int k = 0; k < 8; ++k) out.sample[k] = -1;
    } else {
        for (int k = 0; k < 9; ++k) m[k] = rec.E[k];
        if (status == REFINE_NO_MODEL) rep.num = 0;
        rep.cost_final = rep.cost_start;
    }
    for (int k = 0; k < 9; ++k) rep.model[k] = m[k];
    rep.status = status;
    a.out_rec[p] = out;
    a.report[p] = rep;
}

}  // namespace sfm
