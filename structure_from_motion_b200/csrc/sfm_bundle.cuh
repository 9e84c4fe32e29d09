// Bundle adjustment (sfm_bundle_adjust): joint Levenberg-Marquardt over the free poses of V registered views and the
// points of their tracks, with the point blocks eliminated by a Schur complement.
//
// Problem.
//   cameras     K[V][9] fixed (upper triangular, K[2,2] = 1); Rt[V][12] the start, world to camera, x_cam = R X + t.
//               1 <= V <= kBaMaxViews.
//   tracks      the CSR of sfm_triangulate_tracks (offsets, view, x), at most kBaMaxTrack observations per track; X[T][3]
//               the start point of every track.  A track whose start X has a non-finite entry is not a parameter.
//   list        formed once under the start (the given Rt and X) and fixed while the solver runs: the observations
//               passing the PnP record rule pnp_exact(pnp_projection(K_c, Rt_c), {X, u, v}, thr), of the tracks with
//               at least 2 such observations (the parameter points).  The other tracks are reported unchanged, bits
//               included, and none of their observations is in the list.
//   gauge       fixed[V] marks the poses held constant (at least one).  scale_view (-1 = none), a free view: the
//               component of its start t with the largest |value| (lowest index on ties) is held constant.  Fixed
//               views, that component and the non-parameter points come out bit-identical to the input.
//   parameters  per free view R <- R exp([w]x) (refine_rotate), t <- t + dt; per parameter point X <- X + dX.  A free
//               view starts from the rotation nearest its given R (refine_nearest_rotation, as sfm_refine_pnp).  The
//               anchored component is carried as a parameter whose Jacobian column is zero, and a free view with no
//               list observation has a zero Jacobian block: in the Marquardt-scaled damped system their rows are
//               lambda on the diagonal and 0 elsewhere, so their step is exactly 0 and they stay at their (projected)
//               start.  The reduced camera system is therefore 6 F x 6 F, F the number of free views.
//   cost        the sum over the list of r0^2 + r1^2, r0 = p0 / p2 - u, r1 = p1 / p2 - v, p in pnp_terms' FMA order
//               (refine_p_residuals).  A proposal under which a list observation has p2 < 2^-537 or a non-finite
//               residual costs +inf and is rejected; at the start that is REFINE_NONFINITE and the input is reported.
//   control     refine_control's policy and constants (kRefine*): lambda0 1e-3, / 10 on a strictly lower cost, x 10
//               otherwise; Ftol, Xtol on the scaled step |D d| against sqrt(cost), D = sqrt(diag J^T J) (1 where 0 or
//               non-finite); lambda cap (or lambda underflowed to 0) -> stalled; the cost floor kRefineCostFloor sum(u^2 + v^2) over the list;
//               max_iter evaluated proposals; a damped system that is not numerically positive definite (a point's
//               3 x 3 block or the reduced camera system) multiplies lambda by 10 and is solved again.
//   step        (A_hat + lambda I) y = -g_hat, A_hat = D^-1 J^T J D^-1, g_hat = D^-1 g.  Per point p: V_hat_p (+ lambda)
//               is inverted by a 3 x 3 Cholesky; per list observation i of p in a free view, W_hat_i = D_c^-1 J_c^T J_p
//               D_p^-1 and Y_i = W_hat_i V_hat_p^-1.  The reduced camera system S = U_hat + lambda I - sum_p W_hat_p
//               V_hat_p^-1 W_hat_p^T (block (a, c): the sum over observation pairs (i in a, j in c) of one track of
//               Y_i W_hat_j^T) with right-hand side -g_hat_c + sum_i Y_i g_hat_p, factored by a tiled Cholesky whose
//               last tile row carries the right-hand side (so the forward substitution is part of the factor), then
//               L^T y_c = z and y_p = V_hat_p^-1 (-g_hat_p - sum_i W_hat_i^T y_c).  d = y / D.
//   report      BaReport; the reported parameters are the last accepted ones (the input at REFINE_NONFINITE); mask and
//               err of every observation are its pnp_exact decision and value under them.  An empty list is converged
//               at iteration 0 with cost 0 and the projected start.
// Determinism.  Every sum runs in an order fixed by the inputs alone: per point over its observations in track order;
// per view over its observations in ascending index, in chunks of kBaObsChunk; the cost over chunks of kBaBlock
// tracks, added in chunk order; each S block over its observation pairs in ascending track order, in chunks of
// kBaTripleChunk; the Cholesky's updates in fixed k order.  Chunk partials of one view or S block are added by one warp
// (lane j takes chunks j, j + 32, ... in order, then a fixed butterfly): an order fixed by the chunk count.  No
// floating-point atomics; the bits depend neither on the grid nor on the run.  World x 2^k (t and X with it) and pixels
// x 2^k (K's first two rows, threshold x 4^k) change every sum by a power of two that the Marquardt scaling cancels.
//
// Kernels (all chain kernels; the host enqueues max_iter + 1 rounds, and once the problem is finished every later
// launch exits at once):
//   k_ba_init        the projected start rotations, P of the start, the state.
//   k_ba_list        the decisions under the start, the list and parameter flags, the counts and the cost floor.
//   per round        k_ba_eval (one thread per track: residuals, J_c, J_p of the proposal, V_p, g_p, cost partials),
//                    k_ba_views (per view chunk partials of U_c, g_c), k_ba_views_sum (U_c, g_c; the last block accepts
//                    or rejects, as refine_control), k_ba_schur_pts (V_hat_p^-1), k_ba_schur_obs (W_hat_i, Y_i, per
//                    observation), k_ba_schur (S block and right-hand side partials),
//                    k_ba_schur_sum (S, dense), k_ba_chol (one launch per tile column), k_ba_backsolve (L^T y = z),
//                    k_ba_points (y_p, the proposal; the last block checks Xtol and moves the poses).
//   k_ba_finish, k_ba_mask: the report, the reported parameters, mask and err.
// The equations of an evaluated proposal go to the second of two buffers, which becomes current on accept, so a
// rejected step is solved again from the stored equations without new Jacobians.
#pragma once
#include "sfm_device.cuh"
#include "sfm_pnp_model.cuh"
#include "sfm_refine.cuh"

namespace sfm {

constexpr int kBaMaxViews = 256;
constexpr int kBaMaxTrack = 64;
constexpr int kBaBlock = 128;               // tracks per block (and per cost chunk) of the per-track kernels
constexpr int kBaObsChunk = 2 * kBaBlock;   // view-major observations per chunk
constexpr int kBaTripleChunk = 32;          // observation pairs per S-block chunk
constexpr int kBaTile = 32;                 // Cholesky tile
constexpr int kBaCholThreads = 256;
constexpr int kBaSolveSlices = 16;
constexpr int kBaMaxBatches = 64;           // batches of max_iter + 1 rounds the host enqueues at most (sfm_bundle.cu)
enum { BA_EVAL = 0, BA_SOLVE = 1 };

struct BaObsEq { double Jc[2][6], Jp[2][3], r[2]; };          // one observation's rows of J and residuals
struct BaPtEq { double V[6], g[3], pad; };                    // J_p^T J_p (upper, row-major) and J_p^T r of a point
struct BaViewEq { double U[21], g[6], pad; };                 // J_c^T J_c (upper, row-major) and J_c^T r of a free view
struct BaObsSchur { double W[6][3], Y[6][3], e[6]; };         // W_hat_i, Y_i = W_hat_i V_hat_p^-1, Y_i g_hat_p
struct BaPtSolve { double Vi[9], g[3], D[3], pad; };          // V_hat_p^-1 (damped), g_hat_p, D_p

struct BaState {
    double cost, lambda, cost_start, floor;
    unsigned long long num_obs, num_points;
    int iter, evals, rejected, status, done, phase, cur, fail;
};

// layout of sfm_bundle_report (include/sfm_b200.h)
struct BaReport {
    double cost_start, cost_final;
    long long num_observations, num_points;
    int num_free_views, iterations, status, rejected;
};

struct BaArgs {
    const double* K;            // [V][9]
    const double* Rt;           // [V][12] the start
    const int* fidx;            // [V] free index of a view, -1 = fixed
    int V, F, anchor, anchor_comp, npad, max_iter;
    long long T, M;
    const long long* offsets;   // [T+1]
    const int* view;            // [M]
    const double2* x;           // [M]
    const double* X0;           // [T][3]
    const int* otrack;          // [M] the track of each observation
    double thr;
    // structure (host-built)
    const int* vperm;           // observations of the free views, by free view, ascending within a view
    long long nvch;             // view chunks
    const long long* vch_begin; // [nvch+1] into vperm
    const long long* vfirst;    // [F+1] first chunk of each free view
    const int2* triples;        // (i, j) observation pairs of one track, free(view i) >= free(view j), by block
    long long ntch;             // triple chunks
    const long long* tch_begin; // [ntch+1] into triples
    const long long* bfirst;    // [nblk+1] first chunk of each block
    const int* blk_id;          // [F][F] block of (a, c), a >= c, or -1
    const int2* blk_ac;         // [nblk] (a, c) of each block
    long long nblk;
    long long nptch;            // chunks of kBaBlock tracks
    // state
    BaState* st;
    unsigned* ticket;           // [2] zero on entry and exit
    unsigned char* inlist;      // [M]
    unsigned char* param;       // [T]
    double* pose;               // [2][V][12] R[9], t[3]
    double* Pprop;              // [V][12] P of the proposal
    double* Xp;                 // [2][T][3]
    BaObsEq* oeq;               // [2][M]
    BaPtEq* peq;                // [2][T]
    BaViewEq* veq;              // [2][F]
    BaObsSchur* osch;           // [M]
    BaPtSolve* psol;            // [T]
    double* part_pt;            // [nptch]
    double* part_v;             // [nvch][27]
    double* part_t;             // [ntch][36]
    double* part_r;             // [nvch][6]
    double* S;                  // [npad + kBaTile][npad]: lower triangle, then the right-hand side in row npad
    double* Ldiag;              // [npad / kBaTile][kBaTile][kBaTile] the factor's diagonal tiles (k_ba_backsolve's)
    double* y;                  // [npad]
    // outputs
    double* Rt_out;             // [V][12]
    double* Prep;               // [V][12]
    double* X_out;              // [T][3]
    unsigned char* mask;        // [M]
    double* err;                // [M]
    BaReport* report;
};

__device__ __forceinline__ void ba_Rt(const double* pose, double (&m)[12]) {
    m[0] = pose[0]; m[1] = pose[1]; m[2] = pose[2];  m[3] = pose[9];
    m[4] = pose[3]; m[5] = pose[4]; m[6] = pose[5];  m[7] = pose[10];
    m[8] = pose[6]; m[9] = pose[7]; m[10] = pose[8]; m[11] = pose[11];
}

__device__ __forceinline__ double ba_inf() { return __longlong_as_double(0x7ff0000000000000LL); }
__device__ __forceinline__ double ba_nan() { return __longlong_as_double(0x7ff8000000000000LL); }
__device__ __forceinline__ double ba_scale(double d) { return (d > 0.0 && isfinite(d)) ? sqrt(d) : 1.0; }

// indices of the diagonal of a row-major upper triangle of order 6 and 3
__device__ __forceinline__ int ba_d6(int p) { return p * 6 - p * (p - 1) / 2; }
__device__ __forceinline__ int ba_u6(int p, int m) { return p <= m ? ba_d6(p) + m - p : ba_d6(m) + p - m; }
__device__ __forceinline__ int ba_u3(int p, int m) { return p <= m ? p * 3 - p * (p - 1) / 2 + m - p : m * 3 - m * (m - 1) / 2 + p - m; }

// block sum of one value per thread (kBaBlock threads): butterfly per warp, warps in order; valid on thread 0
__device__ __forceinline__ double ba_block_sum(double v, double* s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (lane == 0) s_warp[warp] = v;
    __syncthreads();
    double t = s_warp[0];
#pragma unroll
    for (int w = 1; w < kBaBlock / 32; ++w) t += s_warp[w];
    __syncthreads();
    return t;
}

// the sum of n partials (stride apart) in index order, as kBaBlock ordered segments added in segment order; every
// thread of the block calls it, the result is valid on thread 0.  Depends on n alone.
__device__ __forceinline__ double ba_ordered_sum(const double* p, long long n, int stride, double* s_seg) {
    const int tid = threadIdx.x;
    const long long len = (n + kBaBlock - 1) / kBaBlock;
    const long long lo = tid * len, hi = lo + len < n ? lo + len : n;
    double x = 0.0;
    for (long long i = lo; i < hi; ++i) x += __ldcg(p + i * stride);
    s_seg[tid] = x;
    __syncthreads();
    double t = 0.0;
    if (tid == 0)
        for (int k = 0; k < kBaBlock; ++k) t += s_seg[k];
    __syncthreads();
    return t;
}

// the last block of a launch to arrive (ticket k); resets the ticket
__device__ __forceinline__ bool ba_last_block(unsigned* ticket, int* s_flag) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const bool last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        if (last) *ticket = 0;
        *s_flag = last;
    }
    __syncthreads();
    if (*s_flag) __threadfence();
    return *s_flag;
}

// ---- the start: projected rotations, P, the state (one block) ----
__global__ void __launch_bounds__(256) k_ba_init(const BaArgs a) {
    chain_enter();
    for (int c = threadIdx.x; c < a.V; c += blockDim.x) {
        const double* m = a.Rt + 12 * c;
        double p[12];
        const double M[9] = {m[0], m[1], m[2], m[4], m[5], m[6], m[8], m[9], m[10]};
        if (a.fidx[c] >= 0) {
            double R[9];
            refine_nearest_rotation(M, R);
            for (int k = 0; k < 9; ++k) p[k] = R[k];
        } else {
            for (int k = 0; k < 9; ++k) p[k] = M[k];
        }
        for (int k = 0; k < 3; ++k) p[9 + k] = m[4 * k + 3];
        for (int k = 0; k < 12; ++k) {
            a.pose[12 * c + k] = p[k];
            a.pose[12 * (a.V + c) + k] = p[k];
        }
        double q[12], P[12];
        ba_Rt(p, q);
        pnp_projection(a.K + 9 * c, q, P);
        for (int k = 0; k < 12; ++k) a.Pprop[12 * c + k] = P[k];
    }
    if (threadIdx.x == 0) {
        BaState s;
        s.cost = s.cost_start = ba_nan();
        s.lambda = kRefineLambda0;
        s.floor = 0.0;
        s.num_obs = s.num_points = 0;
        s.iter = s.evals = s.rejected = 0;
        s.status = REFINE_RUNNING;
        s.done = 0;
        s.phase = BA_EVAL;
        s.cur = 0;
        s.fail = 0;
        *a.st = s;
    }
}

// ---- the list under the start: one thread per track ----
__global__ void __launch_bounds__(kBaBlock) k_ba_list(const BaArgs a) {
    chain_enter();
    __shared__ double s_warp[kBaBlock / 32];
    __shared__ double s_seg[kBaBlock];
    __shared__ int s_flag;
    const long long t = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    double sumsq = 0.0;
    unsigned nobs = 0, npt = 0;
    if (t < a.T) {
        const long long o = a.offsets[t];
        const int n = (int)(a.offsets[t + 1] - o);
        const double X[3] = {a.X0[3 * t], a.X0[3 * t + 1], a.X0[3 * t + 2]};
        const bool finite = isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]);
        unsigned long long bits = 0;
        if (finite)
            for (int j = 0; j < n; ++j) {
                const int c = a.view[o + j];
                double P[12];
                pnp_projection(a.K + 9 * c, a.Rt + 12 * c, P);
                const double2 uv = a.x[o + j];
                PnpRec r;
                r.X = X[0]; r.Y = X[1]; r.Z = X[2]; r.u = uv.x; r.v = uv.y; r.pad = 0.0;
                double val;
                if (pnp_exact(P, r, a.thr, val)) bits |= 1ull << j;
            }
        const bool par = finite && __popcll(bits) >= 2;
        if (!par) bits = 0;
        for (int j = 0; j < n; ++j) {
            const bool in = (bits >> j) & 1ull;
            a.inlist[o + j] = in;
            if (in) {
                const double2 uv = a.x[o + j];
                sumsq += fma(uv.x, uv.x, uv.y * uv.y);
            }
        }
        a.param[t] = par;
        nobs = __popcll(bits);
        npt = par;
        for (int k = 0; k < 3; ++k) {
            a.Xp[3 * t + k] = X[k];
            a.Xp[3 * (a.T + t) + k] = X[k];
        }
    }
    nobs = __reduce_add_sync(0xffffffffu, nobs);
    npt = __reduce_add_sync(0xffffffffu, npt);
    if ((threadIdx.x & 31) == 0 && (nobs | npt)) {
        atomicAdd(&a.st->num_obs, (unsigned long long)nobs);
        atomicAdd(&a.st->num_points, (unsigned long long)npt);
    }
    const double bs = ba_block_sum(sumsq, s_warp);
    if (threadIdx.x == 0) a.part_pt[blockIdx.x] = bs;
    if (!ba_last_block(a.ticket, &s_flag)) return;
    const double tot = ba_ordered_sum(a.part_pt, a.nptch, 1, s_seg);
    if (threadIdx.x == 0) a.st->floor = tot;
}

// ---- evaluate the proposal: one thread per track ----
__global__ void __launch_bounds__(kBaBlock) k_ba_eval(const BaArgs a) {
    chain_enter();
    __shared__ double s_warp[kBaBlock / 32];
    if (__ldcg(&a.st->done) || __ldcg(&a.st->phase) != BA_EVAL) return;
    const int nxt = 1 - __ldcg(&a.st->cur);
    const long long t = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    double cost = 0.0;
    if (t < a.T && a.param[t]) {
        const long long o = a.offsets[t];
        const int n = (int)(a.offsets[t + 1] - o);
        const double* Xs = a.Xp + 3 * (nxt * a.T + t);
        const double X = Xs[0], Y = Xs[1], Z = Xs[2];
        double V[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, g[3] = {0.0, 0.0, 0.0};
        for (int j = 0; j < n; ++j) {
            const long long m = o + j;
            if (!a.inlist[m]) continue;
            const int c = a.view[m];
            double P[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) P[k] = a.Pprop[12 * c + k];
            const double2 uv = a.x[m];
            BaObsEq e;
            const double p2 = refine_p_residuals(P, a.K + 9 * c, X, Y, Z, uv.x, uv.y, e.r, e.Jc);
            const double ip = 1.0 / p2;
            const double u0 = fma(P[0], X, fma(P[1], Y, fma(P[2], Z, P[3]))) * ip;
            const double u1 = fma(P[4], X, fma(P[5], Y, fma(P[6], Z, P[7]))) * ip;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                e.Jp[0][k] = fma(-u0, P[8 + k], P[k]) * ip;
                e.Jp[1][k] = fma(-u1, P[8 + k], P[4 + k]) * ip;
            }
            if (c == a.anchor) e.Jc[0][3 + a.anchor_comp] = e.Jc[1][3 + a.anchor_comp] = 0.0;
            a.oeq[nxt * a.M + m] = e;
            if (!(p2 >= 0x1p-537) || !isfinite(e.r[0]) || !isfinite(e.r[1])) {
                cost = ba_inf();
                continue;
            }
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                cost = fma(e.r[k], e.r[k], cost);
                int q = 0;
#pragma unroll
                for (int p = 0; p < 3; ++p)
#pragma unroll
                    for (int mm = p; mm < 3; ++mm, ++q) V[q] = fma(e.Jp[k][p], e.Jp[k][mm], V[q]);
#pragma unroll
                for (int p = 0; p < 3; ++p) g[p] = fma(e.Jp[k][p], e.r[k], g[p]);
            }
        }
        BaPtEq pe;
        for (int k = 0; k < 6; ++k) pe.V[k] = V[k];
        for (int k = 0; k < 3; ++k) pe.g[k] = g[k];
        pe.pad = 0.0;
        a.peq[nxt * a.T + t] = pe;
    }
    const double bs = ba_block_sum(cost, s_warp);
    if (threadIdx.x == 0) a.part_pt[blockIdx.x] = bs;
}

// ---- the per-view sums of the proposal: one block per chunk of kBaObsChunk view-major observations ----
__global__ void __launch_bounds__(kBaBlock) k_ba_views(const BaArgs a) {
    chain_enter();
    constexpr int NV = 27;
    __shared__ double s_w[kBaBlock / 32][NV];
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_EVAL) return;
    const int nxt = 1 - __ldcg(&st->cur);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long ch = blockIdx.x;
    if (ch < a.nvch) {
        double acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = 0.0;
        const long long b0 = a.vch_begin[ch], b1 = a.vch_begin[ch + 1];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const long long i = b0 + half * kBaBlock + tid;
            if (i < b1) {
                const int m = a.vperm[i];
                if (a.inlist[m]) {
                    const BaObsEq& e = a.oeq[nxt * a.M + m];
                    double Jc[2][6], r[2];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        r[k] = e.r[k];
#pragma unroll
                        for (int p = 0; p < 6; ++p) Jc[k][p] = e.Jc[k][p];
                    }
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        int q = 0;
#pragma unroll
                        for (int p = 0; p < 6; ++p)
#pragma unroll
                            for (int mm = p; mm < 6; ++mm, ++q) acc[q] = fma(Jc[k][p], Jc[k][mm], acc[q]);
#pragma unroll
                        for (int p = 0; p < 6; ++p) acc[21 + p] = fma(Jc[k][p], r[k], acc[21 + p]);
                    }
                }
            }
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            double x = acc[v];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
            if (lane == 0) s_w[warp][v] = x;
        }
        __syncthreads();
        if (tid < NV) {
            double x = s_w[0][tid];
#pragma unroll
            for (int w = 1; w < kBaBlock / 32; ++w) x += s_w[w][tid];
            a.part_v[ch * NV + tid] = x;
        }
    }
}

// ---- U_c and g_c of the proposal: one warp per (free view, entry) adds the view's chunk partials (lane j takes chunks
// j, j + 32, ... in order, then a fixed butterfly); the last block accepts or rejects, as refine_control ----
__global__ void __launch_bounds__(kBaBlock) k_ba_views_sum(const BaArgs a) {
    chain_enter();
    constexpr int NV = 27;
    __shared__ double s_seg[kBaBlock];
    __shared__ int s_flag;
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_EVAL) return;
    const int nxt = 1 - __ldcg(&st->cur);
    const int tid = threadIdx.x, lane = tid & 31;
    const long long wi = (long long)blockIdx.x * (kBaBlock / 32) + (tid >> 5);
    if (wi < (long long)a.F * NV) {
        const int f = (int)(wi / NV), v = (int)(wi % NV);
        double x = 0.0;
        for (long long c = a.vfirst[f] + lane; c < a.vfirst[f + 1]; c += 32) x += __ldcg(a.part_v + c * NV + v);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
        if (lane == 0) {
            BaViewEq& ve = a.veq[nxt * a.F + f];
            if (v < 21) ve.U[v] = x;
            else ve.g[v - 21] = x;
        }
    }
    if (!ba_last_block(a.ticket, &s_flag)) return;
    const double c = ba_ordered_sum(a.part_pt, a.nptch, 1, s_seg);
    if (tid != 0) return;
    // refine_control's policy up to the solve
    BaState s = *st;
    bool accept;
    if (s.evals == 0) {
        s.cost_start = c;
        if (!isfinite(c)) {
            s.status = REFINE_NONFINITE;
            s.done = 1;
            s.evals = 1;
            *st = s;
            return;
        }
        accept = true;
    } else {
        s.iter += 1;
        accept = c < s.cost;
    }
    s.evals += 1;
    bool stop = false;
    if (accept) {
        const double before = s.cost;
        s.cur = nxt;
        s.cost = c;
        if (s.iter > 0) {
            s.lambda /= kRefineLambdaFactor;
            if (before - c <= kRefineFtol * before) {
                s.status = REFINE_CONVERGED;
                stop = true;
            }
        }
        if (!stop && c <= kRefineCostFloor * s.floor) {
            s.status = REFINE_CONVERGED;
            stop = true;
        }
    } else {
        s.lambda *= kRefineLambdaFactor;
        s.rejected += 1;
    }
    if (!stop && s.iter >= a.max_iter) {
        s.status = REFINE_MAX_ITER;
        stop = true;
    }
    if (!stop && !(s.lambda <= kRefineLambdaCap)) {
        s.status = REFINE_STALLED;
        stop = true;
    }
    if (stop) s.done = 1;
    else s.phase = BA_SOLVE;
    *st = s;
}

// the Marquardt scales of free view f from the current equations
__device__ __forceinline__ void ba_view_scale(const BaArgs& a, int cur, int f, double (&D)[6]) {
    const double* U = a.veq[cur * a.F + f].U;
#pragma unroll
    for (int p = 0; p < 6; ++p) D[p] = ba_scale(__ldcg(U + ba_d6(p)));
}

// ---- per parameter point: D_p, V_hat_p^-1 and g_hat_p (one thread per track) ----
__global__ void __launch_bounds__(kBaBlock) k_ba_schur_pts(const BaArgs a) {
    chain_enter();
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE) return;
    const long long t = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    if (t >= a.T || !a.param[t]) return;
    const int cur = __ldcg(&st->cur);
    const double lam = __ldcg(&st->lambda);
    const BaPtEq pe = a.peq[cur * a.T + t];
    double Dp[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) Dp[k] = ba_scale(pe.V[ba_u3(k, k)]);
    // Cholesky of the damped scaled 3 x 3 block (refine_solve's rule), then its inverse
    double L[3][3];
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double v = pe.V[ba_u3(i, j)] / (Dp[i] * Dp[j]) + (i == j ? lam : 0.0);
#pragma unroll
            for (int k = 0; k < j; ++k) v = fma(-L[i][k], L[j][k], v);
            if (i == j) {
                if (!(v > 0.0) || !isfinite(v)) ok = false;
                L[i][i] = sqrt(v);
            } else {
                L[i][j] = v / L[j][j];
            }
        }
    if (!ok) {
        st->fail = 1;
        return;
    }
    BaPtSolve ps;
#pragma unroll
    for (int c = 0; c < 3; ++c) {  // column c of the inverse: L z = e_c, L^T x = z
        double z[3], xx[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double v = i == c ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < i; ++k) v = fma(-L[i][k], z[k], v);
            z[i] = v / L[i][i];
        }
#pragma unroll
        for (int i = 2; i >= 0; --i) {
            double v = z[i];
#pragma unroll
            for (int k = i + 1; k < 3; ++k) v = fma(-L[k][i], xx[k], v);
            xx[i] = v / L[i][i];
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) ps.Vi[3 * i + c] = xx[i];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        ps.g[k] = pe.g[k] / Dp[k];
        ps.D[k] = Dp[k];
    }
    ps.pad = 0.0;
    a.psol[t] = ps;
}

// ---- per list observation in a free view: W_hat, Y, e (one thread per observation) ----
__global__ void __launch_bounds__(kBaBlock) k_ba_schur_obs(const BaArgs a) {
    chain_enter();
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE || __ldcg(&st->fail)) return;
    const long long m = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    if (m >= a.M || !a.inlist[m]) return;
    const int f = a.fidx[a.view[m]];
    if (f < 0) return;
    const int cur = __ldcg(&st->cur);
    const BaPtSolve ps = a.psol[a.otrack[m]];
    double Dc[6];
    ba_view_scale(a, cur, f, Dc);
    const BaObsEq& e = a.oeq[cur * a.M + m];
    BaObsSchur sc;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s)
            sc.W[r][s] = fma(e.Jc[1][r], e.Jp[1][s], e.Jc[0][r] * e.Jp[0][s]) / (Dc[r] * ps.D[s]);
#pragma unroll
    for (int r = 0; r < 6; ++r) {
#pragma unroll
        for (int s = 0; s < 3; ++s)
            sc.Y[r][s] = fma(sc.W[r][2], ps.Vi[6 + s], fma(sc.W[r][1], ps.Vi[3 + s], sc.W[r][0] * ps.Vi[s]));
        sc.e[r] = fma(sc.Y[r][2], ps.g[2], fma(sc.Y[r][1], ps.g[1], sc.Y[r][0] * ps.g[0]));
    }
    a.osch[m] = sc;
}

// ---- S-block partials (one thread per chunk of observation pairs) and right-hand side partials (per view chunk) ----
__global__ void __launch_bounds__(kBaBlock) k_ba_schur(const BaArgs a) {
    chain_enter();
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE || __ldcg(&st->fail)) return;
    const long long i = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    if (i < a.ntch) {
        double acc[36];
#pragma unroll
        for (int q = 0; q < 36; ++q) acc[q] = 0.0;
        for (long long k = a.tch_begin[i]; k < a.tch_begin[i + 1]; ++k) {
            const int2 pr = a.triples[k];
            if (!a.inlist[pr.x] || !a.inlist[pr.y]) continue;
            const BaObsSchur& si = a.osch[pr.x];
            const BaObsSchur& sj = a.osch[pr.y];
            double Y[6][3], W[6][3];
#pragma unroll
            for (int r = 0; r < 6; ++r)
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    Y[r][s] = si.Y[r][s];
                    W[r][s] = sj.W[r][s];
                }
#pragma unroll
            for (int r = 0; r < 6; ++r)
#pragma unroll
                for (int s = 0; s < 6; ++s)
                    acc[6 * r + s] = fma(Y[r][2], W[s][2], fma(Y[r][1], W[s][1], fma(Y[r][0], W[s][0], acc[6 * r + s])));
        }
#pragma unroll
        for (int q = 0; q < 36; ++q) a.part_t[i * 36 + q] = acc[q];
    } else if (i < a.ntch + a.nvch) {
        const long long ch = i - a.ntch;
        double e[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (long long p = a.vch_begin[ch]; p < a.vch_begin[ch + 1]; ++p) {
            const int m = a.vperm[p];
            if (!a.inlist[m]) continue;
#pragma unroll
            for (int k = 0; k < 6; ++k) e[k] += a.osch[m].e[k];
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) a.part_r[ch * 6 + k] = e[k];
    }
}

// ---- S (lower triangle) and the right-hand side row.  Threads [0, ntri + n): one per entry outside every S block with
// observation pairs (U_hat + lambda on the diagonal blocks, 0 elsewhere, the identity on the padding).  Then one warp
// per entry of such a block and per right-hand side entry (lane j adds chunks j, j + 32, ... in order, then a fixed
// butterfly). ----
__global__ void __launch_bounds__(256) k_ba_schur_sum(const BaArgs a) {
    chain_enter();
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE || __ldcg(&st->fail)) return;
    const long long n = a.npad, ntri = n * (n + 1) / 2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int cur = __ldcg(&st->cur);
    const int n6 = 6 * a.F;
    if (gid < ntri + n) {
        if (gid >= ntri) {  // right-hand side padding
            if (gid - ntri >= n6) a.S[n * n + (gid - ntri)] = 0.0;
            return;
        }
        long long R = (long long)((sqrt(8.0 * (double)gid + 1.0) - 1.0) * 0.5);
        while (R * (R + 1) / 2 > gid) --R;
        while ((R + 1) * (R + 2) / 2 <= gid) ++R;
        const long long C = gid - R * (R + 1) / 2;
        double v;
        if (R >= n6) {
            v = R == C ? 1.0 : 0.0;
        } else {
            const int fa = (int)(R / 6), fc = (int)(C / 6), r = (int)(R % 6), s = (int)(C % 6);
            if (a.blk_id[fa * a.F + fc] >= 0) return;  // a warp's
            v = 0.0;
            if (fa == fc) {
                double D[6];
                ba_view_scale(a, cur, fa, D);
                v = __ldcg(a.veq[cur * a.F + fa].U + ba_u6(r, s)) / (D[r] * D[s]) + (r == s ? __ldcg(&st->lambda) : 0.0);
            }
        }
        a.S[R * n + C] = v;
        return;
    }
    const long long base = (ntri + n + 31) / 32 * 32;  // the warps start on a warp boundary
    if (gid < base) return;
    const long long w = (gid - base) >> 5;
    const int lane = threadIdx.x & 31;
    if (w < a.nblk * 36) {
        const int b = (int)(w / 36), r = (int)(w % 36) / 6, s = (int)(w % 6);
        const int2 ac = a.blk_ac[b];
        if (ac.x == ac.y && r < s) return;
        double sum = 0.0;
        for (long long ch = a.bfirst[b] + lane; ch < a.bfirst[b + 1]; ch += 32) sum += __ldcg(a.part_t + ch * 36 + 6 * r + s);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
        if (lane) return;
        double v = 0.0;
        if (ac.x == ac.y) {
            double D[6];
            ba_view_scale(a, cur, ac.x, D);
            v = __ldcg(a.veq[cur * a.F + ac.x].U + ba_u6(r, s)) / (D[r] * D[s]) + (r == s ? __ldcg(&st->lambda) : 0.0);
        }
        a.S[(6LL * ac.x + r) * n + 6LL * ac.y + s] = v - sum;
    } else if (w < a.nblk * 36 + n6) {  // right-hand side: -g_hat_c + sum_i Y_i g_hat_p
        const int C = (int)(w - a.nblk * 36), f = C / 6, s = C % 6;
        double sum = 0.0;
        for (long long ch = a.vfirst[f] + lane; ch < a.vfirst[f + 1]; ch += 32) sum += __ldcg(a.part_r + ch * 6 + s);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
        if (lane) return;
        double D[6];
        ba_view_scale(a, cur, f, D);
        a.S[n * n + C] = sum - __ldcg(a.veq[cur * a.F + f].g + s) / D[s];
    }
}

// ---- tiled Cholesky, tile column j: block b factors tile row j + b (left-looking); every block factors the diagonal
// tile itself (the same bits), so one launch per tile column suffices.  Every block of the launch reads A_jj from S, so
// no block may overwrite it: block 0 writes L_jj to Ldiag, which only k_ba_backsolve reads (the later launches read
// only the off-diagonal tiles of S).  The last tile row holds the right-hand side, whose factor row is the forward
// substitution's z. ----
__global__ void __launch_bounds__(kBaCholThreads) k_ba_chol(const BaArgs a, int j) {
    chain_enter();
    constexpr int TT = kBaTile, PER = TT * TT / kBaCholThreads;
    __shared__ double sA[TT][TT + 1], sB[TT][TT + 1], sLj[TT][TT + 1], sLi[TT][TT + 1];
    __shared__ int s_bad;
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE || __ldcg(&st->fail)) return;
    const int tid = threadIdx.x;
    const long long n = a.npad;
    const int i = j + blockIdx.x;
    const bool off = i != j;
    const long long rj = (long long)j * TT, ri = (long long)i * TT;
    double accA[PER], accB[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) {
        const int e = tid + q * kBaCholThreads, r = e / TT, s = e % TT;
        accA[q] = r >= s ? __ldcg(a.S + (rj + r) * n + rj + s) : 0.0;
        accB[q] = off ? __ldcg(a.S + (ri + r) * n + rj + s) : 0.0;
    }
    for (int k = 0; k < j; ++k) {
        const long long ck = (long long)k * TT;
        __syncthreads();
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + q * kBaCholThreads, r = e / TT, s = e % TT;
            sLj[r][s] = __ldcg(a.S + (rj + r) * n + ck + s);
            if (off) sLi[r][s] = __ldcg(a.S + (ri + r) * n + ck + s);
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + q * kBaCholThreads, r = e / TT, s = e % TT;
            double v = accA[q], w = accB[q];
            for (int m = 0; m < TT; ++m) {
                v = fma(-sLj[r][m], sLj[s][m], v);
                if (off) w = fma(-sLi[r][m], sLj[s][m], w);
            }
            accA[q] = v;
            accB[q] = w;
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < PER; ++q) {
        const int e = tid + q * kBaCholThreads, r = e / TT, s = e % TT;
        sA[r][s] = accA[q];
        sB[r][s] = accB[q];
    }
    if (tid == 0) s_bad = 0;
    __syncthreads();
    for (int c = 0; c < TT; ++c) {  // the diagonal tile, right-looking in shared memory
        if (tid == 0) {
            const double piv = sA[c][c];
            if (!(piv > 0.0) || !isfinite(piv)) s_bad = 1;
            sA[c][c] = sqrt(piv);
        }
        __syncthreads();
        if (s_bad) break;
        if (tid > c && tid < TT) sA[tid][c] = sA[tid][c] / sA[c][c];
        __syncthreads();
        for (int e = tid; e < TT * TT; e += kBaCholThreads) {
            const int r = e / TT, s = e % TT;
            if (s > c && r >= s) sA[r][s] = fma(-sA[r][c], sA[s][c], sA[r][s]);
        }
        __syncthreads();
    }
    if (s_bad) {
        if (tid == 0) st->fail = 1;  // every block finds the same pivot: the same store
        return;
    }
    if (!off) {
        for (int e = tid; e < TT * TT; e += kBaCholThreads) {
            const int r = e / TT, s = e % TT;
            a.Ldiag[(long long)j * TT * TT + r * TT + s] = r >= s ? sA[r][s] : 0.0;
        }
        return;
    }
    if (tid < TT) {  // X L_jj^T = B, row by row
        const int r = tid;
        for (int c = 0; c < TT; ++c) {
            double v = sB[r][c];
            for (int m = 0; m < c; ++m) v = fma(-sB[r][m], sA[c][m], v);
            sB[r][c] = v / sA[c][c];
        }
    }
    __syncthreads();
    for (int e = tid; e < TT * TT; e += kBaCholThreads) {
        const int r = e / TT, s = e % TT;
        a.S[(ri + r) * n + rj + s] = sB[r][s];
    }
}

// ---- L^T y = z (one block: kBaSolveSlices slices of the rows below each tile, then one warp sweeps the tile) ----
__global__ void __launch_bounds__(kBaTile * kBaSolveSlices) k_ba_backsolve(const BaArgs a) {
    chain_enter();
    constexpr int TT = kBaTile;
    __shared__ double sy[6 * kBaMaxViews];
    __shared__ double sp[kBaSolveSlices][TT + 1];
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE || __ldcg(&st->fail)) return;
    const int n = a.npad, nt = n / TT, tid = threadIdx.x, r = tid % TT, sl = tid / TT;
    for (int J = nt - 1; J >= 0; --J) {
        const int col = J * TT + r;
        double p = 0.0;
        for (int k = (J + 1) * TT + sl; k < n; k += kBaSolveSlices) p = fma(__ldcg(a.S + (long long)k * n + col), sy[k], p);
        sp[sl][r] = p;
        __syncthreads();
        if (sl == 0) {
            double v = __ldcg(a.S + (long long)n * n + col);
            for (int q = 0; q < kBaSolveSlices; ++q) v -= sp[q][r];
            for (int rr = TT - 1; rr >= 0; --rr) {
                double yv = 0.0;
                if (r == rr) {
                    yv = v / __ldcg(a.Ldiag + (long long)J * TT * TT + r * TT + r);
                    sy[col] = yv;
                }
                yv = __shfl_sync(0xffffffffu, yv, rr);
                if (r < rr) v = fma(-__ldcg(a.Ldiag + (long long)J * TT * TT + rr * TT + r), yv, v);
            }
        }
        __syncthreads();
    }
    for (int k = tid; k < n; k += blockDim.x) a.y[k] = sy[k];
}

// ---- the point steps and the proposal: one thread per track; the last block checks Xtol and moves the poses ----
__global__ void __launch_bounds__(kBaBlock) k_ba_points(const BaArgs a) {
    chain_enter();
    __shared__ double s_warp[kBaBlock / 32];
    __shared__ double s_seg[kBaBlock];
    __shared__ int s_flag;
    BaState* st = a.st;
    if (__ldcg(&st->done) || __ldcg(&st->phase) != BA_SOLVE) return;
    const bool failed = __ldcg(&st->fail) != 0;
    const int cur = __ldcg(&st->cur), nxt = 1 - cur;
    const long long t = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    double n2 = 0.0;
    if (!failed && t < a.T && a.param[t]) {
        const BaPtSolve ps = a.psol[t];
        double acc[3] = {-ps.g[0], -ps.g[1], -ps.g[2]};
        const long long o = a.offsets[t];
        const int n = (int)(a.offsets[t + 1] - o);
        for (int j = 0; j < n; ++j) {
            const long long m = o + j;
            if (!a.inlist[m]) continue;
            const int f = a.fidx[a.view[m]];
            if (f < 0) continue;
            const BaObsSchur& sc = a.osch[m];
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int r = 0; r < 6; ++r) acc[k] = fma(-sc.W[r][k], __ldcg(a.y + 6 * f + r), acc[k]);
        }
        const BaPtEq& pe = a.peq[cur * a.T + t];
        const double* X = a.Xp + 3 * (cur * a.T + t);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double yk = fma(ps.Vi[3 * k + 2], acc[2], fma(ps.Vi[3 * k + 1], acc[1], ps.Vi[3 * k] * acc[0]));
            n2 = fma(yk, yk, n2);
            a.Xp[3 * (nxt * a.T + t) + k] = X[k] + yk / ba_scale(pe.V[ba_u3(k, k)]);
        }
    }
    const double bs = ba_block_sum(n2, s_warp);
    if (threadIdx.x == 0) a.part_pt[blockIdx.x] = bs;
    if (!ba_last_block(a.ticket, &s_flag)) return;
    if (failed) {  // not numerically positive definite: lambda x 10 and solve again
        if (threadIdx.x == 0) {
            st->fail = 0;
            const double lam = st->lambda * kRefineLambdaFactor;
            st->lambda = lam;
            if (!(lam > 0.0 && lam <= kRefineLambdaCap)) {  // lambda underflowed to 0 (accepts) cannot grow: stalled
                st->status = REFINE_STALLED;
                st->done = 1;
            }
        }
        return;
    }
    const double pts = ba_ordered_sum(a.part_pt, a.nptch, 1, s_seg);
    __shared__ int s_conv;
    if (threadIdx.x == 0) {
        double c2 = 0.0;
        for (int k = 0; k < 6 * a.F; ++k) {
            const double yk = __ldcg(a.y + k);
            c2 = fma(yk, yk, c2);
        }
        const double tot = c2 + pts;
        s_conv = sqrt(tot) <= kRefineXtol * sqrt(st->cost);
        if (s_conv) {
            st->status = REFINE_CONVERGED;
            st->done = 1;
        }
    }
    __syncthreads();
    if (s_conv) return;
    for (int c = threadIdx.x; c < a.V; c += kBaBlock) {
        const int f = a.fidx[c];
        if (f < 0) continue;
        double D[6], d[6];
        ba_view_scale(a, cur, f, D);
#pragma unroll
        for (int k = 0; k < 6; ++k) d[k] = __ldcg(a.y + 6 * f + k) / D[k];
        const double* p = a.pose + 12 * (cur * a.V + c);
        double q[12];
        refine_rotate(p, d, q);
#pragma unroll
        for (int k = 0; k < 3; ++k) q[9 + k] = (c == a.anchor && k == a.anchor_comp) ? p[9 + k] : p[9 + k] + d[3 + k];
        double* pn = a.pose + 12 * (nxt * a.V + c);
        for (int k = 0; k < 12; ++k) pn[k] = q[k];
        double m[12], P[12];
        ba_Rt(q, m);
        pnp_projection(a.K + 9 * c, m, P);
        for (int k = 0; k < 12; ++k) a.Pprop[12 * c + k] = P[k];
    }
    if (threadIdx.x == 0) st->phase = BA_EVAL;
}

// ---- the reported parameters and the report (one block) ----
__global__ void __launch_bounds__(256) k_ba_finish(const BaArgs a) {
    chain_enter();
    const BaState s = *a.st;
    const bool keep = s.status == REFINE_NONFINITE;
    for (int c = threadIdx.x; c < a.V; c += blockDim.x) {
        double m[12], P[12];
        if (keep) {
            for (int k = 0; k < 12; ++k) m[k] = a.Rt[12 * c + k];
        } else {
            ba_Rt(a.pose + 12 * (s.cur * a.V + c), m);
        }
        pnp_projection(a.K + 9 * c, m, P);
        for (int k = 0; k < 12; ++k) {
            a.Rt_out[12 * c + k] = m[k];
            a.Prep[12 * c + k] = P[k];
        }
    }
    if (threadIdx.x == 0) {
        BaReport r;
        r.cost_start = s.cost_start;
        r.cost_final = keep ? s.cost_start : s.cost;
        r.num_observations = (long long)s.num_obs;
        r.num_points = (long long)s.num_points;
        r.num_free_views = a.F;
        r.iterations = s.iter;
        r.status = s.status;
        r.rejected = s.rejected;
        *a.report = r;
    }
}

// ---- the reported points, mask and err: one thread per track ----
__global__ void __launch_bounds__(kBaBlock) k_ba_mask(const BaArgs a) {
    chain_enter();
    const long long t = (long long)blockIdx.x * kBaBlock + threadIdx.x;
    if (t >= a.T) return;
    const bool keep = __ldcg(&a.st->status) == REFINE_NONFINITE;
    const double* Xs = keep ? a.X0 + 3 * t : a.Xp + 3 * (__ldcg(&a.st->cur) * a.T + t);
    const double X[3] = {Xs[0], Xs[1], Xs[2]};
    for (int k = 0; k < 3; ++k) a.X_out[3 * t + k] = X[k];
    const long long o = a.offsets[t];
    const int n = (int)(a.offsets[t + 1] - o);
    for (int j = 0; j < n; ++j) {
        const int c = a.view[o + j];
        double P[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) P[k] = __ldcg(a.Prep + 12 * c + k);
        const double2 uv = a.x[o + j];
        PnpRec r;
        r.X = X[0]; r.Y = X[1]; r.Z = X[2]; r.u = uv.x; r.v = uv.y; r.pad = 0.0;
        double val;
        a.mask[o + j] = pnp_exact(P, r, a.thr, val);
        a.err[o + j] = val;
    }
}

}  // namespace sfm
