// Multi-view triangulation of tracks (sfm_triangulate_tracks): one 3-D point per track, from the track's observations
// in V registered views, with outlier observations rejected.
//
// Inputs.  Cameras K[V][9] (upper triangular, K[2,2] = 1) and Rt[V][12] (world to camera, x_cam = R X + t, the PnP
// convention); P_c = pnp_projection(K_c, Rt_c).  Tracks in CSR form: offsets int64[T+1] (offsets[0] = 0, non-decreasing),
// view int32[M], x double[M][2] (pixels).  A track has at most kMaxTrack observations.
//
// Decision.  Observation (u, v) of view c under a point X: pnp_exact(P_c, {X, u, v}, thr) - p2 >= 2^-537 (in front of
// the camera), F < inf and F <= thr p2^2 - with the value F / p2^2 (px^2).  The PnP scorer's pinned evaluation, not a
// copy of it.
//
// Per track, in this order:
//   1. pair search   every pair (i < j) of the track's observations, in lexicographic order, triangulated by
//                    dlt_triangulate(P_i, P_j).  A pair is a candidate iff both its observations pass under its point.
//                    The winner is the candidate with the most passing observations of the track; ties go to the
//                    smaller sum of the passing values (summed in observation order), then to the lower pair index.
//                    No candidate: NO_PAIR; fewer than 2 observations: SHORT (both with X = NaN).
//   2. linear point  the N-view DLT over the winner's passing observations: the rows of dlt_triangulate, two per
//                    observation in observation order, reduced to a 4x4 triangular factor by Givens rotations (a
//                    streaming QR: never the normal equations), whose null vector null_vector4_fast gives (Jacobi SVD
//                    fallback, as in dlt_triangulate).  Two passing observations: the pair's point itself.  A
//                    non-finite result (a null vector at infinity) also keeps the pair's point.
//   3. refinement    only with max_iter > 0: Levenberg-Marquardt on X (MODEL_X of sfm_refine.cuh, 3 parameters, the
//                    shared refine_control).  The list is the observations passing under the linear point, fixed
//                    while it runs; the residuals are p0 / p2 - u and p1 / p2 - v, with p in pnp_terms' FMA order; a
//                    proposal under which a list observation has p2 < 2^-537 or a non-finite residual costs +inf.  The
//                    cost floor is kRefineCostFloor times the sum of u^2 + v^2 over the list.  Report: TrackRefineReport.
//   4. report        everything is a function of the reported X (refined, else linear) and the inputs: the mask and
//                    value of every observation, their count, the angle - the largest, over pairs of passing
//                    observations, between the lines of sight from the camera centres C = -R^T t to X,
//                    atan2(|a x b|, |a . b|) in [0, pi/2]: rays in opposite directions (a point on the baseline between
//                    two centres) are as degenerate as parallel ones - and the status: OK iff count >= min_views and
//                    angle >= min_angle, else FEW_INLIERS (count short) or SMALL_ANGLE.
//
// Frame.  All of it runs in one frame for the whole call: P's fourth column (K t) and the camera centres of every view
// are scaled by 2^-s, s the binary exponent of the largest |t| entry over all views, so that t is of the magnitude of R;
// X is reported times 2^s.  p changes by exactly 2^-s, so no decision or value changes.  The DLT's algebraic minimum
// does depend on the frame (scaling a column of its system), which is why it is fixed by t alone: a world scaled by
// 2^k (t with it) runs in the same frame and its report is bit-identical after exact rescaling, and pixels and K's
// first two rows scaled by 2^k leave the frame and, with the threshold scaled by 4^k, every decision unchanged.
//
// Mapping.  k_track_pairs: one thread per (track, pair) item of the tracks of 3 or more observations - short tracks
// fill warps with other tracks' items; the item's track is found by binary search over the item offsets.  It writes the
// pair's point, its passing set, count and sum, and whether it is a candidate.  k_track_solve: one thread per track -
// the pair search of a 2-observation track (its one pair), or the winner among the track's items (a scan in pair
// order); the linear point; the refinement (all iterations in this launch: tracks are independent); the report.  The
// bits of a track depend only on its own observations and the cameras: not on the grid, the other tracks or how a
// batch is split.
#pragma once
#include "sfm_pnp_model.cuh"
#include "sfm_pose_math.cuh"
#include "sfm_refine.cuh"

namespace sfm {

constexpr int kMaxTrack = 64;  // observations per track (the passing sets are 64-bit masks)
constexpr int kTrackBlock = 128;

enum { TRACK_OK = 0, TRACK_SHORT = 1, TRACK_NO_PAIR = 2, TRACK_FEW_INLIERS = 3, TRACK_SMALL_ANGLE = 4 };

// one registered view in the call's frame: P with its fourth column scaled by 2^-s, the camera centre scaled by 2^-s
struct TrackView {
    double P[12];
    double C[3];
    double pad;
};

// one (track, pair) item of the pair search
struct TrackPair {
    double X[3];
    double sum;   // passing values of the track, summed in observation order
    unsigned long long bits;  // the passing observations
    int count;    // their number
    int cand;     // both of the pair's observations pass
};

// layout of sfm_track_refinement (include/sfm_b200.h)
struct TrackRefineReport {
    double cost_start, cost_final;
    int num, iterations, status, rejected;
};

struct TrackArgs {
    const double* K;          // [V][9]
    const double* Rt;         // [V][12]
    int V;
    TrackView* views;         // [V]
    int* frame;               // [1] s
    const long long* offsets; // [T+1]
    const long long* pbase;   // [T+1] first item of each track
    const int* view;          // [M]
    const double2* x;         // [M]
    long long T, items;
    TrackPair* pairs;         // [items]
    double thr, min_angle;    // min_angle in radians
    int min_views, max_iter;
    double* X;                // [T][3]
    int* status;              // [T]
    int* num_inliers;         // [T]
    double* angle;            // [T]
    unsigned char* mask;      // [M]
    double* err;              // [M]
    TrackRefineReport* report;  // [T] or null (max_iter == 0)
};

__device__ __forceinline__ void track_load_P(const TrackView* v, double (&P)[12]) {
#pragma unroll
    for (int k = 0; k < 12; ++k) P[k] = __ldg(v->P + k);
}

// the decision and value of one observation under X (the call's frame)
__device__ __forceinline__ bool track_decide(const TrackView* v, double2 uv, const double (&X)[3], double thr, double& value) {
    double P[12];
    track_load_P(v, P);
    PnpRec r;
    r.X = X[0];
    r.Y = X[1];
    r.Z = X[2];
    r.u = uv.x;
    r.v = uv.y;
    r.pad = 0.0;
    return pnp_exact(P, r, thr, value);
}

// ---- the frame: P and C of every view, scaled by 2^-s (one block) ----
__global__ void __launch_bounds__(256) k_track_views(const TrackArgs a) {
    __shared__ double s_big[256];
    const int tid = threadIdx.x;
    double big = 0.0;
    for (int c = tid; c < a.V; c += blockDim.x)
#pragma unroll
        for (int r = 0; r < 3; ++r) big = fmax(big, fabs(a.Rt[12 * c + 4 * r + 3]));
    s_big[tid] = big;
    __syncthreads();
    for (int w = blockDim.x / 2; w > 0; w >>= 1) {  // max: any order gives the same bits
        if (tid < w) s_big[tid] = fmax(s_big[tid], s_big[tid + w]);
        __syncthreads();
    }
    big = s_big[0];
    const int s = big > 0.0 ? ilogb(big) : 0;
    if (tid == 0) *a.frame = s;
    for (int c = tid; c < a.V; c += blockDim.x) {
        const double* m = a.Rt + 12 * c;
        TrackView v;
        pnp_projection(a.K + 9 * c, m, v.P);
#pragma unroll
        for (int r = 0; r < 3; ++r) v.P[4 * r + 3] = scalbn(v.P[4 * r + 3], -s);
#pragma unroll
        for (int k = 0; k < 3; ++k)  // C = -R^T t
            v.C[k] = scalbn(-fma(m[8 + k], m[11], fma(m[4 + k], m[7], m[k] * m[3])), -s);
        v.pad = 0.0;
        a.views[c] = v;
    }
}

// ---- 1. pair search: one thread per (track, pair) item ----
__global__ void __launch_bounds__(kTrackBlock) k_track_pairs(const TrackArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.items) return;
    long long lo = 0, hi = a.T;  // pbase[lo] <= i < pbase[hi]: the track is the last with pbase <= i
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(a.pbase + mid) <= i) lo = mid;
        else hi = mid;
    }
    const long long o = __ldg(a.offsets + lo);
    const int n = (int)(__ldg(a.offsets + lo + 1) - o);
    int k = (int)(i - __ldg(a.pbase + lo)), p = 0;
    while (k >= n - 1 - p) {  // lexicographic pair index k -> (p, q)
        k -= n - 1 - p;
        ++p;
    }
    const int q = p + 1 + k;
    const double2 up = __ldg(a.x + o + p), uq = __ldg(a.x + o + q);
    double X[3];  // P straight from global memory: local copies would go to the stack for the non-inlined call
    dlt_triangulate(up.x, up.y, uq.x, uq.y, a.views[__ldg(a.view + o + p)].P, a.views[__ldg(a.view + o + q)].P, X);
    int count = 0;
    double sum = 0.0;
    unsigned long long bits = 0;
    for (int j = 0; j < n; ++j) {
        double val;
        if (track_decide(a.views + __ldg(a.view + o + j), __ldg(a.x + o + j), X, a.thr, val)) {
            ++count;
            sum += val;
            bits |= 1ull << j;
        }
    }
    TrackPair r;
    r.X[0] = X[0];
    r.X[1] = X[1];
    r.X[2] = X[2];
    r.sum = sum;
    r.bits = bits;
    r.count = count;
    r.cand = ((bits >> p) & (bits >> q) & 1ull) != 0;
    a.pairs[i] = r;
}

// the passing set of a track under X, as a bit mask over its observations, and its mask and err outputs
__device__ __forceinline__ unsigned long long track_judge(const TrackArgs& a, long long o, int n, const double (&X)[3]) {
    unsigned long long bits = 0;
    for (int j = 0; j < n; ++j) {
        double val;
        const bool ok = track_decide(a.views + __ldg(a.view + o + j), __ldg(a.x + o + j), X, a.thr, val);
        bits |= (unsigned long long)ok << j;
        a.mask[o + j] = ok;
        a.err[o + j] = val;
    }
    return bits;
}

// adds one row to the upper triangular factor R (row-major 4x4) by Givens rotations
__device__ __forceinline__ void track_givens(double (&R)[16], double (&r)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (r[k] == 0.0) continue;
        const double h = hypot(R[5 * k], r[k]);
        const double c = R[5 * k] / h, s = r[k] / h;
        R[5 * k] = h;
#pragma unroll
        for (int m = k + 1; m < 4; ++m) {
            const double rk = R[4 * k + m];
            R[4 * k + m] = fma(c, rk, s * r[m]);
            r[m] = fma(c, r[m], -s * rk);
        }
    }
}

// the N-view DLT over the observations in bits (the rows of dlt_triangulate, in observation order)
__device__ __forceinline__ void track_linear(const TrackArgs& a, long long o, unsigned long long bits, double (&X)[3]) {
    double R[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) R[k] = 0.0;
    while (bits) {
        const int j = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        double P[12];
        track_load_P(a.views + __ldg(a.view + o + j), P);
        const double2 uv = __ldg(a.x + o + j);
        double r0[4], r1[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            r0[c] = __dsub_rn(__dmul_rn(uv.y, P[8 + c]), P[4 + c]);  // v P[2,:] - P[1,:]
            r1[c] = __dsub_rn(P[c], __dmul_rn(uv.x, P[8 + c]));      // P[0,:] - u P[2,:]
        }
        track_givens(R, r0);
        track_givens(R, r1);
    }
    dlt_null_point(R, X);
}

// the residuals of one observation under X and their rows of the Jacobian (p in pnp_terms' FMA order); returns p2
__device__ __forceinline__ double track_residuals(const double (&P)[12], const double* X, double u, double v, double (&r)[2],
                                                  double (&J)[2][3]) {
    const double p0 = __fma_rn(P[0], X[0], __fma_rn(P[1], X[1], __fma_rn(P[2], X[2], P[3])));
    const double p1 = __fma_rn(P[4], X[0], __fma_rn(P[5], X[1], __fma_rn(P[6], X[2], P[7])));
    const double p2 = __fma_rn(P[8], X[0], __fma_rn(P[9], X[1], __fma_rn(P[10], X[2], P[11])));
    const double ip = 1.0 / p2;
    const double u0 = p0 * ip, u1 = p1 * ip;
    r[0] = u0 - u;
    r[1] = u1 - v;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        J[0][k] = fma(-u0, P[8 + k], P[k]) * ip;
        J[1][k] = fma(-u1, P[8 + k], P[4 + k]) * ip;
    }
    return p2;
}

// the totals refine_control<MODEL_X> takes (refine_nv layout) for the point x over the list, in observation order
__device__ __noinline__ inline void track_refine_eval(const TrackArgs& a, long long o, unsigned long long list, const double* x,
                                               double (&tot)[refine_nv<MODEL_X>()]) {
#pragma unroll
    for (int k = 0; k < refine_nv<MODEL_X>(); ++k) tot[k] = 0.0;
    while (list) {
        const int j = __ffsll((long long)list) - 1;
        list &= list - 1;
        double P[12];
        track_load_P(a.views + __ldg(a.view + o + j), P);
        const double2 uv = __ldg(a.x + o + j);
        tot[2] += fma(uv.x, uv.x, uv.y * uv.y);
        double r[2], J[2][3];
        const double p2 = track_residuals(P, x, uv.x, uv.y, r, J);
        if (!(p2 >= 0x1p-537) || !isfinite(r[0]) || !isfinite(r[1])) {
            tot[0] = __longlong_as_double(0x7ff0000000000000LL);
            continue;
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            tot[0] = fma(r[k], r[k], tot[0]);
            int q = 3;
#pragma unroll
            for (int p = 0; p < 3; ++p)
#pragma unroll
                for (int m = p; m < 3; ++m, ++q) tot[q] = fma(J[k][p], J[k][m], tot[q]);
#pragma unroll
            for (int p = 0; p < 3; ++p) tot[q + p] = fma(J[k][p], r[k], tot[q + p]);
        }
    }
}

// ---- 2-4. winner, linear point, refinement and report: one thread per track ----
__global__ void __launch_bounds__(kTrackBlock) k_track_solve(const TrackArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.T) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const long long o = a.offsets[t];
    const int n = (int)(a.offsets[t + 1] - o);
    const int s = *a.frame;
    int status = n < 2 ? TRACK_SHORT : TRACK_NO_PAIR;
    // the winner and its passing set; `fresh`: mask and err hold the decisions under X
    double X[3];
    unsigned long long in = 0;
    bool have = false, fresh = false;
    if (n == 2) {  // one pair: no item, the pair search is this thread's
        const TrackView* v0 = a.views + a.view[o];
        const TrackView* v1 = a.views + a.view[o + 1];
        const double2 x0 = a.x[o], x1 = a.x[o + 1];
        dlt_triangulate(x0.x, x0.y, x1.x, x1.y, v0->P, v1->P, X);
        in = track_judge(a, o, n, X);
        have = in == 3ull;
        fresh = true;
    } else if (n > 2) {
        long long best = -1;
        int bc = -1;
        double bs = 0.0;
        for (long long i = a.pbase[t]; i < a.pbase[t + 1]; ++i) {
            const TrackPair& r = a.pairs[i];
            if (r.cand && (r.count > bc || (r.count == bc && r.sum < bs))) {
                best = i;
                bc = r.count;
                bs = r.sum;
            }
        }
        if (best >= 0) {
            const TrackPair& r = a.pairs[best];
            X[0] = r.X[0];
            X[1] = r.X[1];
            X[2] = r.X[2];
            in = r.bits;
            have = true;
        }
    }
    TrackRefineReport rep;
    rep.cost_start = rep.cost_final = nan;
    rep.num = 0;
    rep.iterations = 0;
    rep.status = REFINE_NO_MODEL;
    rep.rejected = 0;
    if (!have) {
        for (int j = 0; j < n; ++j) {
            a.mask[o + j] = 0;
            a.err[o + j] = nan;
        }
        a.X[3 * t] = a.X[3 * t + 1] = a.X[3 * t + 2] = nan;
        a.status[t] = status;
        a.num_inliers[t] = 0;
        a.angle[t] = nan;
        if (a.report) a.report[t] = rep;
        return;
    }
    if (__popcll(in) > 2) {
        double L[3];
        track_linear(a, o, in, L);
        if (isfinite(L[0]) && isfinite(L[1]) && isfinite(L[2])) {
            X[0] = L[0];
            X[1] = L[1];
            X[2] = L[2];
            fresh = false;
        }
    }
    if (a.max_iter > 0) {
        if (!fresh) {
            in = track_judge(a, o, n, X);
            fresh = true;
        }
        const unsigned long long list = in;
        RefineState st;
        for (int k = 0; k < 12; ++k) st.x[k] = st.px[k] = 0.0;
        st.px[0] = X[0];
        st.px[1] = X[1];
        st.px[2] = X[2];
        st.cost = st.cost_ransac = st.cost_start = nan;
        st.lambda = kRefineLambda0;
        st.num = __popcll(list);
        st.iter = st.evals = st.rejected = st.pad = 0;
        st.status = REFINE_RUNNING;
        st.done = 0;
        double tot[refine_nv<MODEL_X>()];
        do {
            track_refine_eval(a, o, list, st.px, tot);
            refine_control<MODEL_X>(st, tot, a.max_iter);
        } while (!st.done);
        rep.cost_start = st.cost_start;
        rep.num = (int)st.num;
        rep.iterations = st.iter;
        rep.status = st.status;
        rep.rejected = st.rejected;
        if (st.status == REFINE_NONFINITE) {
            rep.cost_final = st.cost_start;
        } else {
            rep.cost_final = st.cost;
            X[0] = st.x[0];
            X[1] = st.x[1];
            X[2] = st.x[2];
            fresh = false;
        }
    }
    // the report under X
    if (!fresh) in = track_judge(a, o, n, X);
    double ang = 0.0;
    for (unsigned long long bi = in; bi; bi &= bi - 1) {
        const int i = __ffsll((long long)bi) - 1;
        const TrackView* vi = a.views + a.view[o + i];
        const double ra[3] = {X[0] - vi->C[0], X[1] - vi->C[1], X[2] - vi->C[2]};
        for (unsigned long long bj = bi & (bi - 1); bj; bj &= bj - 1) {
            const int j = __ffsll((long long)bj) - 1;
            const TrackView* vj = a.views + a.view[o + j];
            const double rb[3] = {X[0] - vj->C[0], X[1] - vj->C[1], X[2] - vj->C[2]};
            double cr[3];
            refine_cross(ra, rb, cr);
            const double sn = sqrt(fma(cr[0], cr[0], fma(cr[1], cr[1], cr[2] * cr[2])));
            const double cs = fma(ra[0], rb[0], fma(ra[1], rb[1], ra[2] * rb[2]));
            ang = fmax(ang, atan2(sn, fabs(cs)));
        }
    }
    const int cnt = __popcll(in);
    status = cnt < a.min_views ? TRACK_FEW_INLIERS : (ang >= a.min_angle ? TRACK_OK : TRACK_SMALL_ANGLE);
    a.X[3 * t] = scalbn(X[0], s);
    a.X[3 * t + 1] = scalbn(X[1], s);
    a.X[3 * t + 2] = scalbn(X[2], s);
    a.status[t] = status;
    a.num_inliers[t] = cnt;
    a.angle[t] = ang;
    if (a.report) a.report[t] = rep;
}

}  // namespace sfm
