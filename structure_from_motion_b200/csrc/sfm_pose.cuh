// K5 — essential-matrix decomposition, cheirality vote and DLT triangulation.
#pragma once
#include "sfm_device.cuh"
#include "sfm_pose_math.cuh"
#include "sfm_types.h"

namespace sfm {

__global__ void k_decompose(const double* __restrict__ E, const Best* __restrict__ best,
                            long long idx_offset, PoseSet* __restrict__ out, int npairs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs) return;
    const double* src = E + 9 * (long long)i;
    if (best) {  // single-pair pipeline: decompose the RANSAC winner in place on the device
        const long long local = best->idx - idx_offset;
        if (local < 0) { out[i].best = -2; return; }
        src = E + 9 * local;
    }
    double e[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) e[k] = src[k];
    decompose_essential(e, out[i]);
}

// _cheirality_check for the 4 candidates of one pair (lib/epipolar/eight_point.py:449-488,
// looped as in :210-230).  One thread per (correspondence, candidate pose): the four poses of a
// correspondence sit in four consecutive lanes (the 4x4 Jacobi SVDs are latency-bound, so the pose loop
// is spread over lanes instead of running in sequence).  pass[i] bit p = correspondence i passes pose p.
// counts follow the reference's np.count_nonzero(passing_indices) (:228-230): correspondence 0 never counts.
__global__ void __launch_bounds__(128)
k_cheirality(const Corr* __restrict__ pts, long long m, const long long* __restrict__ gather,
             const long long* __restrict__ m_dev, PoseSet* __restrict__ poses, double dist_thr,
             uint8_t* __restrict__ pass, const int32_t* __restrict__ quirk_row,
             const Best* __restrict__ quirk_best = nullptr, long long quirk_offset = 0) {
    // quirk_best != null: quirk_row is the BASE of the sample table and the winner's row is looked up on the device
    if (quirk_best) quirk_row = quirk_best->idx >= 0 ? quirk_row + 8 * (quirk_best->idx - quirk_offset) : nullptr;
    // gather != null: correspondence i is pts[gather[i]] and the count lives on the device
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long i = t >> 2;
    const int p = (int)(t & 3);
    if (m_dev) m = *m_dev;
    __shared__ int s_cnt[4];
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    bool ok = false, counts = false;
    if (i < m) {
        const long long gi = gather ? gather[i] : i;
        const Corr c = pts[gi];
        const double P1[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};  // Transform3D.identity() (:473)
        double P2[12];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            P2[4 * r + 0] = poses->R[p][3 * r + 0];
            P2[4 * r + 1] = poses->R[p][3 * r + 1];
            P2[4 * r + 2] = poses->R[p][3 * r + 2];
            P2[4 * r + 3] = poses->t[p][r];
        }
        double X1[3];
        dlt_triangulate(c.xa, c.ya, c.xb, c.yb, P1, P2, X1);
        const double z2 = fma(P2[8], X1[0], fma(P2[9], X1[1], fma(P2[10], X1[2], P2[11])));  // :476
        const double nrm = sqrt(fma(X1[2], X1[2], fma(X1[1], X1[1], X1[0] * X1[0])));
        ok = (X1[2] >= -kCheiralityTolerance) && (z2 >= -kCheiralityTolerance) && (nrm <= dist_thr);  // :478-487
        // the count_nonzero-of-indices quirk (:228-230): the correspondence at list position 0
        // never counts.  In the fused pipeline position 0 is the winner's first sample point
        // (lib/ransac/ransac.py:76 returns the samples first).
        const bool has_row = quirk_row && quirk_row[0] >= 0;  // a row of -1 = no sample table
        counts = ok && !(has_row ? (gi == quirk_row[0]) : (i == 0));
    }
    const unsigned lane = threadIdx.x & 31u;
    const unsigned okb = __ballot_sync(0xffffffffu, ok);
    if (i < m && p == 0) pass[i] = (uint8_t)((okb >> (lane & ~3u)) & 0xfu);
    const unsigned cb = __ballot_sync(0xffffffffu, counts);
    if (lane < 4) {
        const int n = __popc(cb & (0x11111111u << lane));  // lanes with pose == lane
        if (n) atomicAdd(&s_cnt[lane], n);
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_cnt[threadIdx.x])
        atomicAdd((unsigned long long*)&poses->counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

// np.argmax(num_good_correspondences) (:237): first maximum.
__global__ void k_vote(PoseSet* poses) {
    if (threadIdx.x || blockIdx.x) return;
    int b = 0;
    for (int p = 1; p < 4; ++p)
        if (poses->counts[p] > poses->counts[b]) b = p;
    poses->best = b;
}

// triangulate_points (lib/epipolar/triangulation.py:42-62), pixel coordinates.
// When use_vote != 0 the second camera is K [R|t] of the voted pose (built on the device)
// and only correspondences passing that pose are triangulated (others get NaN) — the fused
// tail of the single-pair pipeline (apps/sfm.py:133-186).
__global__ void __launch_bounds__(128)
k_triangulate(const double* __restrict__ xa, const double* __restrict__ ya, const double* __restrict__ xb,
              const double* __restrict__ yb, long long stride, long long m, const long long* __restrict__ m_dev,
              const double* __restrict__ P1g, const double* __restrict__ P2g, const double* __restrict__ Kmat,
              const PoseSet* __restrict__ poses, const uint8_t* __restrict__ pass, int use_vote,
              double* __restrict__ X, const long long* __restrict__ gather = nullptr) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (m_dev) m = *m_dev;
    if (i >= m) return;
    const long long gi = gather ? gather[i] : i;
    double P1[12], P2[12];
    if (use_vote) {
        const int b = poses->best;
        const double* R = poses->R[b];
        const double* t = poses->t[b];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                // K_ext @ Tmat: K[r,:] . [R|t][:,c]
                const double a0 = (c < 3) ? R[c] : t[0], a1 = (c < 3) ? R[3 + c] : t[1],
                             a2 = (c < 3) ? R[6 + c] : t[2];
                P2[4 * r + c] = fma(Kmat[3 * r + 2], a2, fma(Kmat[3 * r + 1], a1, Kmat[3 * r] * a0));
                P1[4 * r + c] = (c < 3) ? Kmat[3 * r + c] : 0.0;
            }
        if (!((pass[i] >> b) & 1u)) {
            const double nan = __longlong_as_double(0x7ff8000000000000LL);
            X[3 * i] = nan; X[3 * i + 1] = nan; X[3 * i + 2] = nan;
            return;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) { P1[k] = P1g[k]; P2[k] = P2g[k]; }
    }
    double Xo[3];
    dlt_triangulate(xa[gi * stride], ya[gi * stride], xb[gi * stride], yb[gi * stride], P1, P2, Xo);
    X[3 * i] = Xo[0];
    X[3 * i + 1] = Xo[1];
    X[3 * i + 2] = Xo[2];
}

}  // namespace sfm
