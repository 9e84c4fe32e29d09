// Homography RANSAC: the 4-point fitter, the transfer-error scorer and the mask of one homography.
//
// Model.  H is 3x3 in pixel coordinates, maps image-A points to image-B points (x_b ~ H x_a) and is stored divided by
// H[2,2].  The backward map is adj(H) (homography_adj, sfm_device.cuh): the error is scale-invariant, so no inverse.
//
// Error.  The symmetric transfer error in px^2, d^2 = |x_b - pi(H x_a)|^2 + |x_a - pi(adj(H) x_b)|^2.  With p = H a~ and
// q = adj(H) b~:  F = (p0 - xb p2)^2 + (p1 - yb p2)^2,  G = (q0 - xa q2)^2 + (q1 - ya q2)^2,  P = p2^2,  Q = q2^2.
//   inlier   <=>  p2 != 0 && q2 != 0 && F Q + G P <= (thr P) Q     (every evaluation; division-free)
//   value     =   F / P + G / Q                                    (inliers only; summed)
// Both are pinned to one rounding order with __fma_rn/__dmul_rn/__dadd_rn/__ddiv_rn (transfer_terms and friends in
// sfm_device.cuh); oracle/transfer_exact.c evaluates the same order with fma() under -ffp-contract=off, so decisions and
// values are bit-identical to the oracle.  The mask is defined by the decision, not by "value <= thr".
//
// FP64 issue slots of one evaluation (the scorer's hot loop, counted from the source, one per DFMA/DMUL):
//   p = H a~ 6, q = adj(H) b~ 6, the four differences 4, F and G 4 (two DMUL + two DFMA), P and Q 2,
//   F Q + G P 2, (thr P) Q 2, the compare 1                                                    = 27
// The two "!= 0" tests read the bit patterns (integer pipe).  Pipe floor at the measured 18.35e12 DFMA/s per B200:
// 0.68e12 evaluations/s.  An inlier adds two divisions and the fixed-point conversion on top.
//
// RANSAC semantics (fit_with_ransac with model_fit_data_count = 4, lib/ransac/ransac.py:19-93): the 4 samples are
// columns 0-3 of the shared int32[H][8] sample table (reference sampler: perm[:4] of the same cumulative shuffle;
// device sampler: the first 4 of 8 distinct Philox draws, a uniform 4-subset), never counted as extra inliers and
// always in the error; K3 (k_finalise<MODEL_H>) applies the same selection rules as for E.  A sample with three
// collinear points in either image, or whose H[2,2] is 0 or not finite, is invalid: never a candidate, counted in
// num_invalid / first_invalid.
#pragma once
#include "sfm_device.cuh"
#include "sfm_fit.cuh"
#include "sfm_score.cuh"

namespace sfm {

// |2 x triangle area| below this (Hartley-normalised coordinates: mean distance sqrt(2) from the centroid) = collinear
constexpr double kCollinear = 1e-8;

// Hartley normalisation of 4 points: centroid, scale = sqrt(2) / mean distance; false when three are collinear
__device__ __forceinline__ bool hartley4(const double (&x)[4], const double (&y)[4], double (&nx)[4], double (&ny)[4],
                                         double& scale, double& cx, double& cy) {
    cx = __dadd_rn(__dadd_rn(__dadd_rn(x[0], x[1]), x[2]), x[3]) / 4.0;
    cy = __dadd_rn(__dadd_rn(__dadd_rn(y[0], y[1]), y[2]), y[3]) / 4.0;
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        nx[i] = __dsub_rn(x[i], cx);
        ny[i] = __dsub_rn(y[i], cy);
        s = __dadd_rn(s, sqrt(__dadd_rn(__dmul_rn(nx[i], nx[i]), __dmul_rn(ny[i], ny[i]))));
    }
    scale = sqrt(2.0) / (s / 4.0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        nx[i] = __dmul_rn(nx[i], scale);
        ny[i] = __dmul_rn(ny[i], scale);
    }
    bool ok = true;
#pragma unroll
    for (int o = 0; o < 4; ++o) {  // the triangle that leaves out point o
        const int i = o == 0 ? 1 : 0, j = o <= 1 ? 2 : 1, k = o <= 2 ? 3 : 2;
        const double area2 = fma(nx[j] - nx[i], ny[k] - ny[i], -((ny[j] - ny[i]) * (nx[k] - nx[i])));
        ok = ok && (fabs(area2) > kCollinear);  // NaN (coincident points: scale = inf) fails too
    }
    return ok;
}

// The exact 4-point solve: DLT A^T (9x8, two columns per correspondence) in Hartley-normalised coordinates, its
// Householder null vector (householder_qr_9x8 / householder_null_vector, shared with the eight-point fit), then
// H = T_b^-1 Hn T_a and H /= H[2,2].  Returns validity.
__device__ __forceinline__ bool homography_fit4(const Corr (&c)[4], double (&H)[9]) {
    double s1, c1x, c1y, s2, c2x, c2y;
    double M[9][8];
    bool ok;
    {
        double xa[4], ya[4], xb[4], yb[4], nxa[4], nya[4], nxb[4], nyb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            xa[i] = c[i].xa; ya[i] = c[i].ya; xb[i] = c[i].xb; yb[i] = c[i].yb;
        }
        ok = hartley4(xa, ya, nxa, nya, s1, c1x, c1y);
        ok = hartley4(xb, yb, nxb, nyb, s2, c2x, c2y) && ok;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double x = nxa[k], y = nya[k], u = nxb[k], v = nyb[k];
            // u (h6 x + h7 y + h8) - (h0 x + h1 y + h2) = 0  and  v (...) - (h3 x + h4 y + h5) = 0
            M[0][2 * k] = -x;  M[1][2 * k] = -y;  M[2][2 * k] = -1.0;
            M[3][2 * k] = 0.0; M[4][2 * k] = 0.0; M[5][2 * k] = 0.0;
            M[6][2 * k] = u * x; M[7][2 * k] = u * y; M[8][2 * k] = u;
            M[0][2 * k + 1] = 0.0; M[1][2 * k + 1] = 0.0; M[2][2 * k + 1] = 0.0;
            M[3][2 * k + 1] = -x;  M[4][2 * k + 1] = -y;  M[5][2 * k + 1] = -1.0;
            M[6][2 * k + 1] = v * x; M[7][2 * k + 1] = v * y; M[8][2 * k + 1] = v;
        }
    }
    double beta[8], rdiag[8], z[9];
    bool rank_ok = true;
    householder_qr_9x8(M, beta, rdiag, rank_ok);
    householder_null_vector(M, beta, z);
    // H = T_b^-1 Hn T_a,  T = [[s, 0, -s cx], [0, s, -s cy], [0, 0, 1]],  T^-1 = [[1/s, 0, cx], [0, 1/s, cy], [0, 0, 1]]
    const double Ta[9] = {s1, 0.0, -s1 * c1x, 0.0, s1, -s1 * c1y, 0.0, 0.0, 1.0};
    const double Tbi[9] = {1.0 / s2, 0.0, c2x, 0.0, 1.0 / s2, c2y, 0.0, 0.0, 1.0};
    double tmp[9];
    mat3_mul(Tbi, z, tmp);
    mat3_mul(tmp, Ta, H);
    const double h22 = H[8];
    ok = ok && rank_ok && h22 != 0.0 && isfinite(h22);
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        H[i] = H[i] / h22;
        ok = ok && isfinite(H[i]);
    }
    return ok;
}

// K1 for homographies, one thread per hypothesis, everything in registers (the shape of k_fit_qr): clears this
// hypothesis's accumulator column (and, thread 0 of pair 0, the tail words), reads its row from the table or draws it
// with the device sampler (stream stream0 + pair, recording all 8 columns, as k_fit_qr does), fits columns 0-3.
// Batched form as k_fit_qr: blockIdx.y = image pair, pair p owns records [offsets[p], offsets[p+1]) and table rows,
// models and accumulator columns [p h, (p+1) h); its indices are pair-relative.  A pair of fewer than 8 records gets
// invalid models (and zero rows when drawing).  offsets == nullptr: one pair of n records.
constexpr int kFitHThreads = 64;
__global__ void __launch_bounds__(kFitHThreads)
k_fit_homography(const Corr* __restrict__ pts, const long long* __restrict__ offsets, const int32_t* __restrict__ table,
                 long long h, double* __restrict__ H_out, uint8_t* __restrict__ valid_out,
                 unsigned long long* __restrict__ acc, int acc_planes, int acc_tail_words, int draw,
                 unsigned long long seed, unsigned long long stream0, long long hyp_offset, long long n) {
    chain_enter();
    const long long li = blockIdx.x * (long long)kFitHThreads + threadIdx.x;
    if (li >= h) return;
    const long long i = (long long)blockIdx.y * h + li;
    if (acc) {
        const long long htotal = (long long)gridDim.y * h;
        for (int k = 0; k < acc_planes; ++k) acc[(long long)k * htotal + i] = 0ull;
        if (i == 0)
            for (int k = 0; k < acc_tail_words; ++k) acc[(long long)acc_planes * htotal + k] = 0ull;
    }
    if (offsets) {
        n = offsets[blockIdx.y + 1] - offsets[blockIdx.y];
        if (n < 8) {
            for (int k = 0; k < 9; ++k) H_out[9 * i + k] = 0.0;
            valid_out[i] = FIT_INVALID;
            if (draw) {
                int4* t = reinterpret_cast<int4*>(const_cast<int32_t*>(table) + 8 * i);
                t[0] = make_int4(0, 0, 0, 0);
                t[1] = make_int4(0, 0, 0, 0);
            }
            return;
        }
        pts += offsets[blockIdx.y];
    }
    int idx[4];
    if (draw) {
        int32_t row[8];
        philox_sample8(seed, stream0 + blockIdx.y, (unsigned long long)(hyp_offset + li), (unsigned)n, row);
        int4* t = reinterpret_cast<int4*>(const_cast<int32_t*>(table) + 8 * i);
        t[0] = make_int4(row[0], row[1], row[2], row[3]);
        t[1] = make_int4(row[4], row[5], row[6], row[7]);
#pragma unroll
        for (int k = 0; k < 4; ++k) idx[k] = row[k];
    } else {
        const int4 t0 = reinterpret_cast<const int4*>(table + 8 * i)[0];
        idx[0] = t0.x; idx[1] = t0.y; idx[2] = t0.z; idx[3] = t0.w;
    }
    Corr c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = pts[idx[k]];
    double H[9];
    const bool ok = homography_fit4(c, H);
#pragma unroll
    for (int k = 0; k < 9; ++k) H_out[9 * i + k] = ok ? H[k] : 0.0;
    valid_out[i] = ok ? FIT_VALID : FIT_INVALID;
}

// ------------------------------------------------------------------------------------
// K2 for homographies — count and fixed-point sums of the transfer error of every inlier, per hypothesis.
//
// Mapping: lane = hypothesis, HPT homographies (and their adjugates) per thread in registers.  Warps are persistent and
// claim work items (correspondence split x group of 32*HPT hypotheses) from an atomic counter, as K2 does; each warp
// streams its correspondences through its own ring of tiles filled by 1-D bulk async copies (lane 0 issues, the
// warp's own mbarriers complete) and every lane reads the same record (broadcast).  Every evaluation runs the pinned
// division-free decision; an inlier's value is converted to 84-bit fixed point (chunks21) and added to the lane's own
// 32-bit chunk registers - a lane owns its hypothesis within the item, so neither atomics nor shared memory are needed
// until the item ends and the words are folded into the [kAccWords][h] global accumulators.  Integer sums: counts and
// sums are independent of scheduling and of the split, exactly as on the E path, and K3 reads them unchanged.
// Batches: items are (pair, split, group) as K2's are.  A split is cut within the pair's own records, the pair's models
// are H[p h, (p+1) h) and its sums go to accumulator columns p h + hypothesis, so each pair's counts and sums are those
// of the single-pair call on that pair alone.
// ------------------------------------------------------------------------------------
constexpr int kHScoreThreads = 128;
constexpr int kHScoreWarps = kHScoreThreads / 32;
constexpr int kHTile = 64;
constexpr int kHStages = 3;
constexpr int kHScoreHpt = 2;

struct HScoreArgs {
    const Corr* pts;          // pixel coordinates (K = I)
    const long long* offsets; // [P+1] or null (one pair of n records)
    const double* H;          // [P][h][9]
    long long n, h, htotal;   // htotal = P h: the stride of the accumulator planes
    double thr;
    double scale1, scale2;    // 2^(63-e), 2^(63-2e): every inlier's value < 2^e
    int sums;                 // SUM_S1 | SUM_S2
    long long chunk;          // correspondences per split (multiple of kHTile, <= kMaxItemPoints)
    int hblocks, nsplit;
    long long total_items;
    unsigned* work_counter;
    unsigned long long* acc;  // [kAccWords][htotal], cleared by k_fit_homography
};

struct alignas(128) HScoreWarpSmem {
    Corr tile[kHStages][kHTile];
    unsigned long long full_bar[kHStages];
};

template <int HPT>
__global__ void __launch_bounds__(kHScoreThreads, 3) k_score_homography(const HScoreArgs a) {
    chain_enter();
    extern __shared__ __align__(128) unsigned char hscore_smem[];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(full, (int)(threadIdx.x >> 5), 0);
    HScoreWarpSmem& ws = reinterpret_cast<HScoreWarpSmem*>(hscore_smem)[warp];
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kHStages; ++s) mbar_init(&ws.full_bar[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    unsigned gt = 0;  // tiles consumed so far by this warp (stage + parity)
    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(a.work_counter, 1u);
        item = __shfl_sync(full, item, 0);
        if (item >= a.total_items) break;
        const int hw = (int)(item % (unsigned)a.hblocks);
        const unsigned rest = item / (unsigned)a.hblocks;
        const int split = (int)(rest % (unsigned)a.nsplit);
        const int pair = (int)(rest / (unsigned)a.nsplit);
        const long long pbase = a.offsets ? a.offsets[pair] : 0;
        const long long plen = a.offsets ? a.offsets[pair + 1] - pbase : a.n;
        long long begin = (long long)split * a.chunk;
        if (begin > plen) begin = plen;
        const long long end = pbase + ((begin + a.chunk < plen) ? begin + a.chunk : plen);
        begin += pbase;
        const int ntiles = (int)((end - begin + kHTile - 1) / kHTile);
        auto issue = [&](int t) {  // lane 0 only
            const int s = (int)((gt + (unsigned)t) % kHStages);
            const long long first = begin + (long long)t * kHTile;
            const long long rem = end - first;
            const uint32_t bytes = (uint32_t)((rem < kHTile ? rem : kHTile) * sizeof(Corr));
            mbar_expect_tx(&ws.full_bar[s], bytes);
            bulk_g2s(&ws.tile[s][0], a.pts + first, bytes, &ws.full_bar[s]);
        };
        if (lane == 0)
            for (int t = 0; t < kHStages && t < ntiles; ++t) issue(t);

        // this lane's hypotheses hyp_w + 32 j + lane; padding lanes hold H = 0 (p2 = 0: never an inlier)
        const long long hyp_w = (long long)hw * (32 * HPT);
        const double* Hp = a.H + 9 * (long long)pair * a.h;
        double hm[HPT][9], am[HPT][9];
        unsigned cw[HPT][kAccWords];
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = hyp_w + 32 * j + lane;
#pragma unroll
            for (int k = 0; k < 9; ++k) hm[j][k] = hyp < a.h ? Hp[9 * hyp + k] : 0.0;
            homography_adj(hm[j], am[j]);
#pragma unroll
            for (int k = 0; k < kAccWords; ++k) cw[j][k] = 0u;
        }

        for (int t = 0; t < ntiles; ++t) {
            const unsigned gti = gt + (unsigned)t;
            const int s = (int)(gti % kHStages);
            mbar_wait(&ws.full_bar[s], (gti / kHStages) & 1u);
            const long long first = begin + (long long)t * kHTile;
            const int np = (int)((end - first < kHTile) ? (end - first) : kHTile);
            const Corr* tp = &ws.tile[s][0];
            for (int p = 0; p < np; ++p) {
                const Corr c = tp[p];
#pragma unroll
                for (int j = 0; j < HPT; ++j) {
                    const TransferTerms r = transfer_terms(hm[j], am[j], c.xa, c.ya, c.xb, c.yb);
                    if (transfer_inlier(r, a.thr)) {
                        const double v = transfer_value(r);
                        unsigned ch[kChunks];
                        cw[j][0] += 1u;
                        if (a.sums & SUM_S1) {
                            chunks21(v, a.scale1, ch);
#pragma unroll
                            for (int kk = 0; kk < kChunks; ++kk) cw[j][1 + kk] += ch[kk];
                        }
                        if (a.sums & SUM_S2) {
                            chunks21(__dmul_rn(v, v), a.scale2, ch);
#pragma unroll
                            for (int kk = 0; kk < kChunks; ++kk) cw[j][1 + kChunks + kk] += ch[kk];
                        }
                    }
                }
            }
            __syncwarp();  // every lane is done with the stage: refill it
            if (lane == 0 && t + kHStages < ntiles) issue(t + kHStages);
        }
        gt += (unsigned)ntiles;
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = (long long)pair * a.h + hyp_w + 32 * j + lane;
            if (cw[j][0]) {  // only real hypotheses can have inliers
#pragma unroll
                for (int k = 0; k < kAccWords; ++k)
                    if (cw[j][k]) atomicAdd(a.acc + (long long)k * a.htotal + hyp, (unsigned long long)cw[j][k]);
            }
        }
    }
}

// K4 for homographies: the pinned decision and value of every correspondence under one H - the winner of the last
// estimate (best != null: taken straight from K3's output) or a caller-supplied model (best == null).
__global__ void k_homography_mask(const Corr* __restrict__ pts, long long n, const double* __restrict__ H,
                                  const Best* __restrict__ best, double thr, uint8_t* __restrict__ mask,
                                  double* __restrict__ err) {
    chain_enter();
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long local = best ? best->idx : 0;
    if (local < 0) {
        mask[i] = 0;
        err[i] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    double h[9], adj[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) h[k] = H[9 * local + k];
    homography_adj(h, adj);
    const Corr c = pts[i];
    double v;
    mask[i] = transfer_exact(h, adj, c.xa, c.ya, c.xb, c.yb, thr, v) ? 1 : 0;
    err[i] = v;
}

}  // namespace sfm
