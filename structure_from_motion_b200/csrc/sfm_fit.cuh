// K0 (K-normalisation), the device sampler and K1 (batched eight-point fitter).
#pragma once
#include "sfm_device.cuh"
#include "sfm_linalg.cuh"

namespace sfm {

// ------------------------------------------------------------------------------------
// K0 — to_normalized_image_coords (lib/epipolar/eight_point.py:127-133) once per
// correspondence instead of twice per evaluation (lib/epipolar/epipolar_ransac.py:21-22).
// IEEE subtract + divide, bit-identical to the reference.  Packs SoA/strided pixel input
// into the 32-byte Corr records every other kernel consumes.
// ------------------------------------------------------------------------------------
// Batched form: blockIdx.y = image pair; pair p owns records [offsets[p], offsets[p+1]) and
// its own intrinsics Ks[p] (row-major 3x3).  offsets == nullptr means one pair of n records.
__global__ void k_normalise(const double* __restrict__ xa, const double* __restrict__ ya,
                            const double* __restrict__ xb, const double* __restrict__ yb,
                            long long stride, long long n, const long long* __restrict__ offsets,
                            const double* __restrict__ Ks, Corr* __restrict__ out,
                            unsigned long long* __restrict__ bounds /* [2] or null, zero on entry */) {
    const long long base = offsets ? offsets[blockIdx.y] : 0;
    const long long len = offsets ? offsets[blockIdx.y + 1] - base : n;
    const long long li = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    double a2 = 0.0, b2 = 0.0;
    if (li < len) {
        const long long i = base + li;
        const double* K = Ks + 9 * (long long)blockIdx.y;
        const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
        Corr c;
        c.xa = __ddiv_rn(__dsub_rn(xa[i * stride], cx), fx);
        c.ya = __ddiv_rn(__dsub_rn(ya[i * stride], cy), fy);
        c.xb = __ddiv_rn(__dsub_rn(xb[i * stride], cx), fx);
        c.yb = __ddiv_rn(__dsub_rn(yb[i * stride], cy), fy);
        out[i] = c;
        if (isfinite(c.xa) && isfinite(c.ya) && isfinite(c.xb) && isfinite(c.yb)) {
            a2 = fma(c.xa, c.xa, fma(c.ya, c.ya, 1.0));
            b2 = fma(c.xb, c.xb, fma(c.yb, c.yb, 1.0));
        }
    }
    if (!bounds) return;
    // max |(x, y, 1)|^2 per image over the correspondences with four finite coordinates: the rounding bound kappa of
    // the K2 screens (sfm_score.cuh).  A record with a NaN or infinite coordinate is left out: its sed is inf or NaN
    // (every product with an infinite coordinate is inf or NaN and reaches r or a line norm), so it is never an inlier
    // at the thresholds K2 scores (<= 1e100), whatever its test decides.  Non-negative doubles order like their bits.
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        a2 = fmax(a2, __shfl_xor_sync(0xffffffffu, a2, d));
        b2 = fmax(b2, __shfl_xor_sync(0xffffffffu, b2, d));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(bounds, (unsigned long long)__double_as_longlong(a2));
        atomicMax(bounds + 1, (unsigned long long)__double_as_longlong(b2));
    }
}

// ------------------------------------------------------------------------------------
// Device sampler: table[h] = 8 distinct indices in [0, n) from Philox keyed by
// (seed, stream=pair, global hypothesis index) — independent of how hypotheses are
// sharded over GPUs.  Replaces the O(N) random.shuffle per iteration of
// lib/ransac/ransac.py:62 for the large configurations (documented deviation; the
// faithful sampler is sfm_mt_shuffle_table on the host).
// ------------------------------------------------------------------------------------
__global__ void k_sample(unsigned long long seed, unsigned long long stream0,
                         long long hyp_offset, long long h, long long n,
                         const long long* __restrict__ offsets, int32_t* __restrict__ table) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= h) return;
    const long long len = offsets ? offsets[blockIdx.y + 1] - offsets[blockIdx.y] : n;
    int32_t idx[8];
    if (len >= 8) {
        philox_sample8(seed, stream0 + blockIdx.y, (unsigned long long)(hyp_offset + i), (unsigned)len, idx);
    } else {
        for (int k = 0; k < 8; ++k) idx[k] = 0;
    }
    int4* t = reinterpret_cast<int4*>(table + 8 * ((long long)blockIdx.y * h + i));
    t[0] = make_int4(idx[0], idx[1], idx[2], idx[3]);
    t[1] = make_int4(idx[4], idx[5], idx[6], idx[7]);
}

// ------------------------------------------------------------------------------------
// K1 reference-arithmetic path — eight-point fit through Y^T Y, one thread per hypothesis.
// Runs for the hypotheses the fast path (k_fit_qr above) flags as ambiguous, and for every
// hypothesis when the eigenvalues are requested (sfm_fit with eig_out).
//
// Restates estimate_fundamental_mat (lib/epipolar/eight_point.py:136-170):
//   Hartley normalisation (:308-338) -> Y^T Y (:363-393) -> eigenvector of the smallest
//   |eigenvalue| with the "only one small eigenvalue" validity test (:396-427) -> rank-2
//   projection (:430-446) -> E = T2^T F T1 (:163) -> E /= E[2,2] (:166).
//
// The 9x9 symmetric eigenproblem is solved by cyclic Jacobi with the matrix and the
// eigenvector matrix in shared memory, element-major ([element][thread]) so that a warp's
// accesses are conflict-free; one thread owns one hypothesis, which keeps all 32 lanes of
// a warp doing rotations (a warp-per-hypothesis mapping would idle most lanes in the
// scalar rotation-angle computation and costs ~20x more issue slots per fit).
// The rank-2 projection uses a one-sided Jacobi SVD of the 3x3 estimate in registers.
// ------------------------------------------------------------------------------------
constexpr int kFitThreads = 64;
constexpr int kFitSmemDoubles = 162;  // A[81] + V[81] per thread

__device__ __forceinline__ void hartley(const double (&x)[8], const double (&y)[8], double (&nx)[8],
                                        double (&ny)[8], double& scale, double& cx, double& cy) {
    // np.mean(coords, axis=0): rows added in order (eight_point.py:320)
    double sx = x[0], sy = y[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) {
        sx = __dadd_rn(sx, x[i]);
        sy = __dadd_rn(sy, y[i]);
    }
    cx = sx / 8.0;
    cy = sy / 8.0;
    double nrm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        nx[i] = __dsub_rn(x[i], cx);
        ny[i] = __dsub_rn(y[i], cy);
        nrm[i] = sqrt(__dadd_rn(__dmul_rn(nx[i], nx[i]), __dmul_rn(ny[i], ny[i])));  // :323
    }
    // np.mean over 8 contiguous values: numpy's pairwise tree (eight_point.py:324)
    const double s = __dadd_rn(__dadd_rn(__dadd_rn(nrm[0], nrm[1]), __dadd_rn(nrm[2], nrm[3])),
                               __dadd_rn(__dadd_rn(nrm[4], nrm[5]), __dadd_rn(nrm[6], nrm[7])));
    scale = sqrt(2.0) / (s / 8.0);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        nx[i] = __dmul_rn(nx[i], scale);
        ny[i] = __dmul_rn(ny[i], scale);
    }
}

// Rank-2 projection (:430-446), E = T2^T F T1 (:163), E /= E[2,2] (:166) — shared by both fitters.
__device__ __forceinline__ void finish_fit(double (&F)[9], double s1, double c1x, double c1y, double s2,
                                           double c2x, double c2y, double (&E)[9]) {
    // one-sided Jacobi SVD of F; the column of F V with the
    // smallest norm is sigma_3 u_3, so F' = F - (sigma_3 u_3) v_3^T zeroes the smallest
    // singular value without ever dividing by it.
    {
        double G[9], W[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) G[i] = F[i];
        jacobi_svd_onesided<3, 3, true>(G, W, 30);
        double nrm[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) nrm[j] = fma(G[6 + j], G[6 + j], fma(G[3 + j], G[3 + j], G[j] * G[j]));
        int k3 = 0;
        if (nrm[1] < nrm[0]) k3 = 1;
        if (nrm[2] < (k3 == 0 ? nrm[0] : nrm[1])) k3 = 2;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double g = (k3 == 0) ? G[i * 3] : ((k3 == 1) ? G[i * 3 + 1] : G[i * 3 + 2]);
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double w = (k3 == 0) ? W[j * 3] : ((k3 == 1) ? W[j * 3 + 1] : W[j * 3 + 2]);
                F[i * 3 + j] = fma(-g, w, F[i * 3 + j]);
            }
        }
    }
    // E = T2^T F T1 (:163), T = [[s,0,-s cx],[0,s,-s cy],[0,0,1]] (:329-336)
    const double T1[9] = {s1, 0.0, -s1 * c1x, 0.0, s1, -s1 * c1y, 0.0, 0.0, 1.0};
    const double T2t[9] = {s2, 0.0, 0.0, 0.0, s2, 0.0, -s2 * c2x, -s2 * c2y, 1.0};
    double tmp[9];
    mat3_mul(T2t, F, tmp);
    mat3_mul(tmp, T1, E);
    const double e22 = E[8];
#pragma unroll
    for (int i = 0; i < 9; ++i) E[i] = E[i] / e22;  // (:166)
}

// ------------------------------------------------------------------------------------
// K1 fast path — the same fit without forming Y^T Y.
//
// The 8x9 design matrix Y (:363-393) has rank 8 for a non-degenerate sample, and the
// eigenvector the reference takes (smallest |eigenvalue| of Y^T Y, :423-425) is Y's null
// vector.  Householder QR of Y^T (9x8, one reflector per correspondence) gives it as
// Q e_9 = H_1 ... H_8 e_9 with a backward error of order eps * kappa(Y) — the reference's
// own route through Y^T Y costs eps * kappa(Y)^2, so this path is the more accurate of the
// two.  Everything is statically indexed and lives in registers (no shared memory, no
// local memory): ~1.3k FP64 instructions per hypothesis instead of ~30k for the 9x9 Jacobi.
//
// Validity (:414-421) needs lambda_2(Y^T Y) = sigma_min(R)^2 against 1e-10.  R is the 8x8
// triangular factor:  1/|R^-1|_F <= sigma_min(R) <= min |r_ii|,  so
//     1/|R^-1|_F^2 > 1.001e-10   => valid,       min r_ii^2 < 0.999e-10  => degenerate,
// and the (very rare: P ~ 1e-7 per sample) in-between case is flagged 2 and re-done by the
// Jacobi kernel below, which follows the reference's Y^T Y arithmetic.
// ------------------------------------------------------------------------------------
enum { FIT_INVALID = 0, FIT_VALID = 1, FIT_AMBIGUOUS = 2 };

// Householder QR of a 9x8 matrix in registers (M[i][k]: column k is one design row), shared by the eight-point fit
// and the homography DLT (whose A^T has the same shape: two rows per correspondence, four correspondences).  On
// return column k holds the reflector v_k on and below the diagonal (H_k = I - beta_k v_k v_k^T), R's strictly upper
// part is above it and its diagonal is rdiag; rank_ok is cleared when a column is exactly zero.
__device__ __forceinline__ void householder_qr_9x8(double (&M)[9][8], double (&beta)[8], double (&rdiag)[8], bool& rank_ok) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        // reflector for x = M[k..8][k]:  v = x - alpha e_1, alpha = -sign(x_0) |x|, H = I - beta v v^T
        double n2 = 0.0;
#pragma unroll
        for (int i = k; i < 9; ++i) n2 = fma(M[i][k], M[i][k], n2);
        const double nrm = sqrt(n2);
        const double x0 = M[k][k];
        const double alpha = (x0 > 0.0) ? -nrm : nrm;
        const double v0 = x0 - alpha;                       // |v0| = |x0| + |x|: no cancellation
        const double vtv = 2.0 * fma(nrm, fabs(x0), n2);     // v^T v = 2 |x| (|x| + |x0|)
        rank_ok = rank_ok && (n2 > 0.0);
        beta[k] = (n2 > 0.0) ? 2.0 / vtv : 0.0;
        rdiag[k] = alpha;
        M[k][k] = v0;  // column k below the diagonal now holds v_k
#pragma unroll
        for (int j = k + 1; j < 8; ++j) {
            double w = 0.0;
#pragma unroll
            for (int i = k; i < 9; ++i) w = fma(M[i][k], M[i][j], w);
            w *= beta[k];
#pragma unroll
            for (int i = k; i < 9; ++i) M[i][j] = fma(-w, M[i][k], M[i][j]);
        }
    }
}

// null vector z = H_1 ... H_8 e_9 of the factored matrix
__device__ __forceinline__ void householder_null_vector(const double (&M)[9][8], const double (&beta)[8], double (&z)[9]) {
#pragma unroll
    for (int i = 0; i < 9; ++i) z[i] = (i == 8) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 7; k >= 0; --k) {
        double w = 0.0;
#pragma unroll
        for (int i = k; i < 9; ++i) w = fma(M[i][k], z[i], w);
        w *= beta[k];
#pragma unroll
        for (int i = k; i < 9; ++i) z[i] = fma(-w, M[i][k], z[i]);
    }
}

__device__ __forceinline__ int eight_point_fit_qr(const Corr (&c)[8], double (&E)[9]) {
    double s1, c1x, c1y, s2, c2x, c2y;
    double M[9][8];  // M[i][k] = y_k[i]: column k is the design row of correspondence k
    {
        double xa[8], ya[8], xb[8], yb[8], nxa[8], nya[8], nxb[8], nyb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            xa[i] = c[i].xa; ya[i] = c[i].ya; xb[i] = c[i].xb; yb[i] = c[i].yb;
        }
        hartley(xa, ya, nxa, nya, s1, c1x, c1y);
        hartley(xb, yb, nxb, nyb, s2, c2x, c2y);
#pragma unroll
        for (int k = 0; k < 8; ++k) {  // eight_point.py:376-393
            M[0][k] = __dmul_rn(nxb[k], nxa[k]); M[1][k] = __dmul_rn(nxb[k], nya[k]); M[2][k] = nxb[k];
            M[3][k] = __dmul_rn(nyb[k], nxa[k]); M[4][k] = __dmul_rn(nyb[k], nya[k]); M[5][k] = nyb[k];
            M[6][k] = nxa[k]; M[7][k] = nya[k]; M[8][k] = 1.0;
        }
    }
    double beta[8], rdiag[8];
    bool rank_ok = true;
    householder_qr_9x8(M, beta, rdiag, rank_ok);
    // sigma_min(R)^2 bounds; R = rdiag on the diagonal, M[i][j] (i < j) above it
    double min_r2 = rdiag[0] * rdiag[0];
#pragma unroll
    for (int k = 1; k < 8; ++k) min_r2 = fmin(min_r2, rdiag[k] * rdiag[k]);
    int status;
    if (!rank_ok || !(min_r2 >= 0.999 * kVerySmall)) {
        status = FIT_INVALID;
    } else {
        // X = R^-1 (upper triangular), column by column; only its Frobenius norm is needed
        double rinv[8], f2 = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) rinv[k] = 1.0 / rdiag[k];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double x[8];
            x[j] = rinv[j];
            f2 = fma(x[j], x[j], f2);
#pragma unroll
            for (int i = j - 1; i >= 0; --i) {
                double acc = 0.0;
#pragma unroll
                for (int k = i + 1; k <= j; ++k) acc = fma(M[i][k], x[k], acc);
                x[i] = -acc * rinv[i];
                f2 = fma(x[i], x[i], f2);
            }
        }
        status = (1.0 / f2 > 1.001 * kVerySmall) ? FIT_VALID : FIT_AMBIGUOUS;
    }
    // null vector z = H_1 ... H_8 e_9
    double z[9];
    householder_null_vector(M, beta, z);
    finish_fit(z, s1, c1x, c1y, s2, c2x, c2y, E);  // v_min.reshape((3,3)) (:424-425)
    return status;
}

constexpr int kFitQrThreads = 64;
// 168 registers + 0.5 KB of L1-resident spills: 12 warps/SM hide the sqrt/div latency chains better than 8 warps without
// spills (222 registers: config 4 0.39 vs 0.34 ms) or 14 warps with 1 KB of spills (144 registers: 0.38 ms)
constexpr int kFitQrMinBlocks = 6;

__global__ void __launch_bounds__(kFitQrThreads, kFitQrMinBlocks)
k_fit_qr(const Corr* __restrict__ pts, const long long* __restrict__ offsets, const int32_t* __restrict__ table,
         long long h, double* __restrict__ E_out, uint8_t* __restrict__ valid_out,
         unsigned* __restrict__ ambiguous_count, ModelRow* __restrict__ rows,
         unsigned long long* __restrict__ acc, int acc_planes, int acc_tail_words,
         int draw, unsigned long long seed, unsigned long long stream0, long long hyp_offset, long long n) {
    chain_enter();
    const long long li = blockIdx.x * (long long)kFitQrThreads + threadIdx.x;
    if (li >= h) return;
    const long long i = (long long)blockIdx.y * h + li;  // blockIdx.y = image pair
    if (acc) {
        // K2's exact integer accumulators of this hypothesis start at zero (saves the scoring call a 4.7 MB memset);
        // the first thread also clears the work counter / rescore counter / K3 tickets behind the planes
        const long long htotal = (long long)gridDim.y * h;
        for (int k = 0; k < acc_planes; ++k) acc[(long long)k * htotal + i] = 0ull;
        if (i == 0)
            for (int k = 0; k < acc_tail_words; ++k) acc[(long long)acc_planes * htotal + k] = 0ull;
    }
    if (offsets) {
        if (offsets[blockIdx.y + 1] - offsets[blockIdx.y] < 8) {
            for (int k = 0; k < 9; ++k) E_out[9 * i + k] = 0.0;
            valid_out[i] = FIT_INVALID;
            if (rows) { const double z[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; store_model_row(rows, i, z, false); }
            if (draw) {  // a pair too short to sample from gets a row of zeros, as k_sample writes
                int4* t = reinterpret_cast<int4*>(const_cast<int32_t*>(table) + 8 * i);
                t[0] = make_int4(0, 0, 0, 0);
                t[1] = make_int4(0, 0, 0, 0);
            }
            return;
        }
        pts += offsets[blockIdx.y];
    }
    Corr c[8];
    int idx[8];
    if (draw) {
        // the device sampler (k_sample) folded in: this hypothesis draws its own row and records it in the table
        const long long len = offsets ? offsets[blockIdx.y + 1] - offsets[blockIdx.y] : n;
        int32_t row[8];
        philox_sample8(seed, stream0 + blockIdx.y, (unsigned long long)(hyp_offset + li), (unsigned)len, row);
        int4* t = reinterpret_cast<int4*>(const_cast<int32_t*>(table) + 8 * i);
        t[0] = make_int4(row[0], row[1], row[2], row[3]);
        t[1] = make_int4(row[4], row[5], row[6], row[7]);
#pragma unroll
        for (int k = 0; k < 8; ++k) idx[k] = row[k];
    } else {
        const int4 t0 = reinterpret_cast<const int4*>(table + 8 * i)[0];
        const int4 t1 = reinterpret_cast<const int4*>(table + 8 * i)[1];
        idx[0] = t0.x; idx[1] = t0.y; idx[2] = t0.z; idx[3] = t0.w;
        idx[4] = t1.x; idx[5] = t1.y; idx[6] = t1.z; idx[7] = t1.w;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) c[k] = pts[idx[k]];
    double E[9];
    const int status = eight_point_fit_qr(c, E);
#pragma unroll
    for (int k = 0; k < 9; ++k) E_out[9 * i + k] = (status == FIT_VALID) ? E[k] : 0.0;
    if (rows) store_model_row(rows, i, E, status == FIT_VALID);  // padded copy for K2's survivor path
    valid_out[i] = (uint8_t)status;
    if (status == FIT_AMBIGUOUS) atomicAdd(ambiguous_count, 1u);
}

// Fit one hypothesis from 8 correspondences.  sm points at this thread's column of the
// element-major shared scratch (stride = kFitThreads doubles).  Returns validity.
__device__ inline bool eight_point_fit(const Corr (&c)[8], double* sm, double (&E)[9],
                                       double* eig_out /* 9 or nullptr */) {
    constexpr int S = kFitThreads;
#define A_(i, j) sm[((i) * 9 + (j)) * S]
#define V_(i, j) sm[(81 + (i) * 9 + (j)) * S]
    double s1, c1x, c1y, s2, c2x, c2y;
    {
        double xa[8], ya[8], xb[8], yb[8], nxa[8], nya[8], nxb[8], nyb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            xa[i] = c[i].xa; ya[i] = c[i].ya; xb[i] = c[i].xb; yb[i] = c[i].yb;
        }
        hartley(xa, ya, nxa, nya, s1, c1x, c1y);
        hartley(xb, yb, nxb, nyb, s2, c2x, c2y);
        // Y^T Y = sum_k y_k y_k^T, products rounded then accumulated in point order (:363-375)
        for (int i = 0; i < 9; ++i)
            for (int j = i; j < 9; ++j) A_(i, j) = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            double y[9];
            y[0] = __dmul_rn(nxb[k], nxa[k]); y[1] = __dmul_rn(nxb[k], nya[k]); y[2] = nxb[k];
            y[3] = __dmul_rn(nyb[k], nxa[k]); y[4] = __dmul_rn(nyb[k], nya[k]); y[5] = nyb[k];
            y[6] = nxa[k]; y[7] = nya[k]; y[8] = 1.0;
#pragma unroll
            for (int i = 0; i < 9; ++i)
#pragma unroll
                for (int j = i; j < 9; ++j) A_(i, j) = __dadd_rn(A_(i, j), __dmul_rn(y[i], y[j]));
        }
    }
    for (int i = 0; i < 9; ++i)
        for (int j = 0; j < 9; ++j) V_(i, j) = (i == j) ? 1.0 : 0.0;

    // cyclic Jacobi on the upper triangle
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < 9; ++i) {
            diag += fabs(A_(i, i));
            for (int j = i + 1; j < 9; ++j) off += fabs(A_(i, j));
        }
        if (off <= 1e-300 || off <= 1e-24 * diag) break;
        for (int p = 0; p < 8; ++p) {
            for (int q = p + 1; q < 9; ++q) {
                const double apq = A_(p, q);
                if (apq == 0.0) continue;
                const double app = A_(p, p), aqq = A_(q, q);
                const double g = 1e3 * fabs(apq);
                if (fabs(app) + g == fabs(app) && fabs(aqq) + g == fabs(aqq)) {
                    A_(p, q) = 0.0;
                    continue;
                }
                double cs, sn, t;
                sym_schur(app, aqq, apq, cs, sn, t);
                A_(p, p) = fma(-t, apq, app);
                A_(q, q) = fma(t, apq, aqq);
                A_(p, q) = 0.0;
                for (int k = 0; k < p; ++k) {
                    const double x = A_(k, p), y = A_(k, q);
                    A_(k, p) = fma(cs, x, -sn * y);
                    A_(k, q) = fma(sn, x, cs * y);
                }
                for (int k = p + 1; k < q; ++k) {
                    const double x = A_(p, k), y = A_(k, q);
                    A_(p, k) = fma(cs, x, -sn * y);
                    A_(k, q) = fma(sn, x, cs * y);
                }
                for (int k = q + 1; k < 9; ++k) {
                    const double x = A_(p, k), y = A_(q, k);
                    A_(p, k) = fma(cs, x, -sn * y);
                    A_(q, k) = fma(sn, x, cs * y);
                }
                for (int k = 0; k < 9; ++k) {
                    const double x = V_(k, p), y = V_(k, q);
                    V_(k, p) = fma(cs, x, -sn * y);
                    V_(k, q) = fma(sn, x, cs * y);
                }
            }
        }
    }
    // validity (:414-421): after sorting, every eigenvalue but the smallest must exceed 1e-10
    int nsmall = 0, imin = 0;
    double wmin = fabs(A_(0, 0));
    for (int i = 0; i < 9; ++i) {
        const double w = A_(i, i);
        if (eig_out) eig_out[i] = w;
        nsmall += (w <= kVerySmall) ? 1 : 0;
        if (fabs(w) < wmin) { wmin = fabs(w); imin = i; }  // np.argmin(np.abs(w)) (:423)
    }
    const bool valid = nsmall <= 1;
    double F[9];
    for (int i = 0; i < 9; ++i) F[i] = V_(i, imin);  // v_min.reshape((3,3)) (:424-425)
#undef A_
#undef V_
    finish_fit(F, s1, c1x, c1y, s2, c2x, c2y, E);
    return valid;
}

__global__ void __launch_bounds__(kFitThreads)
k_fit(const Corr* __restrict__ pts, const long long* __restrict__ offsets,
      const int32_t* __restrict__ table, long long h, double* __restrict__ E_out,
      uint8_t* __restrict__ valid_out, double* __restrict__ eig_out,
      const unsigned* __restrict__ only_ambiguous /* null = fit everything */, ModelRow* __restrict__ rows) {
    chain_enter();
    extern __shared__ double fit_smem[];
    if (only_ambiguous && *only_ambiguous == 0u) return;  // the usual case: nothing was flagged
    const long long li = blockIdx.x * (long long)kFitThreads + threadIdx.x;
    if (li >= h) return;
    const long long i = (long long)blockIdx.y * h + li;  // blockIdx.y = image pair
    if (only_ambiguous && valid_out[i] != FIT_AMBIGUOUS) return;
    bool enough = true;
    if (offsets) {
        enough = offsets[blockIdx.y + 1] - offsets[blockIdx.y] >= 8;
        pts += offsets[blockIdx.y];
    }
    if (!enough) {
        for (int k = 0; k < 9; ++k) E_out[9 * i + k] = 0.0;
        valid_out[i] = 0;
        if (rows) { const double z[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; store_model_row(rows, i, z, false); }
        return;
    }
    Corr c[8];
    const int4 t0 = reinterpret_cast<const int4*>(table + 8 * i)[0];
    const int4 t1 = reinterpret_cast<const int4*>(table + 8 * i)[1];
    const int idx[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) c[k] = pts[idx[k]];
    double E[9], eig[9];
    const bool valid = eight_point_fit(c, fit_smem + threadIdx.x, E, eig_out ? eig : nullptr);
#pragma unroll
    for (int k = 0; k < 9; ++k) E_out[9 * i + k] = valid ? E[k] : 0.0;
    if (rows) store_model_row(rows, i, E, valid);
    valid_out[i] = valid ? 1 : 0;
    if (eig_out)
        for (int k = 0; k < 9; ++k) eig_out[9 * i + k] = eig[k];
}

}  // namespace sfm
