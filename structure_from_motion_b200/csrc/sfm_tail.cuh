// The tail of the path after the selection (apps/sfm.py:118-186), three launches, one image pair per blockIdx.y:
//   T1 k_tail_mask        inlier mask of the winner (ransac.py:70-79, exact scorer) + its sample points (ransac.py:76)
//                         -> ordered stream compaction (single pass, decoupled look-back) + decomposition of E
//                         (eight_point.py:245-280)
//   T2 k_tail_cheirality  4-pose cheirality test of every inlier (eight_point.py:210-230, 449-488) + the vote
//                         (eight_point.py:237), taken by the last block of the pair
//   T3 k_tail_triangulate DLT in pixel coordinates of the inliers passing the voted pose (triangulation.py:9-62)
// The winner (model, sample row, index) is read from a SelectRecord on the device: K3's for the fused single-GPU call
// and the batch, the merged one of a hypothesis-sharded run, or one built from a host-chosen winner.
//
// T1 and T2 take the model kind as a template parameter.  MODEL_E: sed_exact, the 8 sample points, decompose_essential,
// K-normalised records, and the vote with the reference's index-0 rule.  MODEL_H (single pair): the pinned transfer
// decision of k_homography_mask, the 4 sample points, decompose_homography (sfm_hpose.cuh) of K^-1 H K with the
// caller's K in Ks, records in pixel coordinates (T2 normalises them with k_normalise's IEEE operations), every passing
// inlier counts, and T2 does nothing but clear the pass bits when the pair is rotation-only.  T3 serves both.
#pragma once
#include "sfm_device.cuh"
#include "sfm_hpose.cuh"
#include "sfm_pose_math.cuh"
#include "sfm_types.h"

namespace sfm {

constexpr int kTailBlock = 256;
constexpr int kTailPerBlock = 1024;  // correspondences per block of T1
constexpr unsigned long long kAggFlag = 1ull << 62;

struct TailArgs {
    const Corr* pts;             // K-normalised correspondences (all pairs)
    const long long* offsets;    // [P+1] or null (one pair of n)
    long long n;
    const SelectRecord* rec;     // [P]
    double thr, dist_thr;
    uint8_t* mask;               // [n_total] sed <= thr (pure: the forced sample points are NOT set here)
    double* sed;                 // [n_total]
    long long* idx;              // [n_total] compacted inlier indices (pair-relative, ascending) from offsets[p]
    long long* num;              // [P] inliers per pair (samples included)
    unsigned long long* agg;     // [P][nblk] look-back state, zero on entry and on exit
    unsigned* ticket;            // [P] zero on entry and on exit
    unsigned* done;              // [P] zero on entry and on exit
    PoseSet* poses;              // [P]
    uint8_t* pass;               // [n_total] bit p = inlier k passes pose p (at compact position offsets[p] + k)
    // triangulation
    const double* xa; const double* ya; const double* xb; const double* yb;  // pixel coordinates
    long long stride;
    const double* Ks;            // [P][9]
    double* X;                   // [n_total][3] at compact positions
    // MODEL_H only
    HPlane* planes;              // [P] normals, distances, rotation flag beside poses
    double rot_tol;              // rotation-only below this s1 - s3
};

// Build a record for a winner chosen by the host (sfm_set_winner / sfm_get_best): E from device memory, row from the
// table or null.
__global__ void k_make_record(const double* __restrict__ E, const int32_t* __restrict__ row, long long idx,
                              SelectRecord* __restrict__ rec) {
    if (threadIdx.x || blockIdx.x) return;
    rec->best.err = 0.0; rec->best.idx = idx; rec->best.count = 0; rec->best.pad = 0;
    rec->num_invalid = 0; rec->first_invalid = -1;
    for (int k = 0; k < 9; ++k) rec->E[k] = E[k];
    for (int k = 0; k < 8; ++k) rec->sample[k] = row ? row[k] : -1;
}

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}

template <int KIND>
__global__ void __launch_bounds__(kTailBlock) k_tail_mask(const TailArgs a) {
    chain_enter();
    __shared__ unsigned s_bid;
    __shared__ int warp_cnt[4][8];
    __shared__ long long s_prefix;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pair = blockIdx.y, nblk = gridDim.x;
    if (tid == 0) s_bid = atomicAdd(&a.ticket[pair], 1u);  // ticket order = start order: predecessors are running
    __syncthreads();
    const int bid = (int)s_bid;
    const long long pbase = a.offsets ? a.offsets[pair] : 0;
    const long long plen = a.offsets ? a.offsets[pair + 1] - pbase : a.n;
    const SelectRecord& rec = a.rec[pair];
    const bool have = rec.best.idx >= 0;
    double e[9];
    int row[8];
#pragma unroll
    for (int k = 0; k < 9; ++k) e[k] = rec.E[k];
#pragma unroll
    for (int k = 0; k < 8; ++k) row[k] = rec.sample[k];
    constexpr int kSample = KIND == MODEL_H ? 4 : 8;  // points of a minimal sample
    double adj[9];
    if constexpr (KIND == MODEL_H) homography_adj(e, adj);
    const long long base = (long long)bid * kTailPerBlock;
    bool f[4];
    unsigned b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long i = base + k * kTailBlock + tid;
        f[k] = false;
        if (i < plen) {
            const Corr c = a.pts[pbase + i];
            double sv;
            bool in;
            if constexpr (KIND == MODEL_E) {
                sv = have ? sed_exact(e, c.xa, c.ya, c.xb, c.yb) : __longlong_as_double(0x7ff8000000000000LL);
                in = have && (sv <= a.thr);  // ransac.py:73
            } else {  // k_homography_mask's decision and value
                sv = __longlong_as_double(0x7ff8000000000000LL);
                in = have && transfer_exact(e, adj, c.xa, c.ya, c.xb, c.yb, a.thr, sv);
            }
            if (a.sed) a.sed[pbase + i] = sv;
            if (a.mask) a.mask[pbase + i] = in ? 1 : 0;
            bool smp = false;  // ransac.py:76: the sample points belong to the model's inliers whatever their score
#pragma unroll
            for (int q = 0; q < kSample; ++q) smp |= ((long long)row[q] == i);
            f[k] = in || (have && smp);
        }
        b[k] = __ballot_sync(0xffffffffu, f[k]);
        if (lane == 0) warp_cnt[k][warp] = __popc(b[k]);
    }
    __syncthreads();
    int total = 0;
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            for (int w = 0; w < 8; ++w) total += warp_cnt[k][w];
        // publish this block's count (value and flag in one word), then sum the predecessors'
        atomicExch(&a.agg[(long long)pair * nblk + bid], (unsigned long long)total | kAggFlag);
    }
    if (warp == 0) {
        long long sum = 0;
        const unsigned long long* ag = a.agg + (long long)pair * nblk;
        for (int j0 = 0; j0 < bid; j0 += 32) {
            const int j = j0 + lane;
            long long v = 0;
            if (j < bid) {
                unsigned long long w;
                do { w = ld_volatile_u64(ag + j); } while (!(w & kAggFlag));
                v = (long long)(w & ~kAggFlag);
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
        for (int w = 0; w < 8; ++w) {
            if (w < warp) o += warp_cnt[k][w];
            off += warp_cnt[k][w];
        }
        if (f[k]) a.idx[pbase + o + __popc(b[k] & ((1u << lane) - 1u))] = base + k * kTailBlock + tid;
    }
    if (bid == nblk - 1 && tid == 0) a.num[pair] = s_prefix + total;  // blocks past the end contribute 0
    // everybody past the look-back: the last one to get here clears the state for the next launch
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(&a.done[pair], 1u) == (unsigned)(nblk - 1)) {
            for (int j = 0; j < nblk; ++j) a.agg[(long long)pair * nblk + j] = 0;
            a.ticket[pair] = 0;
            a.done[pair] = 0;
        }
    }
    // the decomposition of the winner rides along (one thread of the first block, after it has published)
    if (bid == 0 && tid == 32) {
        if constexpr (KIND == MODEL_E) {
            if (have) decompose_essential(e, a.poses[pair]);
            else {
                PoseSet& p = a.poses[pair];
                for (int q = 0; q < 4; ++q) p.counts[q] = 0;
                p.best = -2;
                p.pad = 0;
            }
        } else {
            if (have) {
                double hn[9];
                homography_normalise_k(e, a.Ks + 9 * (long long)pair, hn);
                decompose_homography(hn, a.rot_tol, a.poses[pair], a.planes[pair]);
            } else {
                homography_no_model(a.poses[pair], a.planes[pair]);
            }
        }
    }
}

// DLT of inlier i of the pair in pixel coordinates under the voted pose b (triangulation.py:42-62); NaN when the inlier
// does not pass that pose.
__device__ __forceinline__ void tail_triangulate_one(const TailArgs& a, int pair, long long pbase, long long i, int b,
                                                     uint8_t passbits) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double* Xo = a.X + 3 * (pbase + i);
    if (b < 0 || !((passbits >> b) & 1u)) {
        Xo[0] = nan; Xo[1] = nan; Xo[2] = nan;
        return;
    }
    const PoseSet* poses = a.poses + pair;
    const double* Kmat = a.Ks + 9 * (long long)pair;
    const double* R = poses->R[b];
    const double* t = poses->t[b];
    double P1[12], P2[12];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            // K_ext @ Tmat: K[r,:] . [R|t][:,c]   (triangulation.py:52-56)
            const double a0 = (c < 3) ? R[c] : t[0], a1 = (c < 3) ? R[3 + c] : t[1], a2 = (c < 3) ? R[6 + c] : t[2];
            P2[4 * r + c] = fma(Kmat[3 * r + 2], a2, fma(Kmat[3 * r + 1], a1, Kmat[3 * r] * a0));
            P1[4 * r + c] = (c < 3) ? Kmat[3 * r + c] : 0.0;
        }
    const long long gi = (pbase + a.idx[pbase + i]) * a.stride;
    double Xr[3];
    dlt_triangulate(a.xa[gi], a.ya[gi], a.xb[gi], a.yb[gi], P1, P2, Xr);
    Xo[0] = Xr[0]; Xo[1] = Xr[1]; Xo[2] = Xr[2];
}

constexpr long long kTailSmallTri = 512;  // up to this many inliers the block that takes the vote also triangulates

// Grid-stride: the grid is sized for the machine, not for the (unknown to the host) number of inliers - a config-3
// winner has ~100 inliers, and 3 000 blocks that only find that out cost 30 us.
template <int KIND>
__global__ void __launch_bounds__(128) k_tail_cheirality(const TailArgs a) {
    chain_enter();
    __shared__ int s_cnt[4];
    __shared__ int s_last;
    const int pair = blockIdx.y;
    const long long pbase = a.offsets ? a.offsets[pair] : 0;
    const long long m = a.num[pair];
    PoseSet* poses = a.poses + pair;
    double fx = 1.0, fy = 1.0, cx = 0.0, cy = 0.0, sk = 0.0;
    if constexpr (KIND == MODEL_H) {
        if (a.planes[pair].rotation_only) {  // no vote: nothing passes, best stays -1 and T3 writes NaN points
            for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x)
                a.pass[pbase + i] = 0;
            return;
        }
        const double* K = a.Ks + 9 * (long long)pair;
        fx = K[0]; fy = K[4]; cx = K[2]; cy = K[5]; sk = K[1];
    }
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int r0 = a.rec[pair].sample[0];
    for (long long t0 = blockIdx.x * (long long)blockDim.x; t0 < 4 * m; t0 += (long long)gridDim.x * blockDim.x) {
        const long long t = t0 + threadIdx.x;
        const long long i = t >> 2;
        const int p = (int)(t & 3);
        bool ok = false, counts = false;
        if (i < m) {
            const long long gi = a.idx[pbase + i];
            Corr c = a.pts[pbase + gi];
            if constexpr (KIND == MODEL_H) {
                // pixel records through K^-1, the camera the decomposition and T3 use (hpose_args has checked that K
                // is upper triangular with K[2,2] = 1): y first, then x minus the skew's share.  With no skew this is
                // k_normalise's (x - cx) / fx (eight_point.py:127-133), bit for bit.
                c.ya = __ddiv_rn(__dsub_rn(c.ya, cy), fy);
                c.yb = __ddiv_rn(__dsub_rn(c.yb, cy), fy);
                c.xa = __ddiv_rn(__dsub_rn(__dsub_rn(c.xa, cx), __dmul_rn(sk, c.ya)), fx);
                c.xb = __ddiv_rn(__dsub_rn(__dsub_rn(c.xb, cx), __dmul_rn(sk, c.yb)), fx);
            }
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
            ok = (X1[2] >= -kCheiralityTolerance) && (z2 >= -kCheiralityTolerance) && (nrm <= a.dist_thr);  // :478-487
            // np.count_nonzero of the passing INDICES (:228-230): list position 0 never counts.  The list is the RANSAC
            // inlier list (apps/sfm.py:118-133), whose position 0 is the winner's first sample (ransac.py:76); without
            // a sample row it is the first correspondence.
            if constexpr (KIND == MODEL_E) counts = ok && !(r0 >= 0 ? (gi == (long long)r0) : (i == 0));
            else counts = ok;  // a homography's vote counts every passing inlier
        }
        const unsigned lane = threadIdx.x & 31u;
        const unsigned okb = __ballot_sync(0xffffffffu, ok);
        if (i < m && p == 0) a.pass[pbase + i] = (uint8_t)((okb >> (lane & ~3u)) & 0xfu);
        const unsigned cb = __ballot_sync(0xffffffffu, counts);
        if (lane < 4) {
            const int n = __popc(cb & (0x11111111u << lane));  // lanes with pose == lane
            if (n) atomicAdd(&s_cnt[lane], n);
        }
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_cnt[threadIdx.x])
        atomicAdd((unsigned long long*)&poses->counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
    // np.argmax(num_good_correspondences) (:237), first maximum: by the last block of the pair
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&a.done[pair], 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    __shared__ int s_best;
    if (threadIdx.x == 0) {
        a.done[pair] = 0;
        int bst = poses->best;
        if (bst != -2) {
            const volatile long long* cn = poses->counts;
            bst = 0;
            for (int q = 1; q < 4; ++q)
                if (cn[q] > cn[bst]) bst = q;
            poses->best = bst;
        }
        s_best = bst;
        poses->pad = (m <= kTailSmallTri) ? 1 : 0;  // tells T3 that the pair is already triangulated
    }
    __syncthreads();
    // a short inlier list is triangulated right here (same code, already in the instruction cache); a long one by T3
    if (m <= kTailSmallTri) {
        const int bst = s_best;
        for (long long i = threadIdx.x; i < m; i += blockDim.x)
            tail_triangulate_one(a, pair, pbase, i, bst, __ldcg(a.pass + pbase + i));
    }
}

__global__ void __launch_bounds__(128) k_tail_triangulate(const TailArgs a) {
    chain_enter();
    const int pair = blockIdx.y;
    if (a.poses[pair].pad) return;  // T2 already did it
    const long long pbase = a.offsets ? a.offsets[pair] : 0;
    const long long m = a.num[pair];
    const int b = a.poses[pair].best;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x)
        tail_triangulate_one(a, pair, pbase, i, b, a.pass[pbase + i]);
}

// ---- batch: per-pair results packed densely for the copy back to the host -------------------
// out_off[p] = sum of num[q], q < p (single block); out_off[P] = total.
__global__ void __launch_bounds__(1024) k_batch_offsets(const long long* __restrict__ num, int npairs, long long* __restrict__ out_off) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < npairs; base += 1024) {
        const int i = base + threadIdx.x;
        const long long v = (i < npairs) ? num[i] : 0;
        long long x = v;
        for (int d = 1; d < 32; d <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) warp_tot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long w = warp_tot[lane];
            for (int d = 1; d < 32; d <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += y;
            }
            warp_tot[lane] = w;
        }
        __syncthreads();
        const long long before = carry + (warp ? warp_tot[warp - 1] : 0) + x - v;
        if (i < npairs) out_off[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) out_off[npairs] = carry;
}

__global__ void __launch_bounds__(256) k_batch_pack(const long long* __restrict__ offsets, const long long* __restrict__ num,
                                                    const long long* __restrict__ out_off, const long long* __restrict__ idx,
                                                    const uint8_t* __restrict__ pass, const double* __restrict__ X,
                                                    int32_t* __restrict__ idx_out, uint8_t* __restrict__ pass_out,
                                                    double* __restrict__ X_out) {
    const int pair = blockIdx.y;
    const long long m = num[pair], src = offsets[pair], dst = out_off[pair];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        idx_out[dst + i] = (int32_t)idx[src + i];
        pass_out[dst + i] = pass[src + i];
        X_out[3 * (dst + i)] = X[3 * (src + i)];
        X_out[3 * (dst + i) + 1] = X[3 * (src + i) + 1];
        X_out[3 * (dst + i) + 2] = X[3 * (src + i) + 2];
    }
}

}  // namespace sfm
