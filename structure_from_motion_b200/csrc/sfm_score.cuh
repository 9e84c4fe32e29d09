// K2 (scoring), K3 (finalise + select) and K4 (inlier mask of one hypothesis).
#pragma once
#include <type_traits>

#include "sfm_device.cuh"
#include "sfm_types.h"

namespace sfm {

// ------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA) primitives, raw PTX for sm_100a
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
// 1-D bulk async copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, void* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ------------------------------------------------------------------------------------
// K2 — score H hypotheses against N correspondences.
//
// Restates the inner loop of fit_with_ransac (lib/ransac/ransac.py:66-82) with
// calculate_sed_inlier_score (lib/epipolar/epipolar_ransac.py:18-25, lib/epipolar/sed.py:7-30)
// as the scorer: for every hypothesis, the number of correspondences with sed <= thr and
// the sums of sed and sed^2 over them.  (The 8 sample points are scored like any other
// point here; K3 applies the "samples are not thresholded but always counted in the
// error" rule of ransac.py:63-64,76.)
//
// Mapping: lane = hypothesis.  Each thread keeps HPT essential matrices in registers and
// streams correspondences from shared-memory tiles (every lane reads the same 32-byte record:
// two broadcast LDS.128).  Every WARP is an autonomous worker: it claims work items
// (pair, correspondence split, group of 32*HPT hypotheses) from an atomic counter and streams
// its correspondences through its own kStages-deep ring of tiles filled by 1-D bulk async
// copies (TMA, issued by lane 0, completion on the warp's own mbarriers).  There is no
// block-level barrier anywhere: a warp that meets many survivors delays nobody.
// Persistent: the grid is one wave (SMs x resident blocks).
//
// Two-level evaluation.  Every (hypothesis, correspondence) gets a cheap division-free
// test; the sign bits of a BATCH of HPT*G (<= 32) tests are collected in one register per
// lane and the warp votes once per batch.  Lanes with survivors (~1 % of the tests survive)
// append one {mask, origin} record to a 64-record per-warp ring (ballot-compacted, positions
// are warp-uniform registers: no atomics); whenever 32 records are queued all lanes expand
// the records and process them 32 at a time (dense, no divergence): the exact reference-order
// SED is evaluated and compared with thr.
//
//   SCREEN (default), 9 FP64 issue slots per evaluation.  sed <= thr implies
//   r^2 <= thr * nb  (drop the image-A term), nb = lb0^2 + lb1^2, lb = E^T b, r = lb . a.
//   nb depends on the image-B point only.  K2 streams its own copy of a single pair's correspondences,
//   sorted by a Morton key of (xb, yb) at upload (k2_order_*, sfm_ransac.cu: k2_order), and every tile of kTile
//   records comes with the box of its B points: centre (cx, cy), half-widths (wx, wy) with
//   |xb - cx| <= wx and |yb - cy| <= wy for every record of the tile.  Once per (tile, hypothesis):
//       l_i = lb_i(cx, cy),  m_i = |l_i| + |E_0i| wx + |E_1i| wy  (i = 0, 1)      (8 DFMA)
//       T = thr' (m0^2 + m1^2) + kappa                                             (3 DFMA)
//   and per test
//       lb0, lb1, lb2   (6 DFMA)      r = lb0 xa + lb1 ya + lb2   (2 DFMA)      d = r^2 - T   (1 DFMA)
//   with "d < 0" (sign bit) as the test.  thr' = thr (1 + 3e-9) and
//   kappa_h = 4.2e-20 (1 + thr) |E_h|_F^2 A^2 B^2  (A, B = max |(x, y, 1)| over each image).
//   Why no inlier of the exact scorer is ever screened out, at any threshold:
//   (a) the reference's r and nb against the exact ones: |r_screen - r_ref| <= 32 u |E| A B =: eps
//       and 2 |r| eps <= 1e-9 r^2 + 1e9 eps^2 (AM-GM), the same for the absolute errors of the
//       reference's lb0, lb1 inside its nb: 4e-20 (1 + thr) |E|^2 A^2 B^2 of kappa and a relative
//       1e-9 of thr' (the bound of the 11-slot screen this body replaced, which had the larger
//       screen-side rounding: it also rounded (xa, ya) / sqrt(thr')).
//   (b) the box bound against the exact nb of every record of the tile: lb_i is affine in b, so
//       |lb_i(b)| <= |lb_i(c)| + |E_0i| wx + |E_1i| wy exactly.  The computed l_i is within
//       delta_i <= 2.0001 u |E_.i| |(cx, cy, 1)| of lb_i(c), and |(cx, cy, 1)|^2 <= 2 B^2, so
//       (|l_i| + delta_i + w_i)^2 <= (1 + 1e-9) (|l_i| + w_i)^2 + 1.000001e9 delta_i^2 leaves
//       1e-22 thr |E|^2 B^2 <= 0.0025 * 4e-20 (1 + thr) |E|^2 A^2 B^2 absolute and 1e-9 relative;
//       the seven roundings of m_i, m0^2 + m1^2 and T are downward by at most (1 - 8u) on sums of
//       non-negative terms, covered by the remaining 1e-9 of thr'.  kappa's 0.2e-20 covers both.
//   A T that is NaN becomes +inf, a second line behind the range guard below (only a NaN model can make one: T's
//   terms are non-negative and thr' >= 1e-280, so an infinite box gives T = +inf).  Padding lanes have E = 0
//   and kappa = -1, so T = -1 and d = 1 > 0 (boxes are finite: a tile with a non-finite B
//   coordinate gets centre 0 and half-widths DBL_MAX).  The screen is written
//   hypothesis-innermost so that consecutive DFMAs share the correspondence operand (a DFMA
//   with three fresh 64-bit register operands issues at 2/3 rate on sm_100, measured by
//   tools/fp64_micro.cu).
//   SCREEN11: the 11-slot one-sided screen for uploads without the sorted copy (batches, short pairs: their boxes
//   are wide, see k2_order in sfm_ransac.cu).  With s = sqrt(thr'), E has columns 0 and 1 pre-multiplied by s and the
//   records are a copy with (xa, ya) pre-divided by s (k_screen_pts64), so that
//       lb0' = s lb0, lb1' = s lb1, lb2 (6 DFMA)   r (2 DFMA)   m = lb1'^2 + kappa; m = lb0'^2 + m (2)   d = r^2 - m (1)
//   with the same thr' and kappa ((a) above covers it: its nb is the computed one).
//   FULL: the 21-slot two-sided division-free decision on the unscaled data (survivors ~
//   inliers); identical results; the like-for-like arithmetic baseline AND the body the AUTO
//   variant switches to above 9 % survivors.  Its survivor path differs: one ring ENTRY per
//   survivor (handed out in ballot-compacted rounds) instead of one record per lane and batch,
//   and models and correspondences gathered from shared memory (ScoreWarpSmemFS).
//   SCREEN32 (reported separately, never the fp64 headline): the same 11-slot test in fp32 on
//   E/|E|_F and fp32 copies of the correspondences — a PRE-FILTER only: every survivor is still
//   decided and summed by the exact fp64 scorer, so counts, sums and the winner are bit-identical
//   to the fp64 variants.  With u = 2^-24: |r32 - r| <= eps = 16 u A B, |lb' - s lb| <= 4 u s B;
//   (|r| + eps)^2 <= (1+l) r^2 + (1+1/l) eps^2 and the same for nb with l = 1/64 give the test
//   r32^2 < thr32 nb32 + kappa32, thr32 = 1.0316 thr, kappa32 = 1.2e-10 (1+thr) A^2 B^2
//   (>= u^2 [2113 thr B^2 + 16640 A^2 B^2]); ~2 % more survivors than the fp64 screen.
//
// Range guard, every body.  The arguments above model each rounding as relative (1 + delta, |delta| <= u); they hold
// while no quantity of a screen or of the reference leaves the normal range.  With F = |E_h|_F^2 and A^2, B^2 >= 1 (the
// bounds of k_normalise, over records with four finite coordinates; a non-finite record has sed = inf or NaN and is
// never an inlier at thr <= 1e100, the largest threshold K2 scores):
//   |lb_i| <= |E| B, |la_i| <= |E| A, |r| <= |E| A B, so na, nb, r^2 <= F A^2 B^2 and na nb <= (F A^2 B^2)^2.
//   Over:  FULL's largest terms are r^2 (na + nb) <= 2 (F A^2 B^2)^2 and thr' na nb <= 1.01e100 (F A^2 B^2)^2; the
//          one-sided T <= 1.01e100 * 8 F B^2 + kappa.  F A^2 B^2 <= 2^200 keeps all of them below 2^740, clear of
//          overflow - and keeps the reference's na, nb finite, so it has none of the sed = 0 "inliers" it reports when
//          na and nb overflow while r^2 does not (|E| near 1e154 on unit coordinates).
//   Under: an underflowing operation adds an absolute error of at most 2^-1075 instead.  In the one-sided bodies such
//          errors reach d as at most ~1e3 (1 + thr) 2^-1075 (through thr' NB+ and the squares; through r and lb only
//          as squares, by the AM-GM step of (a)), covered by kappa's spare 0.2e-20 (1 + thr) F A^2 B^2 once F >= 2^-200.
//          FULL's decision is homogeneous of degree 4 in E with the same absolute slack 1e-22 na nb, so it decides as
//          at unit scale while na nb stays normal: F >= 2^-200 keeps na nb ~ F^2 |a|^2 |b|^2 above 2^-400 for records
//          off the epipoles (below the range, at |E| ~ 1e-80 on unit coordinates, both r^2 (na + nb) and thr' na nb
//          underflow to 0, d = +0 and inliers were screened out).  SCREEN32 normalises E by rsqrt(F),
//          which needs F normal.
// A model outside kRangeLo = 2^-200 <= F, F A^2 B^2 <= kRangeHi = 2^200 (an inf or NaN one included) gets every test
// survive: one OR of a per-item mask into each batch's survivor bits, no work per test.  Models of the eight-point
// fit (e_22 = 1 on coordinates of order 1) sit far inside; the guard costs only hypotheses that are degenerate anyway.
//
// Order-independent accumulation.  An inlier's sed (or sed^2 — only the sum the aggregation
// method needs is accumulated unless both are requested) is converted to an 84-bit fixed-point
// integer scaled so that thr < 2^e maps below 2^84, split into four 21-bit chunks and added with
// native 32-bit shared-memory atomics (a word cannot overflow within an item of <= 2^11
// correspondences); chunks are folded into 64-bit global accumulators at the end of the item.
// Integer addition is associative, so the sums are independent of warp scheduling, split count
// and GPU count — run-to-run deterministic by construction; every term >= thr * 2^-10 enters
// without rounding, smaller ones are truncated at 2^-84 of the scale (<= 6e-26 thr per term).
// ------------------------------------------------------------------------------------
constexpr int kScoreThreads = 128;
constexpr int kScoreWarps = kScoreThreads / 32;
constexpr int kTile = 64;     // correspondences per stage (2 KB)
constexpr int kStages = 3;
constexpr int kRing = 64;     // survivor records per warp: < 32 pending + <= 32 new
constexpr unsigned kMaxPoints = 1u << 25;
constexpr int kChunks = 4;             // 21-bit chunks of an 84-bit fixed-point term
constexpr int kFixedBits = 21 * kChunks;  // 2^kFixedBits = scaled value of 2^e (thr < 2^e)
constexpr int kChunkBits = 21;
constexpr int kAccWords = 1 + 2 * kChunks;  // count, sum(sed), sum(sed^2)
constexpr long long kMaxItemPoints = 1ll << 11;  // 2^11 adds of < 2^21 cannot overflow a 32-bit word
enum { SUM_S1 = 1, SUM_S2 = 2 };       // which sums a launch accumulates
enum { MODE_FULL = 0, MODE_SCREEN = 1, MODE_SCREEN32 = 2, MODE_SCREEN11 = 3 };
constexpr double kKappaCoef = 4.2e-20;
constexpr double kThrScreenFactor = 1.0 + 3e-9;  // thr' of the fp64 screen, see the K2 header
constexpr double kKappa32Coef = 1.2e-10;   // fp32 pre-filter, see the K2 header
constexpr double kThr32Factor = 1.0316;   // (1 + 1/64)^2 (1 + 1e-4)
constexpr double kRangeLo = 0x1p-200;      // range guard on |E|_F^2, see the K2 header
constexpr double kRangeHi = 0x1p200;       // range guard on |E|_F^2 A^2 B^2


__global__ void __launch_bounds__(256) k_pad_models(const double* __restrict__ E, long long htotal, ModelRow* __restrict__ rows) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= htotal) return;
    const double* e = E + 9 * i;
    ModelRow r;
    r.a = make_double4(e[0], e[1], e[2], e[3]);
    r.b = make_double4(e[4], e[5], e[6], e[7]);
    r.c = make_double4(e[8], 0.0, 0.0, 0.0);
    rows[i] = r;
}

struct ScoreArgs {
    const Corr* pts;           // K-normalised correspondences: K2's sorted copy (the 9-slot SCREEN), else in input order
    const void* spts;          // streamed records: pts, or its scaled copy (SCREEN11: Corr, SCREEN32: Corr32)
    const double* bounds;      // [2]: max (xa^2+ya^2+1), max (xb^2+yb^2+1) over all correspondences
    long long n;
    const long long* offsets;  // [npairs+1] or null (single pair of n records)
    const double* E;           // [npairs][h][9]
    const ModelRow* rows;      // [npairs][h] padded copies of E for the survivor path
    long long h;
    double thr, thr_pre, s;    // s = sqrt(thr_pre) (SCREEN32)
    double kappa_coef;         // kKappaCoef * (1 + thr)
    double kappa32_coef;       // kKappa32Coef * (1 + thr)
    double scale1, scale2;     // 2^(63-e), 2^(63-2e) with thr < 2^e
    int sums;                  // SUM_S1 | SUM_S2
    long long chunk;           // correspondences per split (multiple of kTile)
    int hblocks, nsplit;
    long long total_items;
    long long htotal;          // npairs * h
    unsigned* work_counter;
    unsigned long long* acc;   // [kAccWords][htotal] exact integer accumulators (pre-zeroed)
    const int* mode_flag;      // AUTO variant: the MODE the pilot selected (k_score_auto runs that body); else null
    const double4* boxes;      // SCREEN (single pairs only): (cx, cy, wx, wy) of the B points of tile t of pts at [t]
};

__device__ __forceinline__ unsigned atom_add_acq_rel_shared(unsigned* p, unsigned v) {
    unsigned old;
    asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(p)), "r"(v) : "memory");
    return old;
}
// one step of a warp inclusive scan: v += shfl_up(v, d) where the source lane exists
__device__ __forceinline__ int scan_step(int v, int d) {
    asm volatile("{ .reg .pred p; .reg .b32 t; shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff; @p add.s32 %0, %0, t; }"
                 : "+r"(v) : "r"(d));
    return v;
}
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// four 21-bit chunks of V = floor(x * 2^(84-e)) < 2^84 (x <= thr < 2^e; `scale` = 2^(63-e)): c[3] is the most
// significant.  The top 63 bits come from one conversion, the low 21 from the exact remainder, so terms down to
// 2^-84 of the threshold scale enter the sum (a 63-bit term lost up to 1e-7 of a sum of squares whose inliers were
// a thousand times tighter than the threshold).  Truncation keeps every chunk < 2^21.
__device__ __forceinline__ void chunks21(double x, double scale, unsigned (&c)[kChunks]) {
    const double t = x * scale;                            // < 2^63
    const unsigned long long v = __double2ull_rz(t);       // floor (t >= 0)
    const double rem = t - __ull2double_rz(v);             // exact: v == t when t >= 2^53
    c[0] = (unsigned)__double2uint_rz(rem * 2097152.0);    // 2^21
    c[1] = (unsigned)v & 0x1fffffu;
    c[2] = (unsigned)(v >> kChunkBits) & 0x1fffffu;
    c[3] = (unsigned)(v >> (2 * kChunkBits));
}

// fp32 twin of the screening record
struct __align__(16) Corr32 {
    float xa, ya, xb, yb;
};

// T = thr' NB+ + kappa of one hypothesis over one tile: NB+ >= lb0^2 + lb1^2 at every B point of the box (K2 header);
// a NaN bound (a NaN model) becomes +inf, so that every test of the tile survives and the exact scorer decides
__device__ __forceinline__ double tile_bound(const double (&e)[9], double4 box, double thr_pre, double kap) {
    const double l0 = fma(box.x, e[0], fma(box.y, e[3], e[6]));
    const double l1 = fma(box.x, e[1], fma(box.y, e[4], e[7]));
    const double m0 = fma(fabs(e[0]), box.z, fma(fabs(e[3]), box.w, fabs(l0)));
    const double m1 = fma(fabs(e[1]), box.z, fma(fabs(e[4]), box.w, fabs(l1)));
    const double t = fma(thr_pre, fma(m0, m0, m1 * m1), kap);
    return t == t ? t : __longlong_as_double(0x7ff0000000000000LL);
}

// ---- K2's copy of the correspondences (at upload; it depends on nothing else) ----------------------------------
// Order-preserving 64-bit image of a double (NaN excluded by the callers): unsigned order = numeric order.
__device__ __forceinline__ unsigned long long k2_ordered(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double k2_unordered(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// Bounding box of the pair's B points: bb = {~min xb, ~min yb, max xb, max yb} as ordered keys (zero on entry; minima
// complemented so that every word is an atomicMax).  NaN coordinates are left out.
__global__ void __launch_bounds__(256) k2_order_bbox(const Corr* __restrict__ pts, long long n,
                                                     unsigned long long* __restrict__ bb) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    unsigned long long v[4] = {0ull, 0ull, 0ull, 0ull};
    if (i < n) {
        const Corr c = pts[i];
        if (c.xb == c.xb) { v[0] = ~k2_ordered(c.xb); v[2] = k2_ordered(c.xb); }
        if (c.yb == c.yb) { v[1] = ~k2_ordered(c.yb); v[3] = k2_ordered(c.yb); }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, v[k], d);
            v[k] = o > v[k] ? o : v[k];
        }
    }
    if ((threadIdx.x & 31) == 0 && i < n)
#pragma unroll
        for (int k = 0; k < 4; ++k) atomicMax(bb + k, v[k]);
}

// one axis quantised to 16 bits inside [lo, hi]; a degenerate or non-finite range (or a NaN coordinate) maps to 0
__device__ __forceinline__ unsigned k2_quantise(double x, double lo, double hi) {
    const double sc = 65535.0 / (hi - lo);
    const double q = (sc > 0.0 && sc < 1e308) ? (x - lo) * sc : 0.0;
    return (unsigned)fmin(fmax(q, 0.0), 65535.0);  // fmax(NaN, 0) = 0
}
__device__ __forceinline__ unsigned k2_spread16(unsigned v) {  // bit k -> bit 2k
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    return (v | (v << 1)) & 0x55555555u;
}
// sort keys (Morton code of (xb, yb) in the pair's box) and the identity permutation
__global__ void __launch_bounds__(256) k2_order_keys(const Corr* __restrict__ pts, long long n,
                                                     const unsigned long long* __restrict__ bb,
                                                     unsigned* __restrict__ keys, int* __restrict__ idx) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Corr c = pts[i];
    const unsigned qx = k2_quantise(c.xb, k2_unordered(~bb[0]), k2_unordered(bb[2]));
    const unsigned qy = k2_quantise(c.yb, k2_unordered(~bb[1]), k2_unordered(bb[3]));
    keys[i] = (k2_spread16(qy) << 1) | k2_spread16(qx);
    idx[i] = (int)i;
}

// One warp per tile: gather the tile's records in sorted order and write its box (K2 header).  cx is the rounded
// midpoint and wx = max(hi - cx, cx - lo) rounded up, so |xb - cx| <= wx holds exactly for every record.
constexpr int kOrderWarps = 4;
__global__ void __launch_bounds__(32 * kOrderWarps) k2_order_gather(const Corr* __restrict__ pts, long long n,
                                                                   const int* __restrict__ idx, Corr* __restrict__ out,
                                                                   double4* __restrict__ boxes) {
    const long long t = (long long)blockIdx.x * kOrderWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t * kTile >= n) return;
    double lo[2] = {__longlong_as_double(0x7ff0000000000000LL), __longlong_as_double(0x7ff0000000000000LL)};
    double hi[2] = {-lo[0], -lo[1]};
#pragma unroll
    for (int k = lane; k < kTile; k += 32) {
        const long long i = t * kTile + k;
        if (i < n) {
            const Corr c = pts[idx[i]];
            out[i] = c;
            lo[0] = fmin(lo[0], c.xb); hi[0] = fmax(hi[0], c.xb);  // fmin/fmax drop NaN
            lo[1] = fmin(lo[1], c.yb); hi[1] = fmax(hi[1], c.yb);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], d));
            hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], d));
        }
    if (lane == 0) {
        double cw[4];
        bool finite = true;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            cw[k] = 0.5 * lo[k] + 0.5 * hi[k];
            cw[2 + k] = fmax(__dsub_ru(hi[k], cw[k]), __dsub_ru(cw[k], lo[k]));
            finite = finite && fabs(cw[k]) <= 1.7976931348623157e308 && fabs(cw[2 + k]) <= 1.7976931348623157e308;
        }
        // a tile with an infinite B coordinate (or only NaN ones): the box of every finite point
        boxes[t] = finite ? make_double4(cw[0], cw[1], cw[2], cw[3])
                          : make_double4(0.0, 0.0, 1.7976931348623157e308, 1.7976931348623157e308);
    }
}

// For the AUTO variant, the PILOT that chooses between the one-sided and the two-sided fp64 screen: kPilotBlocks blocks
// run the one-sided test that K2 will run (9-slot against the tile bounds, or 11-slot) on a sample (64 hypotheses spread
// over the range x ~1 000 correspondences of the first pair, 8 tests per thread) and the last of them to finish turns
// the pass rate into the MODE the scoring kernel checks.  Above ~9 % survivors the exact evaluation of the survivors
// dominates and the 21-slot two-sided screen (survivors = inliers) wins; below, the one-sided screen does (DESIGN.md,
// table against the threshold).
constexpr int kPilotBlocks = 32;
constexpr int kPilotHyps = 64;
constexpr int kPilotPts = 1024;
constexpr double kPilotFullAbove = 0.09;  // measured crossover of the two bodies (tools/auto_crossover.py)
struct PilotArgs {
    const double* E;      // models of the first pair
    long long h;          // hypotheses per pair
    long long plen;       // correspondences of the first pair
    double thr_pre;
    const double* bounds; // [2] A^2, B^2 (k_normalise)
    double kappa_coef;    // kKappaCoef * (1 + thr)
    const double4* boxes; // the tile boxes of K2's sorted copy (BOXES pilot only)
    unsigned* counters;   // [0] passes, [1] ticket (zero on entry)
    int* mode_flag;       // out
};
// the pilot's work in one of nb blocks (block-uniform: every thread of the block calls it); BOXES: the 9-slot test
// against the tile bounds, else the 11-slot one
template <bool BOXES>
__device__ __forceinline__ void pilot_block(const Corr* __restrict__ pts, const PilotArgs& pa, int nb) {
    // thread t of block b -> hypothesis (t % 64) of the sample, correspondences (b * 4 + t / 64) + 32 k
    const long long nh = pa.h < kPilotHyps ? pa.h : kPilotHyps;
    const int hs = threadIdx.x % kPilotHyps;
    int pass = 0, tests = 0;
    if (hs < nh && pa.plen > 0) {
        const long long hyp = (pa.h / nh) * hs;
        double e[9], f2 = 0.0;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            e[k] = pa.E[9 * hyp + k];
            f2 = fma(e[k], e[k], f2);
        }
        const double kap = f2 * (pa.bounds[0] * pa.bounds[1] * pa.kappa_coef);  // as K2's kappa
        const long long np = pa.plen < kPilotPts ? pa.plen : kPilotPts;
        const long long step = pa.plen / np;
        const int lanes = nb * (256 / kPilotHyps);
        // at most 8 correspondences per thread, loads issued back to back (the kernel is pure latency otherwise)
        Corr cs[8];
        double4 bx[8];
        int got = 0;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const long long q = blockIdx.x * (256 / kPilotHyps) + threadIdx.x / kPilotHyps + (long long)u * lanes;
            if (q < np) {
                cs[u] = pts[q * step];
                if constexpr (BOXES) bx[u] = pa.boxes[q * step / kTile];
                got = u + 1;
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (u < got) {
                const double lb0 = fma(cs[u].xb, e[0], fma(cs[u].yb, e[3], e[6]));
                const double lb1 = fma(cs[u].xb, e[1], fma(cs[u].yb, e[4], e[7]));
                const double lb2 = fma(cs[u].xb, e[2], fma(cs[u].yb, e[5], e[8]));
                const double r = fma(cs[u].xa, lb0, fma(cs[u].ya, lb1, lb2));
                double t;
                if constexpr (BOXES) t = tile_bound(e, bx[u], pa.thr_pre, kap);
                else t = pa.thr_pre * fma(lb0, lb0, lb1 * lb1);
                pass += fma(r, r, -t) < 0.0 ? 1 : 0;
                tests += 1;
            }
    }
    // pack (passes, tests) into one 64-bit add: tests <= 2^17 per launch
    unsigned long long v = ((unsigned long long)pass << 32) | (unsigned)tests;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    __shared__ unsigned long long s_sum;
    __shared__ int s_last;
    if (threadIdx.x == 0) s_sum = 0ull;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_sum, v);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long* tot = reinterpret_cast<unsigned long long*>(pa.counters);
        atomicAdd(tot, s_sum);
        __threadfence();
        s_last = atomicAdd(pa.counters + 2, 1u) == (unsigned)(nb - 1);
        if (s_last) {
            __threadfence();
            const unsigned long long t = *reinterpret_cast<volatile unsigned long long*>(tot);
            const double rate = (unsigned)t ? (double)(t >> 32) / (double)(unsigned)t : 0.0;
            *pa.mode_flag = rate > kPilotFullAbove ? MODE_FULL : MODE_SCREEN;
        }
    }
}
// the 9-slot screen's pilot on its own (K2's sorted copy needs no per-call copy)
__global__ void __launch_bounds__(256) k_pilot(const Corr* __restrict__ pts, const PilotArgs pa) {
    chain_enter();
    pilot_block<true>(pts, pa, gridDim.x);
}

// 11-slot screen only: Corr copy with (xa, ya) pre-divided by s = sqrt(thr') (thr-dependent, so it runs at the head of
// every such scoring call; scaling the tiles inside K2 instead costs 5 %: profiles/r2_scale_modes.txt).  AUTO: its
// first kPilotBlocks blocks also run the pilot of the 11-slot screen (pa.mode_flag set).
__global__ void __launch_bounds__(256) k_screen_pts64(const Corr* __restrict__ pts, long long n, double inv_s,
                                                      Corr* __restrict__ spts, const PilotArgs pa) {
    chain_enter();
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) {
        Corr c = pts[i];
        c.xa *= inv_s;
        c.ya *= inv_s;
        spts[i] = c;
    }
    if (!pa.mode_flag || blockIdx.x >= kPilotBlocks) return;
    pilot_block<false>(pts, pa, gridDim.x < kPilotBlocks ? gridDim.x : kPilotBlocks);
}

// fp32 pre-filter only: Corr32 copy of the correspondences with (xa, ya) pre-divided by s (thr-dependent, so it runs
// at the head of every SCREEN32 scoring call).  The coordinate bounds used by kappa come from k_normalise.
__global__ void __launch_bounds__(256) k_screen_pts32(const Corr* __restrict__ pts, long long n, double inv_s,
                                                      Corr32* __restrict__ spts) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Corr c = pts[i];
    Corr32 f;
    f.xa = (float)(c.xa * inv_s); f.ya = (float)(c.ya * inv_s); f.xb = (float)c.xb; f.yb = (float)c.yb;
    spts[i] = f;
}

// Per-warp shared-memory state: every warp is an autonomous worker (own tile ring, own
// mbarriers, own survivor ring and accumulators); there is no block-level barrier anywhere.
template <int HPT>
struct alignas(128) ScoreWarpSmem {
    Corr tile[kStages][kTile];
    unsigned sacc[HPT][kAccWords][32];
    uint2 ring[kRing];
    unsigned short own[32];
    unsigned long long full_bar[kStages];
};
// The 9-slot body's layout: the same, plus the tile boxes and kappa.  Only it pays for them: the other one-sided
// bodies keep the smaller layout and with it their blocks per SM (SCREEN32 at hpt 4 fits 5 blocks only without them).
template <int HPT>
struct alignas(128) ScoreWarpSmemBox : ScoreWarpSmem<HPT> {
    double4 box[kStages];  // the box of the tile in the same stage, delivered by the same mbarrier
    double kap[HPT][32];   // kappa of (slot, lane), read once per tile (registers are the screen's)
};

// Two-sided body (the survivor-rich regime: AUTO sends > 9 % survivors here): the drain gathers nothing
// from global memory.  Its models sit in shared memory (component-major: a gather of 32 models is nine LDS.64) and
// its correspondences are read from the tile ring itself - the two-sided screen streams the UNSCALED records, and a
// stage is refilled only after every record that points into it has been drained (one tile of slack: see the tile
// loop).  Tiles are 32 records so that ring + models fit the same five blocks per SM.  ncu before this layout (17 %
// inliers): 73 % of the drain's gathers missed L1 (60 KB next to 180 KB of shared memory, against 120 KB of model
// rows per SM) and the first DMUL behind them carried 13 % of all stall samples.
constexpr int kTileFS = 32;
constexpr int kStagesFS = 3;
template <int HPT>
struct alignas(128) ScoreWarpSmemFS {
    Corr tile[kStagesFS][kTileFS];
    double model[32 * HPT][10];  // 80-byte rows: a gather is four LDS.128 + one LDS.64 per lane
    unsigned sacc[HPT][kAccWords][32];  // column of (slot j, lane l) = l ^ 16 j: the two slots of a lane in different banks
    uint2 ring[kRing];
    unsigned long long full_bar[kStagesFS];
};

// resident blocks per SM the register budget is shaped for (HPT 2 / 1): 20 / 32 warps.  Measured on config 3: HPT 2
// at 96 registers (5 blocks) beats 80 registers (6 blocks) by ~1.5 %: the extra registers let ptxas keep more
// independent DFMA chains in flight, which is what the FP64 pipe's ~25-cycle latency needs.
constexpr int score_min_blocks(int hpt) { return hpt == 2 ? 5 : 8; }


__device__ __forceinline__ int sign_word(double d) { return __double2hiint(d); }
__device__ __forceinline__ int sign_word(float f) { return __float_as_int(f); }

template <int HPT, int G, int MODE>
__device__ __forceinline__ void score_body(const ScoreArgs& a) {
    constexpr bool SCREEN = MODE != MODE_FULL;
    constexpr bool F32 = MODE == MODE_SCREEN32;
    constexpr bool SCALED = F32 || MODE == MODE_SCREEN11;  // columns 0, 1 of E times s, records (xa, ya) / s
    using T = typename std::conditional<F32, float, double>::type;       // arithmetic of the per-test work
    using P = typename std::conditional<F32, Corr32, Corr>::type;       // record streamed through shared memory
    constexpr int NB = HPT * G;  // tests per lane and batch = survivor bits per vote
    // two-sided: a survivor ring of per-survivor entries instead of per-lane records, drained from shared memory only
    constexpr bool ENTRY = MODE == MODE_FULL;
    constexpr bool BOX = MODE == MODE_SCREEN;  // 9-slot screen against the tile's bound
    constexpr int TILE = ENTRY ? kTileFS : kTile;
    constexpr int STAGES = ENTRY ? kStagesFS : kStages;
    constexpr int AHEAD = ENTRY ? STAGES - 1 : STAGES;  // tiles in flight; ENTRY keeps the previous tile's stage for the drain
    using WS = typename std::conditional<ENTRY, ScoreWarpSmemFS<HPT>,
                                         typename std::conditional<BOX, ScoreWarpSmemBox<HPT>, ScoreWarpSmem<HPT>>::type>::type;
    static_assert(NB <= 32 && (TILE % G) == 0 && (kTile % TILE) == 0, "a batch is at most 32 tests and divides a tile");
    static_assert(!ENTRY || HPT <= 2, "the two-sided body's bank swizzle of sacc holds two slots");
    extern __shared__ __align__(128) unsigned char score_smem[];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(full, (int)(threadIdx.x >> 5), 0);  // tells the compiler it is warp-uniform
    const unsigned lt = lanemask_lt();
    // The pilot's flag (AUTO only) never disagrees here: k_score_auto branches on it first.  The test stays because
    // without it ptxas spills 16-28 bytes in both k_score_auto kernels at the same 96 registers (k2_shapes_sass_check).
    if (a.mode_flag && (*a.mode_flag == MODE_FULL) != (MODE == MODE_FULL)) return;
    WS& ws = reinterpret_cast<WS*>(score_smem)[warp];

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(&ws.full_bar[s], 1);
        mbar_fence_init();
    }
#pragma unroll
    for (int j = 0; j < HPT; ++j)
#pragma unroll
        for (int k = 0; k < kAccWords; ++k) ws.sacc[j][k][lane] = 0;
    __syncwarp();
    uint2* q = ws.ring;
    unsigned head = 0, tail = 0;  // ring positions (records): warp-uniform, monotone, tail - head < 64
    unsigned gt = 0;              // tiles consumed so far by this warp (drives stage + parity)
    const double abnd = a.bounds[0] * a.bounds[1];  // A^2 B^2
    const double ab2 = SCREEN ? abnd * (F32 ? a.kappa32_coef : a.kappa_coef) : 0.0;

    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(a.work_counter, 1u);
        item = __shfl_sync(full, item, 0);
        if (item >= a.total_items) break;
        const int hw = (int)(item % (unsigned)a.hblocks);  // group of 32*HPT hypotheses
        const unsigned rest = item / (unsigned)a.hblocks;
        const int split = (int)(rest % (unsigned)a.nsplit);
        const int pair = (int)(rest / (unsigned)a.nsplit);

        const long long pbase = a.offsets ? a.offsets[pair] : 0;
        const long long plen = a.offsets ? a.offsets[pair + 1] - pbase : a.n;
        long long begin = (long long)split * a.chunk;
        if (begin > plen) begin = plen;
        const long long end = pbase + ((begin + a.chunk < plen) ? begin + a.chunk : plen);
        begin += pbase;
        const int ntiles = (int)((end - begin + TILE - 1) / TILE);
        // this warp's hypotheses: lane l, slot j  ->  hyp_w + 32*j + l
        const long long hyp_w = (long long)hw * (32 * HPT);
        const double* Ep = a.E + 9 * (long long)pair * a.h;
        const ModelRow* Rw = a.rows + (long long)pair * a.h + hyp_w;  // this warp's models, padded (survivor path)
        const Corr* pbeg = a.pts + begin;    // this item's correspondences (exact copies)
        const P* src = reinterpret_cast<const P*>(a.spts);
        const int box0 = (int)(begin / kTile);  // BOX: a single pair (pbase = 0), items start on tiles

        auto issue = [&](int t) {  // lane 0 only
            const int s = (int)((gt + (unsigned)t) % STAGES);
            const long long first = begin + (long long)t * TILE;
            const long long rem = end - first;
            const uint32_t bytes = (uint32_t)((rem < TILE ? rem : TILE) * sizeof(P));
            mbar_expect_tx(&ws.full_bar[s], bytes + (BOX ? (uint32_t)sizeof(double4) : 0u));
            bulk_g2s(&ws.tile[s][0], src + first, bytes, &ws.full_bar[s]);
            if constexpr (BOX) bulk_g2s(&ws.box[s], a.boxes + box0 + t, (uint32_t)sizeof(double4), &ws.full_bar[s]);
        };
        if (lane == 0) {
            for (int t = 0; t < AHEAD && t < ntiles; ++t) issue(t);
        }

        // register-resident models; SCREEN: kappa per hypothesis, the tile's bound T per hypothesis;
        // SCREEN11: columns 0 and 1 scaled by s, kappa per hypothesis;
        // SCREEN32: as SCREEN11, normalised to |E|_F = 1 (sed is scale-invariant in E) and rounded to fp32
        T e[HPT][9], kap[HPT], tb[HPT];
        unsigned fpat = 0u;  // bit HPT-1-j: slot j holds a model outside the range guard, every one of its tests survives
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = hyp_w + 32 * j + lane;
            const bool real = hyp < a.h;
            double v[9], f2 = 0.0;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                v[k] = real ? Ep[9 * hyp + k] : 0.0;
                f2 = fma(v[k], v[k], f2);
            }
            if constexpr (ENTRY) {  // the previous item's drains are complete (queue emptied at its end)
                double2* mp = reinterpret_cast<double2*>(&ws.model[32 * j + lane][0]);
                mp[0] = make_double2(v[0], v[1]);
                mp[1] = make_double2(v[2], v[3]);
                mp[2] = make_double2(v[4], v[5]);
                mp[3] = make_double2(v[6], v[7]);
                ws.model[32 * j + lane][8] = v[8];
            }
            // range guard (K2 header): the bodies are sound for kRangeLo <= |E|^2 and |E|^2 A^2 B^2 <= kRangeHi; outside
            // (a 0, inf or NaN norm included) the model's tests all survive and the exact scorer decides
            if (real && !(f2 >= kRangeLo && f2 * abnd <= kRangeHi)) fpat |= 1u << (HPT - 1 - j);
            const double nrm = F32 ? rsqrt(f2) : 1.0;
#pragma unroll
            for (int k = 0; k < 9; ++k) e[j][k] = (T)((SCALED && (k % 3) != 2) ? v[k] * nrm * a.s : v[k] * nrm);
            // padding lanes can never produce a survivor: m = T = -1, d = r^2 + 1 > 0
            kap[j] = (T)(real ? (F32 ? ab2 : f2 * ab2) : -1.0);
            if constexpr (BOX) ws.kap[j][lane] = kap[j];  // the previous item's tiles are done with it
        }
        // the guard's bits in every group of a batch (bit NB-1-i <-> test i = g * HPT + j, see the one-sided bodies)
        unsigned frep = 0u;
#pragma unroll
        for (int g = 0; g < G; ++g) frep |= 1u << (HPT * g);
        const unsigned fmask = fpat * frep;

        // Exact evaluation of <= 32 survivors, one per lane (the reference's arithmetic, sed_exact), and the sums.
        auto accumulate = [&](bool act, double sv, int slot, int owner) {
            if (act && (sv <= a.thr)) {  // ransac.py:73  score <= threshold
                unsigned ch[kChunks];
                // same-address atomics serialise; ENTRY also keeps the two slots of an owner in different banks
                unsigned* dst = &ws.sacc[slot][0][ENTRY ? (owner ^ (slot << 4)) : owner];
                atomicAdd(dst, 1u);
                if (a.sums & SUM_S1) {
                    chunks21(sv, a.scale1, ch);
#pragma unroll
                    for (int kk = 0; kk < kChunks; ++kk) atomicAdd(dst + 32 * (1 + kk), ch[kk]);
                }
                if (a.sums & SUM_S2) {
                    chunks21(__dmul_rn(sv, sv), a.scale2, ch);
#pragma unroll
                    for (int kk = 0; kk < kChunks; ++kk) atomicAdd(dst + 32 * (1 + kChunks + kk), ch[kk]);
                }
            }
        };
        // candidate's E and correspondence: from global memory (L1/L2 hits) by index, or - ENTRY - from shared memory
        auto survivor_sed = [&](unsigned hl, unsigned pos) -> double {
            double eo[9];
            Corr c;
            if constexpr (ENTRY) {
                const double2* mp = reinterpret_cast<const double2*>(&ws.model[hl][0]);
                const double2 m0 = mp[0], m1 = mp[1], m2 = mp[2], m3 = mp[3];
                eo[0] = m0.x; eo[1] = m0.y; eo[2] = m1.x; eo[3] = m1.y;
                eo[4] = m2.x; eo[5] = m2.y; eo[6] = m3.x; eo[7] = m3.y;
                eo[8] = ws.model[hl][8];
                c = (&ws.tile[0][0])[pos];
            } else {
                const ModelRow* er = Rw + hl;  // padding hypotheses never survive the screen: an active entry is real
                const double4 r0 = er->a, r1 = er->b;
                eo[0] = r0.x; eo[1] = r0.y; eo[2] = r0.z; eo[3] = r0.w;
                eo[4] = r1.x; eo[5] = r1.y; eo[6] = r1.z; eo[7] = r1.w;
                eo[8] = er->c.x;
                c = pbeg[pos];
            }
            return sed_exact(eo, c.xa, c.ya, c.xb, c.yb);
        };

        // ---- two-sided body: one ring ENTRY per survivor ------------------------------------------------------------
        // {owner lane << 14 | slot << 11 | position}: position = the correspondence's place in the tile ring.  A drain is "lane l takes entry head + l": no prefix sum over record counts, no search
        // for the n-th set bit, no record straddling a drain.  The bits of a batch are handed out in rounds, one bit per
        // lane and round (ballot-compacted): ~12 instructions per round, as many rounds as the fullest lane has
        // survivors.  ncu of the record scheme below at 17 % inliers: 130 of the drain's 237 instructions were that
        // bookkeeping, the n-th-set-bit search its longest dependent chain (0.30 -> 0.37e12 evaluations/s).  In the
        // one-sided body (1 % survivors, 1.3 bits per record) the rounds cost more than they save (-5 %), so it keeps
        // the records.
        unsigned* qe = reinterpret_cast<unsigned*>(ws.ring);
        constexpr int LH = HPT == 4 ? 2 : (HPT == 2 ? 1 : 0);  // slot bits, kept at the top of an entry
        const unsigned ln = (unsigned)__popc(lt);  // the lane index again, from a live register (ptxas re-reads SR_TID otherwise)
        auto drain_entries = [&]() {
            const unsigned navail = tail - head;  // 1..63
            const bool act = ln < navail;
            const unsigned en = act ? qe[(head + ln) & (kRing - 1)] : 0u;
            const int owner = (int)((en >> 14) & 31u), slot = LH ? (int)(en >> (32 - (LH ? LH : 1))) : 0;
            accumulate(act, survivor_sed((unsigned)(32 * slot + owner), en & 0x7ffu), slot, owner);
            head += navail < 32u ? navail : 32u;
            __syncwarp();
        };
        // pm: bit NB-1-i <-> test i = g * HPT + j of the batch whose first correspondence has position pos0;
        // entry = {slot i % HPT at the top | owner lane << 14 | pos0 + i / HPT}: a rotation of i added to a per-batch base
        auto push_entries = [&](unsigned pm, unsigned pos0) {
            const unsigned base = (ln << 14) | pos0;
            unsigned vote;
            while ((vote = __ballot_sync(full, pm != 0u)) != 0u) {
                const unsigned top = 0x80000000u >> __clz(pm | 1u);           // highest set bit (bit 0 for an empty mask)
                const unsigned i = (unsigned)(NB - 32) + (unsigned)__clz(pm | 1u);  // NB - 1 - bit
                const unsigned en = base + __funnelshift_r(i, i, LH);
                if (pm) qe[(tail + __popc(vote & lt)) & (kRing - 1)] = en;
                pm &= ~top;
                tail += __popc(vote);
                __syncwarp();
                if (tail - head >= 32u) drain_entries();
            }
        };

        // ---- one-sided bodies: one ring RECORD per (lane, batch) with survivors ------------------------------------
        // {batch mask pm, owner lane << 27 | item-relative index of the batch's first correspondence}; bit NB-1-i of pm
        // <-> test i = g*HPT + j.  drain_records() expands the first <= 32 records into <= 32 survivors, one per lane:
        // prefix sum of the popcounts, then an owner table in shared memory {record, bit position} that every record
        // fills for the survivor slots it owns (1.3 bits per record at a 1 % survivor rate).
        auto drain_records = [&]() {
            const unsigned nrec = tail - head;  // 1..63
            uint2 rec = make_uint2(0u, 0u);
            if ((unsigned)lane < nrec) rec = q[(head + lane) & (kRing - 1)];
            const int cnt = __popc(rec.x);
            int incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) incl = scan_step(incl, d);
            const int total = __shfl_sync(full, incl, 31);
            const int m = total < 32 ? total : 32;  // survivors handled now
            const int excl = incl - cnt;
            // ring bookkeeping: records entirely inside the first 32 survivors are retired
            const unsigned done_mask = __ballot_sync(full, (unsigned)lane < nrec && incl <= 32);
            const int ndone = __popc(done_mask);
            const bool act = lane < m;
            unsigned o = 0u;  // {record (low byte), bit position of this lane's survivor in it}
            uint2 rj = make_uint2(0u, 0u);
            if constexpr (!ENTRY) {
                // the record's set bits are handed out lowest first, so what is left in pmw afterwards is exactly what a
                // record that straddles the 32-survivor boundary keeps for the next drain
                unsigned pmw = rec.x;
                for (int t = excl; pmw && t < 32; ++t) {
                    ws.own[t] = (unsigned short)(lane | ((__ffs(pmw) - 1) << 8));
                    pmw &= pmw - 1u;
                }
                __syncwarp();
                o = act ? ws.own[lane] : 0u;
                rj = q[(head + (o & 255u)) & (kRing - 1)];
                __syncwarp();
                if (lane == ndone && (unsigned)lane < nrec) q[(head + lane) & (kRing - 1)].x = pmw;  // first record not retired
            }
            const int i = NB - 1 - (int)(o >> 8);  // test index in the batch: g * HPT + j
            const int owner = (int)(rj.y >> 27), slot = i % HPT;
            const unsigned rel = act ? (rj.y & 0x3fffffu) + (unsigned)(i / HPT) : 0u;
            accumulate(act, survivor_sed(act ? (unsigned)(32 * slot + owner) : 0u, rel), slot, owner);
            head += (unsigned)ndone;
            __syncwarp();
        };
        // one record per lane with survivors in this batch (ballot-compacted: no atomics, no loop).  The queue is
        // drained whenever 32 RECORDS are waiting - every record holds at least one survivor, so a drain always finds
        // its 32 survivors, retires at least one record, and the ring (< 32 waiting + <= 32 new) cannot overflow; the
        // trigger needs no reduction over the lanes (a REDUX per batch sat on the critical path before)
        auto push_records = [&](unsigned vote, unsigned pm, unsigned rel0) {
            if (pm) q[(tail + __popc(vote & lt)) & (kRing - 1)] = make_uint2(pm, ((unsigned)lane << 27) | rel0);
            tail += __popc(vote);
            __syncwarp();
            while (tail - head >= 32u) drain_records();
        };
        auto drain = [&]() {
            if constexpr (ENTRY) drain_entries();
            else drain_records();
        };

        unsigned mark = tail;  // ENTRY: queue position behind the last record of the previous tile
        for (int t = 0; t < ntiles; ++t) {
            const unsigned gti = gt + (unsigned)t;
            const int s = (int)(gti % STAGES);
            mbar_wait(&ws.full_bar[s], (gti / STAGES) & 1u);
            const long long first = begin + (long long)t * TILE;
            const int np = (int)((end - first < TILE) ? (end - first) : TILE);
            const P* tp = reinterpret_cast<const P*>(&ws.tile[s][0]);
            if constexpr (BOX) {
                const double4 bx = ws.box[s];
#pragma unroll
                for (int j = 0; j < HPT; ++j) tb[j] = tile_bound(e[j], bx, a.thr_pre, ws.kap[j][lane]);
            }
            for (int p = 0; p < np; p += G) {
                unsigned pm = 0;
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const P c = tp[p + g];
                    T d[HPT];
                    if constexpr (BOX) {
                        // hypothesis-innermost: consecutive FMAs share c.yb / c.xb / c.ya / c.xa
                        double t0[HPT], t1[HPT], t2[HPT];
#pragma unroll
                        for (int j = 0; j < HPT; ++j) {
                            t0[j] = fma(c.yb, e[j][3], e[j][6]);
                            t1[j] = fma(c.yb, e[j][4], e[j][7]);
                            t2[j] = fma(c.yb, e[j][5], e[j][8]);
                        }
#pragma unroll
                        for (int j = 0; j < HPT; ++j) {
                            t0[j] = fma(c.xb, e[j][0], t0[j]);  // lb0
                            t1[j] = fma(c.xb, e[j][1], t1[j]);  // lb1
                            t2[j] = fma(c.xb, e[j][2], t2[j]);  // lb2
                        }
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t2[j] = fma(c.ya, t1[j], t2[j]);
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t2[j] = fma(c.xa, t0[j], t2[j]);  // r
#pragma unroll
                        for (int j = 0; j < HPT; ++j) d[j] = fma(t2[j], t2[j], -tb[j]);
                    } else if (SCREEN) {
                        // hypothesis-innermost: consecutive FMAs share c.yb / c.xb / c.ya / c.xa
                        T t0[HPT], t1[HPT], t2[HPT];
#pragma unroll
                        for (int j = 0; j < HPT; ++j) {
                            t0[j] = fma(c.yb, e[j][3], e[j][6]);
                            t1[j] = fma(c.yb, e[j][4], e[j][7]);
                            t2[j] = fma(c.yb, e[j][5], e[j][8]);
                        }
#pragma unroll
                        for (int j = 0; j < HPT; ++j) {
                            t0[j] = fma(c.xb, e[j][0], t0[j]);  // s lb0 / |E|
                            t1[j] = fma(c.xb, e[j][1], t1[j]);  // s lb1 / |E|
                            t2[j] = fma(c.xb, e[j][2], t2[j]);  // lb2
                        }
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t2[j] = fma(c.ya, t1[j], t2[j]);
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t2[j] = fma(c.xa, t0[j], t2[j]);  // r
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t1[j] = fma(t1[j], t1[j], kap[j]);
#pragma unroll
                        for (int j = 0; j < HPT; ++j) t1[j] = fma(t0[j], t0[j], t1[j]);  // thr' nb + kappa
#pragma unroll
                        for (int j = 0; j < HPT; ++j) d[j] = fma(t2[j], t2[j], -t1[j]);
                    } else if constexpr (!SCREEN) {
#pragma unroll
                        for (int j = 0; j < HPT; ++j) d[j] = sed_full_decision(e[j], c.xa, c.ya, c.xb, c.yb, a.thr_pre);
                    }
#pragma unroll
                    for (int j = 0; j < HPT; ++j) pm = __funnelshift_l((unsigned)sign_word(d[j]), pm, 1);
                }
                pm |= fmask;
                const int v = np - p;  // a partial last batch evaluated stale records: drop their bits
                if (v < G) pm &= 0xffffffffu << (NB - v * HPT);
                const unsigned vote = __ballot_sync(full, pm != 0u);
                if (vote) {
                    if constexpr (ENTRY) push_entries(pm, (unsigned)(s * TILE + p));
                    else push_records(vote, pm, (unsigned)(first - begin) + (unsigned)p);
                }
            }
            if constexpr (ENTRY) {
                // the stage of tile t - 1 is refilled next: records that still point into it go first (never the case in
                // the survivor-rich regime - a tile leaves < 32 records behind and they are its own)
                while ((int)(mark - head) > 0) drain();
                mark = tail;
            }
            // every lane is done with the stage: refill it (ENTRY: the previous tile's) with the tile AHEAD tiles on
            __syncwarp();
            if (lane == 0 && t + AHEAD < ntiles) issue(t + AHEAD);
        }
        gt += (unsigned)ntiles;

        // tail of the queue, then publish this item's exact sums
        while (tail != head) drain();
#pragma unroll
        for (int j = 0; j < HPT; ++j) {
            const long long hyp = hyp_w + 32 * j + lane;
            const int col = ENTRY ? (lane ^ ((j & 1) << 4)) : lane;
            const unsigned cnt = ws.sacc[j][0][col];
            if (cnt) {  // only real hypotheses can have inliers
                unsigned long long* dst = a.acc + (long long)pair * a.h + hyp;
                atomicAdd(dst, (unsigned long long)cnt);
                ws.sacc[j][0][col] = 0;
#pragma unroll
                for (int k = 1; k < kAccWords; ++k) {
                    const unsigned v = ws.sacc[j][k][col];
                    if (v) {
                        atomicAdd(dst + (long long)k * a.htotal, (unsigned long long)v);
                        ws.sacc[j][k][col] = 0;
                    }
                }
            }
        }
        __syncwarp();
    }
}

template <int HPT, int G, int MODE>
__global__ void __launch_bounds__(kScoreThreads, score_min_blocks(MODE == MODE_SCREEN32 ? HPT / 2 : HPT))
k_score(const ScoreArgs a) {
    chain_enter();
    score_body<HPT, G, MODE>(a);
}

// AUTO variant: the pilot's verdict (k_pilot, or the one riding on k_screen_pts64) picks the body.  Both bodies live
// in one kernel; the register budget is the larger of the two.
template <int HPT, int G, int SMODE>
__global__ void __launch_bounds__(kScoreThreads, score_min_blocks(HPT)) k_score_auto(const ScoreArgs a, const ScoreArgs a_full) {
    chain_enter();
    if (*a.mode_flag == MODE_FULL) score_body<HPT, G, MODE_FULL>(a_full);
    else score_body<HPT, G, SMODE>(a);
}

// ------------------------------------------------------------------------------------
// K3 — finalise + select (lib/ransac/ransac.py:70-86, 96-108).
//
// Per hypothesis: combine the per-split partials in split order; apply the sample rule
// (ransac.py:63-64,76: the 8 sample points are excluded from the threshold count and
// included unconditionally in the error); n = 8 + count_extra; aggregate
// (SUM / SQUARE / MEAN / RMS); candidate iff valid and min_extra <= count_extra
// (ransac.py:75; min_extra may be fractional).  Then argmin of the error with the lowest
// index winning ties (ransac.py:83: strict <, earliest iteration kept).  mode 1 selects by
// maximum inlier count instead (lowest index on ties; non-default); mode 2 by the MSAC cost
// sum_i min(sed_i, thr) over ALL correspondences of the pair (non-default; err then holds that cost).
// ------------------------------------------------------------------------------------
enum { AGG_SUM = 0, AGG_SQUARE = 1, AGG_MEAN = 2, AGG_RMS = 3 };
enum { SELECT_MIN_ERROR = 0, SELECT_MAX_INLIERS = 1, SELECT_MSAC = 2 };

__device__ __forceinline__ bool better(const Best& x, const Best& y, int mode) {
    // is x better than y ?
    if (y.idx < 0) return x.idx >= 0;
    if (x.idx < 0) return false;
    if (mode == SELECT_MAX_INLIERS) {
        if (x.count != y.count) return x.count > y.count;
        return x.idx < y.idx;
    }
    if (x.err != y.err) return x.err < y.err;
    return x.idx < y.idx;
}

__device__ __forceinline__ Best shfl_best(const Best& b, int src_delta) {
    Best r;
    r.err = __shfl_down_sync(0xffffffffu, b.err, src_delta);
    r.idx = __shfl_down_sync(0xffffffffu, b.idx, src_delta);
    r.count = __shfl_down_sync(0xffffffffu, b.count, src_delta);
    r.pad = 0;
    return r;
}

__device__ __forceinline__ Best block_best(Best b, int mode, Best* sm /* 32 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const Best o = shfl_best(b, d);
        if (better(o, b, mode)) b = o;
    }
    if (lane == 0) sm[warp] = b;
    __syncthreads();
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        Best x;
        if (lane < nw) x = sm[lane];
        else { x.err = 0.0; x.idx = -1; x.count = 0; x.pad = 0; }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const Best o = shfl_best(x, d);
            if (better(o, x, mode)) x = o;
        }
        b = x;
    }
    return b;  // valid in thread 0
}

// ---- double-double helpers for the exact rescore (error-free transformations, Knuth two-sum) ----
struct dd { double hi, lo; };
__device__ __forceinline__ void dd_add(dd& s, double x) {
    const double t = __dadd_rn(s.hi, x);
    const double bb = __dsub_rn(t, s.hi);
    const double e = __dadd_rn(__dsub_rn(s.hi, __dsub_rn(t, bb)), __dsub_rn(x, bb));
    s.hi = t;
    s.lo = __dadd_rn(s.lo, e);
}
__device__ __forceinline__ void dd_merge(dd& s, const dd& o) {
    dd_add(s, o.hi);
    s.lo = __dadd_rn(s.lo, o.lo);
    const double t = __dadd_rn(s.hi, s.lo);  // renormalise
    s.lo = __dsub_rn(s.lo, __dsub_rn(t, s.hi));
    s.hi = t;
}

// exact 128-bit value of a fixed-point sum: sum_k plane[k] * 2^(21k)
__device__ __forceinline__ unsigned __int128 fixed_value(const unsigned long long* acc, long long stride) {
    unsigned __int128 v = 0;
#pragma unroll
    for (int k = kChunks - 1; k >= 0; --k) v = (v << kChunkBits) + acc[(long long)k * stride];
    return v;
}
__device__ __forceinline__ double u128_to_double(unsigned __int128 v) {
    const unsigned long long hi = (unsigned long long)(v >> 64), lo = (unsigned long long)v;
    return fma((double)hi, 18446744073709551616.0, (double)lo);
}

struct FinalArgs {
    const void* pts;       // ExactModel<KIND>::Rec records
    const long long* offsets;
    const double* E;       // [npairs][h][ExactModel<KIND>::kStride]
    const uint8_t* valid;
    const int32_t* table;  // may be null: no sample rule
    long long h;
    long long n;           // correspondences of the pair when offsets is null
    long long idx_offset;  // global index of hypothesis 0 (hypothesis-sharded runs)
    long long htotal;                 // npairs * h (stride of the accumulator planes)
    const unsigned long long* acc;    // [kAccWords][htotal] exact sums from K2
    double inv_scale1, inv_scale2;    // 2^(e-84), 2^(2e-84)
    int sums;                         // which sums K2 accumulated (the other one is reported as NaN)
    int force_rescore;                // K2 did not run (threshold outside the fixed-point range): rescore everything
    double thr, min_extra;
    int agg, mode;
    int32_t* count_extra;
    double* S1;
    double* S2;
    double* err;
    Best* block_out;
    long long* block_inv;  // [npairs][blocks][2]: invalid hypotheses in the block, smallest global index among them
    unsigned* tickets;     // [npairs], zero on entry, zero again on exit
    Best* out;             // [npairs]
    long long* invalid_out;  // [npairs][2]
    SelectRecord* record;    // [npairs]
    unsigned long long* rescored;  // [1] number of hypotheses that went through the exact rescore (diagnostic)
    unsigned* fitflag;             // K1's ambiguous-sample counter: reset here for the next fit (may be null)
    const double* K;               // MODEL_P: the camera of the new view [9]
};

// What K3 needs of a model kind: its record type, model stride, sample size and exact scorer (MODEL_P: sfm_pnp.cuh)
template <int KIND> struct ExactModel;
template <> struct ExactModel<MODEL_E> {
    using Rec = Corr;
    static constexpr int kSample = 8;
    static constexpr int kStride = 9;
    double e[9];
    __device__ __forceinline__ void load(const double* m, const double*) {
#pragma unroll
        for (int k = 0; k < 9; ++k) e[k] = m[k];
    }
    __device__ __forceinline__ bool eval(const Corr& c, double thr, double& v) const {
        v = sed_exact(e, c.xa, c.ya, c.xb, c.yb);
        return v <= thr;  // ransac.py:73
    }
};
template <> struct ExactModel<MODEL_H> {
    using Rec = Corr;
    static constexpr int kSample = 4;
    static constexpr int kStride = 9;
    double h[9], adj[9];
    __device__ __forceinline__ void load(const double* m, const double*) {
#pragma unroll
        for (int k = 0; k < 9; ++k) h[k] = m[k];
        homography_adj(h, adj);
    }
    __device__ __forceinline__ bool eval(const Corr& c, double thr, double& v) const {
        return transfer_exact(h, adj, c.xa, c.ya, c.xb, c.yb, thr, v);
    }
};

// the sample rule + aggregation + candidate test of one hypothesis (ransac.py:63-64, 70-76, 96-108), given the count and
// the sums over ALL correspondences with sed <= thr
template <int KIND>
__device__ __forceinline__ bool finalise_one(const FinalArgs& a, const typename ExactModel<KIND>::Rec* pts, long long i,
                                             long long npts, bool valid, long long cnt, double s1, double s2,
                                             double& err_out, long long& cnt_out, double& s1_out, double& s2_out) {
    constexpr int KS = ExactModel<KIND>::kSample;
    const double msac = __dadd_rn(s1, __dmul_rn(a.thr, (double)(npts - cnt)));  // K2 saw every correspondence
    if (a.table && valid) {
        ExactModel<KIND> m;
        m.load(a.E + ExactModel<KIND>::kStride * i, a.K);
        for (int k = 0; k < KS; ++k) {
            const typename ExactModel<KIND>::Rec c = pts[a.table[8 * i + k]];
            double sv;
            if (m.eval(c, a.thr, sv)) {
                cnt -= 1;  // was counted by K2, but samples are not "extra" inliers
            } else {
                s1 = __dadd_rn(s1, sv);  // not counted by K2, but always part of the error
                s2 = __dadd_rn(s2, __dmul_rn(sv, sv));
            }
        }
    }
    const double n = (double)((a.table ? KS : 0) + cnt);
    double err;
    switch (a.agg) {
        case AGG_SUM: err = s1; break;
        case AGG_SQUARE: err = s2; break;
        case AGG_MEAN: err = s1 / n; break;
        default: err = sqrt(s2 / n); break;
    }
    if (a.mode == SELECT_MSAC) err = msac;
    err_out = err; cnt_out = cnt; s1_out = s1; s2_out = s2;
    return valid && (a.min_extra <= (double)cnt) && (err == err);
}

// K3, one launch.  Thread per hypothesis: integer accumulators -> one rounding, sample rule, aggregation, candidate
// test.  A hypothesis whose fixed-point sum carries fewer than 53 significant bits per term (its inliers are more than
// 2^31 times tighter than the threshold - noise-free data, the reference's own RANSAC test) is RESCORED by the whole
// block: exact scorer over all correspondences, double-double sums in a fixed order (strided partials, fixed tree), so
// the result is still independent of scheduling, sharding and scoring variant.  Block arg-min, then the last block of
// the pair to finish (ticket) reduces the per-block results into the selection record.
template <int KIND>
__global__ void __launch_bounds__(256) k_finalise(const FinalArgs a) {
    chain_enter();
    __shared__ Best sm[32];
    __shared__ int s_list[256];
    __shared__ int s_nlist;
    __shared__ dd s_dd[2][8];
    __shared__ long long s_cnt[8];
    __shared__ long long s_first;
    __shared__ int s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long li = blockIdx.x * (long long)blockDim.x + tid;
    const long long i = (long long)blockIdx.y * a.h + li;  // blockIdx.y = image pair
    using Rec = typename ExactModel<KIND>::Rec;
    const Rec* pts = static_cast<const Rec*>(a.pts) + (a.offsets ? a.offsets[blockIdx.y] : 0);
    const long long npts = a.offsets ? a.offsets[blockIdx.y + 1] - a.offsets[blockIdx.y] : a.n;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    const double pinf = __longlong_as_double(0x7ff0000000000000LL);
    if (tid == 0) { s_nlist = 0; s_first = 0x7fffffffffffffffLL; }
    __syncthreads();
    Best b;
    b.err = 0.0; b.idx = -1; b.count = 0; b.pad = 0;
    if (li < a.h) {
        const bool valid = a.valid ? (a.valid[i] != 0) : true;
        const long long cnt = (long long)a.acc[i];
        const unsigned __int128 v1 = (a.sums & SUM_S1) ? fixed_value(a.acc + 1 * a.htotal + i, a.htotal) : 0;
        const unsigned __int128 v2 = (a.sums & SUM_S2) ? fixed_value(a.acc + (1 + kChunks) * a.htotal + i, a.htotal) : 0;
        // truncation loses < 1 unit per term: the sum is good to 2^-53 relative iff V >= cnt * 2^53
        const unsigned __int128 need = (unsigned __int128)(unsigned long long)cnt << 53;
        bool coarse = cnt > 0 && (((a.sums & SUM_S1) && v1 < need) || ((a.sums & SUM_S2) && v2 < need));
        // a 4-point fit reproduces its own samples to rounding level, so nearly every homography has a coarse sum (its
        // samples and little else): those that cannot be candidates (count_extra <= cnt < min_extra) are not rescored;
        // the same holds for a P3P pose and its 4 samples
        if constexpr (KIND != MODEL_E) coarse = coarse && !((double)cnt < a.min_extra);
        if (valid && (a.force_rescore || coarse)) {
            s_list[atomicAdd(&s_nlist, 1)] = tid;
        } else {
            const double s1 = (a.sums & SUM_S1) ? u128_to_double(v1) * a.inv_scale1 : qnan;
            const double s2 = (a.sums & SUM_S2) ? u128_to_double(v2) * a.inv_scale2 : qnan;
            double err, s1o, s2o;
            long long c2;
            const bool cand = finalise_one<KIND>(a, pts, i, npts, valid, cnt, s1, s2, err, c2, s1o, s2o);
            a.count_extra[i] = valid ? (int32_t)c2 : -1;
            a.S1[i] = s1o;
            a.S2[i] = s2o;
            a.err[i] = cand ? err : pinf;
            if (cand) { b.err = err; b.idx = a.idx_offset + li; b.count = (int)c2; }
        }
    }
    __syncthreads();
    // exact rescore of the listed hypotheses, one after the other, by all threads of the block
    const int nlist = s_nlist;
    for (int q = 0; q < nlist; ++q) {
        const int owner = s_list[q];
        const long long hi_ = (long long)blockIdx.y * a.h + blockIdx.x * (long long)blockDim.x + owner;
        ExactModel<KIND> m;
        m.load(a.E + ExactModel<KIND>::kStride * hi_, a.K);
        dd p1{0.0, 0.0}, p2{0.0, 0.0};
        long long pc = 0;
        for (long long j = tid; j < npts; j += 256) {
            const Rec c = pts[j];
            double sv;
            if (m.eval(c, a.thr, sv)) {
                pc += 1;
                dd_add(p1, sv);
                dd_add(p2, __dmul_rn(sv, sv));
            }
        }
        // fixed reduction tree: lanes (xor 16..1), then warps 0..7 in order
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            dd o1, o2;
            o1.hi = __shfl_xor_sync(0xffffffffu, p1.hi, d); o1.lo = __shfl_xor_sync(0xffffffffu, p1.lo, d);
            o2.hi = __shfl_xor_sync(0xffffffffu, p2.hi, d); o2.lo = __shfl_xor_sync(0xffffffffu, p2.lo, d);
            pc += __shfl_xor_sync(0xffffffffu, pc, d);
            // keep the merge symmetric so that both partners compute the same value: lower lane's partial first
            if (lane & d) { dd t1 = o1, t2 = o2; dd_merge(t1, p1); dd_merge(t2, p2); p1 = t1; p2 = t2; }
            else { dd_merge(p1, o1); dd_merge(p2, o2); }
        }
        if (lane == 0) { s_dd[0][warp] = p1; s_dd[1][warp] = p2; s_cnt[warp] = pc; }
        __syncthreads();
        if (tid == owner) {
            dd t1 = s_dd[0][0], t2 = s_dd[1][0];
            long long c = s_cnt[0];
            for (int w = 1; w < 8; ++w) { dd_merge(t1, s_dd[0][w]); dd_merge(t2, s_dd[1][w]); c += s_cnt[w]; }
            double err, s1o, s2o;
            long long c2;
            const bool cand = finalise_one<KIND>(a, pts, hi_, npts, true, c, (a.sums & SUM_S1) ? t1.hi : qnan,
                                           (a.sums & SUM_S2) ? t2.hi : qnan, err, c2, s1o, s2o);
            a.count_extra[hi_] = (int32_t)c2;
            a.S1[hi_] = s1o;
            a.S2[hi_] = s2o;
            a.err[hi_] = cand ? err : pinf;
            if (cand) { b.err = err; b.idx = a.idx_offset + (hi_ - (long long)blockIdx.y * a.h); b.count = (int)c2; }
        }
        __syncthreads();
    }
    if (tid == 0 && nlist) atomicAdd(a.rescored, (unsigned long long)nlist);
    // invalid hypotheses of this block (ransac.py:65 has no try/except: one degenerate sample aborts the reference run,
    // so the host needs their number and the earliest one)
    const bool inv = (li < a.h) && a.valid && (a.valid[i] == 0);
    const int ninv = __syncthreads_count(inv);
    if (inv) atomicMin(&s_first, a.idx_offset + li);
    b = block_best(b, a.mode, sm);
    __syncthreads();
    const int nblocks = gridDim.x;
    if (tid == 0) {
        const long long blk = (long long)blockIdx.y * nblocks + blockIdx.x;
        a.block_out[blk] = b;
        a.block_inv[2 * blk] = ninv;
        a.block_inv[2 * blk + 1] = s_first;
        __threadfence();
        s_last = (atomicAdd(&a.tickets[blockIdx.y], 1u) == (unsigned)(nblocks - 1)) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    // ---- last block of the pair: reduce the per-block results into the selection record ----
    __threadfence();
    __shared__ long long s_ninv, s_first2;
    if (tid == 0) {
        s_ninv = 0; s_first2 = 0x7fffffffffffffffLL; a.tickets[blockIdx.y] = 0;
        if (a.fitflag && blockIdx.y == 0) *a.fitflag = 0u;
    }
    __syncthreads();
    const volatile Best* blocks = a.block_out + (long long)blockIdx.y * nblocks;
    const volatile long long* binv = a.block_inv + 2 * (long long)blockIdx.y * nblocks;
    Best g;
    g.err = 0.0; g.idx = -1; g.count = 0; g.pad = 0;
    long long tn = 0, tf = 0x7fffffffffffffffLL;
    for (int k = tid; k < nblocks; k += 256) {
        Best o;
        o.err = blocks[k].err; o.idx = blocks[k].idx; o.count = blocks[k].count; o.pad = 0;
        if (better(o, g, a.mode)) g = o;
        tn += binv[2 * k];
        const long long f = binv[2 * k + 1];
        if (f < tf) tf = f;
    }
    if (tn) {
        atomicAdd((unsigned long long*)&s_ninv, (unsigned long long)tn);
        atomicMin(&s_first2, tf);
    }
    g = block_best(g, a.mode, sm);
    __syncthreads();
    if (tid == 0) {
        a.out[blockIdx.y] = g;
        a.invalid_out[2 * blockIdx.y] = s_ninv;
        a.invalid_out[2 * blockIdx.y + 1] = s_ninv ? s_first2 : -1;
        // everything the host wants about this pair in one record (one D2H copy, one synchronisation)
        SelectRecord& r = a.record[blockIdx.y];
        r.best = g;
        r.num_invalid = s_ninv;
        r.first_invalid = s_ninv ? s_first2 : -1;
        const long long w = (long long)blockIdx.y * a.h + (g.idx >= 0 ? g.idx - a.idx_offset : 0);
        // a pose does not fit E[9]: its winner is read from the models by the index (k_pnp_mask), E reads zero
        for (int k = 0; k < 9; ++k) r.E[k] = (KIND != MODEL_P && g.idx >= 0) ? a.E[ExactModel<KIND>::kStride * w + k] : 0.0;
        for (int k = 0; k < 8; ++k)
            r.sample[k] = (a.table && g.idx >= 0 && k < ExactModel<KIND>::kSample) ? a.table[8 * w + k] : -1;
    }
}

// SURVEY.md H1: candidates whose error is within rel_tol of the winner's (ransac.py:83 compares errors that were
// summed in list order; the host re-evaluates near-ties in that order).  Appends up to cap local indices, unordered.
__global__ void __launch_bounds__(256) k_near_ties(const double* __restrict__ err, long long h, const SelectRecord* __restrict__ rec,
                                                   double rel_tol, int cap, long long* __restrict__ out, unsigned* __restrict__ count) {
    const double best = rec->best.err;
    if (rec->best.idx < 0) return;
    const double lim = best + fabs(best) * rel_tol;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < h; i += (long long)gridDim.x * blockDim.x) {
        if (err[i] <= lim) {
            const unsigned pos = atomicAdd(count, 1u);
            if (pos < (unsigned)cap) out[pos] = i;
        }
    }
}

// Hypothesis-sharded runs (SURVEY.md 8(e)): every rank's SelectRecord, gathered by one NCCL all-gather, is merged on
// the device with the reference's rule (smallest error, earliest GLOBAL iteration on ties, ransac.py:83; or the
// non-default modes) so that the tail can be enqueued without a host round trip.  One thread.
//   merged      : winner with its global index (idx = owner * hyps_per_rank + local idx), its model and sample row,
//                 this rank's invalid counters
//   winner_E    : the winning model (the tail reads it from here whichever rank fitted it)
//   local_best  : Best whose idx is this rank's local index if it owns the winner, else -1 (sample-row lookups)
__global__ void k_merge_records(const SelectRecord* __restrict__ gathered, int world, int rank, long long hyps_per_rank,
                                int mode, SelectRecord* __restrict__ merged, int* __restrict__ owner_out,
                                double* __restrict__ winner_E, Best* __restrict__ local_best) {
    if (threadIdx.x || blockIdx.x) return;
    Best b;
    b.err = 0.0; b.idx = -1; b.count = 0; b.pad = 0;
    int owner = -1;
    for (int r = 0; r < world; ++r) {
        Best o = gathered[r].best;
        if (o.idx >= 0) o.idx += (long long)r * hyps_per_rank;
        if (better(o, b, mode)) { b = o; owner = r; }
    }
    merged->best = b;
    merged->num_invalid = gathered[rank].num_invalid;
    merged->first_invalid = gathered[rank].first_invalid;
    for (int k = 0; k < 9; ++k) {
        const double v = owner >= 0 ? gathered[owner].E[k] : 0.0;
        merged->E[k] = v;
        winner_E[k] = v;
    }
    // the winner's sample row travels with the record: every rank forces the same 8 points into the inlier set
    // (ransac.py:76) and applies the same index-0 quirk of the vote (eight_point.py:228-230)
    for (int k = 0; k < 8; ++k) merged->sample[k] = owner >= 0 ? gathered[owner].sample[k] : -1;
    *owner_out = owner;
    Best lb = b;
    lb.idx = (owner == rank) ? gathered[rank].best.idx : -1;
    *local_best = lb;
}

// ------------------------------------------------------------------------------------
// K4 — inlier mask + SED values of one hypothesis over all correspondences (the winner):
// the same exact scorer, one thread per correspondence.
// ------------------------------------------------------------------------------------
__global__ void k_inlier_mask(const Corr* __restrict__ pts, long long n, const double* __restrict__ E,
                              const Best* __restrict__ best, long long idx_offset, long long hyp,
                              double thr, uint8_t* __restrict__ mask, double* __restrict__ sed) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long local = hyp;
    if (best) local = best->idx - idx_offset;  // take the winner straight from K3's output
    if (local < 0) {
        mask[i] = 0;
        sed[i] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    double e[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) e[k] = E[9 * local + k];
    const Corr c = pts[i];
    const double sv = sed_exact(e, c.xa, c.ya, c.xb, c.yb);
    sed[i] = sv;
    mask[i] = (sv <= thr) ? 1 : 0;
}

}  // namespace sfm
