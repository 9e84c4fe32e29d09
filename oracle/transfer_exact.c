/* TEST INFRASTRUCTURE ONLY — plain-C restatement of the homography transfer error.
 *
 * The reference has no homography model; this file pins the evaluation order of the device kernels
 * (structure_from_motion_b200/csrc/sfm_homography.cuh, sfm_device.cuh) so that their decisions, values, counts and
 * sums can be checked bit for bit.  Compile with -ffp-contract=off so that only the explicit fma() calls fuse
 * (oracle/ctransfer.py does).
 *
 * Never linked into, or called by, the product library.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>

/* H is row-major and maps image-A points to image-B points; adj(H) maps back without a division (the error is
 * invariant to the scale of either matrix).  With p = H (xa, ya, 1) and q = adj(H) (xb, yb, 1):
 *   F = (p0 - xb p2)^2 + (p1 - yb p2)^2,   G = (q0 - xa q2)^2 + (q1 - ya q2)^2,   P = p2^2,  Q = q2^2
 *   inlier  <=>  p2 != 0 && q2 != 0 && F Q + G P <= (thr P) Q      (division-free)
 *   value    =  F / P + G / Q                                         (the symmetric transfer error in px^2)
 * Every operation below is one IEEE operation or one explicit fma(); compiled with -ffp-contract=off this is
 * bit-identical to the device kernels. */
void oracle_homography_adj(const double *h, double *a) {
    a[0] = fma(h[4], h[8], -(h[5] * h[7]));
    a[1] = fma(h[2], h[7], -(h[1] * h[8]));
    a[2] = fma(h[1], h[5], -(h[2] * h[4]));
    a[3] = fma(h[5], h[6], -(h[3] * h[8]));
    a[4] = fma(h[0], h[8], -(h[2] * h[6]));
    a[5] = fma(h[2], h[3], -(h[0] * h[5]));
    a[6] = fma(h[3], h[7], -(h[4] * h[6]));
    a[7] = fma(h[1], h[6], -(h[0] * h[7]));
    a[8] = fma(h[0], h[4], -(h[1] * h[3]));
}

int oracle_transfer_exact(const double *h, const double *a, double xa, double ya, double xb, double yb,
                          double thr, double *value) {
    const double p0 = fma(h[0], xa, fma(h[1], ya, h[2]));
    const double p1 = fma(h[3], xa, fma(h[4], ya, h[5]));
    const double p2 = fma(h[6], xa, fma(h[7], ya, h[8]));
    const double q0 = fma(a[0], xb, fma(a[1], yb, a[2]));
    const double q1 = fma(a[3], xb, fma(a[4], yb, a[5]));
    const double q2 = fma(a[6], xb, fma(a[7], yb, a[8]));
    const double u = fma(-xb, p2, p0), v = fma(-yb, p2, p1);
    const double s = fma(-xa, q2, q0), t = fma(-ya, q2, q1);
    const double F = fma(u, u, v * v), G = fma(s, s, t * t);
    const double P = p2 * p2, Q = q2 * q2;
    *value = F / P + G / Q;
    return p2 != 0.0 && q2 != 0.0 && fma(F, Q, G * P) <= (thr * P) * Q;
}

/* decision and value of every correspondence under one H (pixel coordinates) */
void oracle_transfer_exact_many(const double *h, const double *xa, const double *ya, const double *xb,
                                const double *yb, int64_t n, double thr, uint8_t *mask, double *value) {
    double a[9];
    oracle_homography_adj(h, a);
    for (int64_t i = 0; i < n; ++i)
        mask[i] = (uint8_t)oracle_transfer_exact(h, a, xa[i], ya[i], xb[i], yb[i], thr, &value[i]);
}

typedef struct {
    const double *H, *xa, *ya, *xb, *yb;
    const int32_t *table; /* [h][8]: the first 4 columns are the sample */
    const uint8_t *valid;
    int64_t n, h0, h1;
    double thr;
    int32_t *count_extra;
    double *s1, *s2;
} hjob_t;

static void *hworker(void *p) {
    hjob_t *j = (hjob_t *)p;
    for (int64_t h = j->h0; h < j->h1; ++h) {
        if (j->valid && !j->valid[h]) {
            j->count_extra[h] = -1;
            j->s1[h] = j->s2[h] = 0.0;
            continue;
        }
        const double *hm = j->H + 9 * h;
        double a[9], v;
        oracle_homography_adj(hm, a);
        int64_t cnt = 0;
        double s1 = 0.0, s2 = 0.0;
        for (int64_t i = 0; i < j->n; ++i) {
            if (oracle_transfer_exact(hm, a, j->xa[i], j->ya[i], j->xb[i], j->yb[i], j->thr, &v)) {
                ++cnt;
                s1 += v;
                s2 += v * v;
            }
        }
        if (j->table) { /* the 4 samples: never counted, always in the error */
            for (int k = 0; k < 4; ++k) {
                int64_t i = j->table[8 * h + k];
                if (oracle_transfer_exact(hm, a, j->xa[i], j->ya[i], j->xb[i], j->yb[i], j->thr, &v)) {
                    --cnt;
                } else {
                    s1 += v;
                    s2 += v * v;
                }
            }
        }
        j->count_extra[h] = (int32_t)cnt;
        j->s1[h] = s1;
        j->s2[h] = s2;
    }
    return 0;
}

/* oracle_score_batch for homographies: count_extra[h] = #{i not in sample_h : inlier}; s1/s2 = sums of the value /
 * value^2 over the 4 samples and the extra inliers.  valid and table may be NULL. */
void oracle_transfer_score_batch(const double *H, const uint8_t *valid, const double *xa, const double *ya,
                                 const double *xb, const double *yb, int64_t n, int64_t h, const int32_t *table,
                                 double thr, int32_t *count_extra, double *s1, double *s2, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    pthread_t th[256];
    hjob_t jobs[256];
    int64_t per = (h + nthreads - 1) / nthreads;
    int used = 0;
    for (int t = 0; t < nthreads; ++t) {
        int64_t h0 = t * per, h1 = h0 + per > h ? h : h0 + per;
        if (h0 >= h1) break;
        jobs[t] = (hjob_t){H, xa, ya, xb, yb, table, valid, n, h0, h1, thr, count_extra, s1, s2};
        pthread_create(&th[t], 0, hworker, &jobs[t]);
        ++used;
    }
    for (int t = 0; t < used; ++t) pthread_join(th[t], 0);
}
