/* TEST INFRASTRUCTURE ONLY — plain-C restatement of the PnP reprojection scorer (csrc/sfm_pnp.cuh).
 *
 * P = K [R | t] and p = P (X, Y, Z, 1), the differences, F = d0^2 + d1^2, W = p2^2, the decision
 * p2 >= 2^-537 && F < inf && F <= thr W and the value F / W, each one IEEE operation or one fma() in the device's pinned order.
 * Compiled with -ffp-contract=off so that no product and sum are fused behind our back: decisions and values are
 * bit-identical to the kernels (k_score_pnp, k_finalise<MODEL_P>, k_pnp_mask). */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>

void oracle_pnp_projection(const double *K, const double *m, double *P) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c)
            P[4 * r + c] = fma(K[3 * r + 0], m[c], fma(K[3 * r + 1], m[4 + c], K[3 * r + 2] * m[8 + c]));
}

static inline int reproj_eval(const double *P, double X, double Y, double Z, double u, double v, double thr,
                              double *value) {
    const double p0 = fma(P[0], X, fma(P[1], Y, fma(P[2], Z, P[3])));
    const double p1 = fma(P[4], X, fma(P[5], Y, fma(P[6], Z, P[7])));
    const double p2 = fma(P[8], X, fma(P[9], Y, fma(P[10], Z, P[11])));
    const double d0 = fma(-u, p2, p0), d1 = fma(-v, p2, p1);
    const double F = fma(d0, d0, d1 * d1);
    const double W = p2 * p2;
    *value = F / W;
    return p2 >= 0x1p-537 && F < INFINITY && F <= thr * W;
}

/* decision and value of every record under one [R | t] (row-major 3 x 4) */
void oracle_reproj_exact_many(const double *Rt, const double *K, const double *X, const double *Y, const double *Z,
                              const double *u, const double *v, int64_t n, double thr, uint8_t *mask, double *val) {
    double P[12];
    oracle_pnp_projection(K, Rt, P);
    for (int64_t i = 0; i < n; ++i) mask[i] = (uint8_t)reproj_eval(P, X[i], Y[i], Z[i], u[i], v[i], thr, &val[i]);
}

typedef struct {
    const double *Rt, *K, *X, *Y, *Z, *u, *v;
    const uint8_t *valid;
    const int32_t *table;
    int64_t n, h0, h1;
    double thr;
    int32_t *cnt;
    double *s1, *s2;
} Job;

static void *run(void *p) {
    const Job *j = (const Job *)p;
    for (int64_t k = j->h0; k < j->h1; ++k) {
        if (j->valid && !j->valid[k]) { j->cnt[k] = -1; j->s1[k] = j->s2[k] = NAN; continue; }
        double P[12];
        oracle_pnp_projection(j->K, j->Rt + 12 * k, P);
        int64_t c = 0;
        double a = 0.0, b = 0.0;
        for (int64_t i = 0; i < j->n; ++i) {
            double val;
            int is_sample = 0;
            if (j->table)
                for (int s = 0; s < 4; ++s) is_sample |= (j->table[8 * k + s] == i);
            const int in = reproj_eval(P, j->X[i], j->Y[i], j->Z[i], j->u[i], j->v[i], j->thr, &val);
            if (in && !is_sample) c += 1;
            if (in || is_sample) { a += val; b += val * val; }
        }
        j->cnt[k] = (int32_t)c;
        j->s1[k] = a;
        j->s2[k] = b;
    }
    return NULL;
}

/* (count_extra, S1, S2) per pose: the 4 samples (table columns 0-3, if a table is given) are never counted and always
 * summed; an invalid pose (valid[k] == 0) reports -1 and NaN. */
void oracle_reproj_score_batch(const double *Rt, const uint8_t *valid, const double *K, const double *X, const double *Y,
                               const double *Z, const double *u, const double *v, int64_t n, int64_t h,
                               const int32_t *table, double thr, int32_t *cnt, double *s1, double *s2, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    pthread_t th[64];
    Job jobs[64];
    if (nthreads > 64) nthreads = 64;
    for (int t = 0; t < nthreads; ++t) {
        Job j = {Rt, K, X, Y, Z, u, v, valid, table, n, h * t / nthreads, h * (t + 1) / nthreads, thr, cnt, s1, s2};
        jobs[t] = j;
        pthread_create(&th[t], NULL, run, &jobs[t]);
    }
    for (int t = 0; t < nthreads; ++t) pthread_join(th[t], NULL);
}
