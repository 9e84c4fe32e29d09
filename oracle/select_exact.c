/* TEST INFRASTRUCTURE ONLY — plain-C restatement of the essential-matrix / homography model scores.
 *
 * The reference has no model selection; this file pins the evaluation order of k_score_models
 * (structure_from_motion_b200/csrc/sfm_select.cuh, with transfer_terms and homography_adj of sfm_device.cuh) so that
 * its per-correspondence errors, fixed-point sums, counts, ratio and choice can be checked bit for bit.  Compile with
 * -ffp-contract=off so that only the explicit fma() calls fuse (oracle/cselect.py does).
 *
 * Never linked into, or called by, the product library.
 */
#include <math.h>
#include <stdint.h>

#define GAMMA 5.99
#define T_E 3.84
#define T_H 5.99
#define FIXED 4294967296.0 /* 2^32 */

/* adj(m), row-major: homography_adj's nine fma's */
static void adj3(const double *h, double *a) {
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

/* F = K^-T E K^-1 with K^-1 = adj(K) / det(K) */
void oracle_fundamental(const double *E, const double *K, double *F) {
    double adj[9], ki[9], m[9];
    adj3(K, adj);
    const double det = fma(K[0], adj[0], fma(K[1], adj[3], K[2] * adj[6]));
    for (int i = 0; i < 9; ++i) ki[i] = adj[i] / det;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            m[3 * i + j] = fma(E[3 * i + 2], ki[6 + j], fma(E[3 * i + 1], ki[3 + j], E[3 * i] * ki[j]));
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            F[3 * i + j] = fma(ki[6 + i], m[6 + j], fma(ki[3 + i], m[3 + j], ki[i] * m[j]));
}

static uint64_t rho(double d2, double s2, double T, int *pass) {
    const double x = d2 / s2;
    *pass = x < T;
    return *pass ? (uint64_t)rint((GAMMA - x) * FIXED) : 0;
}

/* E and H may be NULL (not both).  pp[n][4] = (d2_A,E, d2_B,E, d2_A,H, d2_B,H) or NULL.
 * fixed[2] = (E, H) sums, count[2], scores[3] = (score_e, score_h, ratio_h); returns the model (0 = E, 1 = H). */
int oracle_score_models(const double *E, const double *H, const double *K, const double *xa, const double *ya,
                        const double *xb, const double *yb, int64_t n, double sigma, double ratio, double *pp,
                        uint64_t *fixed, int64_t *count, double *scores) {
    double f[9] = {0}, h[9] = {0}, a[9];
    if (E) oracle_fundamental(E, K, f);
    if (H)
        for (int i = 0; i < 9; ++i) h[i] = H[i];
    adj3(h, a);
    const double s2 = sigma * sigma;
    uint64_t se = 0, sh = 0;
    int64_t ce = 0, ch = 0;
    for (int64_t i = 0; i < n; ++i) {
        double dae = NAN, dbe = NAN, dah = NAN, dbh = NAN;
        int pa, pb;
        if (E) {
            const double la0 = fma(f[0], xa[i], fma(f[1], ya[i], f[2]));
            const double la1 = fma(f[3], xa[i], fma(f[4], ya[i], f[5]));
            const double la2 = fma(f[6], xa[i], fma(f[7], ya[i], f[8]));
            const double lb0 = fma(f[0], xb[i], fma(f[3], yb[i], f[6]));
            const double lb1 = fma(f[1], xb[i], fma(f[4], yb[i], f[7]));
            const double r = fma(xb[i], la0, fma(yb[i], la1, la2));
            const double r2 = r * r;
            dbe = r2 / fma(la0, la0, la1 * la1);
            dae = r2 / fma(lb0, lb0, lb1 * lb1);
            se += rho(dae, s2, T_E, &pa);
            se += rho(dbe, s2, T_E, &pb);
            ce += pa && pb;
        }
        if (H) { /* transfer_terms: p = H a, q = adj(H) b */
            const double p0 = fma(h[0], xa[i], fma(h[1], ya[i], h[2]));
            const double p1 = fma(h[3], xa[i], fma(h[4], ya[i], h[5]));
            const double p2 = fma(h[6], xa[i], fma(h[7], ya[i], h[8]));
            const double q0 = fma(a[0], xb[i], fma(a[1], yb[i], a[2]));
            const double q1 = fma(a[3], xb[i], fma(a[4], yb[i], a[5]));
            const double q2 = fma(a[6], xb[i], fma(a[7], yb[i], a[8]));
            const double u = fma(-xb[i], p2, p0), v = fma(-yb[i], p2, p1);
            const double s = fma(-xa[i], q2, q0), t = fma(-ya[i], q2, q1);
            const double F = fma(u, u, v * v), G = fma(s, s, t * t);
            dbh = F / (p2 * p2);
            dah = G / (q2 * q2);
            sh += rho(dah, s2, T_H, &pa);
            sh += rho(dbh, s2, T_H, &pb);
            ch += pa && pb;
        }
        if (pp) {
            pp[4 * i] = dae;
            pp[4 * i + 1] = dbe;
            pp[4 * i + 2] = dah;
            pp[4 * i + 3] = dbh;
        }
    }
    fixed[0] = se;
    fixed[1] = sh;
    count[0] = ce;
    count[1] = ch;
    const double score_e = (double)se * (1.0 / FIXED), score_h = (double)sh * (1.0 / FIXED);
    const double tot = score_h + score_e;
    scores[0] = score_e;
    scores[1] = score_h;
    scores[2] = tot > 0.0 ? score_h / tot : 0.0;
    return !E ? 1 : (!H ? 0 : scores[2] > ratio);
}
