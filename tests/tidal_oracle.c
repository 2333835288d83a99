/* tidal_oracle.c — fp64 reference for b200nb_tidal and b200nb_tidal_bodies.  TEST INFRASTRUCTURE ONLY.
 *
 * Same conventions as tests/field_oracle.c: float inputs, G = (double)G_f32, soft^2 = (double)soft * soft, OpenMP over
 * targets.  Rows of six in the library's order xx, yy, zz, xy, xz, yz.
 * Build: gcc -O2 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target tidal_oracle). */
#include <math.h>
#include <stdint.h>

static const int IA[6] = {0, 1, 2, 0, 0, 1}, IB[6] = {0, 1, 2, 1, 2, 2};

/* T_ab(p) = sum_{j != skip} G m_j [3 d_a d_b / s^5 - delta_ab / s^3], d = q_j - p, s^2 = |d|^2 + soft^2, into t[6];
 * amag[6] (may be NULL) = sum_j G m_j (3 |d_a d_b| / s^5 + delta_ab / s^3), the cancellation-free scale of each entry;
 * s5[0] (may be NULL) = sum_j G m_j / s^5, the sum of the trace identity tr T = -3 soft^2 sum_j G m_j / s^5. */
static void tidal_at(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, double Gd, double s2,
                     double x, double y, double z, uint64_t skip, double *t, double *amag, double *s5)
{
    double st[6] = {0, 0, 0, 0, 0, 0}, sa[6] = {0, 0, 0, 0, 0, 0}, sum5 = 0.0;
    for (uint64_t j = 0; j < n; j++) {
        if (j == skip) continue;
        const double d[3] = {(double)qx[j] - x, (double)qy[j] - y, (double)qz[j] - z};
        const double r2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + s2;
        const double inv = 1.0 / sqrt(r2);
        const double g3 = Gd * (double)m[j] * inv * inv * inv, g5 = g3 * inv * inv;
        for (int q = 0; q < 6; q++) {
            const double dd = d[IA[q]] * d[IB[q]], diag = q < 3 ? g3 : 0.0;
            st[q] += 3.0 * g5 * dd - diag;
            sa[q] += 3.0 * g5 * fabs(dd) + diag;
        }
        sum5 += g5;
    }
    for (int q = 0; q < 6; q++) {
        t[q] = st[q];
        if (amag) amag[q] = sa[q];
    }
    if (s5) *s5 = sum5;
}

/* over ALL bodies at n_pts points; t, amag: [n_pts][6]; s5: [n_pts]; amag and s5 may be NULL */
void oracle_tidal_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, float G, float soft,
                      uint64_t n_pts, const float *px, const float *py, const float *pz, double *t, double *amag,
                      double *s5)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < (int64_t)n_pts; i++)
        tidal_at(n, qx, qy, qz, m, Gd, s2, px[i], py[i], pz[i], UINT64_MAX, t + 6 * i, amag ? amag + 6 * i : 0,
                 s5 ? s5 + i : 0);
}

/* per body, self pair excluded by index (coincident bodies still see each other), for bodies idx[0..n_idx)
 * (idx == NULL: 0..n_idx-1) */
void oracle_tidal_bodies_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, float G,
                             float soft, const uint64_t *idx, uint64_t n_idx, double *t, double *amag, double *s5)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t k = 0; k < (int64_t)n_idx; k++) {
        const uint64_t i = idx ? idx[k] : (uint64_t)k;
        tidal_at(n, qx, qy, qz, m, Gd, s2, qx[i], qy[i], qz[i], i, t + 6 * k, amag ? amag + 6 * k : 0, s5 ? s5 + k : 0);
    }
}
