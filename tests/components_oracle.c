/* components_oracle.c — fp64 reference for b200nb_component_field and b200nb_component_field_bodies.  TEST
 * INFRASTRUCTURE ONLY.
 *
 * Same conventions as tests/field_oracle.c: float inputs, G = (double)G_f32, soft^2 = (double)soft * soft, OpenMP over
 * targets.  A body with comp[j] >= n_comp (B200NB_NO_GROUP) is a source of nothing.
 * Build: gcc -O2 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target components_oracle). */
#include <math.h>
#include <stdint.h>

/* acc[C][3], phi[C], amag[C] at (x, y, z) over j != skip: the field of each component and sum_{j in h} |a_ij| */
static void components_at(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, const uint32_t *comp,
                          uint32_t C, double Gd, double s2, double x, double y, double z, uint64_t skip, double *acc,
                          double *phi, double *amag)
{
    for (uint32_t h = 0; h < C; h++) {
        acc[3 * h] = acc[3 * h + 1] = acc[3 * h + 2] = 0.0;
        phi[h] = 0.0;
        amag[h] = 0.0;
    }
    for (uint64_t j = 0; j < n; j++) {
        const uint32_t h = comp[j];
        if (j == skip || h >= C) continue;
        const double rx = (double)qx[j] - x, ry = (double)qy[j] - y, rz = (double)qz[j] - z;
        const double r2 = rx * rx + ry * ry + rz * rz;
        const double d = r2 + s2;
        const double gi = Gd * (double)m[j] / sqrt(d);
        const double f = gi / d;
        acc[3 * h] += f * rx;
        acc[3 * h + 1] += f * ry;
        acc[3 * h + 2] += f * rz;
        phi[h] -= gi;
        amag[h] += f * sqrt(r2);
    }
}

/* at n_pts points: acc [n_pts][C][3], phi and amag [n_pts][C] */
void oracle_components_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, const uint32_t *comp,
                           uint32_t C, float G, float soft, uint64_t n_pts, const float *px, const float *py, const float *pz,
                           double *acc, double *phi, double *amag)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t t = 0; t < (int64_t)n_pts; t++)
        components_at(n, qx, qy, qz, m, comp, C, Gd, s2, px[t], py[t], pz[t], UINT64_MAX, acc + 3 * C * t, phi + C * t,
                      amag + C * t);
}

/* per body, self pair excluded by index (coincident bodies still see each other), for bodies idx[0..n_idx) (idx == NULL:
 * 0..n_idx-1) */
void oracle_components_bodies_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m,
                                  const uint32_t *comp, uint32_t C, float G, float soft, const uint64_t *idx, uint64_t n_idx,
                                  double *acc, double *phi, double *amag)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t t = 0; t < (int64_t)n_idx; t++) {
        const uint64_t i = idx ? idx[t] : (uint64_t)t;
        components_at(n, qx, qy, qz, m, comp, C, Gd, s2, qx[i], qy[i], qz[i], i, acc + 3 * C * t, phi + C * t, amag + C * t);
    }
}
