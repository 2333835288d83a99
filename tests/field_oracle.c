/* field_oracle.c — fp64 reference for b200nb_field and b200nb_potential.  TEST INFRASTRUCTURE ONLY.
 *
 * Kept beside the tests rather than in oracle/, whose restatement of the reference is pinned against golden vectors;
 * the field has no reference counterpart.  Same conventions as oracle_accel_f64: float inputs, G = (double)G_f32,
 * soft^2 = (double)soft * soft, OpenMP over targets.
 * Build: gcc -O2 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target field_oracle). */
#include <math.h>
#include <stdint.h>

/* a(p) = sum_j G m_j (q_j - p) / (|q_j - p|^2 + soft^2)^(3/2) and phi(p) = -sum_j G m_j / (|q_j - p|^2 + soft^2)^(1/2)
 * over ALL bodies, at n_pts points.  amag (may be NULL) = sum_j |a_ij|: the cancellation-free scale of the acceleration
 * error bound. */
void oracle_field_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, float G, float soft,
                      uint64_t n_pts, const float *px, const float *py, const float *pz, double *ax, double *ay,
                      double *az, double *phi, double *amag)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t t = 0; t < (int64_t)n_pts; t++) {
        const double x = px[t], y = py[t], z = pz[t];
        double sx = 0.0, sy = 0.0, sz = 0.0, sp = 0.0, sm = 0.0;
        for (uint64_t j = 0; j < n; j++) {
            const double rx = (double)qx[j] - x, ry = (double)qy[j] - y, rz = (double)qz[j] - z;
            const double r2 = rx * rx + ry * ry + rz * rz;
            const double d = r2 + s2;
            const double gi = Gd * (double)m[j] / sqrt(d);
            const double f = gi / d;
            sx += f * rx;
            sy += f * ry;
            sz += f * rz;
            sp += gi;
            sm += f * sqrt(r2);
        }
        ax[t] = sx; ay[t] = sy; az[t] = sz; phi[t] = -sp;
        if (amag) amag[t] = sm;
    }
}

/* phi_i = -sum_{j != i} G m_j / (|r_ij|^2 + soft^2)^(1/2) for bodies idx[0..n_idx) (idx == NULL: 0..n_idx-1); the self
 * pair is excluded by index, so coincident bodies still see each other. */
void oracle_potential_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, float G,
                          float soft, const uint64_t *idx, uint64_t n_idx, double *phi)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(static)
    for (int64_t t = 0; t < (int64_t)n_idx; t++) {
        const uint64_t i = idx ? idx[t] : (uint64_t)t;
        const double x = qx[i], y = qy[i], z = qz[i];
        double sp = 0.0;
        for (uint64_t j = 0; j < n; j++) {
            if (j == i) continue;
            const double rx = (double)qx[j] - x, ry = (double)qy[j] - y, rz = (double)qz[j] - z;
            sp += Gd * (double)m[j] / sqrt(rx * rx + ry * ry + rz * rz + s2);
        }
        phi[t] = -sp;
    }
}
