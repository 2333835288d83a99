/* groups_oracle.c — fp64 reference for b200nb_group_potential and b200nb_unbind.  TEST INFRASTRUCTURE ONLY.
 *
 * Same conventions as field_oracle.c: float inputs, G = (double)G_f32, soft^2 = (double)soft * soft, OpenMP over
 * targets.  Labels are uint32; 0xFFFFFFFF (NO_GROUP) takes no part.
 * Build: gcc -O2 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target groups_oracle). */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NO_GROUP 0xFFFFFFFFu

/* phi_i = -sum_{j != i, group[j] = group[i]} G m_j / (|r_ij|^2 + soft^2)^(1/2) for bodies idx[0..n_idx), 0 for NO_GROUP */
void oracle_group_potential_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m, float G,
                                float soft, const uint32_t *group, const uint64_t *idx, uint64_t n_idx, double *phi)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t t = 0; t < (int64_t)n_idx; t++) {
        const uint64_t i = idx[t];
        const uint32_t g = group[i];
        double sp = 0.0;
        if (g != NO_GROUP) {
            const double x = qx[i], y = qy[i], z = qz[i];
            for (uint64_t j = 0; j < n; j++) {
                if (j == i || group[j] != g) continue;
                const double rx = (double)qx[j] - x, ry = (double)qy[j] - y, rz = (double)qz[j] - z;
                sp += Gd * (double)m[j] / sqrt(rx * rx + ry * ry + rz * rz + s2);
            }
        }
        phi[t] = 0.0 - sp;
    }
}

static const uint32_t *g_lab;
static int by_label(const void *a, const void *b)
{
    const uint64_t i = *(const uint64_t *)a, j = *(const uint64_t *)b;
    if (g_lab[i] != g_lab[j]) return g_lab[i] < g_lab[j] ? -1 : 1;
    return i < j ? -1 : (i > j);
}

/* One unbinding pass over the member set `group` (NO_GROUP: not a member): phi[i] the group potential, E[i] =
 * |v_i - V_g|^2 / 2 + phi_i with V_g = sum m v / sum m over g's members (0 when their mass is 0), both fp64; 0 for
 * non-members.  Returns the number of members. */
uint64_t oracle_unbind_pass_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m,
                                const float *vx, const float *vy, const float *vz, float G, float soft,
                                const uint32_t *group, double *phi, double *E)
{
    const double Gd = (double)G, s2 = (double)soft * (double)soft;
    uint64_t *ord = (uint64_t *)malloc((n + 1) * sizeof(uint64_t));
    uint64_t M = 0;
    for (uint64_t i = 0; i < n; i++) {
        phi[i] = 0.0;
        E[i] = 0.0;
        if (group[i] != NO_GROUP) ord[M++] = i;
    }
    g_lab = group;
    qsort(ord, M, sizeof(uint64_t), by_label);
    /* group ranges [s, e) of ord; frame velocities in index order */
    uint64_t s = 0;
    while (s < M) {
        uint64_t e = s + 1;
        while (e < M && group[ord[e]] == group[ord[s]]) e++;
        double sm = 0.0, sx = 0.0, sy = 0.0, sz = 0.0;
        for (uint64_t k = s; k < e; k++) {
            const uint64_t i = ord[k];
            sm += (double)m[i];
            sx += (double)m[i] * vx[i];
            sy += (double)m[i] * vy[i];
            sz += (double)m[i] * vz[i];
        }
        const double Vx = sm != 0.0 ? sx / sm : 0.0, Vy = sm != 0.0 ? sy / sm : 0.0, Vz = sm != 0.0 ? sz / sm : 0.0;
#pragma omp parallel for schedule(dynamic, 16)
        for (int64_t k = (int64_t)s; k < (int64_t)e; k++) {
            const uint64_t i = ord[k];
            const double x = qx[i], y = qy[i], z = qz[i];
            double sp = 0.0;
            for (uint64_t l = s; l < e; l++) {
                const uint64_t j = ord[l];
                if (j == i) continue;
                const double rx = (double)qx[j] - x, ry = (double)qy[j] - y, rz = (double)qz[j] - z;
                sp += Gd * (double)m[j] / sqrt(rx * rx + ry * ry + rz * rz + s2);
            }
            phi[i] = 0.0 - sp;
            const double dx = (double)vx[i] - Vx, dy = (double)vy[i] - Vy, dz = (double)vz[i] - Vz;
            E[i] = 0.5 * (dx * dx + dy * dy + dz * dz) + phi[i];
        }
        s = e;
    }
    free(ord);
    return M;
}

/* The whole loop: passes until one removes nobody or max_iter passes.  bound[n] = the labels kept; phi[n] = the last
 * pass's potential over the set it used; returns the number of passes, *converged. */
uint32_t oracle_unbind_f64(uint64_t n, const float *qx, const float *qy, const float *qz, const float *m,
                           const float *vx, const float *vy, const float *vz, float G, float soft, const uint32_t *group,
                           uint32_t max_iter, uint32_t *bound, double *phi, int *converged)
{
    double *E = (double *)malloc((n + 1) * sizeof(double));
    uint64_t M = 0;
    for (uint64_t i = 0; i < n; i++) {
        bound[i] = group[i];
        phi[i] = 0.0;
        M += group[i] != NO_GROUP;
    }
    uint32_t t = 0;
    *converged = 1;
    if (M > 0)
        for (;;) {
            oracle_unbind_pass_f64(n, qx, qy, qz, m, vx, vy, vz, G, soft, bound, phi, E);
            t++;
            uint64_t removed = 0;
            for (uint64_t i = 0; i < n; i++)
                if (bound[i] != NO_GROUP && !(E[i] < 0.0)) {
                    bound[i] = NO_GROUP;
                    removed++;
                }
            if (removed == 0) break;
            if (t == max_iter) {
                *converged = 0;
                break;
            }
        }
    free(E);
    return t;
}
