/* The external potential of libb200nb on the host (include/b200nb.h, "external potential"): the evaluator in the operation
 * order csrc/external_sm100.cuh states, and the MUrB and leapfrog updates of a system without self-gravity, whose
 * acceleration is then fp32(a_ext) exactly.  Built with -ffp-contract=off, so every a * b + c below is two roundings
 * unless written as fma / fmaf (libm, correctly rounded): bit for bit the device wherever no log / log1p is involved.
 * TEST INFRASTRUCTURE ONLY. */
#include <math.h>
#include <stdint.h>

#include "../include/b200nb.h"

void ext_eval(uint32_t n_terms, const b200nb_external_term *terms, uint64_t n, const float *px, const float *py,
              const float *pz, double *ax, double *ay, double *az, double *phi)
{
    for (uint64_t i = 0; i < n; i++) {
        double sx = 0.0, sy = 0.0, sz = 0.0, sp = 0.0;
        for (uint32_t m = 0; m < n_terms; m++) {
            const b200nb_external_term *t = &terms[m];
            const double dx = (double)px[i] - t->centre[0], dy = (double)py[i] - t->centre[1], dz = (double)pz[i] - t->centre[2];
            const double R2 = dx * dx + dy * dy, dz2 = dz * dz;
            double p, k, tz;
            if (t->kind == B200NB_EXT_PLUMMER) {
                const double s2 = (R2 + dz2) + t->a * t->a, s = sqrt(s2);
                p = -(t->gm / s);
                k = t->gm / (s2 * s);
                tz = -(k * dz);
            } else if (t->kind == B200NB_EXT_HERNQUIST) {
                const double r = sqrt(R2 + dz2), u = r + t->a;
                p = -(t->gm / u);
                k = r > 0.0 ? t->gm / ((r * u) * u) : 0.0;
                tz = -(k * dz);
            } else if (t->kind == B200NB_EXT_NFW) {
                const double r2 = R2 + dz2, r = sqrt(r2), x = r / t->a, l = log1p(x), xp1 = 1.0 + x;
                double mu;
                if (x < 0.1) {
                    const double y = x / xp1;
                    double s = 1.0 / 18;
                    for (int j = 17; j >= 2; j--) s = 1.0 / j + y * s;
                    mu = (y * y) * s;
                } else {
                    mu = l - x / xp1;
                }
                p = r > 0.0 ? -((t->gm * l) / r) : -(t->gm / t->a);
                k = r > 0.0 ? (t->gm * mu) / (r2 * r) : 0.0;
                tz = -(k * dz);
            } else if (t->kind == B200NB_EXT_MIYAMOTO_NAGAI) {
                const double zeta = sqrt(dz2 + t->b * t->b), w = t->a + zeta, D2 = R2 + w * w, D = sqrt(D2);
                p = -(t->gm / D);
                k = t->gm / (D2 * D);
                tz = -(((k * w) / zeta) * dz);
            } else {
                const double q2 = t->b * t->b, S = (R2 + dz2 / q2) + t->a * t->a;
                p = (0.5 * t->gm) * log(S);
                k = t->gm / S;
                tz = -((k * dz) / q2);
            }
            sx = sx + -(k * dx);
            sy = sy + -(k * dy);
            sz = sz + tz;
            sp = sp + p;
        }
        if (ax) ax[i] = sx;
        if (ay) ay[i] = sy;
        if (az) az[i] = sz;
        if (phi) phi[i] = sp;
    }
}

/* acc[k][i] = fp32(a_ext): the acceleration of a body or tracer when self-gravity is exactly zero */
static void ext_accel(uint32_t n_terms, const b200nb_external_term *terms, uint64_t n, float *const q[3], float *const acc[3])
{
    for (uint64_t i = 0; i < n; i++) {
        double a[3];
        ext_eval(n_terms, terms, 1, q[0] + i, q[1] + i, q[2] + i, a, a + 1, a + 2, 0);
        for (int k = 0; k < 3; k++) acc[k][i] = (float)a[k];
    }
}

/* n_steps of the integrator with a = fp32(a_ext), in the device's operation sequence (integrate_kernel):
 *   MUrB:     adt = a*dt; q = fp32(q + (v + adt*0.5)*dt) in fp64; v = v + adt
 *   leapfrog: v = fmaf(a, dt/2, v); q = fp32(fma(v, dt, q)); a = a(q'); v = fmaf(a, dt/2, v),
 * a(x_0) taken first unless have_acc (then acc holds the stored a(x_n)).  acc is left holding the last acceleration. */
void ext_steps(uint32_t n_terms, const b200nb_external_term *terms, uint64_t n, float *qx, float *qy, float *qz, float *vx,
               float *vy, float *vz, float *ax, float *ay, float *az, float dt, int integrator, int n_steps, int have_acc)
{
    float *q[3] = {qx, qy, qz}, *v[3] = {vx, vy, vz}, *a[3] = {ax, ay, az};
    const float hdt = dt * 0.5f;
    for (int s = 0; s < n_steps; s++) {
        if (integrator == 0) {
            ext_accel(n_terms, terms, n, q, a);
            for (uint64_t i = 0; i < n; i++)
                for (int k = 0; k < 3; k++) {
                    const float adt = a[k][i] * dt;
                    q[k][i] = (float)((double)q[k][i] + ((double)v[k][i] + (double)adt * 0.5) * (double)dt);
                    v[k][i] = v[k][i] + adt;
                }
            continue;
        }
        if (!have_acc) ext_accel(n_terms, terms, n, q, a);
        have_acc = 1;
        for (uint64_t i = 0; i < n; i++)
            for (int k = 0; k < 3; k++) {
                v[k][i] = fmaf(a[k][i], hdt, v[k][i]);
                q[k][i] = (float)fma((double)v[k][i], (double)dt, (double)q[k][i]);
            }
        ext_accel(n_terms, terms, n, q, a);
        for (uint64_t i = 0; i < n; i++)
            for (int k = 0; k < 3; k++) v[k][i] = fmaf(a[k][i], hdt, v[k][i]);
    }
}
