/* The test-particle updates of libb200nb on the host, for SoA arrays and given accelerations, in the exact operation
 * sequence of the device integrator (integrate_kernel in csrc/integrate_sm100.cuh; include/b200nb.h, "test particles").
 * Built with -ffp-contract=off so that every a * b + c below is two roundings unless it is written as fmaf / fma (libm,
 * correctly rounded).  TEST INFRASTRUCTURE ONLY. */
#include <math.h>
#include <stdint.h>

/* MUrB: q += (v + a*dt/2)*dt evaluated in fp64 from the fp32 a*dt and rounded once; v += a*dt in fp32 */
void tracers_murb(uint64_t n, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz, const float *ax,
                  const float *ay, const float *az, float dt)
{
    float *q[3] = {qx, qy, qz}, *v[3] = {vx, vy, vz};
    const float *a[3] = {ax, ay, az};
    for (uint64_t i = 0; i < n; i++)
        for (int k = 0; k < 3; k++) {
            const float adt = a[k][i] * dt;
            q[k][i] = (float)((double)q[k][i] + ((double)v[k][i] + (double)adt * 0.5) * (double)dt);
            v[k][i] = v[k][i] + adt;
        }
}

/* leapfrog first half: v = fmaf(a, dt/2, v); q = fp32(fma(v, dt, q)) in fp64 */
void tracers_kick_drift(uint64_t n, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz, const float *ax,
                        const float *ay, const float *az, float dt)
{
    float *q[3] = {qx, qy, qz}, *v[3] = {vx, vy, vz};
    const float *a[3] = {ax, ay, az};
    const float hdt = dt * 0.5f;
    for (uint64_t i = 0; i < n; i++)
        for (int k = 0; k < 3; k++) {
            v[k][i] = fmaf(a[k][i], hdt, v[k][i]);
            q[k][i] = (float)fma((double)v[k][i], (double)dt, (double)q[k][i]);
        }
}

/* leapfrog closing kick: v = fmaf(a, dt/2, v) */
void tracers_kick(uint64_t n, float *vx, float *vy, float *vz, const float *ax, const float *ay, const float *az, float dt)
{
    float *v[3] = {vx, vy, vz};
    const float *a[3] = {ax, ay, az};
    const float hdt = dt * 0.5f;
    for (uint64_t i = 0; i < n; i++)
        for (int k = 0; k < 3; k++) v[k][i] = fmaf(a[k][i], hdt, v[k][i]);
}
