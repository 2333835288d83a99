// Massless test particles ("tracers", b200nb_set_tracers) advanced inside the step, for sm_100a.
//
// A tracer's acceleration is the field of all bodies at its position, a(p) of b200nb_field bit for bit: the hot pass is
// field_kernel<false> itself with the points pointing into the shard's tracer arrays, and the kernel below sums the
// S chunk rows with field_sum_rows, the summation of field_reduce_kernel, before it rounds once to fp32 and applies the
// update.  The updates are the operation sequences of integrate_kernel (integrate_sm100.cuh), written out again for SoA
// positions: IM_MURB, and the leapfrog's IM_LF_KICK_DRIFT and IM_LF_KICK.  A tracer therefore moves exactly as a host
// evaluation of the same expressions would move it, given the field at its position (tested bit for bit).
//
// Layout, per shard: tr = [9][T] floats, rows qx qy qz vx vy vz ax ay az (the a rows: the stored a(p) of the leapfrog),
// the shard's tracers [rank * T, rank * T + count) in its first `count` columns.  No tracer is ever exchanged: every
// shard holds the full body array after the position exchange.
#pragma once
#include "field_sm100.cuh"
#include "external_sm100.cuh"

namespace b200nb {

enum TracerMode : int {
    TM_MURB = 0,    // a = sum of the rows; q += (v + a*dt/2)*dt; v += a*dt   (IM_MURB)
    TM_LF_ACC = 1,  // a = sum of the rows, stored                             (the leapfrog's one-off a(p_0))
    TM_LF_KICK = 2  // a = sum of the rows, stored; v += a*dt/2                (IM_LF_KICK)
};

struct TracerArgs {
    const float *partial; // [S][4][stride] rows of field_kernel for the `count` tracers starting at `tr`
    uint32_t n_chunks, stride, count;
    float *tr;            // the first tracer of the batch inside the shard's [9][T] arrays
    uint64_t T;           // floats per row of those arrays
    float dt;
    int mode;
};

// after each field_kernel batch: fixed-order fp64 sum, rounded once, then the update.  EXT: the sum is rounded together
// with the external acceleration at the tracer's current position, as integrate_kernel<true> does for the bodies.
// FIELD (with an expansion): e is read from ef = [4][T] rows starting at the batch's first tracer, written by
// ext_total_kernel for the shard's tracers before the pass, instead of evaluated from `ext`.
template <bool EXT, bool FIELD = false>
__global__ void __launch_bounds__(256) tracer_update_kernel(const TracerArgs a, const __grid_constant__ ExtTerms ext,
                                                            const double *__restrict__ ef)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.count) return;
    double s[3];
    field_sum_rows<3>(a.partial, a.n_chunks, a.stride, i, s);
    if constexpr (EXT) {
        double e[3];
        if constexpr (FIELD) {
            e[0] = ef[i]; e[1] = ef[a.T + i]; e[2] = ef[2 * a.T + i];
        } else {
            double phi;
            ext_eval(ext, a.tr[i], a.tr[a.T + i], a.tr[2 * a.T + i], e, &phi);
        }
        s[0] = __dadd_rn(s[0], e[0]); s[1] = __dadd_rn(s[1], e[1]); s[2] = __dadd_rn(s[2], e[2]);
    }
    const float ax = (float)s[0], ay = (float)s[1], az = (float)s[2];
    float *q = a.tr + i;
    const size_t T = a.T;
    float vx = q[3 * T], vy = q[4 * T], vz = q[5 * T];
    if (a.mode == TM_MURB) { // integrate_kernel, IM_MURB
        const float axdt = __fmul_rn(ax, a.dt), aydt = __fmul_rn(ay, a.dt), azdt = __fmul_rn(az, a.dt);
        const double dt = (double)a.dt;
        q[0] = (float)__dadd_rn((double)q[0], __dmul_rn(__dadd_rn((double)vx, __dmul_rn((double)axdt, 0.5)), dt));
        q[T] = (float)__dadd_rn((double)q[T], __dmul_rn(__dadd_rn((double)vy, __dmul_rn((double)aydt, 0.5)), dt));
        q[2 * T] = (float)__dadd_rn((double)q[2 * T], __dmul_rn(__dadd_rn((double)vz, __dmul_rn((double)azdt, 0.5)), dt));
        q[3 * T] = __fadd_rn(vx, axdt);
        q[4 * T] = __fadd_rn(vy, aydt);
        q[5 * T] = __fadd_rn(vz, azdt);
        return;
    }
    q[6 * T] = ax; q[7 * T] = ay; q[8 * T] = az;
    if (a.mode == TM_LF_KICK) { // integrate_kernel, IM_LF_KICK
        const float hdt = __fmul_rn(a.dt, 0.5f);
        q[3 * T] = __fmaf_rn(ax, hdt, vx);
        q[4 * T] = __fmaf_rn(ay, hdt, vy);
        q[5 * T] = __fmaf_rn(az, hdt, vz);
    }
}

// the leapfrog's first half with the stored a(p): integrate_kernel, IM_LF_KICK_DRIFT
__global__ void __launch_bounds__(256) tracer_kick_drift_kernel(float *__restrict__ tr, uint64_t T, uint32_t count, float dt)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float *q = tr + i;
    const float hdt = __fmul_rn(dt, 0.5f);
    const double dtd = (double)dt;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float v = __fmaf_rn(q[(6 + k) * T], hdt, q[(3 + k) * T]);
        q[(3 + k) * T] = v;
        q[k * T] = (float)__fma_rn((double)v, dtd, (double)q[k * T]);
    }
}

} // namespace b200nb
