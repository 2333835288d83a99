// O(N) kernels around the force pass: layout pack/unpack, the fused partial-sum reduction + integrator, energy.
//
// Replaces, from scratch:
//   devUpdatePositionsAndVelocities           src/common/core/CUDABodies.cu:125-153   (MUrB explicit scheme)
//   devLeapfrogFirst/Middle/Last + dispatcher src/common/core/CUDABodies.cu:215-347   (documented intent :172-211)
//   devInitializeDevGM                        src/murb/implem/SimulationNBodyCUDATileFullDevice.cu:41-45
//   devComputeBodiesMetrics + cub::DeviceReduce::Sum
//                                             src/murb/implem/SimulationNBodyCUDAPropertyTracking.cu:217-304,333-364
// All of them are HBM-bound streaming kernels (coalesced, a few dozen bytes per body) and run in microseconds; they
// are fused so one step is: force pass -> one integrator kernel.
#pragma once
#include "force_sm100.cuh"
#include "external_sm100.cuh"

namespace b200nb {

enum IntegrateMode : int {
    IM_REDUCE_ONLY = 0,  // acc = sum of partial rows
    IM_MURB = 1,         // acc = sum of partial rows; q += (v + a*dt/2)*dt; v += a*dt      (Bodies.cpp:259-278)
    IM_LF_KICK_DRIFT = 2,// uses stored acc: v += a*dt/2; q += v*dt                         (leapfrog first half)
    IM_LF_KICK = 3,      // acc = sum of partial rows; v += a*dt/2                          (leapfrog closing kick)
    IM_MURB_STORED = 4   // MUrB update with the stored acc (caller-supplied accelerations)
};

// stream-K launches give every target tile its own number of partial rows (force_sm100.cuh: sk_rows_of_tile)
struct SkRows {
    uint64_t units; // U of the launch (0: launch not used)
    uint32_t G, nb, row0;
};

constexpr int MAX_PUSH_TARGETS = 16;

struct IntegrateArgs {
    const float *bodies;  // blocked full array the current positions are read from
    // Where the new positions of the slice [first, first+L) go.  One entry == `bodies`: in-place update (single GPU,
    // or NCCL all-gather afterwards).  Several entries: the *other* buffer of the double-buffered body array on this
    // GPU and on every peer GPU (peer pointers, stores travel over NVLink) - the integrator is also the exchange step.
    float *out[MAX_PUSH_TARGETS];
    int n_out;
    float *vel;           // [3][L] local velocities
    float *acc;           // [3][L] local accelerations
    const float *partial; // [rows][3][pstride]
    uint32_t rows;
    uint32_t pstride;     // floats per component row of `partial` (slice length rounded up to whole target tiles)
    uint32_t L;           // local slice length == stride of vel / acc
    uint32_t n_local;     // real (non-padding) bodies in the slice
    uint64_t first;       // global index of the first local body (multiple of BLK)
    float dt;
    int mode;
    uint32_t sk_ti;       // 0: chunk-grid rows [0, rows); else target-tile size of the stream-K launches below
    SkRows sk[2];
};

// EXT: the fp64 sum is rounded together with the external acceleration at the body's current position (include/b200nb.h,
// "external potential"); <false> ignores `ext` and `ef` and is the kernel without terms.  FIELD (with an expansion):
// e is read from ef = [4][L], the total external field ext_total_kernel has just written for the slice, instead of
// evaluated from `ext`; it is added at the same place.
template <bool EXT, bool FIELD = false>
__global__ void __launch_bounds__(256) integrate_kernel(const IntegrateArgs a, const __grid_constant__ ExtTerms ext,
                                                        const double *__restrict__ ef)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_local) return;
    const size_t L = a.L, P = a.pstride;

    float ax, ay, az;
    if (a.mode == IM_LF_KICK_DRIFT || a.mode == IM_MURB_STORED) {
        ax = a.acc[i]; ay = a.acc[L + i]; az = a.acc[2 * L + i];
    } else {
        // fixed-order fp64 sum of the chunk partials: deterministic, and the top level of the
        // hierarchical summation that keeps the fp32 error independent of N
        double sx = 0.0, sy = 0.0, sz = 0.0;
        if (a.sk_ti == 0) {
            for (uint32_t r = 0; r < a.rows; ++r) {
                const float *p = a.partial + (size_t)r * 3 * P;
                sx += (double)p[i]; sy += (double)p[P + i]; sz += (double)p[2 * P + i];
            }
        } else {
            const uint32_t t = i / a.sk_ti;
#pragma unroll
            for (int l = 0; l < 2; ++l) {
                if (a.sk[l].units == 0) continue;
                const uint32_t cnt = sk_rows_of_tile(t, a.sk[l].nb, a.sk[l].units, a.sk[l].G);
                for (uint32_t r = 0; r < cnt; ++r) {
                    const float *p = a.partial + (size_t)(a.sk[l].row0 + r) * 3 * P;
                    sx += (double)p[i]; sy += (double)p[P + i]; sz += (double)p[2 * P + i];
                }
            }
        }
        if constexpr (EXT) {
            double e[3];
            if constexpr (FIELD) {
                e[0] = ef[i]; e[1] = ef[L + i]; e[2] = ef[2 * L + i];
            } else {
                const size_t g = a.first + i;
                double phi;
                ext_eval(ext, a.bodies[blk_index(g, 0)], a.bodies[blk_index(g, 1)], a.bodies[blk_index(g, 2)], e, &phi);
            }
            sx = __dadd_rn(sx, e[0]); sy = __dadd_rn(sy, e[1]); sz = __dadd_rn(sz, e[2]);
        }
        ax = (float)sx; ay = (float)sy; az = (float)sz;
        a.acc[i] = ax; a.acc[L + i] = ay; a.acc[2 * L + i] = az;
        if (a.mode == IM_REDUCE_ONLY) return;
    }

    float vx = a.vel[i], vy = a.vel[L + i], vz = a.vel[2 * L + i];
    const size_t g = a.first + i;
    const size_t ix = blk_index(g, 0), iy = blk_index(g, 1), iz = blk_index(g, 2);

    if (a.mode == IM_MURB || a.mode == IM_MURB_STORED) {
        // The reference writes `q + (v + aDt * 0.5) * dt` with a double literal, so for T=float the position update
        // is evaluated in fp64 and rounded once (Bodies.cpp:264-270, CUDABodies.cu:139-141).  Same here, without
        // FMA contraction, so the result is bit-identical to an IEEE host evaluation of the same expression (tested).
        const float axdt = __fmul_rn(ax, a.dt), aydt = __fmul_rn(ay, a.dt), azdt = __fmul_rn(az, a.dt);
        const double dt = (double)a.dt;
        const double qx = (double)a.bodies[ix], qy = (double)a.bodies[iy], qz = (double)a.bodies[iz];
        const float nx = (float)__dadd_rn(qx, __dmul_rn(__dadd_rn((double)vx, __dmul_rn((double)axdt, 0.5)), dt));
        const float ny = (float)__dadd_rn(qy, __dmul_rn(__dadd_rn((double)vy, __dmul_rn((double)aydt, 0.5)), dt));
        const float nz = (float)__dadd_rn(qz, __dmul_rn(__dadd_rn((double)vz, __dmul_rn((double)azdt, 0.5)), dt));
        for (int d = 0; d < a.n_out; ++d) { a.out[d][ix] = nx; a.out[d][iy] = ny; a.out[d][iz] = nz; }
        a.vel[i] = __fadd_rn(vx, axdt);
        a.vel[L + i] = __fadd_rn(vy, aydt);
        a.vel[2 * L + i] = __fadd_rn(vz, azdt);
        return;
    }

    // leapfrog half kick (both modes)
    const float hdt = __fmul_rn(a.dt, 0.5f);
    vx = __fmaf_rn(ax, hdt, vx);
    vy = __fmaf_rn(ay, hdt, vy);
    vz = __fmaf_rn(az, hdt, vz);
    a.vel[i] = vx; a.vel[L + i] = vy; a.vel[2 * L + i] = vz;
    if (a.mode == IM_LF_KICK_DRIFT) { // drift, fp64 like the MUrB position update
        const double dt = (double)a.dt;
        const float nx = (float)__fma_rn((double)vx, dt, (double)a.bodies[ix]);
        const float ny = (float)__fma_rn((double)vy, dt, (double)a.bodies[iy]);
        const float nz = (float)__fma_rn((double)vz, dt, (double)a.bodies[iz]);
        for (int d = 0; d < a.n_out; ++d) { a.out[d][ix] = nx; a.out[d][iy] = ny; a.out[d][iz] = nz; }
    }
}

// ---------------------------------------------------------------------------------------------- pack / unpack
// Host <-> device layout conversion for ONE shard's slice (global bodies [first, first + L)).
// stage: 7 host-layout SoA slices (qx qy qz m vx vy vz), each L floats, the first n_local of each valid.  Writes the
// slice's AoSoA blocks (positions + G*m) into `bodies` and the local velocities and masses.  Padding bodies (slice
// entries past n_local) carry G*m = 0 at (px,py,pz) = the position of the last real body of the system, so they add
// exactly 0 and cannot create a singularity that a real pair does not have.
__global__ void __launch_bounds__(256) pack_slice_kernel(const float *__restrict__ stage, uint32_t L, uint32_t n_local,
                                                        size_t first, float px, float py, float pz, float G,
                                                        float *__restrict__ bodies, float *__restrict__ vel,
                                                        float *__restrict__ mass)
{
    for (uint32_t li = blockIdx.x * blockDim.x + threadIdx.x; li < L; li += gridDim.x * blockDim.x) {
        const bool real = li < n_local;
        const size_t i = first + li;
        const float m = real ? stage[3 * (size_t)L + li] : 0.f;
        bodies[blk_index(i, 0)] = real ? stage[li] : px;
        bodies[blk_index(i, 1)] = real ? stage[(size_t)L + li] : py;
        bodies[blk_index(i, 2)] = real ? stage[2 * (size_t)L + li] : pz;
        bodies[blk_index(i, 3)] = __fmul_rn(G, m); // devInitializeDevGM: GM[i] = G * m[i]
        vel[li] = real ? stage[4 * (size_t)L + li] : 0.f;
        vel[(size_t)L + li] = real ? stage[5 * (size_t)L + li] : 0.f;
        vel[2 * (size_t)L + li] = real ? stage[6 * (size_t)L + li] : 0.f;
        mass[li] = m;
    }
}

// blocked positions of bodies [first, first + count) -> three SoA arrays of `stride` floats (entry 0 = body `first`)
__global__ void __launch_bounds__(256) unpack_positions_kernel(const float *__restrict__ bodies, size_t first, size_t count,
                                                              float *__restrict__ stage, size_t stride)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        stage[i] = bodies[blk_index(first + i, 0)];
        stage[stride + i] = bodies[blk_index(first + i, 1)];
        stage[2 * stride + i] = bodies[blk_index(first + i, 2)];
    }
}

// load caller-supplied accelerations of the slice (host SoA slices staged at `stage`, 3 x stride) into the local acc
__global__ void __launch_bounds__(256) load_acc_kernel(const float *__restrict__ stage, size_t stride, uint32_t n_local,
                                                      float *__restrict__ acc, size_t L)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_local) return;
    acc[i] = stage[i];
    acc[L + i] = stage[stride + i];
    acc[2 * L + i] = stage[2 * stride + i];
}

// ---------------------------------------------------------------------------------------------- metrics
// One pass produces every per-iteration metric of the reference's history (SimulationHistory.hpp:12-15, CSV columns
// :45): the total energy (the only one computed upstream), and the angular momentum and density centre that are
// declared there but never filled in.
//   E_i = m_i |v_i|^2 / 2  -  (m_i / 2) * ( sum_j Gm_j / sqrt(r_ij^2 + soft^2)  -  Gm_i / soft )
//         (definition and self-term handling: SimulationNBodyCUDAPropertyTracking.cu:262-301)
//   L   = sum_i m_i (r_i x v_i)                                  about the origin
//   centre of mass   = sum_i m_i r_i / sum_i m_i
//   density centre   = sum_i w_i r_i / sum_i w_i,  w_i = m_i * (softened potential at body i, self term excluded):
//                      the potential-weighted centre, which follows the densest region instead of the mass mean
// The pair sum uses rsqrt.approx + one Newton step (~1e-7 relative), 128-term fp32 tile sums and an fp64 running sum;
// everything per-body is fp64.  Rows of the raw output (summed over blocks, then over ranks, by the caller):
enum MetricRow { MR_ENERGY = 0, MR_LX, MR_LY, MR_LZ, MR_M, MR_MX, MR_MY, MR_MZ, MR_W, MR_WX, MR_WY, MR_WZ, MR_COUNT };
constexpr int ENERGY_THREADS = 128;

__device__ __forceinline__ float rsqrt_nr(float d)
{
    const float y = rsqrt_approx(d);
    return y * fmaf(-0.5f * d, y * y, 1.5f);
}

// block_out[row * n_blocks + block].  EXT: the energy row adds m_i Phi_ext(q_i); <false> ignores `ext` and `ef`.
// FIELD: Phi_ext is row 3 of ef = [4][L], written by ext_total_kernel for the slice (see integrate_kernel).
template <bool EXT, bool FIELD = false>
__global__ void __launch_bounds__(ENERGY_THREADS) energy_kernel(const float *__restrict__ bodies,
                                                                const float *__restrict__ vel,
                                                                const float *__restrict__ mass, uint32_t L,
                                                                uint32_t n_local, uint64_t first, uint32_t nblk_total,
                                                                float soft2, double *__restrict__ block_out,
                                                                const __grid_constant__ ExtTerms ext,
                                                                const double *__restrict__ ef)
{
    __shared__ __align__(16) float tile[BLK_FLOATS];
    __shared__ double warp_sums[MR_COUNT][ENERGY_THREADS / 32];
    const uint32_t i = blockIdx.x * ENERGY_THREADS + threadIdx.x;
    const bool valid = i < n_local;
    const size_t g = first + (valid ? i : 0);
    const float xi = bodies[blk_index(g, 0)], yi = bodies[blk_index(g, 1)], zi = bodies[blk_index(g, 2)];
    const float gi = bodies[blk_index(g, 3)];

    double pot = 0.0;
    for (uint32_t b = 0; b < nblk_total; ++b) {
        __syncthreads();
        reinterpret_cast<float4 *>(tile)[threadIdx.x] =
            reinterpret_cast<const float4 *>(bodies + (size_t)b * BLK_FLOATS)[threadIdx.x];
        __syncthreads();
        float s = 0.f;
#pragma unroll 8
        for (int j = 0; j < BLK; ++j) {
            const float dx = tile[j] - xi, dy = tile[BLK + j] - yi, dz = tile[2 * BLK + j] - zi;
            const float d = fmaf(dz, dz, fmaf(dy, dy, fmaf(dx, dx, soft2)));
            s = fmaf(tile[3 * BLK + j], rsqrt_nr(d), s);
        }
        pot += (double)s;
    }
    double r[MR_COUNT];
#pragma unroll
    for (int k = 0; k < MR_COUNT; ++k) r[k] = 0.0;
    if (valid) {
        const double vx = vel[i], vy = vel[L + i], vz = vel[2 * (size_t)L + i];
        const double x = xi, y = yi, z = zi;
        const double m = (double)mass[i];
        const double self = (double)gi * (double)rsqrt_nr(soft2);
        const double v2 = vx * vx + vy * vy + vz * vz;
        const double w = m * (pot - self);
        r[MR_ENERGY] = 0.5 * m * v2 - 0.5 * w;
        if constexpr (EXT) {
            double phi;
            if constexpr (FIELD) {
                phi = ef[3 * (size_t)L + i];
            } else {
                double e[3];
                ext_eval(ext, xi, yi, zi, e, &phi);
            }
            r[MR_ENERGY] = __dadd_rn(r[MR_ENERGY], __dmul_rn(m, phi));
        }
        r[MR_LX] = m * (y * vz - z * vy);
        r[MR_LY] = m * (z * vx - x * vz);
        r[MR_LZ] = m * (x * vy - y * vx);
        r[MR_M] = m;  r[MR_MX] = m * x; r[MR_MY] = m * y; r[MR_MZ] = m * z;
        r[MR_W] = w;  r[MR_WX] = w * x; r[MR_WY] = w * y; r[MR_WZ] = w * z;
    }
#pragma unroll
    for (int k = 0; k < MR_COUNT; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r[k] += __shfl_down_sync(0xffffffffu, r[k], o);
        if ((threadIdx.x & 31) == 0) warp_sums[k][threadIdx.x >> 5] = r[k];
    }
    __syncthreads();
    if (threadIdx.x < MR_COUNT) {
        double t = 0.0;
        for (int w = 0; w < ENERGY_THREADS / 32; ++w) t += warp_sums[threadIdx.x][w];
        block_out[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = t;
    }
}

// fixed-order final sum, one block per row (deterministic; replaces cub::DeviceReduce::Sum and its per-call cudaMalloc)
__global__ void __launch_bounds__(256) energy_final_kernel(const double *__restrict__ block_out, uint32_t nb,
                                                          double *__restrict__ out)
{
    __shared__ double sh[256];
    const double *row = block_out + (size_t)blockIdx.x * nb;
    double t = 0.0;
    for (uint32_t k = threadIdx.x; k < nb; k += 256) t += row[k];
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

} // namespace b200nb
