// Tidal tensor (the derivative of the gravitational field) at arbitrary points and per body, for sm_100a.
//
//   T_ab(p)  = sum_j G m_j [ 3 d_a d_b / s^5 - delta_ab / s^3 ],   d = q_j - p,  s^2 = |d|^2 + soft^2   over ALL bodies
//   T_ab,i   = the same sum at p = q_i over j != i                                      per body, self pair excluded BY INDEX
//
// T = da/dp of the softened field of field_sm100.cuh, i.e. minus the Hessian of its potential.  Same law, G*m fold and
// softening, and the same machinery as field_kernel: the replicated AoSoA-128 body array streams through the
// cp.async.bulk + mbarrier pipeline, R targets per thread, two sources per packed f32x2 instruction, per-block folds into
// fp64, and a (target tile x source chunk) grid whose per-chunk rows a small kernel sums in fp64 in a fixed order.
//
// Each target keeps seven sums: S_ab = sum (G m d_a / s^3) (d_b / s^2) for the six pairs ab, and S_3 = sum G m / s^3;
// tidal_reduce_kernel forms T_ab = 3 S_ab - delta_ab S_3 in fp64 and rounds once.
//
// Range: every intermediate stays in fp32's normal range.  The pair is formed as u_b = d_b * inv^2 (|u| <= 1 / s) times
// the field's own pair term f * d_a, f = G m * inv^3 built exactly as field_pair builds it (inv^2 is its first product).
// G m / s^5 is never formed: for the galaxy scheme at 10^3 system radii (s ~ 2e11 m) it is 1e-43..1e-46, below fp32's
// normal range, while f * d ~ 1e-13 and u ~ 5e-12 are not.
//
// Cost per source pair: 3 FADD2 + 9 FFMA2 + 9 FMUL2 + 1 FADD2 + 2 MUFU.RSQ, 22 packed FP32-pipe ops against the force
// pass's 12.  force_sm100.cuh and field_sm100.cuh are used, never edited (see the note at the top of field_sm100.cuh).
//
// Determinism: as for the field, S = field_chunks(N) depends on N only and every target runs the same per-thread code
// whatever tile, batch, shard or rank it lands in, so a value depends only on its target and the bodies.
#pragma once
#include "field_sm100.cuh"

namespace b200nb {

// Shape: 128 threads x R = 2 targets, 4 CTAs (16 warps) per SM: 112 / 118 registers (points / bodies), 0 spill bytes.
// Swept on a B200 (1000 W, N = 200k, one 32768-target launch, G-interactions/s, same per-pair op count): this shape 1406 for points and
// 1365-1404 for bodies; 128 x 2 at 3 CTAs 1406 / 1359; 128 x 4 at 2 CTAs 1390 / 1388; 128 x 4 at 3 CTAs 1339 (and 16
// spill bytes for bodies); 64 x 4 at 6 CTAs 1339.  field_kernel<false> ran at 2329 in the same run.
constexpr int TIDAL_THREADS = 128, TIDAL_R = 2, TIDAL_TJB = 2, TIDAL_ST = 3, TIDAL_MINB = 4;
constexpr int TIDAL_TI = TIDAL_THREADS * TIDAL_R; // targets per CTA tile
constexpr int TIDAL_NQ = 7;                       // partial rows per chunk: xx yy zz xy xz yz, sum G m / s^3
// targets per launch: [S][7][batch] fp32 partial rows stay within 64 * 7 * 32768 * 4 B = 56 MiB
constexpr uint32_t TIDAL_BATCH = 32768;
static_assert(TIDAL_BATCH % TIDAL_TI == 0 && TIDAL_TI % BLK == 0, "batches and tiles cover whole blocks");

constexpr size_t tidal_smem_bytes() { return (size_t)TIDAL_ST * (TIDAL_TJB * BLK_BYTES + 8); }

// one target against one packed source pair; acc = {xx, yy, zz, xy, xz, yz, G m / s^3}.  MASK: lanes whose source is the
// target itself contribute exactly zero.  inv is zeroed after the rsqrt (so soft^2 = 0 cannot leak an inf or NaN), and
// every term carries it.
template <bool MASK>
__device__ __forceinline__ void tidal_pair(const uint64_t (&sj)[3], uint64_t gj, float xi, float yi, float zi,
                                           uint64_t soft2p, uint64_t (&acc)[TIDAL_NQ], bool self_lo, bool self_hi)
{
    const uint64_t dx = sub2(sj[0], pk2(xi, xi));
    const uint64_t dy = sub2(sj[1], pk2(yi, yi));
    const uint64_t dz = sub2(sj[2], pk2(zi, zi));
    uint64_t d = fma2(dx, dx, soft2p);
    d = fma2(dy, dy, d);
    d = fma2(dz, dz, d);
    float d0, d1;
    upk2(d, d0, d1);
    uint64_t inv = pk2(rsqrt_approx(d0), rsqrt_approx(d1));
    if (MASK) {
        float i0, i1;
        upk2(inv, i0, i1);
        inv = pk2(self_lo ? 0.f : i0, self_hi ? 0.f : i1);
    }
    const uint64_t gi = mul2(gj, inv);
    const uint64_t inv2 = mul2(inv, inv);
    const uint64_t f = mul2(inv2, gi);                                             // G m / s^3, as field_pair forms it
    const uint64_t tx = mul2(f, dx), ty = mul2(f, dy), tz = mul2(f, dz);           // the field's pair terms
    const uint64_t ux = mul2(dx, inv2), uy = mul2(dy, inv2), uz = mul2(dz, inv2);  // d / s^2, |u| <= 1 / s
    acc[0] = fma2(tx, ux, acc[0]);
    acc[1] = fma2(ty, uy, acc[1]);
    acc[2] = fma2(tz, uz, acc[2]);
    acc[3] = fma2(tx, uy, acc[3]);
    acc[4] = fma2(tx, uz, acc[4]);
    acc[5] = fma2(ty, uz, acc[5]);
    acc[6] = add2(acc[6], f);
}

// one AoSoA block (128 sources, global indices j0 + [0, 128)) against the R targets of this thread.  MASK: target k is
// body t0 + k * TIDAL_THREADS and rel = t0 - j0, so source j0 + j is target k's own index iff
// j - rel == k * TIDAL_THREADS: one subtraction per source quad against constants, instead of R live target indices.
template <bool MASK>
__device__ __forceinline__ void tidal_block(const float *__restrict__ sb, const float (&xi)[TIDAL_R],
                                            const float (&yi)[TIDAL_R], const float (&zi)[TIDAL_R], uint64_t soft2p,
                                            uint64_t (&acc)[TIDAL_R][TIDAL_NQ], uint32_t rel)
{
#pragma unroll 1
    for (int j = 0; j < BLK; j += 4) {
        const float4 xv = *reinterpret_cast<const float4 *>(sb + j);
        const float4 yv = *reinterpret_cast<const float4 *>(sb + BLK + j);
        const float4 zv = *reinterpret_cast<const float4 *>(sb + 2 * BLK + j);
        const float4 gv = *reinterpret_cast<const float4 *>(sb + 3 * BLK + j);
        const uint64_t s0[3] = {pk2(xv.x, xv.y), pk2(yv.x, yv.y), pk2(zv.x, zv.y)};
        const uint64_t s1[3] = {pk2(xv.z, xv.w), pk2(yv.z, yv.w), pk2(zv.z, zv.w)};
        const uint64_t g0 = pk2(gv.x, gv.y), g1 = pk2(gv.z, gv.w);
        const uint32_t o = (uint32_t)j - rel;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
            for (int k = 0; k < TIDAL_R; ++k)
                tidal_pair<MASK>(h ? s1 : s0, h ? g1 : g0, xi[k], yi[k], zi[k], soft2p, acc[k],
                                 MASK && o == (uint32_t)(k * TIDAL_THREADS - 2 * h),
                                 MASK && o == (uint32_t)(k * TIDAL_THREADS - 2 * h - 1));
        }
    }
}

// grid (ceil(count / TIDAL_TI), S).  SELF = false: targets are the points px/py/pz; SELF = true: targets are the bodies
// self0 + [0, count) and each one skips its own index.  a.partial is [S][7][stride].
template <bool SELF>
__global__ void __launch_bounds__(TIDAL_THREADS, TIDAL_MINB) tidal_kernel(const FieldArgs a)
{
    constexpr int TI = TIDAL_TI, R = TIDAL_R;
    constexpr int STAGE_FLOATS = TIDAL_TJB * BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)TIDAL_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint32_t b_begin = (uint32_t)(((uint64_t)a.src_nblk * c) / a.n_chunks);
    const uint32_t b_end = (uint32_t)(((uint64_t)a.src_nblk * (c + 1)) / a.n_chunks);
    const uint32_t nblk = b_end - b_begin;
    const uint32_t ntiles = (nblk + TIDAL_TJB - 1) / TIDAL_TJB;
    const float *chunk_src = a.src + (size_t)b_begin * BLK_FLOATS;

    if (leader) {
#pragma unroll
        for (int s = 0; s < TIDAL_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) {
        const uint32_t nb = min((uint32_t)TIDAL_TJB, nblk - tile * TIDAL_TJB);
        const uint32_t bytes = nb * BLK_BYTES;
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4), chunk_src + (size_t)tile * STAGE_FLOATS, bytes, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < TIDAL_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    float xi[R], yi[R], zi[R];
    // SELF: target k is body t0 + k * TIDAL_THREADS.  Threads past `count` re-read the last body and their rows are never read,
    // so their mask may miss.
    const uint32_t t0 = (uint32_t)(a.self0 + blockIdx.x * TI + threadIdx.x);
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const uint32_t il = min((uint32_t)(blockIdx.x * TI + k * TIDAL_THREADS + threadIdx.x), a.count - 1);
        if (SELF) {
            const uint64_t g = a.self0 + il;
            xi[k] = __ldg(a.src + blk_index(g, 0));
            yi[k] = __ldg(a.src + blk_index(g, 1));
            zi[k] = __ldg(a.src + blk_index(g, 2));
        } else {
            xi[k] = __ldg(a.px + il);
            yi[k] = __ldg(a.py + il);
            zi[k] = __ldg(a.pz + il);
        }
    }
    // source blocks that can hold a target of this tile (self0 is a multiple of BLK)
    const uint32_t mb0 = (uint32_t)((a.self0 + (uint64_t)blockIdx.x * TI) / BLK);
    const uint32_t mb1 = (uint32_t)((a.self0 + min((uint64_t)blockIdx.x * TI + TI, (uint64_t)a.count) - 1) / BLK);

    double m[R][TIDAL_NQ]; // second-level accumulators
#pragma unroll
    for (int k = 0; k < R; ++k)
#pragma unroll
        for (int q = 0; q < TIDAL_NQ; ++q) m[k][q] = 0.0;
    const uint64_t soft2p = pk2(a.soft2, a.soft2);

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % TIDAL_ST;
        mbar_wait(bar0 + 8 * s, (t / TIDAL_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)TIDAL_TJB, nblk - t * TIDAL_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            uint64_t acc[R][TIDAL_NQ];
#pragma unroll
            for (int k = 0; k < R; ++k)
#pragma unroll
                for (int q = 0; q < TIDAL_NQ; ++q) acc[k][q] = 0ull;
            const uint32_t gb = b_begin + t * TIDAL_TJB + b;
            if (SELF && gb >= mb0 && gb <= mb1)
                tidal_block<true>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, t0 - gb * BLK);
            else
                tidal_block<false>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, 0);
            // fold every block (64 terms per lane) into fp64, as field_kernel does
#pragma unroll
            for (int k = 0; k < R; ++k)
#pragma unroll
                for (int q = 0; q < TIDAL_NQ; ++q) {
                    float lo, hi;
                    upk2(acc[k][q], lo, hi);
                    m[k][q] += (double)(lo + hi);
                }
        }
        if (t + TIDAL_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + TIDAL_ST, s);
        }
    }

    const size_t row = (size_t)c * TIDAL_NQ;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const size_t il = (size_t)blockIdx.x * TI + (size_t)k * TIDAL_THREADS + threadIdx.x;
#pragma unroll
        for (int q = 0; q < TIDAL_NQ; ++q) a.partial[(row + q) * a.stride + il] = (float)m[k][q];
    }
}

// out[i][6] = xx, yy, zz, xy, xz, yz of target i: the fixed-order fp64 sum of the S chunk rows of each of the seven sums,
// T_ab = 3 S_ab - delta_ab S_3 formed in fp64 and rounded once.
__global__ void __launch_bounds__(256) tidal_reduce_kernel(const float *__restrict__ partial, uint32_t n_chunks,
                                                          uint32_t stride, uint32_t count, float *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double s[TIDAL_NQ];
#pragma unroll
    for (int q = 0; q < TIDAL_NQ; ++q) s[q] = 0.0;
    for (uint32_t r = 0; r < n_chunks; ++r)
#pragma unroll
        for (int q = 0; q < TIDAL_NQ; ++q) s[q] += (double)partial[((size_t)r * TIDAL_NQ + q) * stride + i];
    float *o = out + (size_t)i * 6;
#pragma unroll
    for (int q = 0; q < 3; ++q) o[q] = (float)(3.0 * s[q] - s[6]);
#pragma unroll
    for (int q = 3; q < 6; ++q) o[q] = (float)(3.0 * s[q]);
}

} // namespace b200nb
