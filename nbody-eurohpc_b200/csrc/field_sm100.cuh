// Gravitational field (acceleration and potential) at arbitrary points, and the per-body potential, for sm_100a.
//
//   a(p)  = sum_j G m_j (q_j - p) / (|q_j - p|^2 + soft^2)^(3/2)       over ALL bodies
//   phi(p) = -sum_j G m_j / (|q_j - p|^2 + soft^2)^(1/2)
//   phi_i = -sum_{j != i} G m_j / (|r_ij|^2 + soft^2)^(1/2)             per body, self pair excluded BY INDEX
//
// Same law, G*m fold and softening as the force pass (force_sm100.cuh), and the same machinery: the replicated AoSoA-128
// body array is streamed through the cp.async.bulk + mbarrier pipeline, targets are register-blocked R per thread, two
// sources are processed per packed f32x2 instruction, and a (target tile x source chunk) grid writes per-chunk partial
// rows that a small kernel sums in fp64 in a fixed order.  One pair costs the force pass's 14 issue slots plus one
// packed add of G*m*inv (already formed for the force factor) into a potential accumulator: 15 per two interactions.
//
// Why this is a separate kernel and not a mode of force_kernel: the default force variant's hot loop is re-ordered
// after ptxas and fingerprinted (tools/sass_resched.py); any change to force_sm100.cuh rebuilds that cubin, and a
// changed loop silently drops the re-ordering.  This file only reuses the helpers of force_sm100.cuh and leaves its
// code untouched.
//
// Determinism: the value for a target depends only on that target and the bodies.  The source-chunk split S is a
// function of N alone (field_chunks) and every target is summed by the same per-thread code whatever tile, batch,
// shard or rank it lands in, so results are bit-identical for any set of points, batching and shard count.
//
// Self pair: at small softening the self term G m_i / soft dwarfs the rest (3000x for the galaxy scheme at soft = 1e4),
// so subtracting it after an fp32 sum would lose every significant digit.  It is excluded inside the kernel: only the
// source blocks that hold the tile's own targets take a masked path that zeroes the self lane's terms.
#pragma once
#include "force_sm100.cuh"

namespace b200nb {

__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b)
{
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// Shape: 128 threads x R = 4 targets, 3 CTAs (12 warps) per SM.  Four accumulators per target (x, y, z, potential)
// plus fp64 second-level sums do not fit next to R = 8 at a useful occupancy.  Measured on a B200 (1000 W, N = 200k),
// against the force pass in the same run: this shape 0.81-0.83 of its interactions/s; 4 CTAs per SM (128 registers)
// 0.74; R = 8 with 128 / 64 / 32 threads 0.77 / 0.75 / 0.74; 32 threads x R = 4 0.72.
constexpr int FIELD_THREADS = 128, FIELD_R = 4, FIELD_TJB = 2, FIELD_ST = 3, FIELD_MINB = 3;
constexpr int FIELD_TI = FIELD_THREADS * FIELD_R; // targets per CTA tile
constexpr uint32_t FIELD_CHUNK_BLKS = 32;         // source blocks per chunk (before the cap below)
constexpr uint32_t FIELD_MAX_CHUNKS = 64;
constexpr uint32_t FIELD_BATCH = 128 * FIELD_TI;  // targets per launch: bounds the scratch ([S][4][batch] partial rows)
static_assert(FIELD_TI % BLK == 0, "target tile must cover whole blocks");

// S, the number of source chunks: a function of N only (see the determinism note above)
__host__ __device__ inline uint32_t field_chunks(uint64_t n)
{
    const uint64_t nblk = (n + BLK - 1) / BLK;
    const uint64_t s = (nblk + FIELD_CHUNK_BLKS - 1) / FIELD_CHUNK_BLKS;
    return (uint32_t)(s < 1 ? 1 : (s > FIELD_MAX_CHUNKS ? FIELD_MAX_CHUNKS : s));
}

struct FieldArgs {
    const float *src;          // blocked bodies (the full replicated array)
    const float *px, *py, *pz; // SoA target points (field mode)
    uint64_t self0;            // potential mode: global body index of target 0 (targets are read from `src`)
    float *partial;            // [S][4][stride]: x, y, z, G*m*inv sums per chunk
    uint32_t stride;           // floats per component row of `partial`: `count` rounded up to whole tiles
    uint32_t count;            // targets of this launch; threads of the last tile past it re-read the last target
    uint32_t src_nblk;         // blocks that hold real bodies: ceil(N / BLK)
    uint32_t n_chunks;         // S = field_chunks(N)
    float soft2;
};

constexpr size_t field_smem_bytes() { return (size_t)FIELD_ST * (FIELD_TJB * BLK_BYTES + 8); }

// one target against one packed source pair; acc = {x, y, z, G*m*inv}.  MASK: lanes whose source is the target itself
// contribute exactly zero (selected after the math, so even soft^2 underflowing to 0 cannot leak an inf or NaN)
template <bool MASK>
__device__ __forceinline__ void field_pair(const uint64_t (&sj)[3], uint64_t gj, float xi, float yi, float zi,
                                           uint64_t soft2p, uint64_t (&acc)[4], bool self_lo, bool self_hi)
{
    const uint64_t dx = sub2(sj[0], pk2(xi, xi));
    const uint64_t dy = sub2(sj[1], pk2(yi, yi));
    const uint64_t dz = sub2(sj[2], pk2(zi, zi));
    uint64_t d = fma2(dx, dx, soft2p);
    d = fma2(dy, dy, d);
    d = fma2(dz, dz, d);
    float d0, d1;
    upk2(d, d0, d1);
    const uint64_t inv = pk2(rsqrt_approx(d0), rsqrt_approx(d1));
    uint64_t gi = mul2(gj, inv);
    uint64_t f = mul2(mul2(inv, inv), gi);
    if (MASK) {
        float g0, g1, f0, f1;
        upk2(gi, g0, g1);
        upk2(f, f0, f1);
        gi = pk2(self_lo ? 0.f : g0, self_hi ? 0.f : g1);
        f = pk2(self_lo ? 0.f : f0, self_hi ? 0.f : f1);
    }
    acc[0] = fma2(f, dx, acc[0]);
    acc[1] = fma2(f, dy, acc[1]);
    acc[2] = fma2(f, dz, acc[2]);
    acc[3] = add2(acc[3], gi);
}

// one AoSoA block (128 sources, global indices j0 + [0, 128)) against the R targets of this thread
template <bool MASK>
__device__ __forceinline__ void field_block(const float *__restrict__ sb, const float (&xi)[FIELD_R],
                                            const float (&yi)[FIELD_R], const float (&zi)[FIELD_R], uint64_t soft2p,
                                            uint64_t (&acc)[FIELD_R][4], uint32_t j0, const uint32_t (&tg)[FIELD_R])
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
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
            for (int k = 0; k < FIELD_R; ++k) {
                const uint32_t js = j0 + (uint32_t)(j + 2 * h);
                field_pair<MASK>(h ? s1 : s0, h ? g1 : g0, xi[k], yi[k], zi[k], soft2p, acc[k], MASK && tg[k] == js,
                                 MASK && tg[k] == js + 1);
            }
        }
    }
}

// grid (ceil(count / FIELD_TI), S).  SELF = false: targets are the points px/py/pz; SELF = true: targets are the bodies
// self0 + [0, count) and each one skips its own index.
template <bool SELF>
__global__ void __launch_bounds__(FIELD_THREADS, FIELD_MINB) field_kernel(const FieldArgs a)
{
    constexpr int STAGE_FLOATS = FIELD_TJB * BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)FIELD_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint32_t b_begin = (uint32_t)(((uint64_t)a.src_nblk * c) / a.n_chunks);
    const uint32_t b_end = (uint32_t)(((uint64_t)a.src_nblk * (c + 1)) / a.n_chunks);
    const uint32_t nblk = b_end - b_begin;
    const uint32_t ntiles = (nblk + FIELD_TJB - 1) / FIELD_TJB;
    const float *chunk_src = a.src + (size_t)b_begin * BLK_FLOATS;

    if (leader) {
#pragma unroll
        for (int s = 0; s < FIELD_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) {
        const uint32_t nb = min((uint32_t)FIELD_TJB, nblk - tile * FIELD_TJB);
        const uint32_t bytes = nb * BLK_BYTES;
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4), chunk_src + (size_t)tile * STAGE_FLOATS, bytes, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < FIELD_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    float xi[FIELD_R], yi[FIELD_R], zi[FIELD_R];
    uint32_t tg[FIELD_R]; // SELF: global body index of each target
#pragma unroll
    for (int k = 0; k < FIELD_R; ++k) {
        const uint32_t il = min((uint32_t)(blockIdx.x * FIELD_TI + k * FIELD_THREADS + threadIdx.x), a.count - 1);
        if (SELF) {
            const uint64_t g = a.self0 + il;
            tg[k] = (uint32_t)g;
            xi[k] = __ldg(a.src + blk_index(g, 0));
            yi[k] = __ldg(a.src + blk_index(g, 1));
            zi[k] = __ldg(a.src + blk_index(g, 2));
        } else {
            tg[k] = 0;
            xi[k] = __ldg(a.px + il);
            yi[k] = __ldg(a.py + il);
            zi[k] = __ldg(a.pz + il);
        }
    }
    // source blocks that can hold a target of this tile (self0 is a multiple of BLK)
    const uint32_t mb0 = (uint32_t)((a.self0 + (uint64_t)blockIdx.x * FIELD_TI) / BLK);
    const uint32_t mb1 = (uint32_t)((a.self0 + min((uint64_t)blockIdx.x * FIELD_TI + FIELD_TI, (uint64_t)a.count) - 1) / BLK);

    double m[FIELD_R][4]; // second-level accumulators
#pragma unroll
    for (int k = 0; k < FIELD_R; ++k) m[k][0] = m[k][1] = m[k][2] = m[k][3] = 0.0;
    const uint64_t soft2p = pk2(a.soft2, a.soft2);

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % FIELD_ST;
        mbar_wait(bar0 + 8 * s, (t / FIELD_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)FIELD_TJB, nblk - t * FIELD_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            uint64_t acc[FIELD_R][4];
#pragma unroll
            for (int k = 0; k < FIELD_R; ++k) acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0ull;
            const uint32_t gb = b_begin + t * FIELD_TJB + b;
            if (SELF && gb >= mb0 && gb <= mb1)
                field_block<true>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tg);
            else
                field_block<false>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tg);
            // fold every block (64 terms per lane) into fp64: a potential is a sum of same-sign terms, often one of
            // them (a central mass) much larger than the rest, and fp32 folds onto it lose ~1e-6 over a few hundred
#pragma unroll
            for (int k = 0; k < FIELD_R; ++k)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float lo, hi;
                    upk2(acc[k][q], lo, hi);
                    m[k][q] += (double)(lo + hi);
                }
        }
        if (t + FIELD_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + FIELD_ST, s);
        }
    }

    const size_t row = (size_t)c * 4;
#pragma unroll
    for (int k = 0; k < FIELD_R; ++k) {
        const size_t il = (size_t)blockIdx.x * FIELD_TI + (size_t)k * FIELD_THREADS + threadIdx.x;
#pragma unroll
        for (int q = 0; q < 4; ++q) a.partial[(row + q) * a.stride + il] = (float)m[k][q];
    }
}

// s[q] = the fixed-order fp64 sum of the S chunk rows of component q < NQ (0..2: x, y, z; 3: G*m*inv) of target i.
// The one summation behind every field value: b200nb_field and the test-particle step (tracers_sm100.cuh) both use it,
// which is what makes a tracer's acceleration bit-identical to b200nb_field at its position.
template <int NQ>
__device__ __forceinline__ void field_sum_rows(const float *__restrict__ partial, uint32_t n_chunks, uint32_t stride,
                                               uint32_t i, double (&s)[NQ])
{
#pragma unroll
    for (int q = 0; q < NQ; ++q) s[q] = 0.0;
    for (uint32_t r = 0; r < n_chunks; ++r)
#pragma unroll
        for (int q = 0; q < NQ; ++q) s[q] += (double)partial[((size_t)r * 4 + q) * stride + i];
}

// out[q * stride + i], q = 0..3: ax, ay, az, phi.  Fixed-order fp64 sum of the S chunk rows, rounded once.
__global__ void __launch_bounds__(256) field_reduce_kernel(const float *__restrict__ partial, uint32_t n_chunks,
                                                          uint32_t stride, uint32_t count, float *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double s[4];
    field_sum_rows<4>(partial, n_chunks, stride, i, s);
#pragma unroll
    for (int q = 0; q < 3; ++q) out[(size_t)q * stride + i] = (float)s[q];
    out[(size_t)3 * stride + i] = (float)-s[3];
}

} // namespace b200nb
