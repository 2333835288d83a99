// Gravitational field by source component, at arbitrary points and per body, for sm_100a.
//
//   a^h(p)   = sum_{j: comp[j] = h} G m_j (q_j - p) / (|q_j - p|^2 + soft^2)^(3/2)
//   phi^h(p) = -sum_{j: comp[j] = h} G m_j / (|q_j - p|^2 + soft^2)^(1/2)
//   per body i: the same sums at p = q_i, self pair excluded BY INDEX
//
// The pair math, the per-block fp64 fold and the reduction are field_sm100.cuh's own (field_block, field_sum_rows): only
// the source array and its chunk cut differ.  force_sm100.cuh and field_sm100.cuh are used, never edited.
//
// Member order.  The host sorts the bodies by (component, index) (a stable counting sort) and the members of component h
// are packed in that order into an AoSoA-128 source array from a block boundary on; its last block is padded with
// G*m = 0 lanes at the position of h's last member, the convention of b200nb_upload for the body array.
//
// Chunks.  Component h's nblk_h blocks are cut into S_h = field_chunks(M_h) chunks at b = nblk_h * c / S_h, field_kernel's
// formula, so the cut depends on M_h alone.  The grid is (target tiles x sum_h S_h); a table maps blockIdx.y to its
// packed block range.  With one component holding every body, the packed array and the cut are field_kernel's, so a
// value is bit-identical to b200nb_field / b200nb_potential; in general a value depends only on the target and on h's
// members in index order.
//
// Bodies mode.  Targets are the bodies in index order (run_targets' slices), read from the body array; each one carries
// its packed position (or COMP_NONE), and a lane is its own iff the packed positions match.  The source blocks that hold
// a target of the tile are no longer one range when labels interleave, so every CTA first marks them in a shared-memory
// bitmap over its chunk; only marked blocks take field_block's masked path, a CTA-uniform branch as in field_kernel<true>.
#pragma once
#include "field_sm100.cuh"

namespace b200nb {

constexpr uint32_t COMP_MAX = 64;
constexpr uint32_t COMP_NONE = 0xFFFFFFFFu; // B200NB_NO_GROUP; also "no packed position"
constexpr uint32_t COMP_PAD = 0x80000000u;  // in the member map: a padding lane at this body's position (bodies < 2^31)
constexpr uint32_t COMP_PARTIAL_FLOATS = 1u << 24; // [sum S][4][batch] partial rows stay within 64 MiB

struct CompArgs {
    const float *src;          // packed components, AoSoA-128 (x, y, z, G*m)
    const float *bodies;       // bodies mode: the replicated body array, where the targets are read
    const uint32_t *pos;       // bodies mode: packed position of every body (COMP_NONE: source of nothing)
    const float *px, *py, *pz; // points mode: SoA target points
    const uint2 *chunk;        // per blockIdx.y: packed blocks [x, y) of that chunk
    uint64_t self0;            // bodies mode: global body index of target 0
    float *partial;            // [sum S][4][stride]: x, y, z, G*m*inv sums per chunk
    uint32_t stride;           // floats per component row of `partial`
    uint32_t count;            // targets of this launch; threads of the last tile past it re-read the last target
    float soft2;
};

// dynamic shared memory: field_kernel's ring, then (bodies mode) one bit per block of the longest chunk
inline size_t comp_smem_bytes(uint32_t max_chunk_blks) { return field_smem_bytes() + 4 * (size_t)((max_chunk_blks + 31) / 32); }

// grid (ceil(count / FIELD_TI), sum_h S_h).  SELF = false: targets are the points px/py/pz; SELF = true: targets are the
// bodies self0 + [0, count) and each one skips its own index.
template <bool SELF>
__global__ void __launch_bounds__(FIELD_THREADS, FIELD_MINB) component_field_kernel(const CompArgs a)
{
    constexpr int STAGE_FLOATS = FIELD_TJB * BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)FIELD_ST * STAGE_FLOATS * 4);
    // SELF: the blocks of this chunk that hold a target of the tile, after the ring (field_smem_bytes())
    uint32_t *own = reinterpret_cast<uint32_t *>(smem_raw + (size_t)FIELD_ST * (STAGE_FLOATS * 4 + 8));
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint2 ch = a.chunk[c];
    const uint32_t b_begin = ch.x;
    const uint32_t nblk = ch.y - ch.x;
    const uint32_t ntiles = (nblk + FIELD_TJB - 1) / FIELD_TJB;
    const float *chunk_src = a.src + (size_t)b_begin * BLK_FLOATS;

    if (SELF)
        for (uint32_t w = threadIdx.x; w < (nblk + 31) / 32; w += FIELD_THREADS) own[w] = 0;
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
    uint32_t tg[FIELD_R]; // SELF: packed position of each target
#pragma unroll
    for (int k = 0; k < FIELD_R; ++k) {
        const uint32_t il = min((uint32_t)(blockIdx.x * FIELD_TI + k * FIELD_THREADS + threadIdx.x), a.count - 1);
        if (SELF) {
            const uint64_t g = a.self0 + il;
            tg[k] = __ldg(a.pos + g);
            xi[k] = __ldg(a.bodies + blk_index(g, 0));
            yi[k] = __ldg(a.bodies + blk_index(g, 1));
            zi[k] = __ldg(a.bodies + blk_index(g, 2));
            const uint32_t b = tg[k] / BLK - b_begin; // wraps past nblk for COMP_NONE and blocks before the chunk
            if (tg[k] != COMP_NONE && b < nblk) atomicOr(own + b / 32, 1u << (b % 32));
        } else {
            tg[k] = 0;
            xi[k] = __ldg(a.px + il);
            yi[k] = __ldg(a.py + il);
            zi[k] = __ldg(a.pz + il);
        }
    }
    if (SELF) __syncthreads(); // the bitmap is complete

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
            const uint32_t lb = t * FIELD_TJB + b, gb = b_begin + lb;
            if (SELF && ((own[lb / 32] >> (lb % 32)) & 1u))
                field_block<true>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tg);
            else
                field_block<false>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tg);
            // every block folds into fp64, as in field_kernel
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

// acc[i][h][3], phi[i][h] of target i < count, component h = blockIdx.y: field_sum_rows over h's chunk rows
// [chunk0[h], chunk0[h + 1]) in order, rounded once (a component without members gives 0 and phi = -0)
__global__ void __launch_bounds__(256) component_reduce_kernel(const float *__restrict__ partial, const uint32_t *__restrict__ chunk0,
                                                              uint32_t stride, uint32_t count, uint32_t n_comp,
                                                              float *__restrict__ acc, float *__restrict__ phi)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t h = blockIdx.y;
    if (i >= count) return;
    const uint32_t r0 = chunk0[h];
    double s[4];
    field_sum_rows<4>(partial + (size_t)r0 * 4 * stride, chunk0[h + 1] - r0, stride, i, s);
    float *o = acc + ((size_t)i * n_comp + h) * 3;
#pragma unroll
    for (int q = 0; q < 3; ++q) o[q] = (float)s[q];
    phi[(size_t)i * n_comp + h] = (float)-s[3];
}

// src[p], p < count: the member map[p] (x, y, z, G*m), or for map[p] = body | COMP_PAD that body's position with G*m = 0
__global__ void __launch_bounds__(256) component_pack_kernel(const float *__restrict__ bodies, const uint32_t *__restrict__ map,
                                                            uint32_t count, float *__restrict__ src)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= count) return;
    const uint32_t e = map[p], i = e & ~COMP_PAD;
#pragma unroll
    for (int q = 0; q < 3; ++q) src[blk_index(p, q)] = __ldg(bodies + blk_index(i, q));
    src[blk_index(p, 3)] = (e & COMP_PAD) ? 0.f : __ldg(bodies + blk_index(i, 3));
}

} // namespace b200nb
