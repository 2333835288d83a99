// k nearest bodies of every body, and of arbitrary points, for sm_100a.
//
// Definition (include/b200nb.h): fp32 d2 = fma(dz, dz, fma(dy, dy, dx * dx)) with d = q_j - p, no softening, candidates
// ordered by the key (d2, j), so the k smallest keys are unique and the answer is a pure function of the fp32 positions.
//
// Same machinery as the field pass (field_sm100.cuh): the replicated AoSoA-128 body array is streamed through the
// cp.async.bulk + mbarrier pipeline, targets are register-blocked R per thread and two sources go through every packed
// f32x2 instruction.  One pair costs 3 FADD2 + 1 FMUL2 + 2 FFMA2 and one threshold test per target, against the force
// pass's 12 packed ops + 2 MUFU.  force_sm100.cuh is only included for its helpers; its code stays as it is.
//
// Keys in registers: d2 is >= 0 (or +inf, or NaN for non-finite positions), so its bit pattern as uint32 orders like the
// float.  Every target keeps its KB smallest keys of the current source chunk as a sorted list (d2 bits, index) in
// registers, updated by a fully unrolled compare-and-shift with static indices only.  An empty slot holds NB_EMPTY_D2 =
// 0x7F800001, above +inf: a pair whose d2 overflowed to +inf is still a candidate and keeps its (d2, j) place.  Masked
// lanes (the target itself in bodies mode, padding bodies j >= N) get 0xFFFFFFFF, which is never below any threshold.
//
// Within a chunk a thread meets sources in increasing index (lanes lo before hi, blocks in order), so the strict test
// d2 < (current KB-th d2) selects exactly in key order without an index compare, and a new entry goes after every
// stored entry of equal d2.  Chunk lists are then merged by nb_merge_kernel on 64-bit keys (d2 bits << 32 | j).
//
// Chunk count: after j sources a target inserts with probability ~KB/j and a warp takes the insertion branch when any
// of its 32 lanes does, so the insertion work per chunk grows like 32*KB*(1 + ln(chunk / (32*KB))) and the total like
// S times that.  The result does not depend on S, so S is chosen (nb_chunks) to fill the GPU with few, long chunks.
#pragma once
#include "force_sm100.cuh"

namespace b200nb {

constexpr uint32_t NB_EMPTY_D2 = 0x7F800001u;  // key of an empty slot: above every finite or infinite d2
constexpr uint32_t NB_MASKED_D2 = 0xFFFFFFFFu; // key of a masked lane: never inserted
constexpr uint32_t NB_NONE = 0xFFFFFFFFu;      // index of an empty slot
constexpr int NB_K_MAX = 32;
constexpr int NB_THREADS = 128, NB_TJB = 2, NB_ST = 3, NB_MINB = 4;
constexpr uint64_t NB_CAND_CAP = 1ull << 23;   // candidate entries ([S][KB][batch], 8 bytes each) per launch: 64 MiB
constexpr uint32_t NB_BATCH_CHUNKS = 4;        // a full batch still leaves room for this many chunks
constexpr uint32_t NB_BATCH_MAX = 1u << 20;    // targets per launch, whatever KB
constexpr uint32_t NB_MAX_CHUNKS = 64;
constexpr uint32_t NB_MIN_CHUNK_BLKS = 16;     // a chunk holds at least 2048 sources (if N allows)

// k buckets: the kernel keeps KB >= k keys; R targets per thread keeps the lists at 64 registers per thread or fewer
__host__ __device__ constexpr int nb_bucket(int k) { return k <= 1 ? 1 : k <= 8 ? 8 : k <= 16 ? 16 : 32; }
__host__ __device__ constexpr int nb_r(int kb) { return kb == 1 ? 8 : kb == 8 ? 4 : kb == 16 ? 2 : 1; }
__host__ __device__ constexpr uint32_t nb_tile(int kb) { return (uint32_t)(NB_THREADS * nb_r(kb)); }

// targets per launch for bucket KB: a multiple of the target tile
inline uint32_t nb_batch(int kb)
{
    const uint64_t b = NB_CAND_CAP / ((uint64_t)kb * NB_BATCH_CHUNKS);
    return (uint32_t)((b < NB_BATCH_MAX ? b : NB_BATCH_MAX) / nb_tile(kb) * nb_tile(kb));
}

// S for one launch of `cnt` targets out of a batch of `cap`.  The CTAs run in rounds of `slots` (4 per SM), so S0 =
// ceil(slots / tiles) chunks fill the first round; among S0..2*S0 the S whose last round is fullest wins (the smallest on
// a tie), because a part-filled last round costs as much as a full one.  Measured on a B200 (1000 W) at N = 200k, k = 8,
// 391 tiles: S = 2 (1.32 rounds) ran at 0.73 of the force pass's rate, S = 3 (1.98 rounds, this rule) at 0.91.
// Also: no chunk shorter than NB_MIN_CHUNK_BLKS blocks, candidate rows within NB_CAND_CAP.
inline uint32_t nb_chunks(int kb, uint32_t cnt, uint32_t cap, uint32_t src_nblk, uint32_t slots)
{
    const uint64_t tiles = (cnt + nb_tile(kb) - 1) / nb_tile(kb);
    uint64_t lim = (uint64_t)src_nblk / NB_MIN_CHUNK_BLKS;
    lim = lim < NB_CAND_CAP / ((uint64_t)kb * cap) ? lim : NB_CAND_CAP / ((uint64_t)kb * cap);
    lim = lim < NB_MAX_CHUNKS ? lim : NB_MAX_CHUNKS;
    if (lim < 1) lim = 1;
    const uint64_t s0 = (slots + tiles - 1) / tiles;
    uint64_t best = 1;
    double best_fill = 0.0;
    for (uint64_t s = s0; s <= 2 * s0; ++s) {
        const uint64_t ss = s < lim ? s : lim, ctas = tiles * ss;
        const double fill = (double)ctas / (double)(((ctas + slots - 1) / slots) * slots);
        if (fill > best_fill + 1e-9) {
            best_fill = fill;
            best = ss;
        }
    }
    return (uint32_t)best;
}
// the largest S any launch of a batch of `cap` can take (scratch sizing)
inline uint32_t nb_max_chunks(int kb, uint32_t cap)
{
    const uint64_t s = NB_CAND_CAP / ((uint64_t)kb * cap);
    return s < 1 ? 1u : (s > NB_MAX_CHUNKS ? NB_MAX_CHUNKS : (uint32_t)s);
}

struct NbArgs {
    const float *src;          // blocked bodies (the full replicated array)
    const float *px, *py, *pz; // SoA target points (points mode)
    uint64_t self0;            // bodies mode: global body index of target 0 (a multiple of BLK)
    uint32_t *cd2, *cidx;      // [S][KB][stride] candidate d2 bits and indices per chunk
    uint32_t stride;           // `count` rounded up to whole tiles
    uint32_t count;            // targets of this launch; threads of the last tile past it re-read the last target
    uint32_t n;                // real bodies: lanes j >= n are padding
    uint32_t src_nblk;         // ceil(n / BLK)
    uint32_t n_chunks;         // S
};

constexpr size_t nb_smem_bytes() { return (size_t)NB_ST * (NB_TJB * BLK_FLOATS * 4 + 8); }

// insert (d, j) into the sorted list (dl, il), knowing d < dl[KB-1] and that j exceeds every stored index: it goes after
// every entry of d2 <= d.  Descending p reads dl[p-1] before it is overwritten.
template <int KB>
__device__ __forceinline__ void nb_insert(uint32_t (&dl)[KB], uint32_t (&il)[KB], uint32_t d, uint32_t j)
{
#pragma unroll
    for (int p = KB - 1; p > 0; --p) {
        const bool up = dl[p - 1] > d;
        const bool here = !up && dl[p] > d;
        il[p] = up ? il[p - 1] : (here ? j : il[p]);
        dl[p] = up ? dl[p - 1] : (here ? d : dl[p]);
    }
    if (dl[0] > d) {
        dl[0] = d;
        il[0] = j;
    }
}

// one AoSoA block (sources j0 + [0, 128)) against the R targets of this thread.  MASK: lanes that are the target itself
// (tg, SELF only) or padding (>= n) never become candidates.
template <int KB, int R, bool SELF, bool MASK>
__device__ __forceinline__ void nb_block(const float *__restrict__ sb, const float (&xi)[R], const float (&yi)[R],
                                         const float (&zi)[R], uint32_t (&dl)[R][KB], uint32_t (&il)[R][KB], uint32_t j0,
                                         const uint32_t (&tg)[R], uint32_t n)
{
#pragma unroll 1
    for (int j = 0; j < BLK; j += 4) {
        const float4 xv = *reinterpret_cast<const float4 *>(sb + j);
        const float4 yv = *reinterpret_cast<const float4 *>(sb + BLK + j);
        const float4 zv = *reinterpret_cast<const float4 *>(sb + 2 * BLK + j);
        const uint64_t sx[2] = {pk2(xv.x, xv.y), pk2(xv.z, xv.w)};
        const uint64_t sy[2] = {pk2(yv.x, yv.y), pk2(yv.z, yv.w)};
        const uint64_t sz[2] = {pk2(zv.x, zv.y), pk2(zv.z, zv.w)};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t js = j0 + (uint32_t)(j + 2 * h);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t dx = sub2(sx[h], pk2(xi[r], xi[r]));
                const uint64_t dy = sub2(sy[h], pk2(yi[r], yi[r]));
                const uint64_t dz = sub2(sz[h], pk2(zi[r], zi[r]));
                uint64_t d = mul2(dx, dx);
                d = fma2(dy, dy, d);
                d = fma2(dz, dz, d);
                float f0, f1;
                upk2(d, f0, f1);
                uint32_t d0 = __float_as_uint(f0), d1 = __float_as_uint(f1);
                if (MASK) {
                    if (js >= n || (SELF && tg[r] == js)) d0 = NB_MASKED_D2;
                    if (js + 1 >= n || (SELF && tg[r] == js + 1)) d1 = NB_MASKED_D2;
                }
                if (min(d0, d1) < dl[r][KB - 1]) {
                    if (d0 < dl[r][KB - 1]) nb_insert<KB>(dl[r], il[r], d0, js);
                    if (d1 < dl[r][KB - 1]) nb_insert<KB>(dl[r], il[r], d1, js + 1);
                }
            }
        }
    }
}

// grid (ceil(count / (NB_THREADS * R)), S).  SELF = false: targets are the points px/py/pz; SELF = true: targets are
// the bodies self0 + [0, count).  Writes each target's sorted KB-list of its chunk.
template <int KB, bool SELF>
__global__ void __launch_bounds__(NB_THREADS, NB_MINB) neighbors_kernel(const NbArgs a)
{
    constexpr int R = nb_r(KB);
    constexpr int TI = NB_THREADS * R;
    constexpr int STAGE_FLOATS = NB_TJB * BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)NB_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint32_t b_begin = (uint32_t)(((uint64_t)a.src_nblk * c) / a.n_chunks);
    const uint32_t b_end = (uint32_t)(((uint64_t)a.src_nblk * (c + 1)) / a.n_chunks);
    const uint32_t nblk = b_end - b_begin;
    const uint32_t ntiles = (nblk + NB_TJB - 1) / NB_TJB;
    const float *chunk_src = a.src + (size_t)b_begin * BLK_FLOATS;

    if (leader) {
#pragma unroll
        for (int s = 0; s < NB_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) {
        const uint32_t nb = min((uint32_t)NB_TJB, nblk - tile * NB_TJB);
        const uint32_t bytes = nb * BLK_BYTES;
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4), chunk_src + (size_t)tile * STAGE_FLOATS, bytes, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < NB_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    float xi[R], yi[R], zi[R];
    uint32_t tg[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t il = min((uint32_t)(blockIdx.x * TI + r * NB_THREADS + threadIdx.x), a.count - 1);
        if (SELF) {
            const uint64_t g = a.self0 + il;
            tg[r] = (uint32_t)g;
            xi[r] = __ldg(a.src + blk_index(g, 0));
            yi[r] = __ldg(a.src + blk_index(g, 1));
            zi[r] = __ldg(a.src + blk_index(g, 2));
        } else {
            tg[r] = 0;
            xi[r] = __ldg(a.px + il);
            yi[r] = __ldg(a.py + il);
            zi[r] = __ldg(a.pz + il);
        }
    }
    // source blocks that need the masked path: those that can hold a target of this tile, and the last one when it
    // ends in padding
    const uint32_t mb0 = SELF ? (uint32_t)((a.self0 + (uint64_t)blockIdx.x * TI) / BLK) : 0xFFFFFFFFu;
    const uint32_t mb1 = SELF ? (uint32_t)((a.self0 + min((uint64_t)blockIdx.x * TI + TI, (uint64_t)a.count) - 1) / BLK) : 0u;
    const uint32_t pad_blk = (a.n % BLK) ? a.src_nblk - 1 : 0xFFFFFFFFu;

    uint32_t dl[R][KB], il[R][KB];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int p = 0; p < KB; ++p) {
            dl[r][p] = NB_EMPTY_D2;
            il[r][p] = NB_NONE;
        }

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % NB_ST;
        mbar_wait(bar0 + 8 * s, (t / NB_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)NB_TJB, nblk - t * NB_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t gb = b_begin + t * NB_TJB + b;
            if ((SELF && gb >= mb0 && gb <= mb1) || gb == pad_blk)
                nb_block<KB, R, SELF, true>(sb + b * BLK_FLOATS, xi, yi, zi, dl, il, gb * BLK, tg, a.n);
            else
                nb_block<KB, R, SELF, false>(sb + b * BLK_FLOATS, xi, yi, zi, dl, il, gb * BLK, tg, a.n);
        }
        if (t + NB_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + NB_ST, s);
        }
    }

#pragma unroll
    for (int r = 0; r < R; ++r) {
        const size_t t = (size_t)blockIdx.x * TI + (size_t)r * NB_THREADS + threadIdx.x;
#pragma unroll
        for (int p = 0; p < KB; ++p) {
            const size_t o = ((size_t)c * KB + p) * a.stride + t;
            a.cd2[o] = dl[r][p];
            a.cidx[o] = il[r][p];
        }
    }
}

// Merge the S sorted chunk lists of each target into its k smallest keys (d2 bits << 32 | j) and write the rows
// idx[t][k], dist[t][k] (dist = sqrt(d2) correctly rounded; empty slots: NB_NONE, +inf).
template <int KB>
__global__ void __launch_bounds__(128) nb_merge_kernel(const uint32_t *__restrict__ cd2, const uint32_t *__restrict__ cidx,
                                                       uint32_t n_chunks, uint32_t stride, uint32_t count, uint32_t k,
                                                       uint32_t *__restrict__ idx, float *__restrict__ dist)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    constexpr uint64_t EMPTY = ((uint64_t)NB_EMPTY_D2 << 32) | NB_NONE;
    uint64_t key[KB];
#pragma unroll
    for (int p = 0; p < KB; ++p) key[p] = EMPTY;
    for (uint32_t c = 0; c < n_chunks; ++c) {
        for (int q = 0; q < KB; ++q) {
            const size_t o = ((size_t)c * KB + q) * stride + t;
            const uint64_t v = ((uint64_t)cd2[o] << 32) | cidx[o];
            if (v >= key[KB - 1]) break; // the chunk's list is sorted
#pragma unroll
            for (int p = KB - 1; p > 0; --p) {
                const bool up = key[p - 1] > v;
                key[p] = up ? key[p - 1] : (key[p] > v ? v : key[p]);
            }
            if (key[0] > v) key[0] = v;
        }
    }
#pragma unroll
    for (int p = 0; p < KB; ++p)
        if ((uint32_t)p < k) {
            const uint32_t d = (uint32_t)(key[p] >> 32), j = (uint32_t)key[p];
            const bool empty = key[p] == EMPTY;
            idx[(size_t)t * k + p] = empty ? NB_NONE : j;
            dist[(size_t)t * k + p] = empty ? __int_as_float(0x7F800000) : __fsqrt_rn(__uint_as_float(d));
        }
}

} // namespace b200nb
