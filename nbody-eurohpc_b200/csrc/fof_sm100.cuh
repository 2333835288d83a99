// Friends-of-friends groups of the bodies for sm_100a.
//
// Definition (include/b200nb.h): bodies i != j are linked iff the fp32 d2 = fma(dz, dz, fma(dy, dy, dx * dx)), d = q_j -
// q_i, satisfies d2 <= b2 (b2 = b * b in fp32); groups are the connected components, labelled by their smallest body
// index.  fp32 subtraction is exactly antisymmetric, so d2(i, j) and d2(j, i) are bitwise equal and every unordered pair
// needs to be visited from one side only.
//
// Same machinery as the neighbour search (neighbors_sm100.cuh): the replicated AoSoA-128 body array is streamed through
// the cp.async.bulk + mbarrier pipeline, R targets per thread, two sources per packed f32x2 instruction; one pair costs
// 3 FADD2 + 1 FMUL2 + 2 FFMA2 and one threshold test on the bits of d2 (d2 >= 0 or NaN: its bits order like the float,
// NaN above +inf).  force_sm100.cuh is only included for its helpers; its code stays as it is.
//
// Each pair once, every tile the same work.  With nb = ceil(n / 128) source blocks, a target in block bt visits source
// block bs iff delta = (bs - bt) mod nb is in [1, nb / 2], or delta = 0 and j > i.  For two distinct blocks delta(a -> b) +
// delta(b -> a) = nb, so one of the two is at most nb / 2 and every pair is covered (pairs at exactly nb / 2 twice, which
// union tolerates).  Target r of a thread lies in block bt0 + r, so a tile streams the min(nb / 2 + R, nb) consecutive
// blocks bt0, bt0 + 1, ... (wrapping at nb) and at stream position pos target r has delta = (pos - r) mod nb: the
// predicate is uniform across the CTA, and only the R own blocks (pos == r: j > i) and the block that ends in padding
// (j < n) take the masked path.  Every tile, and so every shard, does the same work whatever slice it owns.
//
// Union-find (the ECL-CC / Jayanti-Tarjan lock-free scheme) on a forest parent[] with parent[x] <= x: find halves the
// path, union hooks the larger root under the smaller with one CAS and retries when another thread hooked it first.
// Every pointer goes to a smaller index, so a root is the smallest index of its tree, the roots after the last union are
// the component minima and the labels do not depend on the order in which the atomics land.  parent[] is read with
// relaxed device-scope atomics, never through the non-coherent path.  Each thread caches a node of each target's set
// (its last known root) and only calls union when find(j) differs from it, so a dense clump costs one find per linked
// pair rather than a CAS.
//
// Shape: 128 threads x R = 8 targets (1024-target tiles), 2-block stages, 3 stages.  -Xptxas -v: 101 registers, 0 spill
// bytes, so the 4 CTAs of 128 threads per SM that __launch_bounds__ asks for fit.
#pragma once
#include <cuda/atomic>

#include "force_sm100.cuh"

namespace b200nb {

constexpr int FOF_THREADS = 128, FOF_R = 8, FOF_TJB = 2, FOF_ST = 3, FOF_MINB = 4;
constexpr uint32_t FOF_TI = FOF_THREADS * FOF_R; // targets per tile: R consecutive AoSoA blocks
constexpr uint32_t FOF_MAX_CHUNKS = 64;
constexpr uint32_t FOF_MIN_CHUNK_BLKS = 16;      // a chunk streams at least 2048 sources (if there are that many)
constexpr uint32_t FOF_MASKED = 0xFFFFFFFFu;     // d2 bits of a masked lane: never below a threshold

struct FofArgs {
    const float *src;  // blocked bodies (the full replicated array)
    uint32_t *parent;  // this shard's forest
    uint32_t first;    // global index of the shard's first target (a multiple of BLK)
    uint32_t count;    // the shard's real targets; lanes past them are never linked
    uint32_t n;        // real bodies: lanes j >= n are padding
    uint32_t nb;       // ceil(n / BLK) source blocks
    uint32_t stream;   // blocks a tile streams: min(nb / 2 + R, nb)
    uint32_t n_chunks; // S: each CTA streams a contiguous part of the tile's blocks
    uint32_t thr;      // bits(b2) + 1: linked iff bits(d2) < thr
};

constexpr size_t fof_smem_bytes() { return (size_t)FOF_ST * (FOF_TJB * BLK_FLOATS * 4 + 8); }

// S for `tiles` tiles of `stream` blocks each, the rule of nb_chunks: CTAs run in rounds of `slots` (4 per SM), so among
// S0 = ceil(slots / tiles) .. 2 * S0 the S whose last round is fullest wins (the smallest on a tie).  No chunk shorter than
// FOF_MIN_CHUNK_BLKS blocks.  The labels do not depend on S.
inline uint32_t fof_chunks(uint32_t tiles, uint32_t stream, uint32_t slots)
{
    uint64_t lim = stream / FOF_MIN_CHUNK_BLKS;
    lim = lim < FOF_MAX_CHUNKS ? lim : FOF_MAX_CHUNKS;
    if (lim < 1) lim = 1;
    const uint64_t s0 = (slots + tiles - 1) / tiles;
    uint64_t best = 1;
    double best_fill = 0.0;
    for (uint64_t s = s0; s <= 2 * s0; ++s) {
        const uint64_t ss = s < lim ? s : lim, ctas = (uint64_t)tiles * ss;
        const double fill = (double)ctas / (double)(((ctas + slots - 1) / slots) * slots);
        if (fill > best_fill + 1e-9) {
            best_fill = fill;
            best = ss;
        }
    }
    return (uint32_t)best;
}

using fof_ref = cuda::atomic_ref<uint32_t, cuda::thread_scope_device>;

__device__ __forceinline__ uint32_t fof_load(uint32_t *p, uint32_t x) { return fof_ref(p[x]).load(cuda::memory_order_relaxed); }

// root of x, halving the path: every node passed on the way points to its grandparent afterwards.  The store is to a
// non-root (a root is only changed by union's CAS) and writes a smaller node of the same tree.
__device__ __forceinline__ uint32_t fof_find(uint32_t *p, uint32_t x)
{
    uint32_t px = fof_load(p, x);
    while (px != x) {
        const uint32_t gp = fof_load(p, px);
        if (gp == px) return px;
        fof_ref(p[x]).store(gp, cuda::memory_order_relaxed);
        x = gp;
        px = fof_load(p, x);
    }
    return x;
}

// join the sets of a and b; returns a node of the joined set (the root that survived the hook)
__device__ __forceinline__ uint32_t fof_union(uint32_t *p, uint32_t a, uint32_t b)
{
    for (;;) {
        a = fof_find(p, a);
        b = fof_find(p, b);
        if (a == b) return a;
        if (a > b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        uint32_t expect = b;
        if (fof_ref(p[b]).compare_exchange_strong(expect, a, cuda::memory_order_relaxed)) return a;
    }
}

// source j against every target r whose bits(d2) d[r] is below its threshold
template <int R>
__device__ __forceinline__ void fof_link(uint32_t *parent, uint32_t j, const uint32_t (&d)[R], const uint32_t (&thr)[R],
                                         uint32_t (&root)[R])
{
    uint32_t rj = FOF_MASKED;
#pragma unroll
    for (int r = 0; r < R; ++r)
        if (d[r] < thr[r]) {
            if (rj == FOF_MASKED) rj = fof_find(parent, j);
            if (rj != root[r]) rj = fof_union(parent, root[r], rj);
            root[r] = rj;
        }
}

// one AoSoA block (sources j0 + [0, 128)) against the R targets of this thread.  MASK: target `self_r` (tg0 + self_r *
// BLK) shares the block and only links sources j > its index; sources j >= n are padding.
template <int R, bool MASK>
__device__ __forceinline__ void fof_block(const float *__restrict__ sb, const float (&xi)[R], const float (&yi)[R],
                                          const float (&zi)[R], const uint32_t (&thr)[R], uint32_t (&root)[R],
                                          uint32_t *parent, uint32_t j0, uint32_t tg0, int self_r, uint32_t n)
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
            uint32_t d0[R], d1[R];
            bool hit = false;
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
                d0[r] = __float_as_uint(f0);
                d1[r] = __float_as_uint(f1);
                if (MASK) {
                    const uint32_t tg = tg0 + (uint32_t)r * BLK;
                    if (js >= n || (r == self_r && js <= tg)) d0[r] = FOF_MASKED;
                    if (js + 1 >= n || (r == self_r && js + 1 <= tg)) d1[r] = FOF_MASKED;
                }
                hit |= min(d0[r], d1[r]) < thr[r];
            }
            if (hit) {
                fof_link<R>(parent, js, d0, thr, root);
                fof_link<R>(parent, js + 1, d1, thr, root);
            }
        }
    }
}

// grid (ceil(count / FOF_TI), S): tile x links its targets first + x * FOF_TI + [0, FOF_TI) against its share of the
// tile's source stream, in the forest a.parent (initialised to parent[i] = i).
__global__ void __launch_bounds__(FOF_THREADS, FOF_MINB) fof_link_kernel(const FofArgs a)
{
    constexpr int R = FOF_R;
    constexpr int STAGE_FLOATS = FOF_TJB * BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)FOF_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint32_t p_begin = (uint32_t)(((uint64_t)a.stream * c) / a.n_chunks);
    const uint32_t p_end = (uint32_t)(((uint64_t)a.stream * (c + 1)) / a.n_chunks);
    const uint32_t nblk = p_end - p_begin;
    const uint32_t ntiles = (nblk + FOF_TJB - 1) / FOF_TJB;
    const uint32_t bt0 = a.first / BLK + blockIdx.x * R; // block of target r = 0; target r is in block bt0 + r
    auto src_block = [&](uint32_t pos) { // stream position -> source block, wrapping at nb (bt0 < nb, pos < nb)
        const uint32_t bs = bt0 + pos;
        return bs >= a.nb ? bs - a.nb : bs;
    };

    if (leader) {
#pragma unroll
        for (int s = 0; s < FOF_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) { // one copy per block: consecutive positions may wrap
        const uint32_t nb = min((uint32_t)FOF_TJB, nblk - tile * FOF_TJB);
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, nb * BLK_BYTES);
        for (uint32_t b = 0; b < nb; ++b)
            bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4) + b * BLK_BYTES,
                     a.src + (size_t)src_block(p_begin + tile * FOF_TJB + b) * BLK_FLOATS, BLK_BYTES, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < FOF_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    // targets past the shard's real bodies sit at NaN: their d2 is NaN and never below a threshold
    const uint32_t tg0 = bt0 * BLK + threadIdx.x;
    float xi[R], yi[R], zi[R];
    uint32_t root[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t g = tg0 + (uint32_t)r * BLK;
        const bool real = g < a.first + a.count;
        xi[r] = real ? __ldg(a.src + blk_index(g, 0)) : __int_as_float(0x7FFFFFFF);
        yi[r] = real ? __ldg(a.src + blk_index(g, 1)) : __int_as_float(0x7FFFFFFF);
        zi[r] = real ? __ldg(a.src + blk_index(g, 2)) : __int_as_float(0x7FFFFFFF);
        root[r] = g;
    }
    const uint32_t half = a.nb / 2;
    const uint32_t pad_blk = (a.n % BLK) ? a.nb - 1 : 0xFFFFFFFFu;

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % FOF_ST;
        mbar_wait(bar0 + 8 * s, (t / FOF_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)FOF_TJB, nblk - t * FOF_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t pos = p_begin + t * FOF_TJB + b, bs = src_block(pos);
            uint32_t thr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) { // delta = (pos - r) mod nb; targets r >= nb are never real
                const uint32_t delta = pos >= (uint32_t)r ? pos - r : pos + a.nb - r;
                thr[r] = delta <= half ? a.thr : 0u;
            }
            if (pos < (uint32_t)R || bs == pad_blk)
                fof_block<R, true>(sb + b * BLK_FLOATS, xi, yi, zi, thr, root, a.parent, bs * BLK, tg0, (int)pos, a.n);
            else
                fof_block<R, false>(sb + b * BLK_FLOATS, xi, yi, zi, thr, root, a.parent, bs * BLK, tg0, R, a.n);
        }
        if (t + FOF_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + FOF_ST, s);
        }
    }
}

// parent[x] = x for x < count
__global__ void __launch_bounds__(256) fof_init_kernel(uint32_t *__restrict__ parent, uint32_t count)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < count) parent[x] = x;
}

// Fold the forests[1 .. n_forests) (stride `stride` entries) into forests[0]: x and parent_p[x] are in the same set of
// forest p, so union(x, parent_p[x]) over every x carries all of its connectivity over.
__global__ void __launch_bounds__(256) fof_merge_kernel(uint32_t *forests, uint32_t n_forests, size_t stride, uint32_t n)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    for (uint32_t p = 1; p < n_forests; ++p) {
        const uint32_t y = forests[p * stride + x];
        if (y != x) fof_union(forests, x, y);
    }
}

// parent[x] = root of x = the smallest index of its group.  Reads only on the way up: a thread stores only its own
// entry, and only the root, so every entry read by another thread is still a node of the same tree.
__global__ void __launch_bounds__(256) fof_finalize_kernel(uint32_t *parent, uint32_t n)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    uint32_t r = x, q;
    while ((q = fof_load(parent, r)) != r) r = q;
    fof_ref(parent[x]).store(r, cuda::memory_order_relaxed);
}

} // namespace b200nb
