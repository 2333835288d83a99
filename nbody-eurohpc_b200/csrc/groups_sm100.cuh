// Self-potential of body groups and unbinding, for sm_100a.
//
// Definition (include/b200nb.h): for a body i with label g != NO_GROUP,
//   phi^g_i = -sum_{j != i, group[j] = g} G m_j / (|r_ij|^2 + soft^2)^(1/2),
// with the G*m fold, softening, fp32 pair terms and fp64 second-level sums of field_sm100.cuh.
//
// Member order.  The bodies of every label except NO_GROUP are sorted by (label, index) (CUB's stable radix sort of the
// labels with the indices as values) and packed in that order into an AoSoA-128 source array (x, y, z, G*m) read from
// the replicated blocked body array.  A label's members are then one range [lo, hi) of sorted positions, and a tile of
// sorted targets only has to stream the union of its targets' ranges: a tile inside one big group streams that group,
// a tile across many small groups streams them all (at most ~TI extra sources per target).
//
// Potential kernel: the field_kernel skeleton (cp.async.bulk + mbarrier ring, R targets per thread, two sources per
// packed f32x2 instruction), with a potential-only pair: 3 FADD2 + 3 FFMA2 for d^2, 2 MUFU.RSQ, one FFMA2 of G*m*inv
// into the accumulator.  Lanes outside a target's range, and its own lane, get inv = 0 after the math (fma(g, 0, acc) ==
// acc; a NaN of another group cannot leak).  Only blocks that are not inside every target's range, or that hold the
// tile's own targets, take that masked path; in-range lanes compute the same FFMA2 on both paths.
//
// Determinism.  Source chunks are cut at absolute block positions of the sorted array, gp_chunk_blks(M) blocks each, a
// function of the member count M alone.  A target's chunk row is the fp64 sum, in block order, of per-block fp32 sums in
// which lanes outside its range add exactly zero, so it does not depend on which tile, batch or shard the target lands
// in, nor on which of the tile's blocks were streamed.  group_reduce_kernel sums the target's own chunks in fp64 in
// chunk order.  The unbinding step (frame velocities, energies, flags, stable compaction) runs identically on every
// device on identical inputs.
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include "force_sm100.cuh"

namespace b200nb {

constexpr uint32_t GP_NONE = 0xFFFFFFFFu; // B200NB_NO_GROUP

// Shape: 128 threads x R = 8 targets (1024-target tiles), 2-block stages, 3 stages, 4 CTAs per SM (-Xptxas -v: 127
// registers, 0 spill bytes).  Measured on a B200 (1000 W, N = 200k, one label): 3911 G-pairs/s, 1.33x the force pass's
// interactions/s in the same run (profiles/groups_bench_1gpu_200k.json).  No other shape was measured.
constexpr int GP_THREADS = 128, GP_R = 8, GP_TJB = 2, GP_ST = 3, GP_MINB = 4;
constexpr uint32_t GP_TI = GP_THREADS * GP_R;  // targets per CTA tile
constexpr uint32_t GP_MIN_CHUNK_BLKS = 16;     // a chunk streams at least 2048 sources (if there are that many)
constexpr uint32_t GP_MAX_CHUNKS = 64;
constexpr uint32_t GP_BATCH = 256 * GP_TI;     // targets per launch: bounds the [chunks][batch] partial rows (64 MiB)
constexpr uint32_t GP_PIECE = 256;             // sorted positions per thread of the frame-velocity sums
static_assert(GP_TI % BLK == 0, "target tile must cover whole blocks");

// blocks per source chunk for M members: a function of M alone (see the determinism note above)
__host__ __device__ inline uint32_t gp_chunk_blks(uint32_t m)
{
    const uint32_t nblk = (m + BLK - 1) / BLK;
    uint32_t s = (nblk + GP_MIN_CHUNK_BLKS - 1) / GP_MIN_CHUNK_BLKS;
    s = s < 1 ? 1 : (s > GP_MAX_CHUNKS ? GP_MAX_CHUNKS : s);
    const uint32_t cb = (nblk + s - 1) / s;
    return cb < 1 ? 1 : cb;
}

struct GpArgs {
    const float *src;        // members in sorted order, AoSoA-128 (x, y, z, G*m); G*m = 0 past the last member
    const uint32_t *lo, *hi; // per sorted position: the range [lo, hi) of its label
    float *partial;          // [chunk][stride]: per-chunk sums of G*m*inv
    uint32_t stride;         // floats per chunk row: the batch, a multiple of GP_TI
    uint32_t t0;             // sorted position of this launch's first target (a multiple of GP_TI)
    uint32_t count;          // targets of this launch; threads of the last tile past it re-read the last target
    uint32_t cb;             // gp_chunk_blks(M)
    float soft2;
};

constexpr size_t gp_smem_bytes() { return (size_t)GP_ST * (GP_TJB * BLK_BYTES + 8); }

// one AoSoA block (sorted positions j0 + [0, 128)) against the R targets of this thread.  MASK: lane j counts for target
// k iff tlo[k] <= j < thi[k] and j != tp[k]; the others get inv = 0.
template <bool MASK>
__device__ __forceinline__ void gp_block(const float *__restrict__ sb, const float (&xi)[GP_R], const float (&yi)[GP_R],
                                         const float (&zi)[GP_R], uint64_t soft2p, uint64_t (&acc)[GP_R], uint32_t j0,
                                         const uint32_t (&tp)[GP_R], const uint32_t (&tlo)[GP_R], const uint32_t (&thi)[GP_R])
{
#pragma unroll 1
    for (int j = 0; j < BLK; j += 4) {
        const float4 xv = *reinterpret_cast<const float4 *>(sb + j);
        const float4 yv = *reinterpret_cast<const float4 *>(sb + BLK + j);
        const float4 zv = *reinterpret_cast<const float4 *>(sb + 2 * BLK + j);
        const float4 gv = *reinterpret_cast<const float4 *>(sb + 3 * BLK + j);
        const uint64_t sx[2] = {pk2(xv.x, xv.y), pk2(xv.z, xv.w)};
        const uint64_t sy[2] = {pk2(yv.x, yv.y), pk2(yv.z, yv.w)};
        const uint64_t sz[2] = {pk2(zv.x, zv.y), pk2(zv.z, zv.w)};
        const uint64_t sg[2] = {pk2(gv.x, gv.y), pk2(gv.z, gv.w)};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
            for (int k = 0; k < GP_R; ++k) {
                const uint64_t dx = sub2(sx[h], pk2(xi[k], xi[k]));
                const uint64_t dy = sub2(sy[h], pk2(yi[k], yi[k]));
                const uint64_t dz = sub2(sz[h], pk2(zi[k], zi[k]));
                uint64_t d = fma2(dx, dx, soft2p);
                d = fma2(dy, dy, d);
                d = fma2(dz, dz, d);
                float d0, d1;
                upk2(d, d0, d1);
                float i0 = rsqrt_approx(d0), i1 = rsqrt_approx(d1);
                if (MASK) {
                    const uint32_t js = j0 + (uint32_t)(j + 2 * h);
                    if (!(js >= tlo[k] && js < thi[k] && js != tp[k])) i0 = 0.f;
                    if (!(js + 1 >= tlo[k] && js + 1 < thi[k] && js + 1 != tp[k])) i1 = 0.f;
                }
                acc[k] = fma2(sg[h], pk2(i0, i1), acc[k]);
            }
        }
    }
}

// grid (ceil(count / GP_TI), chunks of M).  CTA (x, c) streams the blocks of chunk c that intersect the union of its
// targets' ranges and writes their chunk-c sums; a CTA whose chunk misses that union returns at once.
__global__ void __launch_bounds__(GP_THREADS, GP_MINB) group_potential_kernel(const GpArgs a)
{
    constexpr int STAGE_FLOATS = GP_TJB * BLK_FLOATS;
    const uint32_t p0 = a.t0 + blockIdx.x * GP_TI;
    const uint32_t plast = a.t0 + min((blockIdx.x + 1) * GP_TI, a.count) - 1;
    const uint32_t ulo = __ldg(a.lo + p0), uhi = __ldg(a.hi + plast); // union of the tile's ranges (sorted targets)
    const uint32_t ilo = __ldg(a.lo + plast), ihi = __ldg(a.hi + p0); // their intersection (empty unless one label)
    const uint32_t c = blockIdx.y;
    const uint32_t b_begin = max(c * a.cb, ulo / BLK);
    const uint32_t b_end = min((c + 1) * a.cb, (uhi - 1) / BLK + 1);
    if (b_begin >= b_end) return; // uniform over the CTA, before any barrier
    const uint32_t nblk = b_end - b_begin;
    const uint32_t ntiles = (nblk + GP_TJB - 1) / GP_TJB;
    const float *chunk_src = a.src + (size_t)b_begin * BLK_FLOATS;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)GP_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);
    if (leader) {
#pragma unroll
        for (int s = 0; s < GP_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) {
        const uint32_t nb = min((uint32_t)GP_TJB, nblk - tile * GP_TJB);
        const uint32_t bytes = nb * BLK_BYTES;
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4), chunk_src + (size_t)tile * STAGE_FLOATS, bytes, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < GP_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    float xi[GP_R], yi[GP_R], zi[GP_R];
    uint32_t tp[GP_R], tlo[GP_R], thi[GP_R];
#pragma unroll
    for (int k = 0; k < GP_R; ++k) {
        const uint32_t il = min((uint32_t)(blockIdx.x * GP_TI + k * GP_THREADS + threadIdx.x), a.count - 1);
        const uint32_t p = a.t0 + il;
        tp[k] = p;
        tlo[k] = __ldg(a.lo + p);
        thi[k] = __ldg(a.hi + p);
        xi[k] = __ldg(a.src + blk_index(p, 0));
        yi[k] = __ldg(a.src + blk_index(p, 1));
        zi[k] = __ldg(a.src + blk_index(p, 2));
    }
    const uint32_t tb0 = p0 / BLK, tb1 = plast / BLK; // blocks that hold the tile's own targets

    double m[GP_R];
#pragma unroll
    for (int k = 0; k < GP_R; ++k) m[k] = 0.0;
    const uint64_t soft2p = pk2(a.soft2, a.soft2);

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % GP_ST;
        mbar_wait(bar0 + 8 * s, (t / GP_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)GP_TJB, nblk - t * GP_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            uint64_t acc[GP_R];
#pragma unroll
            for (int k = 0; k < GP_R; ++k) acc[k] = 0ull;
            const uint32_t gb = b_begin + t * GP_TJB + b;
            const bool masked = (gb >= tb0 && gb <= tb1) || gb * BLK < ilo || (gb + 1) * BLK > ihi;
            if (masked)
                gp_block<true>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tp, tlo, thi);
            else
                gp_block<false>(sb + b * BLK_FLOATS, xi, yi, zi, soft2p, acc, gb * BLK, tp, tlo, thi);
            // every block (64 terms per lane) folds into fp64, as in field_kernel
#pragma unroll
            for (int k = 0; k < GP_R; ++k) {
                float lo, hi;
                upk2(acc[k], lo, hi);
                m[k] += (double)(lo + hi);
            }
        }
        if (t + GP_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + GP_ST, s);
        }
    }
#pragma unroll
    for (int k = 0; k < GP_R; ++k) {
        const size_t il = (size_t)blockIdx.x * GP_TI + (size_t)k * GP_THREADS + threadIdx.x;
        a.partial[(size_t)c * a.stride + il] = (float)m[k];
    }
}

// phi[t0 + i] = -(fixed-order fp64 sum of the target's own chunk rows), +0 when nothing was summed
__global__ void __launch_bounds__(256) group_reduce_kernel(const float *__restrict__ partial, uint32_t stride, uint32_t t0,
                                                           uint32_t count, uint32_t cb, const uint32_t *__restrict__ lo,
                                                           const uint32_t *__restrict__ hi, float *__restrict__ phi)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t p = t0 + i, span = cb * BLK;
    const uint32_t c0 = lo[p] / span, c1 = (hi[p] - 1) / span;
    double s = 0.0;
    for (uint32_t c = c0; c <= c1; ++c) s += (double)partial[(size_t)c * stride + i];
    phi[p] = (float)(0.0 - s);
}

// ------------------------------------------------------------------------------------------------ member set
__global__ void __launch_bounds__(256) gp_iota_kernel(uint32_t *__restrict__ v, uint32_t n)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = i;
}

// mem[p] = (label << 32) | index from the sorted (label, index) pairs; info[0] = M, the members before the first
// NO_GROUP label (info[0] must be 0 beforehand: nobody writes it when there is no member)
__global__ void __launch_bounds__(256) gp_members_kernel(const uint32_t *__restrict__ key, const uint32_t *__restrict__ val,
                                                         uint32_t n, uint64_t *__restrict__ mem, uint32_t *__restrict__ info)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t k = key[p];
    mem[p] = ((uint64_t)k << 32) | val[p];
    if (k != GP_NONE && (p + 1 == n || key[p + 1] == GP_NONE)) info[0] = p + 1;
}

__device__ __forceinline__ uint32_t gp_lower_bound(const uint64_t *mem, uint32_t lo, uint32_t hi, uint64_t key)
{
    while (lo < hi) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (mem[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// For the info[0] = M members of mem: the packed sources (positions up to the end of the last block; G*m = 0 past M)
// and every member's label range.  Grid over `bound` >= M positions.
__global__ void __launch_bounds__(256) gp_pack_kernel(const float *__restrict__ bodies, const uint64_t *__restrict__ mem,
                                                      const uint32_t *__restrict__ info, uint32_t bound, float *__restrict__ src,
                                                      uint32_t *__restrict__ lo, uint32_t *__restrict__ hi)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t M = info[0];
    if (p >= bound || p >= (M + BLK - 1) / BLK * BLK) return;
    if (p >= M) {
        for (int q = 0; q < 4; ++q) src[blk_index(p, q)] = 0.f;
        return;
    }
    const uint64_t e = mem[p];
    const uint32_t idx = (uint32_t)e;
    for (int q = 0; q < 4; ++q) src[blk_index(p, q)] = __ldg(bodies + blk_index(idx, q));
    const uint64_t lab = e >> 32;
    lo[p] = gp_lower_bound(mem, 0, p, lab << 32);
    hi[p] = gp_lower_bound(mem, p + 1, M, (lab + 1) << 32);
}

// Cost split of the info[0] = M members' tiles over P shards: split[k] (info[1 + k]) is the first tile of shard k.  A
// tile's cost is the number of source blocks it streams; tile t goes to shard floor(P * cost before t / total).  One
// CTA, a fixed partition of the tiles over its threads: the split is a pure function of the ranges.
constexpr int GP_SPLIT_THREADS = 1024;
__global__ void __launch_bounds__(GP_SPLIT_THREADS) gp_split_kernel(const uint32_t *__restrict__ lo, const uint32_t *__restrict__ hi,
                                                                    uint32_t *__restrict__ info, uint32_t P)
{
    __shared__ unsigned long long part[GP_SPLIT_THREADS], total_s;
    const uint32_t M = info[0];
    const uint32_t T = (M + GP_TI - 1) / GP_TI;
    uint32_t *split = info + 1;
    auto cost = [&](uint32_t t) -> uint64_t {
        const uint32_t a = t * GP_TI, b = min(a + GP_TI, M) - 1;
        return (uint64_t)((hi[b] - 1) / BLK - lo[a] / BLK + 1);
    };
    const uint32_t tid = threadIdx.x;
    const uint32_t ta = (uint32_t)((uint64_t)T * tid / GP_SPLIT_THREADS), tb = (uint32_t)((uint64_t)T * (tid + 1) / GP_SPLIT_THREADS);
    uint64_t mine = 0;
    for (uint32_t t = ta; t < tb; ++t) mine += cost(t);
    part[tid] = mine;
    for (uint32_t k = tid; k <= P; k += GP_SPLIT_THREADS) split[k] = k == 0 ? 0u : T;
    __syncthreads();
    if (tid == 0) { // exclusive prefix over the threads, in order
        uint64_t run = 0;
        for (int i = 0; i < GP_SPLIT_THREADS; ++i) {
            const uint64_t v = part[i];
            part[i] = run;
            run += v;
        }
        total_s = run;
    }
    __syncthreads();
    const uint64_t total = total_s;
    uint64_t before = part[tid];
    if (total == 0) return;
    auto shard_of = [&](uint64_t b) { const uint64_t s = b * P / total; return (uint32_t)(s < P - 1 ? s : P - 1); };
    uint32_t prev = ta == 0 ? 0u : shard_of(before - cost(ta - 1));
    for (uint32_t t = ta; t < tb; ++t) {
        const uint32_t sh = shard_of(before);
        for (uint32_t k = prev + 1; k <= sh; ++k) split[k] = t;
        prev = sh;
        before += cost(t);
    }
}

// ------------------------------------------------------------------------------------------------ unbinding step
struct alignas(32) GpSum {
    double m, x, y, z;
};

// velocity component q (3: mass) of body i from the gathered [P][4][L] array
__device__ __forceinline__ float gp_vm(const float *vm, uint32_t L, uint32_t i, int q)
{
    return __ldg(vm + ((size_t)(i / L) * 4 + q) * L + i % L);
}

// Thread k sums (m, m vx, m vy, m vz) in fp64 over sorted positions [k * GP_PIECE, (k + 1) * GP_PIECE) in order, one sum
// per label piece, stored at the piece's first position.  A label's pieces start at its first position and at every
// multiple of GP_PIECE inside its range.
__global__ void __launch_bounds__(256) gp_piece_kernel(const uint64_t *__restrict__ mem, const uint32_t *__restrict__ info,
                                                       const float *__restrict__ vm, uint32_t L, GpSum *__restrict__ piece)
{
    const uint32_t M = info[0];
    const uint32_t p0 = (blockIdx.x * blockDim.x + threadIdx.x) * GP_PIECE;
    if (p0 >= M) return;
    const uint32_t p1 = min(p0 + GP_PIECE, M);
    uint32_t q = p0;
    uint64_t lab = mem[p0] >> 32;
    GpSum s{0.0, 0.0, 0.0, 0.0};
    for (uint32_t p = p0; p < p1; ++p) {
        const uint64_t e = mem[p];
        if (e >> 32 != lab) {
            piece[q] = s;
            q = p;
            lab = e >> 32;
            s = GpSum{0.0, 0.0, 0.0, 0.0};
        }
        const uint32_t i = (uint32_t)e;
        const double mi = gp_vm(vm, L, i, 3);
        s.m += mi;
        s.x += mi * gp_vm(vm, L, i, 0);
        s.y += mi * gp_vm(vm, L, i, 1);
        s.z += mi * gp_vm(vm, L, i, 2);
    }
    piece[q] = s;
}

// At every label's first position: V = sum m v / sum m over its pieces in order (0 when the mass is 0), stored over the
// first piece's (x, y, z).
__global__ void __launch_bounds__(256) gp_frame_kernel(const uint32_t *__restrict__ lo, const uint32_t *__restrict__ hi,
                                                       const uint32_t *__restrict__ info, GpSum *__restrict__ piece)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= info[0] || lo[p] != p) return;
    const uint32_t e = hi[p];
    GpSum s = piece[p];
    for (uint32_t q = (p / GP_PIECE + 1) * GP_PIECE; q < e; q += GP_PIECE) {
        const GpSum t = piece[q];
        s.m += t.m;
        s.x += t.x;
        s.y += t.y;
        s.z += t.z;
    }
    const bool has = s.m != 0.0;
    piece[p] = GpSum{s.m, has ? s.x / s.m : 0.0, has ? s.y / s.m : 0.0, has ? s.z / s.m : 0.0};
}

// Member p of the current set: phi_out[i] = phi[p]; with vm (unbinding), E = |v - V|^2 / 2 + phi in fp64, stays iff
// E < 0: flags[p], bound[i] = label or NO_GROUP.
__global__ void __launch_bounds__(256) gp_finish_kernel(const uint64_t *__restrict__ mem, const uint32_t *__restrict__ info,
                                                        const uint32_t *__restrict__ lo, const float *__restrict__ vm, uint32_t L,
                                                        const GpSum *__restrict__ piece, const float *__restrict__ phi,
                                                        unsigned char *__restrict__ flags, uint32_t *__restrict__ bound,
                                                        float *__restrict__ phi_out)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= info[0]) return;
    const uint64_t e = mem[p];
    const uint32_t i = (uint32_t)e;
    phi_out[i] = phi[p];
    if (!vm) return;
    const GpSum V = piece[lo[p]];
    const double dx = (double)gp_vm(vm, L, i, 0) - V.x, dy = (double)gp_vm(vm, L, i, 1) - V.y,
                 dz = (double)gp_vm(vm, L, i, 2) - V.z;
    const double E = 0.5 * (dx * dx + dy * dy + dz * dz) + (double)phi[p];
    const bool stays = E < 0.0;
    flags[p] = stays;
    bound[i] = stays ? (uint32_t)(e >> 32) : GP_NONE;
}

} // namespace b200nb
