// Phase-space friends-of-friends groups of the bodies for sm_100a.
//
// Definition (include/b200nb.h): with s_x = 1 / b_x and s_v = 1 / b_v (fp32, correctly rounded; b = +inf gives 0), the
// scaled coordinates are X = fl(x * s_x), Y, Z and U = fl(v_x * s_v), V, W.  Bodies i != j are linked iff the fp32
// d2 = fma(dW, dW, fma(dV, dV, fma(dU, dU, fma(dZ, dZ, fma(dY, dY, dX * dX))))), d = scaled j - scaled i, satisfies
// d2 <= 1.  fp32 subtraction is exactly antisymmetric, so d2(i, j) and d2(j, i) are bitwise equal and the pair-once
// scheme of fof_sm100.cuh holds unchanged; groups are labelled by their smallest body index.
//
// The scaled coordinates are packed once per call (phase_fof_pack_kernel) into a 6-float AoSoA-128 array, X | Y | Z | U
// | V | W per block (3 KiB), which the placement replicates like the body array.  phase_fof_link_kernel is
// fof_link_kernel with six coordinates: the same cp.async.bulk + mbarrier ring, the same stream of min(nb / 2 + R, nb)
// blocks per tile with only the R own blocks and the padding block on the masked path, R targets per thread and two
// sources per packed f32x2 instruction.  One source pair costs 6 FADD2 + 1 FMUL2 + 5 FFMA2 and the threshold test on
// the bits of d2 (d2 >= 0 or NaN: its bits order like the float, NaN above +inf), against bits(1.0f) + 1.  The forest,
// union-find, merge, finalize and chunk rule are fof_sm100.cuh's, used as they are; that file stays as it is.
//
// Shape: FoF's, 128 threads x R = 8 targets, 2-block stages (6 KiB), 3 stages, 4 CTAs/SM.  Six coordinates per target
// double the target registers of position FoF (101 registers); it still fits under the 128-register cap, so no other
// shape was needed.  -Xptxas -v (CUDA 12.9, sm_100a) and tools/phase_fof_bench.py at N = 200k on a B200 at 1000 W:
//   R   CTAs/SM   registers   spills   sparse setting, galaxy / random
//   8   4         117         0        2222 / 2272 G-pairs/s (profiles/phase_fof_bench_1gpu_200k.json)
#pragma once
#include "fof_sm100.cuh"

namespace b200nb {

constexpr int PF_THREADS = 128, PF_R = 8, PF_TJB = 2, PF_ST = 3, PF_MINB = 4;
constexpr uint32_t PF_TI = PF_THREADS * PF_R;  // targets per tile: R consecutive AoSoA blocks
constexpr int PF_BLK_FLOATS = 6 * BLK;         // X | Y | Z | U | V | W
constexpr int PF_BLK_BYTES = PF_BLK_FLOATS * 4;
constexpr uint32_t PF_THR = 0x3F800001u;       // bits(1.0f) + 1: linked iff bits(d2) < PF_THR

struct PhaseFofArgs {
    const float *src;  // the replicated 6-float AoSoA array of every body
    uint32_t *parent;  // this shard's forest
    uint32_t first;    // global index of the shard's first target (a multiple of BLK)
    uint32_t count;    // the shard's real targets; lanes past them are never linked
    uint32_t n;        // real bodies: lanes j >= n are padding
    uint32_t nb;       // ceil(n / BLK) source blocks
    uint32_t stream;   // blocks a tile streams: min(nb / 2 + R, nb)
    uint32_t n_chunks; // S: each CTA streams a contiguous part of the tile's blocks (fof_chunks)
};

constexpr size_t phase_fof_smem_bytes() { return (size_t)PF_ST * (PF_TJB * PF_BLK_FLOATS * 4 + 8); }

// float index of scaled coordinate `comp` (0..5 = X Y Z U V W) of body i in the 6-float array
__host__ __device__ __forceinline__ size_t pf_index(size_t i, int comp)
{
    return (i / BLK) * (size_t)PF_BLK_FLOATS + (size_t)comp * BLK + (i % BLK);
}

// The shard's slice [first, first + L) of the 6-float array: positions from the blocked body array, velocities from the
// shard's own [3][L] rows.  Lanes past the n_local real bodies are 0 (padding: never linked).
__global__ void __launch_bounds__(256) phase_fof_pack_kernel(const float *__restrict__ bodies, const float *__restrict__ vel,
                                                             float *__restrict__ dst, uint32_t first, uint32_t L,
                                                             uint32_t n_local, float sx, float sv)
{
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= L) return;
    const size_t g = (size_t)first + li;
    const bool real = li < n_local;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        dst[pf_index(g, k)] = real ? __fmul_rn(bodies[blk_index(g, k)], sx) : 0.f;
        dst[pf_index(g, 3 + k)] = real ? __fmul_rn(vel[(size_t)k * L + li], sv) : 0.f;
    }
}

// one AoSoA block (sources j0 + [0, 128)) against the R targets of this thread; MASK as in fof_block
template <int R, bool MASK>
__device__ __forceinline__ void phase_fof_block(const float *__restrict__ sb, const float (&ti)[6][R],
                                                const uint32_t (&thr)[R], uint32_t (&root)[R], uint32_t *parent,
                                                uint32_t j0, uint32_t tg0, int self_r, uint32_t n)
{
#pragma unroll 1
    for (int j = 0; j < BLK; j += 4) {
        uint64_t s[6][2];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const float4 v = *reinterpret_cast<const float4 *>(sb + k * BLK + j);
            s[k][0] = pk2(v.x, v.y);
            s[k][1] = pk2(v.z, v.w);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t js = j0 + (uint32_t)(j + 2 * h);
            uint32_t d0[R], d1[R];
            bool hit = false;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t dx = sub2(s[0][h], pk2(ti[0][r], ti[0][r]));
                const uint64_t dy = sub2(s[1][h], pk2(ti[1][r], ti[1][r]));
                const uint64_t dz = sub2(s[2][h], pk2(ti[2][r], ti[2][r]));
                const uint64_t du = sub2(s[3][h], pk2(ti[3][r], ti[3][r]));
                const uint64_t dv = sub2(s[4][h], pk2(ti[4][r], ti[4][r]));
                const uint64_t dw = sub2(s[5][h], pk2(ti[5][r], ti[5][r]));
                uint64_t d = mul2(dx, dx);
                d = fma2(dy, dy, d);
                d = fma2(dz, dz, d);
                d = fma2(du, du, d);
                d = fma2(dv, dv, d);
                d = fma2(dw, dw, d);
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

// grid (ceil(count / PF_TI), S): tile x links its targets first + x * PF_TI + [0, PF_TI) against its share of the
// tile's source stream, in the forest a.parent (initialised to parent[i] = i).  fof_link_kernel with six coordinates.
__global__ void __launch_bounds__(PF_THREADS, PF_MINB) phase_fof_link_kernel(const PhaseFofArgs a)
{
    constexpr int R = PF_R;
    constexpr int STAGE_FLOATS = PF_TJB * PF_BLK_FLOATS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *stages = reinterpret_cast<float *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)PF_ST * STAGE_FLOATS * 4);
    const bool leader = threadIdx.x == 0;
    const uint32_t stages_u32 = smem_u32(stages);
    const uint32_t bar0 = smem_u32(bars);

    const uint32_t c = blockIdx.y;
    const uint32_t p_begin = (uint32_t)(((uint64_t)a.stream * c) / a.n_chunks);
    const uint32_t p_end = (uint32_t)(((uint64_t)a.stream * (c + 1)) / a.n_chunks);
    const uint32_t nblk = p_end - p_begin;
    const uint32_t ntiles = (nblk + PF_TJB - 1) / PF_TJB;
    const uint32_t bt0 = a.first / BLK + blockIdx.x * R; // block of target r = 0; target r is in block bt0 + r
    auto src_block = [&](uint32_t pos) { // stream position -> source block, wrapping at nb (bt0 < nb, pos < nb)
        const uint32_t bs = bt0 + pos;
        return bs >= a.nb ? bs - a.nb : bs;
    };

    if (leader) {
#pragma unroll
        for (int s = 0; s < PF_ST; ++s) mbar_init(bar0 + 8 * s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](uint32_t tile, uint32_t stage) { // one copy per block: consecutive positions may wrap
        const uint32_t nb = min((uint32_t)PF_TJB, nblk - tile * PF_TJB);
        const uint32_t bar = bar0 + 8 * stage;
        mbar_arrive_expect_tx(bar, nb * PF_BLK_BYTES);
        for (uint32_t b = 0; b < nb; ++b)
            bulk_g2s(stages_u32 + stage * (STAGE_FLOATS * 4) + b * PF_BLK_BYTES,
                     a.src + (size_t)src_block(p_begin + tile * PF_TJB + b) * PF_BLK_FLOATS, PF_BLK_BYTES, bar);
    };
    if (leader) {
#pragma unroll
        for (int s = 0; s < PF_ST; ++s)
            if ((uint32_t)s < ntiles) issue(s, s);
    }

    // targets past the shard's real bodies sit at NaN: their d2 is NaN and never below the threshold
    const uint32_t tg0 = bt0 * BLK + threadIdx.x;
    float ti[6][R];
    uint32_t root[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t g = tg0 + (uint32_t)r * BLK;
        const bool real = g < a.first + a.count;
#pragma unroll
        for (int k = 0; k < 6; ++k) ti[k][r] = real ? __ldg(a.src + pf_index(g, k)) : __int_as_float(0x7FFFFFFF);
        root[r] = g;
    }
    const uint32_t half = a.nb / 2;
    const uint32_t pad_blk = (a.n % BLK) ? a.nb - 1 : 0xFFFFFFFFu;

    for (uint32_t t = 0; t < ntiles; ++t) {
        const uint32_t s = t % PF_ST;
        mbar_wait(bar0 + 8 * s, (t / PF_ST) & 1u);
        const float *sb = stages + (size_t)s * STAGE_FLOATS;
        const uint32_t nb = min((uint32_t)PF_TJB, nblk - t * PF_TJB);
        for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t pos = p_begin + t * PF_TJB + b, bs = src_block(pos);
            uint32_t thr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) { // delta = (pos - r) mod nb; targets r >= nb are never real
                const uint32_t delta = pos >= (uint32_t)r ? pos - r : pos + a.nb - r;
                thr[r] = delta <= half ? PF_THR : 0u;
            }
            if (pos < (uint32_t)R || bs == pad_blk)
                phase_fof_block<R, true>(sb + b * PF_BLK_FLOATS, ti, thr, root, a.parent, bs * BLK, tg0, (int)pos, a.n);
            else
                phase_fof_block<R, false>(sb + b * PF_BLK_FLOATS, ti, thr, root, a.parent, bs * BLK, tg0, R, a.n);
        }
        if (t + PF_ST < ntiles) { // refill the stage just drained
            __syncthreads();
            if (leader) issue(t + PF_ST, s);
        }
    }
}

} // namespace b200nb
