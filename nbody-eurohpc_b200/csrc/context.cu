// libb200nb: context, sharding, streams/events, NCCL exchange and the C ABI declared in include/b200nb.h.
//
// One context drives one or more "shards" (one per GPU).  A shard owns a contiguous range of L targets and keeps
//   bodies  : the FULL system as AoSoA blocks (positions + G*m), 16 B/body, replicated on every GPU
//   vel/acc : SoA [3][L] for its own targets,  mass [L],  partial [S][3][L] chunk partial sums
// State replication + target sharding is the reference's only distributed strategy
// (src/murb/implem/SimulationNBodyMultiNode.cpp:76-148: MPI_Allgatherv of qx,qy,qz,m then of ax,ay,az); here the
// exchange is ONE in-place ncclAllGather of the blocked slice per step on a communication stream, overlapped with
// the force pass over the rank's own (already resident) source chunks, and no acceleration gather at all because
// every GPU integrates only its own targets.
#include <cuda.h>
#include <dlfcn.h>
#include <nccl.h>

#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200nb.h"
#include "field_sm100.cuh"
#include "neighbors_sm100.cuh"
#include "fof_sm100.cuh"
#include "phase_fof_sm100.cuh"
#include "groups_sm100.cuh"
#include "tracers_sm100.cuh"
#include "tidal_sm100.cuh"
#include "components_sm100.cuh"
#include "integrate_sm100.cuh"
#include "external_sm100.cuh"
#include "scf_sm100.cuh"
#include "plan.hpp"
// The default force-kernel variant once more, as a cubin whose hot loop has been re-ordered after ptxas by
// tools/sass_resched.py (same instructions, same registers, same arithmetic: bit-identical results, ~5 % faster; the
// order was found with the GPU as the cost function and is kept in csrc/resched/*.order.json).  Generated at build time;
// the array is empty when this compiler's loop is not the one the order was derived from.
#include "generated/force_resched_cubin.inc"

using namespace b200nb;

namespace {

// ------------------------------------------------------------------------------------------------ NCCL (lazy)
// Loaded with dlopen only when more than one rank is requested, so single-GPU use has no NCCL dependency.
struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
    bool load()
    {
        if (handle) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) { err = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return false; }
#define LOADSYM(field, sym)                                                                                            \
    field = reinterpret_cast<decltype(field)>(dlsym(handle, sym));                                                     \
    if (!field) { err = std::string("missing NCCL symbol ") + sym; return false; }
        LOADSYM(GetUniqueId, "ncclGetUniqueId");
        LOADSYM(CommInitRank, "ncclCommInitRank");
        LOADSYM(CommDestroy, "ncclCommDestroy");
        LOADSYM(GroupStart, "ncclGroupStart");
        LOADSYM(GroupEnd, "ncclGroupEnd");
        LOADSYM(AllGather, "ncclAllGather");
        LOADSYM(AllReduce, "ncclAllReduce");
        LOADSYM(GetErrorString, "ncclGetErrorString");
#undef LOADSYM
        return true;
    }
};
NcclApi g_nccl;
thread_local std::string g_create_error;

// ------------------------------------------------------------------------------------------------ driver API (lazy)
// Only used to load and launch the re-ordered cubin; resolved with dlopen so the library links against cudart alone.
struct DriverApi {
    void *handle = nullptr;
    bool tried = false;
    CUresult (*ModuleLoadData)(CUmodule *, const void *) = nullptr;
    CUresult (*ModuleUnload)(CUmodule) = nullptr;
    CUresult (*ModuleGetFunction)(CUfunction *, CUmodule, const char *) = nullptr;
    CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int) = nullptr;
    CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void **, void **) = nullptr;
    bool load()
    {
        if (tried) return handle != nullptr;
        tried = true;
        void *h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return false;
#define LOADDRV(field, sym)                                                                                            \
    field = reinterpret_cast<decltype(field)>(dlsym(h, sym));                                                          \
    if (!field) { dlclose(h); return false; }
        LOADDRV(ModuleLoadData, "cuModuleLoadData");
        LOADDRV(ModuleUnload, "cuModuleUnload");
        LOADDRV(ModuleGetFunction, "cuModuleGetFunction");
        LOADDRV(FuncSetAttribute, "cuFuncSetAttribute");
        LOADDRV(LaunchKernel, "cuLaunchKernel");
#undef LOADDRV
        handle = h;
        return true;
    }
};
DriverApi g_drv;

// ------------------------------------------------------------------------------------------------ kernel table
typedef void (*ForceKernelFn)(const ForceArgs);
typedef void (*ForceKernelSkFn)(const ForceArgsSK);
struct KernelVariant {
    const char *name;
    ForceKernelFn fn;
    int threads, r, tjb, st;
    size_t smem;
    double int_per_clk_sm; // measured steady-state rate (profiles/), used to choose between variants for small N
    ForceKernelSkFn fn_sk; // stream-K decomposition of the same inner loop (nullptr: not built for this variant)
    size_t smem_sk;
};
#define VARIANT(NAME, THREADS, R, TJB, ST, MATH, WP, U, MINB, RATE)                                                  \
    KernelVariant { NAME, force_kernel<THREADS, R, TJB, ST, MATH, WP, U, MINB>, THREADS, R, TJB, ST,                 \
                    force_smem_bytes<THREADS, R, TJB, ST, WP>(), RATE, nullptr, 0 }
#define VARIANT_SK(NAME, THREADS, R, TJB, ST, U, MINB, RATE)                                                         \
    KernelVariant { NAME, force_kernel<THREADS, R, TJB, ST, 1, false, U, MINB>, THREADS, R, TJB, ST,                 \
                    force_smem_bytes<THREADS, R, TJB, ST, false>(), RATE, force_kernel_sk<THREADS, R, TJB, ST, U, MINB>, \
                    force_sk_smem_bytes<THREADS, R, TJB, ST>() }
const KernelVariant g_variants[] = {
    // default first; chosen from the B200 sweep in profiles/ (tools/kbench)
    // 8 targets per thread and only 2 warps per scheduler: the operand-reuse cache keeps hitting while one warp keeps
    // issuing, which is what gets the accumulate FFMA2 triples back to 2 cycles (DESIGN.md section 3.1)
    VARIANT_SK("pk_t128_r8_tj2_st3_cta_u1_mb2", 128, 8, 2, 3, 1, 2, 9.53),
    // small systems: 256-target tiles and 1-block stages give enough CTAs to fill 148 SMs below N ~ 30k
    VARIANT_SK("pk_t128_r2_tj1_st3_cta_u2_mb4", 128, 2, 1, 3, 2, 4, 9.2),
    // one-warp CTAs, 8 per SM: the R = 8 inner loop on 256-target tiles.  Same rate as the default at large N (9.53),
    // ahead of it when a rank has few tiles (sharded runs: 25 088 targets x 200k sources 9.40 vs 9.34 vs 9.19 for the
    // R = 2 variant, profiles/r02_kbench_cluster_smalltiles.txt)
    VARIANT("pk_t32_r8_tj2_st2_cta_u1_mb8", 32, 8, 2, 2, 1, false, 1, 8, 9.53),
    VARIANT("pk_t128_r8_tj4_st2_cta_u1_mb2", 128, 8, 4, 2, 1, false, 1, 2, 9.5),
    VARIANT("pk_t256_r8_tj2_st3_cta_u1_mb1", 256, 8, 2, 3, 1, false, 1, 1, 9.5),
    VARIANT("pk_t256_r2_tj2_st3_cta_u2_mb3", 256, 2, 2, 3, 1, false, 2, 3, 9.0),
    VARIANT("sc_t256_r4_tj2_st3_cta_u1_mb2", 256, 4, 2, 3, 0, false, 1, 2, 8.2),
};
constexpr int N_VARIANTS = sizeof(g_variants) / sizeof(g_variants[0]);
constexpr uint64_t SLICE_ALIGN = 256;  // slice length granularity: a multiple of BLK; target tiles round up on their own (Lp)
constexpr uint32_t MAX_ROWS = 256; // upper bound on partial rows (the 1 GiB cap in max_rows_for usually binds first for big N)
constexpr int N_TIMER_SLOTS = 8;

struct Shard {
    int rank = 0, device = 0;
    cudaStream_t s_compute = nullptr, s_comm = nullptr;
    cudaEvent_t ev_integrated = nullptr, ev_gathered = nullptr;
    cudaEvent_t ev_pushed = nullptr; // p2p exchange: this shard's integrator has stored its new positions on every GPU
    float *bodies_next = nullptr;    // p2p exchange: the other half of the double-buffered body array
    cudaEvent_t timer[N_TIMER_SLOTS] = {};
    float *bodies = nullptr, *vel = nullptr, *acc = nullptr, *mass = nullptr, *partial = nullptr;
    float *stage = nullptr;      // 7 host-layout SoA slices of L floats (H2D / D2H staging of the shard's own bodies)
    float *stage_full = nullptr; // one rank per process only: 3 x stage_stride floats for a full-system position download (lazy)
    double *energy_blocks = nullptr, *energy_out = nullptr;
    void *l2_scratch = nullptr;
    // scratch of the field / potential / neighbours / friends-of-friends / group calls (grow-only)
    unsigned char *query_buf = nullptr;
    uint64_t query_bytes = 0;
    // test particles (b200nb_set_tracers): tr = [9][tr_T] rows qx qy qz vx vy vz ax ay az of the shard's tracers, the
    // first tr_local columns real; tr_part = the [S][4][tr_cap] partial rows of their field pass.  Both are owned by the
    // tracer set, never by query_buf: a captured step graph bakes their addresses in.
    float *tr = nullptr, *tr_part = nullptr;
    uint32_t tr_local = 0;
    uint64_t tr_bytes = 0;
    // the external expansion (b200nb_set_external_scf): ext_coef = tables | [S | T] (grow-only, ext_coef_bytes), and the
    // [4][L] and [4][tr_T] fp64 rows (ax, ay, az, phi) ext_total_kernel writes for the slice and the tracers before use
    unsigned char *ext_coef = nullptr;
    uint64_t ext_coef_bytes = 0;
    double *ext_body = nullptr, *ext_tr = nullptr;
    ncclComm_t comm = nullptr;
    CUmodule resched_mod = nullptr;   // the re-ordered cubin of the default variant on this device (nullptr: not in use)
    CUfunction resched_fn = nullptr;
    int n_sms = 0, occ = 0, occ_sk = 0;
    uint32_t n_local = 0; // real bodies in the slice
    // profiling mode: event pairs (start, stop) around force launches.  In-flight pairs are folded into prof_ms and
    // recycled once PROF_RING of them are pending, so a long profiled run neither grows nor creates events per launch.
    std::vector<cudaEvent_t> prof, prof_free;
    double prof_ms = 0.0;
    uint64_t prof_n = 0;
    uint64_t bytes = 0;
};

} // namespace

// A captured run of `steps` consecutive iterations (force + integrator launches) for one (integrator, dt).
struct StepGraph {
    int integrator = 0;
    float dt = 0.f;
    int steps = 0;
    uint64_t launches = 0; // kernels inside the graph
    cudaGraphExec_t exec = nullptr;
};
constexpr int GRAPH_STEPS = 16;     // iterations per graph launch
constexpr int GRAPH_MIN_STEPS = 32; // only worth capturing for longer runs
constexpr size_t GRAPH_CACHE_MAX = 4; // executable graphs kept per context (oldest evicted)

struct b200nb_ctx {
    std::vector<StepGraph> graphs;
    uint64_t n = 0;
    int n_ranks = 1;
    uint64_t L = 0, total_pad = 0, stage_stride = 0, total_pad_hint = 0;
    uint64_t Lp = 0; // L rounded up to whole target tiles of the chosen variant: grid size and stride of the partial rows
    uint32_t nblk_total = 0;
    float G = 0.f, soft = 0.f, soft2 = 0.f;
    const KernelVariant *kv = nullptr;
    uint32_t k_per_slice = 1, rows = 1; // S = k_per_slice * n_ranks
    std::string kname;                  // variant name (+ "+sk" in stream-K mode)
    bool stream_k = false;              // stream-K decomposition instead of the (tile x chunk) grid
    bool p2p = false;                   // exchange = peer stores from the integrator (in-process multi-GPU) instead of NCCL
    bool merge_launches = true;         // one force launch when the exchange has already landed at enqueue time (B200NB_SPLIT_LAUNCHES=1: never)
    uint32_t sk_grid = 0;               // CTAs per stream-K launch (resident slots)
    uint32_t sk_rows_own = 0, sk_rows_rem = 0;
    std::vector<Shard> shards;
    bool uploaded = false, acc_valid = false, profiling = false;
    // test particles: M in all, T per shard (ceil(M / P) in whole FIELD_TI tiles), batch of one field launch; the stored
    // tracer a(p) is valid for the current positions (the leapfrog's counterpart of acc_valid, kept apart from it)
    uint64_t m_tracers = 0, tr_T = 0;
    uint32_t tr_cap = 0;
    bool tr_acc_valid = false;
    ExtTerms ext{}; // the external potential (b200nb_set_external); ext.n == 0: none
    // the external expansion (b200nb_set_external_scf) as set, for b200nb_get_external_scf; on == false: none
    struct {
        bool on = false;
        uint32_t nmax = 0, lmax = 0, K = 0;
        double a = 0.0, centre[3] = {};
        std::vector<double> coef; // [S | T], K each
    } scf;
    uint64_t launches = 0;
    std::string err;
};

namespace {

struct DeviceGuard {
    int saved = -1;
    DeviceGuard() { if (cudaGetDevice(&saved) != cudaSuccess) saved = -1; }
    ~DeviceGuard() { if (saved >= 0) cudaSetDevice(saved); }
};

int fail(b200nb_ctx *c, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CU(c, call)                                                                                                    \
    do {                                                                                                               \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
            return fail(c, B200NB_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);  \
    } while (0)
#define NC(c, call)                                                                                                    \
    do {                                                                                                               \
        ncclResult_t r_ = (call);                                                                                      \
        if (r_ != ncclSuccess)                                                                                         \
            return fail(c, B200NB_ENCCL, "%s failed: %s (%s:%d)", #call, g_nccl.GetErrorString(r_), __FILE__, __LINE__); \
    } while (0)

int alloc_shard(b200nb_ctx *c, Shard &s)
{
    CU(c, cudaSetDevice(s.device));
    cudaDeviceProp prop;
    CU(c, cudaGetDeviceProperties(&prop, s.device));
    if (prop.major < 10)
        return fail(c, B200NB_ECUDA, "device %d is sm_%d%d; libb200nb is built for sm_100a only", s.device, prop.major,
                    prop.minor);
    s.n_sms = prop.multiProcessorCount;
    CU(c, cudaStreamCreateWithFlags(&s.s_compute, cudaStreamNonBlocking));
    CU(c, cudaStreamCreateWithFlags(&s.s_comm, cudaStreamNonBlocking));
    CU(c, cudaEventCreateWithFlags(&s.ev_integrated, cudaEventDisableTiming));
    CU(c, cudaEventCreateWithFlags(&s.ev_gathered, cudaEventDisableTiming));
    CU(c, cudaEventCreateWithFlags(&s.ev_pushed, cudaEventDisableTiming));
    for (auto &t : s.timer) CU(c, cudaEventCreate(&t));
    CU(c, cudaFuncSetAttribute(c->kv->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->kv->smem));
    CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s.occ, c->kv->fn, c->kv->threads, c->kv->smem));
    if (s.occ < 1) return fail(c, B200NB_ECUDA, "force kernel %s cannot be resident on device %d", c->kv->name, s.device);
    if (c->kv->fn_sk) {
        CU(c, cudaFuncSetAttribute(c->kv->fn_sk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->kv->smem_sk));
        CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s.occ_sk, c->kv->fn_sk, c->kv->threads, c->kv->smem_sk));
    }
    const uint64_t first = (uint64_t)s.rank * c->L;
    s.n_local = first >= c->n ? 0u : (uint32_t)std::min<uint64_t>(c->L, c->n - first);
    // the post-ptxas re-ordered build of the default variant (B200NB_NO_RESCHED=1: launch what ptxas scheduled)
    if (c->kv == &g_variants[2] && force_resched_cubin_size > 0 && !getenv("B200NB_NO_RESCHED") && g_drv.load()) {
        CU(c, cudaFree(nullptr)); // make sure the primary context exists and is current
        CUmodule mod = nullptr;
        CUfunction fn = nullptr;
        if (g_drv.ModuleLoadData(&mod, force_resched_cubin) == CUDA_SUCCESS && g_drv.ModuleGetFunction(&fn, mod, force_resched_kernel) == CUDA_SUCCESS &&
            g_drv.FuncSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)c->kv->smem) == CUDA_SUCCESS) {
            s.resched_mod = mod;
            s.resched_fn = fn;
        } else {
            if (mod) g_drv.ModuleUnload(mod);
            fprintf(stderr, "libb200nb: the re-ordered force kernel could not be loaded on device %d; using the ptxas-scheduled one\n", s.device);
        }
    }
    return B200NB_OK;
}

int alloc_buffers(b200nb_ctx *c, Shard &s)
{
    CU(c, cudaSetDevice(s.device));
    const size_t L = c->L;
    auto dmalloc = [&](void **p, size_t bytes) -> cudaError_t { s.bytes += bytes; return cudaMalloc(p, bytes); };
    CU(c, dmalloc((void **)&s.bodies, c->total_pad * 16));
    if (c->p2p) CU(c, dmalloc((void **)&s.bodies_next, c->total_pad * 16));
    CU(c, dmalloc((void **)&s.vel, 3 * L * 4));
    CU(c, dmalloc((void **)&s.acc, 3 * L * 4));
    CU(c, dmalloc((void **)&s.mass, L * 4));
    CU(c, dmalloc((void **)&s.partial, (size_t)c->rows * 3 * c->Lp * 4));
    CU(c, dmalloc((void **)&s.stage, 7 * L * 4));
    const size_t eb = (L + ENERGY_THREADS - 1) / ENERGY_THREADS;
    CU(c, dmalloc((void **)&s.energy_blocks, eb * 8 * MR_COUNT));
    CU(c, dmalloc((void **)&s.energy_out, 8 * MR_COUNT));
    CU(c, cudaMemsetAsync(s.acc, 0, 3 * L * 4, s.s_compute));
    CU(c, cudaMemsetAsync(s.vel, 0, 3 * L * 4, s.s_compute));
    CU(c, cudaEventRecord(s.ev_gathered, s.s_comm)); // "positions are current" before the first step
    return B200NB_OK;
}

const KernelVariant *pick_variant()
{
    const char *e = getenv("B200NB_VARIANT");
    if (e && *e) {
        for (int i = 0; i < N_VARIANTS; ++i)
            if (!strcmp(e, g_variants[i].name)) return &g_variants[i];
        const long idx = strtol(e, nullptr, 10);
        if (idx >= 0 && idx < N_VARIANTS && e[0] >= '0' && e[0] <= '9') return &g_variants[idx];
        fprintf(stderr, "libb200nb: unknown B200NB_VARIANT '%s', choosing automatically\n", e);
    }
    return nullptr; // choose by the planner's time estimate (choose_variant)
}

uint32_t max_rows_for(uint64_t L, int n_ranks)
{
    // rows of partial sums cost 12*L bytes each: never more than MAX_ROWS, never more than 1 GiB in total
    return (uint32_t)std::max<uint64_t>((uint64_t)n_ranks, std::min<uint64_t>(MAX_ROWS, (1ull << 30) / (12ull * L)));
}

// Source blocks the force pass has to visit.  The slice length is rounded up to the launch granularity, so the tail of
// the (last) slice is padding with G*m = 0; on one GPU everything past the last real body's block is skipped outright
// (0.3 % of the pass at N = 200k).  With several ranks every slice keeps its full length so that slices stay congruent.
uint32_t source_blocks(uint64_t n, uint64_t L, int n_ranks)
{
    return n_ranks == 1 ? (uint32_t)((n + BLK - 1) / BLK) : (uint32_t)(L * (uint64_t)n_ranks / BLK);
}

ChunkPlan plan_for(const KernelVariant &kv, uint64_t n, uint64_t L, int n_sms, int occ, int n_ranks)
{
    const uint32_t ti = kv.threads * kv.r;
    return plan_chunks((uint32_t)((L + ti - 1) / ti), source_blocks(n, L, n_ranks) / (uint32_t)n_ranks, (uint32_t)(n_sms * occ),
                       (uint32_t)n_ranks, max_rows_for((L + ti - 1) / ti * ti, n_ranks), (uint32_t)(2 * kv.tjb));
}

// Between the one-warp R = 8 variant (256-target tiles), the 4-warp R = 8 variant (1024-target tiles) and the small R = 2
// variant, take the one the planner expects to finish first (plan.hpp: choose_variant_index).  The one-warp variant is
// listed first: it matches the 4-warp one at large N (N = 200k inside bench.py: 14.52 vs 14.56 ms per launch, with 56
// instead of 74 partial rows; profiles/r02_ncu_force_kernel_*.txt) and its finer tiles win when a rank has few of them.
int choose_variant(b200nb_ctx *c, int device, const KernelVariant **out)
{
    cudaDeviceProp prop;
    CU(c, cudaSetDevice(device)); // the occupancy query below answers for the current device
    CU(c, cudaGetDeviceProperties(&prop, device));
    const KernelVariant *cands[3] = {&g_variants[2], &g_variants[0], &g_variants[1]};
    *out = cands[0];
    const char *mode = getenv("B200NB_MODE");
    if (mode && !strcmp(mode, "sk")) {
        // stream-K: every CTA gets ceil(U/G) (tile x block) units; a unit is TI x 128 interactions at SM rate / occ
        double best_t = 1e300;
        for (const KernelVariant *kv : {&g_variants[0], &g_variants[1]}) {
            int occ_sk = 0;
            CU(c, cudaFuncSetAttribute(kv->fn_sk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kv->smem_sk));
            CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_sk, kv->fn_sk, kv->threads, kv->smem_sk));
            if (occ_sk < 1) continue;
            const uint64_t G = (uint64_t)prop.multiProcessorCount * occ_sk;
            const uint64_t ti = (uint64_t)kv->threads * kv->r;
            const uint64_t U = ((c->L + ti - 1) / ti) * (c->total_pad_hint / BLK);
            const double t = (double)((U + G - 1) / G) * (double)ti * (double)occ_sk / kv->int_per_clk_sm;
            if (t < best_t) { best_t = t; *out = kv; }
        }
        return B200NB_OK;
    }
    VariantShape shapes[3];
    uint32_t max_rows[3];
    for (int i = 0; i < 3; ++i) {
        const KernelVariant *kv = cands[i];
        int occ = 0;
        CU(c, cudaFuncSetAttribute(kv->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kv->smem));
        CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kv->fn, kv->threads, kv->smem));
        shapes[i] = VariantShape{(uint32_t)kv->threads, (uint32_t)kv->r, (uint32_t)kv->tjb, (uint32_t)std::max(occ, 0), kv->int_per_clk_sm};
        const uint64_t ti = (uint64_t)kv->threads * kv->r;
        max_rows[i] = max_rows_for((c->L + ti - 1) / ti * ti, c->n_ranks);
    }
    const int pick = choose_variant_index(shapes, 3, c->L, source_blocks(c->n, c->L, c->n_ranks) / (uint32_t)c->n_ranks,
                                          (uint32_t)prop.multiProcessorCount, (uint32_t)c->n_ranks, max_rows);
    if (pick >= 0) *out = cands[pick];
    return B200NB_OK;
}

int enqueue_gather(b200nb_ctx *c);
int sync_all(b200nb_ctx *c);

constexpr size_t PROF_RING = 512; // pending (start, stop) pairs per shard before they are folded

// fold every pending pair into the running total (joins the stop events) and recycle the events
int prof_drain(b200nb_ctx *c, Shard &s)
{
    for (size_t i = 0; i + 1 < s.prof.size(); i += 2) {
        float ms = 0.f;
        CU(c, cudaEventSynchronize(s.prof[i + 1]));
        CU(c, cudaEventElapsedTime(&ms, s.prof[i], s.prof[i + 1]));
        s.prof_ms += ms;
        s.prof_n++;
    }
    s.prof_free.insert(s.prof_free.end(), s.prof.begin(), s.prof.end());
    s.prof.clear();
    return B200NB_OK;
}

// start event of a profiled launch (recorded on the compute stream); the matching prof_stop records the other one
int prof_start(b200nb_ctx *c, Shard &s)
{
    if (s.prof.size() >= 2 * PROF_RING)
        if (int rc = prof_drain(c, s)) return rc;
    while (s.prof_free.size() < 2) {
        cudaEvent_t ev;
        CU(c, cudaEventCreate(&ev));
        s.prof_free.push_back(ev);
    }
    cudaEvent_t e[2];
    for (auto &ev : e) { ev = s.prof_free.back(); s.prof_free.pop_back(); }
    s.prof.push_back(e[0]);
    s.prof.push_back(e[1]);
    CU(c, cudaEventRecord(e[0], s.s_compute));
    return B200NB_OK;
}
int prof_stop(b200nb_ctx *c, Shard &s)
{
    CU(c, cudaEventRecord(s.prof.back(), s.s_compute));
    return B200NB_OK;
}

// In-process multi-GPU has two exchange steps.  Default: in-place ncclAllGather on a communication stream, which runs
// entirely beside the own-slice force launch.  Alternative (B200NB_EXCHANGE=p2p, and automatically when libnccl cannot
// be loaded): every GPU can address every other one (NVLink / NVSwitch peers), so the integrator stores the new
// positions of its slice straight into the body array of every GPU (integrate_sm100.cuh: IntegrateArgs::out) and one
// event per GPU is the only synchronisation; the body array is double-buffered so that a fast GPU never overwrites
// positions a slower one is still reading.  Measured on 2 B200s the fused form is 0.1-1.4 % *slower*
// (profiles/r01_exchange_p2p_vs_nccl.txt): the peer stores must be flushed before the integrator kernel can retire,
// which puts an NVLink round trip on the compute stream's critical path, while the separate all-gather hides all of
// its latency behind the own-slice launch.  Both paths produce bit-identical results (tested).
int enable_p2p(b200nb_ctx *c)
{
    const char *e = getenv("B200NB_EXCHANGE");
    // several shards on one device ("virtual shards", b200nb_create_sharded): NCCL refuses a communicator with the
    // same GPU twice, and the peer path needs no peer at all there
    bool shared_device = false;
    for (size_t i = 0; i < c->shards.size(); ++i)
        for (size_t j = i + 1; j < c->shards.size(); ++j) shared_device |= c->shards[i].device == c->shards[j].device;
    if (shared_device) {
        if (e && !strcmp(e, "nccl"))
            return fail(c, B200NB_EINVAL, "B200NB_EXCHANGE=nccl cannot be used when several shards share one device");
        e = "p2p";
    }
    if (e && !strcmp(e, "nccl")) return B200NB_OK;
    if (e && *e && strcmp(e, "p2p"))
        return fail(c, B200NB_EINVAL, "B200NB_EXCHANGE must be 'p2p' or 'nccl', not '%s'", e);
    if (!(e && *e)) {
        if (g_nccl.load()) return B200NB_OK; // default
        e = nullptr;                         // no NCCL on this machine: try the peer path before giving up
    }
    if (c->shards.size() > (size_t)MAX_PUSH_TARGETS) {
        if (e) return fail(c, B200NB_EINVAL, "B200NB_EXCHANGE=p2p supports at most %d GPUs", MAX_PUSH_TARGETS);
        return B200NB_OK;
    }
    for (auto &a : c->shards)
        for (auto &b : c->shards) {
            if (a.device == b.device) continue;
            int ok = 0;
            CU(c, cudaDeviceCanAccessPeer(&ok, a.device, b.device));
            if (!ok) {
                if (e) return fail(c, B200NB_ECUDA, "B200NB_EXCHANGE=p2p: device %d cannot access device %d", a.device, b.device);
                return B200NB_OK; // no peer path: NCCL
            }
        }
    for (auto &a : c->shards) {
        CU(c, cudaSetDevice(a.device));
        for (auto &b : c->shards) {
            if (a.device == b.device) continue;
            const cudaError_t r = cudaDeviceEnablePeerAccess(b.device, 0);
            if (r == cudaErrorPeerAccessAlreadyEnabled) { (void)cudaGetLastError(); continue; }
            CU(c, r);
        }
    }
    c->p2p = true;
    return B200NB_OK;
}

int create_common(b200nb_ctx **out, uint64_t n, float G, float soft, int n_ranks, const std::vector<int> &ranks,
                  const std::vector<int> &devices, const void *nccl_id)
{
    if (!out) return fail(nullptr, B200NB_EINVAL, "out is NULL");
    *out = nullptr;
    if (n == 0 || n > (1ull << 31)) return fail(nullptr, B200NB_EINVAL, "n_bodies must be in [1, 2^31]");
    if (!(soft != 0.f)) return fail(nullptr, B200NB_EINVAL, "softening factor can't be equal to 0 (main.cpp:150-155)");
    DeviceGuard guard;
    b200nb_ctx *c = new b200nb_ctx();
    c->n = n; c->n_ranks = n_ranks; c->G = G; c->soft = soft; c->soft2 = soft * soft;
    c->kv = pick_variant();
    c->L = b200nb_slice_length(n, n_ranks);
    c->total_pad_hint = c->L * n_ranks;
    if (!c->kv) {
        if (int rc = choose_variant(c, devices[0], &c->kv)) { g_create_error = c->err; delete c; return rc; }
    }
    c->total_pad = c->L * n_ranks;
    c->nblk_total = (uint32_t)(c->total_pad / BLK);
    c->stage_stride = (n + 3) / 4 * 4;
    c->shards.resize(ranks.size());
    auto bail = [&](int code) {
        g_create_error = c->err;
        b200nb_destroy(c);
        return code;
    };
    for (size_t i = 0; i < ranks.size(); ++i) {
        c->shards[i].rank = ranks[i];
        c->shards[i].device = devices[i];
        if (int rc = alloc_shard(c, c->shards[i])) return bail(rc);
    }
    const Shard &s0 = c->shards[0];
    {
        const uint64_t ti = (uint64_t)c->kv->threads * c->kv->r;
        c->Lp = (c->L + ti - 1) / ti * ti;
    }
    c->k_per_slice = plan_for(*c->kv, c->n, c->L, s0.n_sms, s0.occ, n_ranks).n_chunks;
    c->rows = c->k_per_slice * n_ranks;
    {
        // "grid" (default): dynamic (tile x chunk) grid; "sk": static stream-K split, measured 3-8 % slower on B200
        // (profiles/r01_streamk_vs_grid.txt) and kept as a tested alternative
        const char *mode = getenv("B200NB_MODE");
        const bool want_sk = mode && !strcmp(mode, "sk");
        c->stream_k = want_sk && c->kv->fn_sk && s0.occ_sk >= 1;
        if (want_sk && !c->stream_k) { c->err = "B200NB_MODE=sk: variant has no stream-K kernel"; return bail(B200NB_EINVAL); }
    }
    c->kname = std::string(c->kv->name) + (c->stream_k ? "+sk" : "") + (!c->stream_k && c->shards[0].resched_fn ? "+resched" : "");
    c->merge_launches = getenv("B200NB_SPLIT_LAUNCHES") == nullptr;
    if (c->stream_k) {
        const uint32_t ti = c->kv->threads * c->kv->r;
        const uint32_t n_itiles = (uint32_t)(c->Lp / ti), nbs = (uint32_t)(c->L / BLK);
        const char *w = getenv("B200NB_SK_WAVES"); // experiment: CTAs = waves x resident slots
        c->sk_grid = (uint32_t)(s0.n_sms * s0.occ_sk) * (uint32_t)std::max(1, w ? atoi(w) : 1);
        auto max_rows = [&](uint32_t nb) {
            uint32_t m = 0;
            if (nb == 0) return m;
            const uint64_t U = (uint64_t)n_itiles * nb;
            for (uint32_t t = 0; t < n_itiles; ++t) m = std::max(m, sk_rows_of_tile(t, nb, U, c->sk_grid));
            return m;
        };
        c->sk_rows_own = max_rows(nbs);
        c->sk_rows_rem = max_rows(c->nblk_total - nbs);
        c->rows = c->sk_rows_own + c->sk_rows_rem;
    }
    if (n_ranks > 1 && ranks.size() == (size_t)n_ranks) {
        if (int rc = enable_p2p(c)) return bail(rc);
    }
    for (auto &s : c->shards)
        if (int rc = alloc_buffers(c, s)) return bail(rc);

    if (n_ranks > 1 && !c->p2p) {
        if (!g_nccl.load()) { c->err = g_nccl.err; return bail(B200NB_ENCCL); }
        ncclUniqueId id;
        if (nccl_id) memcpy(&id, nccl_id, sizeof id);
        else if (ranks.size() == (size_t)n_ranks) {
            ncclResult_t r = g_nccl.GetUniqueId(&id);
            if (r != ncclSuccess) { c->err = std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r); return bail(B200NB_ENCCL); }
        } else { c->err = "nccl_id is required when this process does not own every rank"; return bail(B200NB_EINVAL); }
        ncclResult_t r = g_nccl.GroupStart();
        for (auto &s : c->shards) {
            if (r != ncclSuccess) break;
            if (cudaSetDevice(s.device) != cudaSuccess) { r = ncclUnhandledCudaError; break; }
            r = g_nccl.CommInitRank(&s.comm, n_ranks, id, s.rank);
        }
        ncclResult_t r2 = g_nccl.GroupEnd();
        if (r == ncclSuccess) r = r2;
        if (r != ncclSuccess) { c->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r); return bail(B200NB_ENCCL); }
        // NCCL builds its channels lazily on the first collective (hundreds of ms): pay that here, not in step 1
        // of the caller's timed loop (main.cpp:348-371 times every iteration).  The buffer content is irrelevant.
        if (int rc = enqueue_gather(c)) return bail(rc);
        if (int rc = sync_all(c)) return bail(rc);
    }
    *out = c;
    return B200NB_OK;
}

// Have the remote slices of the current positions already landed on shard `s` (host-side query, no waiting)?  True when
// the caller steps synchronously (the CLI joins the device after every iteration, main.cpp:356-368): the exchange of
// the previous step is long over by the time the next force pass is enqueued, there is nothing left to overlap, and
// the pass can be ONE launch over all chunks instead of own-slice + remote launches with a tail each.
bool remote_positions_landed(b200nb_ctx *c, Shard &s)
{
    bool ready = true;
    if (!c->p2p) {
        ready = cudaEventQuery(s.ev_gathered) == cudaSuccess;
    } else {
        for (auto &o : c->shards) {
            if (&o == &s || !ready) continue;
            if (o.device != s.device) (void)cudaSetDevice(o.device); // query an event on the device that owns it
            ready = cudaEventQuery(o.ev_pushed) == cudaSuccess;
        }
        (void)cudaSetDevice(s.device);
    }
    if (!ready) (void)cudaGetLastError(); // cudaErrorNotReady is an answer, not a fault
    return ready;
}

// the compute stream of `s` may not read remote slices before they have landed
int wait_remote_positions(b200nb_ctx *c, Shard &s)
{
    if (!c->p2p) {
        CU(c, cudaStreamWaitEvent(s.s_compute, s.ev_gathered, 0));
        return B200NB_OK;
    }
    for (auto &o : c->shards)
        if (&o != &s) CU(c, cudaStreamWaitEvent(s.s_compute, o.ev_pushed, 0));
    return B200NB_OK;
}

// stream-K launches: one for the rank's own (already resident) source blocks, one for the gathered remote blocks
int enqueue_force_sk(b200nb_ctx *c)
{
    const KernelVariant &kv = *c->kv;
    const uint32_t ti = kv.threads * kv.r;
    const uint32_t nbs = (uint32_t)(c->L / BLK);
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        ForceArgsSK a{};
        a.src = s.bodies; a.tgt = s.bodies; a.partial = s.partial;
        a.tgt_blk0 = (uint32_t)((uint64_t)s.rank * c->L / BLK);
        a.tgt_stride = (uint32_t)c->Lp; a.tgt_count = (uint32_t)c->L;
        a.src_nblk_total = c->nblk_total;
        a.blk_rot = nbs * (uint32_t)s.rank;
        a.n_itiles = (uint32_t)(c->Lp / ti);
        a.soft2 = c->soft2;
        auto launch = [&](uint32_t lb0, uint32_t nb, uint32_t row0) -> int {
            a.lb0 = lb0; a.nb = nb; a.row0 = row0;
            if (c->profiling) if (int rc = prof_start(c, s)) return rc;
            kv.fn_sk<<<c->sk_grid, kv.threads, kv.smem_sk, s.s_compute>>>(a);
            if (c->profiling) if (int rc = prof_stop(c, s)) return rc;
            c->launches++;
            CU(c, cudaGetLastError());
            return B200NB_OK;
        };
        if (int rc = launch(0, nbs, 0)) return rc; // own slice: resident, overlaps the all-gather
        if (c->n_ranks > 1) {
            if (int rc = wait_remote_positions(c, s)) return rc;
            if (int rc = launch(nbs, c->nblk_total - nbs, c->sk_rows_own)) return rc;
        }
    }
    return B200NB_OK;
}

// enqueue the force pass (own chunks, wait for the gather, remote chunks) on every shard's compute stream
int enqueue_force(b200nb_ctx *c)
{
    if (c->stream_k) return enqueue_force_sk(c);
    const KernelVariant &kv = *c->kv;
    const uint32_t ti = kv.threads * kv.r;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        ForceArgs a{};
        a.src = s.bodies; a.tgt = s.bodies; a.partial = s.partial;
        a.tgt_blk0 = (uint32_t)((uint64_t)s.rank * c->L / BLK);
        a.tgt_stride = (uint32_t)c->Lp; a.tgt_count = (uint32_t)c->L;
        a.src_nblk_total = source_blocks(c->n, c->L, c->n_ranks);
        a.n_chunks_total = c->rows;
        a.chunk_rot = c->k_per_slice * (uint32_t)s.rank;
        a.soft2 = c->soft2;
        a.dbg = nullptr;
        const uint32_t n_itiles = (uint32_t)(c->Lp / ti);
        auto launch = [&](uint32_t first, uint32_t count) -> int {
            a.chunk_first = first;
            if (c->profiling) if (int rc = prof_start(c, s)) return rc;
            if (s.resched_fn) {
                void *params[1] = {&a};
                const CUresult r = g_drv.LaunchKernel(s.resched_fn, n_itiles, count, 1, (unsigned)kv.threads, 1, 1, (unsigned)kv.smem,
                                                      (CUstream)s.s_compute, params, nullptr);
                if (r != CUDA_SUCCESS) return fail(c, B200NB_ECUDA, "cuLaunchKernel(re-ordered force kernel) failed: %d", (int)r);
            } else {
                kv.fn<<<dim3(n_itiles, count), kv.threads, kv.smem, s.s_compute>>>(a);
            }
            if (c->profiling) if (int rc = prof_stop(c, s)) return rc;
            c->launches++;
            CU(c, cudaGetLastError());
            return B200NB_OK;
        };
        if (c->n_ranks == 1) {
            if (int rc = launch(0, c->rows)) return rc;
        } else if (c->merge_launches && remote_positions_landed(c, s)) {
            if (int rc = wait_remote_positions(c, s)) return rc; // already complete: orders the stream, costs nothing
            if (int rc = launch(0, c->rows)) return rc;          // same chunks, same rows: bit-identical to the split form
        } else {
            if (int rc = launch(0, c->k_per_slice)) return rc; // own slice: resident, overlaps the exchange
            if (int rc = wait_remote_positions(c, s)) return rc;
            if (int rc = launch(c->k_per_slice, c->rows - c->k_per_slice)) return rc;
        }
    }
    return B200NB_OK;
}

size_t round256(size_t x) { return (x + 255) / 256 * 256; }

// ext_total_kernel over `count` points of `pts` into out = [4][stride], on the shard's compute stream: one launch
template <class Points>
int enqueue_ext_total(b200nb_ctx *c, Shard &s, const Points &pts, uint32_t count, uint32_t stride, double *out)
{
    ExtScf E{};
    E.tab = reinterpret_cast<const ScfTables *>(s.ext_coef);
    E.coef = reinterpret_cast<const double *>(s.ext_coef + round256(sizeof(ScfTables)));
    E.nmax = c->scf.nmax; E.lmax = c->scf.lmax; E.K = c->scf.K;
    E.cx = c->scf.centre[0]; E.cy = c->scf.centre[1]; E.cz = c->scf.centre[2];
    E.a = c->scf.a;
    ext_total_kernel<Points><<<(count + SCF_EVAL_THREADS - 1) / SCF_EVAL_THREADS, SCF_EVAL_THREADS, scf_field_smem(E.K), s.s_compute>>>(
        c->ext, E, pts, count, stride, out);
    c->launches++;
    CU(c, cudaGetLastError());
    return B200NB_OK;
}

// the total external field at the shard's own bodies, into s.ext_body (the current positions of `bodies`)
int enqueue_ext_total_bodies(b200nb_ctx *c, Shard &s)
{
    return enqueue_ext_total(c, s, BlockedPoints{s.bodies, (uint64_t)s.rank * c->L}, s.n_local, (uint32_t)c->L, s.ext_body);
}

int enqueue_integrate(b200nb_ctx *c, int mode, float dt)
{
    const bool moves = mode == IM_MURB || mode == IM_MURB_STORED || mode == IM_LF_KICK_DRIFT;
    // the modes that sum partial rows add e: with an expansion it is evaluated by one ext_total_kernel launch first
    const bool field = c->scf.on && (mode == IM_MURB || mode == IM_REDUCE_ONLY || mode == IM_LF_KICK);
    const bool push = c->p2p && moves;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        if (push) {
            // the buffers about to be overwritten were last read one position update ago: every GPU's kernels of
            // that time precede its previous push in stream order, so waiting for those pushes is enough
            if (int rc = wait_remote_positions(c, s)) return rc;
        }
        if (s.n_local == 0) continue;
        IntegrateArgs a{};
        a.bodies = s.bodies; a.vel = s.vel; a.acc = s.acc; a.partial = s.partial;
        if (push) {
            a.n_out = 0;
            for (auto &o : c->shards) a.out[a.n_out++] = o.bodies_next;
        } else {
            a.out[0] = s.bodies; a.n_out = 1;
        }
        a.rows = c->rows; a.L = (uint32_t)c->L; a.pstride = (uint32_t)c->Lp; a.n_local = s.n_local;
        a.first = (uint64_t)s.rank * c->L; a.dt = dt; a.mode = mode;
        if (c->stream_k) {
            const uint32_t ti = c->kv->threads * c->kv->r, n_itiles = (uint32_t)(c->Lp / ti), nbs = (uint32_t)(c->L / BLK);
            a.sk_ti = ti;
            a.sk[0] = SkRows{(uint64_t)n_itiles * nbs, c->sk_grid, nbs, 0};
            const uint32_t nbr = c->nblk_total - nbs;
            a.sk[1] = SkRows{(uint64_t)n_itiles * nbr, c->sk_grid, nbr, c->sk_rows_own};
        }
        // caller-supplied accelerations (IM_MURB_STORED) already are the whole acceleration: no terms added
        if (field) {
            if (int rc = enqueue_ext_total_bodies(c, s)) return rc;
            integrate_kernel<true, true><<<(s.n_local + 255) / 256, 256, 0, s.s_compute>>>(a, c->ext, s.ext_body);
        } else if (c->ext.n > 0 && mode != IM_MURB_STORED) {
            integrate_kernel<true><<<(s.n_local + 255) / 256, 256, 0, s.s_compute>>>(a, c->ext, nullptr);
        } else {
            integrate_kernel<false><<<(s.n_local + 255) / 256, 256, 0, s.s_compute>>>(a, c->ext, nullptr);
        }
        c->launches++;
        CU(c, cudaGetLastError());
    }
    if (push) {
        for (auto &s : c->shards) {
            CU(c, cudaSetDevice(s.device));
            CU(c, cudaEventRecord(s.ev_pushed, s.s_compute));
            std::swap(s.bodies, s.bodies_next);
        }
    }
    return B200NB_OK;
}

// positions of the own slice changed: publish them to every other rank (in place, on the comm stream)
int enqueue_gather(b200nb_ctx *c)
{
    if (c->n_ranks == 1 || c->p2p) return B200NB_OK; // p2p: the integrator already stored the positions everywhere
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaEventRecord(s.ev_integrated, s.s_compute));
        CU(c, cudaStreamWaitEvent(s.s_comm, s.ev_integrated, 0));
    }
    NC(c, g_nccl.GroupStart());
    ncclResult_t r = ncclSuccess;
    for (auto &s : c->shards) {
        if (cudaSetDevice(s.device) != cudaSuccess) { r = ncclUnhandledCudaError; break; }
        const size_t count = (size_t)c->L * 4; // floats in one blocked slice
        r = g_nccl.AllGather(s.bodies + (size_t)s.rank * count, s.bodies, count, ncclFloat, s.comm, s.s_comm);
        if (r != ncclSuccess) break;
    }
    ncclResult_t r2 = g_nccl.GroupEnd();
    if (r == ncclSuccess) r = r2;
    if (r != ncclSuccess) return fail(c, B200NB_ENCCL, "ncclAllGather failed: %s", g_nccl.GetErrorString(r));
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaEventRecord(s.ev_gathered, s.s_comm));
    }
    return B200NB_OK;
}

int sync_all(b200nb_ctx *c)
{
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaStreamSynchronize(s.s_compute));
        CU(c, cudaStreamSynchronize(s.s_comm));
    }
    return B200NB_OK;
}

// gather a [3][L] per-rank device array (vel or acc) into host SoA arrays of n floats
int download_sliced(b200nb_ctx *c, float *Shard::*field, float *hx, float *hy, float *hz)
{
    float *dst[3] = {hx, hy, hz};
    const bool all_local = c->shards.size() == (size_t)c->n_ranks;
    if (all_local) {
        for (auto &s : c->shards) {
            if (s.n_local == 0) continue;
            CU(c, cudaSetDevice(s.device));
            for (int k = 0; k < 3; ++k)
                if (dst[k])
                    CU(c, cudaMemcpyAsync(dst[k] + (size_t)s.rank * c->L, (s.*field) + (size_t)k * c->L,
                                          (size_t)s.n_local * 4, cudaMemcpyDeviceToHost, s.s_compute));
        }
        return sync_all(c);
    }
    // one rank per process: all-gather the slices through a temporary [P][3][L] device buffer
    Shard &s = c->shards[0];
    CU(c, cudaSetDevice(s.device));
    struct Scratch { // freed on every exit path
        float *p = nullptr;
        ~Scratch() { if (p) cudaFree(p); }
    } tmp;
    const size_t count = 3 * (size_t)c->L;
    CU(c, cudaMalloc((void **)&tmp.p, count * c->n_ranks * 4));
    CU(c, cudaMemcpyAsync(tmp.p + (size_t)s.rank * count, s.*field, count * 4, cudaMemcpyDeviceToDevice, s.s_compute));
    NC(c, g_nccl.AllGather(tmp.p + (size_t)s.rank * count, tmp.p, count, ncclFloat, s.comm, s.s_compute));
    for (int rk = 0; rk < c->n_ranks; ++rk) {
        const uint64_t first = (uint64_t)rk * c->L;
        if (first >= c->n) break;
        const size_t cnt = (size_t)std::min<uint64_t>(c->L, c->n - first);
        for (int k = 0; k < 3; ++k)
            if (dst[k])
                CU(c, cudaMemcpyAsync(dst[k] + first, tmp.p + (size_t)rk * count + (size_t)k * c->L, cnt * 4,
                                      cudaMemcpyDeviceToHost, s.s_compute));
    }
    CU(c, cudaStreamSynchronize(s.s_compute));
    return B200NB_OK;
}

// Grow-only scratch of the field / potential / neighbours / friends-of-friends calls.
int query_scratch(b200nb_ctx *c, Shard &s, size_t bytes)
{
    if (s.query_bytes >= bytes) return B200NB_OK;
    CU(c, cudaSetDevice(s.device));
    if (s.query_buf) {
        CU(c, cudaFree(s.query_buf));
        s.query_buf = nullptr;
        s.bytes -= s.query_bytes;
        s.query_bytes = 0;
    }
    CU(c, cudaMalloc((void **)&s.query_buf, bytes));
    s.query_bytes = bytes;
    s.bytes += bytes;
    return B200NB_OK;
}

// One result of run_targets: `bytes` per target, written to host rows (host == nullptr: not copied back).
struct TargetOut {
    void *host;
    size_t bytes;
};

// Targets are the points (self == false, m of them) or every body (self == true).  They are cut into one contiguous
// range of Q per rank (points: ceil(m / n_ranks); bodies: the rank's slice) and each range into launches of at most
// `cap` targets, cap = min(batch, Q rounded up to whole tiles).  In-process shards copy their results straight to the
// host.  With one rank per process every rank runs the same number of rounds and each round's results are all-gathered,
// the way download_sliced gathers accelerations.
// Scratch per shard: work_bytes(cap) | [3][cap] points | the outputs' [cap] rows one after another | with one rank per
// process, n_ranks copies of those rows.  launch(s, base, cnt, cap, work, dpts, dout) enqueues on s.s_compute what
// leaves the results of targets base + [0, cnt) in dout.
// Reads only the body array and writes only this scratch: the simulation state and cached step graphs are untouched.
template <class Work, class Launch>
int run_targets(b200nb_ctx *c, bool self, uint64_t m, const float *const pts[3], uint32_t tile, uint32_t batch,
                       const std::vector<TargetOut> &out, Work work_bytes, Launch launch)
{
    DeviceGuard guard;
    const bool gather = c->shards.size() != (size_t)c->n_ranks;
    const uint64_t Q = self ? c->L : (m + c->n_ranks - 1) / c->n_ranks;
    const uint32_t cap = (uint32_t)std::min<uint64_t>(batch, (Q + tile - 1) / tile * tile);
    const uint64_t rounds = (Q + cap - 1) / cap;
    const size_t P = cap;
    size_t row_bytes = 0; // all outputs of one target
    for (auto &o : out) row_bytes += o.bytes;
    const size_t work = work_bytes(cap);
    for (auto &s : c->shards) {
        if (int rc = query_scratch(c, s, work + 3 * 4 * P + (1 + (gather ? c->n_ranks : 0)) * row_bytes * P)) return rc;
        CU(c, cudaSetDevice(s.device));
        // an asynchronous step may still be exchanging positions: the whole body array is read
        if (c->n_ranks > 1)
            if (int rc = wait_remote_positions(c, s)) return rc;
        float *dpts = reinterpret_cast<float *>(s.query_buf + work);
        unsigned char *dout = reinterpret_cast<unsigned char *>(dpts + 3 * P), *dgat = dout + row_bytes * P;
        const uint64_t lo = (uint64_t)s.rank * Q;
        const uint64_t hi = self ? lo + s.n_local : std::min<uint64_t>(lo + Q, m);
        for (uint64_t r = 0; r < rounds; ++r) {
            const uint64_t base = lo + r * cap;
            const uint32_t cnt = base < hi ? (uint32_t)std::min<uint64_t>(cap, hi - base) : 0u;
            if (cnt == 0 && !gather) break;
            if (cnt > 0) {
                if (!self)
                    for (int k = 0; k < 3; ++k)
                        CU(c, cudaMemcpyAsync(dpts + k * P, pts[k] + base, (size_t)cnt * 4, cudaMemcpyHostToDevice, s.s_compute));
                if (int rc = launch(s, base, cnt, cap, s.query_buf, dpts, dout)) return rc;
                CU(c, cudaGetLastError());
            }
            if (!gather) {
                size_t off = 0;
                for (auto &o : out) {
                    if (o.host)
                        CU(c, cudaMemcpyAsync(static_cast<unsigned char *>(o.host) + base * o.bytes, dout + off * P, cnt * o.bytes,
                                              cudaMemcpyDeviceToHost, s.s_compute));
                    off += o.bytes;
                }
                continue;
            }
            NC(c, g_nccl.AllGather(dout, dgat, row_bytes / 4 * P, ncclFloat, s.comm, s.s_compute));
            for (int rk = 0; rk < c->n_ranks; ++rk) {
                const uint64_t rb = (uint64_t)rk * Q + r * cap;
                const uint64_t rhi = std::min<uint64_t>((uint64_t)rk * Q + Q, self ? c->n : m);
                if (rb >= rhi) continue;
                const size_t rcnt = (size_t)std::min<uint64_t>(cap, rhi - rb);
                size_t off = 0;
                for (auto &o : out) {
                    if (o.host)
                        CU(c, cudaMemcpyAsync(static_cast<unsigned char *>(o.host) + rb * o.bytes, dgat + (rk * row_bytes + off) * P,
                                              rcnt * o.bytes, cudaMemcpyDeviceToHost, s.s_compute));
                    off += o.bytes;
                }
            }
        }
    }
    return sync_all(c);
}

template <int KB>
void nb_launch(bool self, const NbArgs &a, uint32_t k, uint32_t *idx, float *dist, cudaStream_t st)
{
    const dim3 grid((a.count + nb_tile(KB) - 1) / nb_tile(KB), a.n_chunks);
    if (self)
        neighbors_kernel<KB, true><<<grid, NB_THREADS, nb_smem_bytes(), st>>>(a);
    else
        neighbors_kernel<KB, false><<<grid, NB_THREADS, nb_smem_bytes(), st>>>(a);
    nb_merge_kernel<KB><<<(a.count + 127) / 128, 128, 0, st>>>(a.cd2, a.cidx, a.n_chunks, a.stride, a.count, k, idx, dist);
}

// ------------------------------------------------------------------------------------------------ test particles
// Device bytes of one shard's tracer set (include/b200nb.h states the same formula)
uint64_t tracer_bytes(uint64_t T, uint32_t cap, uint32_t S) { return 36 * T + 16 * (uint64_t)S * cap; }

// the expansion's [4][tr_T] tracer rows of every shard (callers have joined the streams)
void free_ext_tracers(b200nb_ctx *c)
{
    for (auto &s : c->shards) {
        if (!s.ext_tr) continue;
        cudaSetDevice(s.device);
        cudaFree(s.ext_tr);
        s.ext_tr = nullptr;
        s.bytes -= 32 * c->tr_T;
    }
}

// with an expansion and tracers: the [4][tr_T] tracer rows of every shard that lacks them
cudaError_t alloc_ext_tracers(b200nb_ctx *c)
{
    for (auto &s : c->shards) {
        if (s.ext_tr) continue;
        cudaError_t e = cudaSetDevice(s.device);
        if (e == cudaSuccess) e = cudaMalloc((void **)&s.ext_tr, 32 * c->tr_T);
        if (e != cudaSuccess) { s.ext_tr = nullptr; (void)cudaGetLastError(); return e; }
        s.bytes += 32 * c->tr_T;
    }
    return cudaSuccess;
}

// the context holds no expansion afterwards (callers have joined the streams)
void free_ext_scf(b200nb_ctx *c)
{
    free_ext_tracers(c);
    for (auto &s : c->shards) {
        if (s.ext_coef || s.ext_body) {
            cudaSetDevice(s.device);
            cudaFree(s.ext_coef);
            cudaFree(s.ext_body);
        }
        if (s.ext_body) s.bytes -= 32 * c->L;
        s.bytes -= s.ext_coef_bytes;
        s.ext_coef = nullptr;
        s.ext_body = nullptr;
        s.ext_coef_bytes = 0;
    }
    c->scf.on = false;
    c->scf.coef.clear();
}

// the context holds no tracers afterwards (callers have joined the streams)
void free_tracers(b200nb_ctx *c)
{
    free_ext_tracers(c);
    for (auto &s : c->shards) {
        if (s.tr || s.tr_part) {
            cudaSetDevice(s.device);
            cudaFree(s.tr);
            cudaFree(s.tr_part);
        }
        s.tr = s.tr_part = nullptr;
        s.bytes -= s.tr_bytes;
        s.tr_bytes = 0;
        s.tr_local = 0;
    }
    c->m_tracers = c->tr_T = 0;
    c->tr_cap = 0;
    c->tr_acc_valid = false;
}

// The field of the current body array at every tracer of every shard, in batches of at most FIELD_BATCH targets, each
// batch summed and applied by tracer_update_kernel (TracerMode `mode`).  The pass reads the whole body array, so with
// several ranks it waits for the position exchange itself.
int enqueue_tracer_pass(b200nb_ctx *c, int mode, float dt)
{
    const uint32_t S = field_chunks(c->n);
    for (auto &s : c->shards) {
        if (s.tr_local == 0) continue;
        CU(c, cudaSetDevice(s.device));
        if (c->n_ranks > 1)
            if (int rc = wait_remote_positions(c, s)) return rc;
        if (c->scf.on) // the total external field at every tracer of the shard, before any batch moves one
            if (int rc = enqueue_ext_total(c, s, SoaPoints{s.tr, s.tr + c->tr_T, s.tr + 2 * c->tr_T}, s.tr_local,
                                           (uint32_t)c->tr_T, s.ext_tr))
                return rc;
        for (uint32_t base = 0; base < s.tr_local; base += c->tr_cap) {
            const uint32_t cnt = std::min(c->tr_cap, s.tr_local - base);
            FieldArgs a{};
            a.src = s.bodies;
            a.px = s.tr + base; a.py = s.tr + c->tr_T + base; a.pz = s.tr + 2 * c->tr_T + base;
            a.partial = s.tr_part;
            a.stride = c->tr_cap;
            a.count = cnt;
            a.src_nblk = (uint32_t)((c->n + BLK - 1) / BLK);
            a.n_chunks = S;
            a.soft2 = c->soft2;
            field_kernel<false><<<dim3((cnt + FIELD_TI - 1) / FIELD_TI, S), FIELD_THREADS, field_smem_bytes(), s.s_compute>>>(a);
            TracerArgs u{};
            u.partial = s.tr_part; u.n_chunks = S; u.stride = c->tr_cap; u.count = cnt;
            u.tr = s.tr + base; u.T = c->tr_T; u.dt = dt; u.mode = mode;
            if (c->scf.on)
                tracer_update_kernel<true, true><<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(u, c->ext, s.ext_tr + base);
            else if (c->ext.n > 0)
                tracer_update_kernel<true><<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(u, c->ext, nullptr);
            else
                tracer_update_kernel<false><<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(u, c->ext, nullptr);
            c->launches += 2;
            CU(c, cudaGetLastError());
        }
    }
    return B200NB_OK;
}

// the leapfrog's kick-drift of every tracer with its stored a(p); element-wise, no body is read
int enqueue_tracer_kick_drift(b200nb_ctx *c, float dt)
{
    for (auto &s : c->shards) {
        if (s.tr_local == 0) continue;
        CU(c, cudaSetDevice(s.device));
        tracer_kick_drift_kernel<<<(s.tr_local + 255) / 256, 256, 0, s.s_compute>>>(s.tr, c->tr_T, s.tr_local, dt);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    return B200NB_OK;
}

} // namespace

// =================================================================================================== C ABI
extern "C" {

int b200nb_create(b200nb_ctx **out, uint64_t n_bodies, int n_gpus, float G, float soft)
{
    int cur = 0, visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible < 1)
        return fail(nullptr, B200NB_ECUDA, "no CUDA device visible (libb200nb has no CPU fallback)");
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    if (n_gpus < 0 || n_gpus > visible) return fail(nullptr, B200NB_EINVAL, "n_gpus=%d but %d device(s) visible", n_gpus, visible);
    if (n_gpus == 0) n_gpus = visible;
    std::vector<int> ranks, devices;
    for (int i = 0; i < n_gpus; ++i) {
        ranks.push_back(i);
        devices.push_back(n_gpus == 1 ? cur : i);
    }
    return create_common(out, n_bodies, G, soft, n_gpus, ranks, devices, nullptr);
}

int b200nb_create_sharded(b200nb_ctx **out, uint64_t n_bodies, int n_shards, const int *devices, float G, float soft)
{
    int visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible < 1)
        return fail(nullptr, B200NB_ECUDA, "no CUDA device visible (libb200nb has no CPU fallback)");
    if (n_shards < 1 || n_shards > MAX_PUSH_TARGETS || !devices)
        return fail(nullptr, B200NB_EINVAL, "n_shards must be in [1, %d] with a device list", MAX_PUSH_TARGETS);
    std::vector<int> ranks, devs;
    for (int i = 0; i < n_shards; ++i) {
        if (devices[i] < 0 || devices[i] >= visible) return fail(nullptr, B200NB_EINVAL, "device %d not visible", devices[i]);
        ranks.push_back(i);
        devs.push_back(devices[i]);
    }
    return create_common(out, n_bodies, G, soft, n_shards, ranks, devs, nullptr);
}

int b200nb_create_rank(b200nb_ctx **out, uint64_t n_bodies, float G, float soft, int rank, int n_ranks, int device,
                       const void *nccl_id)
{
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(nullptr, B200NB_EINVAL, "bad rank %d of %d", rank, n_ranks);
    int visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible < 1)
        return fail(nullptr, B200NB_ECUDA, "no CUDA device visible (libb200nb has no CPU fallback)");
    if (device < 0 || device >= visible) return fail(nullptr, B200NB_EINVAL, "device %d not visible", device);
    if (n_ranks > 1 && !nccl_id) return fail(nullptr, B200NB_EINVAL, "nccl_id is required for n_ranks > 1");
    return create_common(out, n_bodies, G, soft, n_ranks, {rank}, {device}, nccl_id);
}

int b200nb_comm_unique_id(void *id128)
{
    if (!id128) return fail(nullptr, B200NB_EINVAL, "id128 is NULL");
    if (!g_nccl.load()) return fail(nullptr, B200NB_ENCCL, "%s", g_nccl.err.c_str());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    ncclResult_t r = g_nccl.GetUniqueId(&id);
    if (r != ncclSuccess) return fail(nullptr, B200NB_ENCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString(r));
    memcpy(id128, &id, sizeof id);
    return B200NB_OK;
}

void b200nb_destroy(b200nb_ctx *c)
{
    if (!c) return;
    DeviceGuard guard;
    for (auto &s : c->shards) { // join before anything the streams may still be using goes away
        if (cudaSetDevice(s.device) != cudaSuccess) continue;
        if (s.s_compute) cudaStreamSynchronize(s.s_compute);
        if (s.s_comm) cudaStreamSynchronize(s.s_comm);
    }
    for (auto &g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    for (auto &s : c->shards) {
        if (cudaSetDevice(s.device) != cudaSuccess) continue;
        if (s.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(s.comm);
        if (s.resched_mod) g_drv.ModuleUnload(s.resched_mod);
        for (auto e : s.prof) cudaEventDestroy(e);
        for (auto e : s.prof_free) cudaEventDestroy(e);
        cudaFree(s.bodies); cudaFree(s.bodies_next); cudaFree(s.vel); cudaFree(s.acc); cudaFree(s.mass); cudaFree(s.partial); cudaFree(s.stage); cudaFree(s.stage_full);
        cudaFree(s.energy_blocks); cudaFree(s.energy_out); cudaFree(s.l2_scratch); cudaFree(s.query_buf);
        cudaFree(s.tr); cudaFree(s.tr_part);
        cudaFree(s.ext_coef); cudaFree(s.ext_body); cudaFree(s.ext_tr);
        for (auto t : s.timer) if (t) cudaEventDestroy(t);
        if (s.ev_integrated) cudaEventDestroy(s.ev_integrated);
        if (s.ev_gathered) cudaEventDestroy(s.ev_gathered);
        if (s.ev_pushed) cudaEventDestroy(s.ev_pushed);
        if (s.s_compute) cudaStreamDestroy(s.s_compute);
        if (s.s_comm) cudaStreamDestroy(s.s_comm);
    }
    delete c;
}

const char *b200nb_last_error(const b200nb_ctx *c) { return c ? c->err.c_str() : g_create_error.c_str(); }

// After an upload every shard holds only its own slice of the blocked array: replicate it everywhere (the same exchange
// a step performs).  p2p: each shard copies its slice into both halves of every shard's double buffer (G*m and the
// padding bodies live in the buffers too); NCCL: the in-place all-gather.
static int publish_slices(b200nb_ctx *c)
{
    if (c->n_ranks == 1) return B200NB_OK;
    if (!c->p2p) return enqueue_gather(c);
    const size_t slice_floats = (size_t)c->L * 4;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        const float *mine = s.bodies + (size_t)s.rank * slice_floats;
        for (auto &o : c->shards) {
            if (&o != &s)
                CU(c, cudaMemcpyAsync(o.bodies + (size_t)s.rank * slice_floats, mine, slice_floats * 4, cudaMemcpyDefault, s.s_compute));
            CU(c, cudaMemcpyAsync(o.bodies_next + (size_t)s.rank * slice_floats, mine, slice_floats * 4, cudaMemcpyDefault, s.s_compute));
        }
        CU(c, cudaEventRecord(s.ev_pushed, s.s_compute));
    }
    return B200NB_OK;
}

int b200nb_upload(b200nb_ctx *c, const float *qx, const float *qy, const float *qz, const float *m, const float *vx,
                  const float *vy, const float *vz)
{
    if (!c) return B200NB_EINVAL;
    if (!qx || !qy || !qz || !m || !vx || !vy || !vz) return fail(c, B200NB_EINVAL, "upload: NULL array");
    DeviceGuard guard;
    const float *src[7] = {qx, qy, qz, m, vx, vy, vz};
    if (c->p2p) { // peers may still be storing positions into this GPU's buffers
        if (int rc = sync_all(c)) return rc;
    }
    const float px = qx[c->n - 1], py = qy[c->n - 1], pz = qz[c->n - 1]; // where the padding bodies sit
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        // the previous step's gather may still be writing remote slices of `bodies`
        CU(c, cudaStreamWaitEvent(s.s_compute, s.ev_gathered, 0));
        // only the shard's own bodies cross the host link (7 x 4 B each); the exchange below replicates the positions
        const size_t first = (size_t)s.rank * c->L;
        if (s.n_local > 0)
            for (int k = 0; k < 7; ++k)
                CU(c, cudaMemcpyAsync(s.stage + (size_t)k * c->L, src[k] + first, (size_t)s.n_local * 4, cudaMemcpyHostToDevice, s.s_compute));
        const int grid = (int)std::min<uint64_t>((c->L + 255) / 256, (uint64_t)s.n_sms * 8);
        pack_slice_kernel<<<grid, 256, 0, s.s_compute>>>(s.stage, (uint32_t)c->L, s.n_local, first, px, py, pz, c->G, s.bodies,
                                                        s.vel, s.mass);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    if (int rc = publish_slices(c)) return rc;
    // host pointers are only borrowed for the call: the copies must have left them (pinned memory is truly async)
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaStreamSynchronize(s.s_compute));
    }
    c->uploaded = true;
    c->acc_valid = false;
    c->tr_acc_valid = false; // the tracers stay, their stored a(p) was taken in the old field
    return B200NB_OK;
}

// positions and velocities of the local shards' own bodies into the global-index host arrays (other entries untouched)
static int download_local(b200nb_ctx *c, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz)
{
    float *q[3] = {qx, qy, qz}, *v[3] = {vx, vy, vz};
    for (auto &s : c->shards) {
        if (s.n_local == 0) continue;
        CU(c, cudaSetDevice(s.device));
        const size_t first = (size_t)s.rank * c->L;
        if (qx || qy || qz) {
            const int grid = (int)std::min<uint64_t>((s.n_local + 255) / 256, (uint64_t)s.n_sms * 8);
            unpack_positions_kernel<<<grid, 256, 0, s.s_compute>>>(s.bodies, first, s.n_local, s.stage, c->L);
            c->launches++;
            CU(c, cudaGetLastError());
        }
        for (int k = 0; k < 3; ++k) {
            if (q[k])
                CU(c, cudaMemcpyAsync(q[k] + first, s.stage + (size_t)k * c->L, (size_t)s.n_local * 4, cudaMemcpyDeviceToHost, s.s_compute));
            if (v[k])
                CU(c, cudaMemcpyAsync(v[k] + first, s.vel + (size_t)k * c->L, (size_t)s.n_local * 4, cudaMemcpyDeviceToHost, s.s_compute));
        }
    }
    return sync_all(c);
}

int b200nb_download_state(b200nb_ctx *c, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "download_state before upload");
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    if (c->shards.size() == (size_t)c->n_ranks) // every shard is local: each one returns its own slice over its own link
        return download_local(c, qx, qy, qz, vx, vy, vz);
    // one rank per process: positions are replicated, so this rank's device has all of them after the gather
    if (qx || qy || qz) {
        Shard &s = c->shards[0];
        CU(c, cudaSetDevice(s.device));
        if (!s.stage_full) {
            CU(c, cudaMalloc((void **)&s.stage_full, 3 * c->stage_stride * 4));
            s.bytes += 3 * c->stage_stride * 4;
        }
        const int grid = (int)std::min<uint64_t>((c->n + 255) / 256, (uint64_t)s.n_sms * 8);
        unpack_positions_kernel<<<grid, 256, 0, s.s_compute>>>(s.bodies, 0, c->n, s.stage_full, c->stage_stride);
        c->launches++;
        CU(c, cudaGetLastError());
        float *dst[3] = {qx, qy, qz};
        for (int k = 0; k < 3; ++k)
            if (dst[k])
                CU(c, cudaMemcpyAsync(dst[k], s.stage_full + (size_t)k * c->stage_stride, c->n * 4, cudaMemcpyDeviceToHost, s.s_compute));
        CU(c, cudaStreamSynchronize(s.s_compute));
    }
    if (vx || vy || vz) return download_sliced(c, &Shard::vel, vx, vy, vz);
    return B200NB_OK;
}

int b200nb_download_slice(b200nb_ctx *c, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "download_slice before upload");
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    return download_local(c, qx, qy, qz, vx, vy, vz);
}

int b200nb_slice_bounds(const b200nb_ctx *c, int local_shard, uint64_t *first, uint64_t *count)
{
    if (!c || local_shard < 0 || (size_t)local_shard >= c->shards.size()) return B200NB_EINVAL;
    const Shard &s = c->shards[local_shard];
    if (first) *first = std::min<uint64_t>((uint64_t)s.rank * c->L, c->n);
    if (count) *count = s.n_local;
    return B200NB_OK;
}

int b200nb_download_accel(b200nb_ctx *c, float *ax, float *ay, float *az)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "download_accel before upload");
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    return download_sliced(c, &Shard::acc, ax, ay, az);
}

// one iteration, enqueued on the compute stream(s).  Tracers (if any) read the body positions of the same instant as the
// bodies' own accelerations: q_n for MUrB, so their pass precedes the integrator, which overwrites the own slice in
// place (or, p2p, swaps `bodies`); q_{n+1} for the leapfrog's closing kick, read from the current `bodies` after the swap.
static int enqueue_one_step(b200nb_ctx *c, float dt, int integrator)
{
    const bool tracers = c->m_tracers > 0;
    if (integrator == B200NB_INTEGRATOR_MURB) {
        if (int rc = enqueue_force(c)) return rc;
        if (tracers)
            if (int rc = enqueue_tracer_pass(c, TM_MURB, dt)) return rc;
        if (int rc = enqueue_integrate(c, IM_MURB, dt)) return rc;
        if (int rc = enqueue_gather(c)) return rc;
        c->acc_valid = false; // acc belongs to the positions before the update
        c->tr_acc_valid = false;
    } else {
        if (!c->acc_valid) { // a(x_0): once after an upload
            if (int rc = enqueue_force(c)) return rc;
            if (int rc = enqueue_integrate(c, IM_REDUCE_ONLY, dt)) return rc;
        }
        if (tracers && !c->tr_acc_valid) // a(p_0; q_0): once after the tracers, the bodies or the scheme changed
            if (int rc = enqueue_tracer_pass(c, TM_LF_ACC, dt)) return rc;
        if (int rc = enqueue_integrate(c, IM_LF_KICK_DRIFT, dt)) return rc;
        if (int rc = enqueue_gather(c)) return rc;
        if (tracers) // beside the exchange
            if (int rc = enqueue_tracer_kick_drift(c, dt)) return rc;
        if (int rc = enqueue_force(c)) return rc;
        if (tracers)
            if (int rc = enqueue_tracer_pass(c, TM_LF_KICK, dt)) return rc;
        if (int rc = enqueue_integrate(c, IM_LF_KICK, dt)) return rc;
        c->acc_valid = true; // acc == a(x_{n+1})
        c->tr_acc_valid = tracers;
    }
    return B200NB_OK;
}

// Long single-GPU runs replay a captured CUDA graph of GRAPH_STEPS iterations: at murb-test sizes (N ~ 2k) an
// iteration is a few microseconds of GPU work behind two launches, so launch latency is the whole cost.
static int get_step_graph(b200nb_ctx *c, float dt, int integrator, StepGraph **out)
{
    for (auto &g : c->graphs)
        if (g.integrator == integrator && g.dt == dt && g.steps == GRAPH_STEPS) { *out = &g; return B200NB_OK; }
    Shard &s = c->shards[0];
    CU(c, cudaSetDevice(s.device));
    const uint64_t before = c->launches;
    const bool acc_valid = c->acc_valid, tr_acc_valid = c->tr_acc_valid;
    CU(c, cudaStreamBeginCapture(s.s_compute, cudaStreamCaptureModeThreadLocal));
    int rc = B200NB_OK;
    for (int i = 0; i < GRAPH_STEPS && rc == B200NB_OK; ++i) rc = enqueue_one_step(c, dt, integrator);
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(s.s_compute, &graph);
    StepGraph g;
    g.integrator = integrator; g.dt = dt; g.steps = GRAPH_STEPS; g.launches = c->launches - before;
    c->launches = before;      // nothing ran yet
    c->acc_valid = acc_valid;
    c->tr_acc_valid = tr_acc_valid;
    if (rc != B200NB_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) return fail(c, B200NB_ECUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
    const cudaError_t ei = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) return fail(c, B200NB_ECUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ei));
    // one executable graph per (integrator, dt): callers that change dt all the time would otherwise grow this
    // list without bound.  Eviction is rare: join the stream first so no launch of the evicted graph is in flight.
    while (c->graphs.size() >= GRAPH_CACHE_MAX) {
        CU(c, cudaStreamSynchronize(s.s_compute));
        cudaGraphExecDestroy(c->graphs.front().exec);
        c->graphs.erase(c->graphs.begin());
    }
    c->graphs.push_back(g);
    *out = &c->graphs.back();
    return B200NB_OK;
}

int b200nb_step(b200nb_ctx *c, float dt, int integrator, int n_steps)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "step before upload");
    if (integrator != B200NB_INTEGRATOR_MURB && integrator != B200NB_INTEGRATOR_LEAPFROG)
        return fail(c, B200NB_EINVAL, "unknown integrator %d", integrator);
    if (n_steps < 0) return fail(c, B200NB_EINVAL, "n_steps < 0");
    DeviceGuard guard;
    int it = 0;
    static const bool no_graph = getenv("B200NB_NO_GRAPH") != nullptr;
    if (c->n_ranks == 1 && !c->profiling && !no_graph && n_steps >= GRAPH_MIN_STEPS) {
        // the one-off a(x_0) and tracer a(p_0) passes stay outside the graph
        if (integrator == B200NB_INTEGRATOR_LEAPFROG && (!c->acc_valid || (c->m_tracers > 0 && !c->tr_acc_valid))) {
            if (int rc = enqueue_one_step(c, dt, integrator)) return rc;
            ++it;
        }
        StepGraph *g = nullptr;
        if (int rc = get_step_graph(c, dt, integrator, &g)) return rc;
        Shard &s = c->shards[0];
        CU(c, cudaSetDevice(s.device));
        for (; it + GRAPH_STEPS <= n_steps; it += GRAPH_STEPS) {
            CU(c, cudaGraphLaunch(g->exec, s.s_compute));
            c->launches += g->launches;
        }
        c->acc_valid = integrator == B200NB_INTEGRATOR_LEAPFROG;
        c->tr_acc_valid = c->acc_valid && c->m_tracers > 0;
    }
    for (; it < n_steps; ++it)
        if (int rc = enqueue_one_step(c, dt, integrator)) return rc;
    return B200NB_OK;
}

int b200nb_accel(b200nb_ctx *c)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "accel before upload");
    DeviceGuard guard;
    if (int rc = enqueue_force(c)) return rc;
    if (int rc = enqueue_integrate(c, IM_REDUCE_ONLY, 0.f)) return rc;
    c->acc_valid = true;
    return B200NB_OK;
}

int b200nb_integrate_host_accel(b200nb_ctx *c, const float *ax, const float *ay, const float *az, float dt)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "integrate before upload");
    if (!ax || !ay || !az) return fail(c, B200NB_EINVAL, "integrate_host_accel: NULL array");
    DeviceGuard guard;
    const float *src[3] = {ax, ay, az};
    for (auto &s : c->shards) {
        if (s.n_local == 0) continue;
        CU(c, cudaSetDevice(s.device));
        // an in-place all-gather of a preceding asynchronous step may still be sending this slice from the comm stream
        if (c->n_ranks > 1 && !c->p2p) CU(c, cudaStreamWaitEvent(s.s_compute, s.ev_gathered, 0));
        for (int k = 0; k < 3; ++k)
            CU(c, cudaMemcpyAsync(s.stage + (size_t)k * c->L, src[k] + (size_t)s.rank * c->L, (size_t)s.n_local * 4,
                                  cudaMemcpyHostToDevice, s.s_compute));
        load_acc_kernel<<<(s.n_local + 255) / 256, 256, 0, s.s_compute>>>(s.stage, c->L, s.n_local, s.acc, c->L);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    if (int rc = enqueue_integrate(c, IM_MURB_STORED, dt)) return rc;
    if (int rc = enqueue_gather(c)) return rc;
    c->acc_valid = false;
    c->tr_acc_valid = false; // the bodies moved, the tracers did not
    return sync_all(c); // borrowed host pointers (see upload)
}

// raw[MR_COUNT]: the metric rows summed over every body of every rank
static int metric_sums(b200nb_ctx *c, double *raw)
{
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "metrics before upload");
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc; // positions gathered, velocities final
    for (int k = 0; k < MR_COUNT; ++k) raw[k] = 0.0;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        const uint32_t nb = (s.n_local + ENERGY_THREADS - 1) / ENERGY_THREADS;
        double part[MR_COUNT];
        if (nb > 0) {
            if (c->scf.on)
                if (int rc = enqueue_ext_total_bodies(c, s)) return rc;
            auto energy = c->scf.on ? energy_kernel<true, true> : c->ext.n > 0 ? energy_kernel<true> : energy_kernel<false>;
            energy<<<nb, ENERGY_THREADS, 0, s.s_compute>>>(s.bodies, s.vel, s.mass, (uint32_t)c->L, s.n_local,
                                                          (uint64_t)s.rank * c->L, c->nblk_total, c->soft2,
                                                          s.energy_blocks, c->ext, s.ext_body);
            energy_final_kernel<<<MR_COUNT, 256, 0, s.s_compute>>>(s.energy_blocks, nb, s.energy_out);
            c->launches += 2;
            CU(c, cudaGetLastError());
        } else {
            CU(c, cudaMemsetAsync(s.energy_out, 0, 8 * MR_COUNT, s.s_compute));
        }
        if (c->shards.size() != (size_t)c->n_ranks) // one rank per process: sum over ranks on the device
            NC(c, g_nccl.AllReduce(s.energy_out, s.energy_out, MR_COUNT, ncclDouble, ncclSum, s.comm, s.s_compute));
        CU(c, cudaMemcpyAsync(part, s.energy_out, 8 * MR_COUNT, cudaMemcpyDeviceToHost, s.s_compute));
        CU(c, cudaStreamSynchronize(s.s_compute));
        for (int k = 0; k < MR_COUNT; ++k) raw[k] += part[k];
    }
    return B200NB_OK;
}

int b200nb_energy(b200nb_ctx *c, double *total)
{
    if (!c || !total) return B200NB_EINVAL;
    double raw[MR_COUNT];
    if (int rc = metric_sums(c, raw)) return rc;
    *total = raw[MR_ENERGY];
    return B200NB_OK;
}

int b200nb_metrics(b200nb_ctx *c, double *out)
{
    if (!c || !out) return B200NB_EINVAL;
    double raw[MR_COUNT];
    if (int rc = metric_sums(c, raw)) return rc;
    out[B200NB_METRIC_ENERGY] = raw[MR_ENERGY];
    out[B200NB_METRIC_ANG_X] = raw[MR_LX];
    out[B200NB_METRIC_ANG_Y] = raw[MR_LY];
    out[B200NB_METRIC_ANG_Z] = raw[MR_LZ];
    out[B200NB_METRIC_MASS] = raw[MR_M];
    for (int k = 0; k < 3; ++k) {
        out[B200NB_METRIC_COM_X + k] = raw[MR_M] != 0.0 ? raw[MR_MX + k] / raw[MR_M] : 0.0;
        out[B200NB_METRIC_DENSITY_X + k] = raw[MR_W] != 0.0 ? raw[MR_WX + k] / raw[MR_W] : out[B200NB_METRIC_COM_X + k];
    }
    return B200NB_OK;
}

// Field at points (self == false) or potential of every body (self == true): [S][4][cap] partial rows, summed into
// four [cap] rows (ax, ay, az, phi).
static int field_run(b200nb_ctx *c, bool self, uint64_t m, const float *const pts[3], float *const out[4])
{
    const uint32_t S = field_chunks(c->n);
    std::vector<TargetOut> outs;
    for (int q = 0; q < 4; ++q) outs.push_back({out[q], 4});
    auto work = [&](uint32_t cap) { return (size_t)S * 4 * cap * 4; };
    auto launch = [&](Shard &s, uint64_t base, uint32_t cnt, uint32_t cap, unsigned char *wk, const float *dpts,
                      unsigned char *dout) -> int {
        FieldArgs a{};
        a.src = s.bodies;
        a.partial = reinterpret_cast<float *>(wk);
        a.stride = cap;
        a.count = cnt;
        a.src_nblk = (uint32_t)((c->n + BLK - 1) / BLK);
        a.n_chunks = S;
        a.soft2 = c->soft2;
        const dim3 grid((cnt + FIELD_TI - 1) / FIELD_TI, S);
        if (self) {
            a.self0 = base; // a multiple of BLK: slices and batches are
            field_kernel<true><<<grid, FIELD_THREADS, field_smem_bytes(), s.s_compute>>>(a);
        } else {
            a.px = dpts; a.py = dpts + cap; a.pz = dpts + 2 * (size_t)cap;
            field_kernel<false><<<grid, FIELD_THREADS, field_smem_bytes(), s.s_compute>>>(a);
        }
        field_reduce_kernel<<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(a.partial, S, cap, cnt, reinterpret_cast<float *>(dout));
        c->launches += 2;
        return B200NB_OK;
    };
    return run_targets(c, self, m, pts, FIELD_TI, FIELD_BATCH, outs, work, launch);
}

int b200nb_field(b200nb_ctx *c, uint64_t n_points, const float *px, const float *py, const float *pz, float *ax, float *ay,
                 float *az, float *phi)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "field before upload");
    if (n_points == 0) return B200NB_OK;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "field: NULL point array");
    const float *pts[3] = {px, py, pz};
    float *out[4] = {ax, ay, az, phi};
    return field_run(c, false, n_points, pts, out);
}

int b200nb_potential(b200nb_ctx *c, float *phi)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "potential before upload");
    if (!phi) return fail(c, B200NB_EINVAL, "potential: phi is NULL");
    float *out[4] = {nullptr, nullptr, nullptr, phi};
    return field_run(c, true, c->n, nullptr, out);
}

// Tidal tensor at points (self == false) or of every body (self == true): [S][7][cap] partial rows, summed into one
// [cap][6] row block (xx, yy, zz, xy, xz, yz).
static int tidal_run(b200nb_ctx *c, bool self, uint64_t m, const float *const pts[3], float *t)
{
    const uint32_t S = field_chunks(c->n);
    const std::vector<TargetOut> outs = {{t, 6 * 4}};
    auto work = [&](uint32_t cap) { return (size_t)S * TIDAL_NQ * cap * 4; };
    auto launch = [&](Shard &s, uint64_t base, uint32_t cnt, uint32_t cap, unsigned char *wk, const float *dpts,
                      unsigned char *dout) -> int {
        FieldArgs a{};
        a.src = s.bodies;
        a.partial = reinterpret_cast<float *>(wk);
        a.stride = cap;
        a.count = cnt;
        a.src_nblk = (uint32_t)((c->n + BLK - 1) / BLK);
        a.n_chunks = S;
        a.soft2 = c->soft2;
        const dim3 grid((cnt + TIDAL_TI - 1) / TIDAL_TI, S);
        if (self) {
            a.self0 = base; // a multiple of BLK: slices and batches are
            tidal_kernel<true><<<grid, TIDAL_THREADS, tidal_smem_bytes(), s.s_compute>>>(a);
        } else {
            a.px = dpts; a.py = dpts + cap; a.pz = dpts + 2 * (size_t)cap;
            tidal_kernel<false><<<grid, TIDAL_THREADS, tidal_smem_bytes(), s.s_compute>>>(a);
        }
        tidal_reduce_kernel<<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(a.partial, S, cap, cnt, reinterpret_cast<float *>(dout));
        c->launches += 2;
        return B200NB_OK;
    };
    return run_targets(c, self, m, pts, TIDAL_TI, TIDAL_BATCH, outs, work, launch);
}

int b200nb_tidal(b200nb_ctx *c, uint64_t n_points, const float *px, const float *py, const float *pz, float *t)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "tidal before upload");
    if (n_points == 0) return B200NB_OK;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "tidal: NULL point array");
    if (!t) return fail(c, B200NB_EINVAL, "tidal: t is NULL");
    const float *pts[3] = {px, py, pz};
    return tidal_run(c, false, n_points, pts, t);
}

int b200nb_tidal_bodies(b200nb_ctx *c, float *t)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "tidal_bodies before upload");
    if (!t) return fail(c, B200NB_EINVAL, "tidal_bodies: t is NULL");
    return tidal_run(c, true, c->n, nullptr, t);
}

// Scratch of the component calls (components_sm100.cuh) ahead of run_targets' points and rows, the same on every shard;
// each array is rounded up to 256 B.
struct CompBufs {
    float *partial, *src;
    uint32_t *map, *pos, *chunk0;
    uint2 *chunk;
    size_t total;
};

static CompBufs comp_carve(unsigned char *base, uint32_t n_chunks, uint32_t cap, uint32_t T, uint32_t n_pos, uint32_t C)
{
    CompBufs b{};
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char *p = base ? base + off : nullptr; off += (bytes + 255) / 256 * 256; return p; };
    b.partial = reinterpret_cast<float *>(take((size_t)16 * n_chunks * cap));
    b.src = reinterpret_cast<float *>(take((size_t)16 * T));
    b.map = reinterpret_cast<uint32_t *>(take((size_t)4 * T));
    b.pos = reinterpret_cast<uint32_t *>(take((size_t)4 * n_pos));
    b.chunk = reinterpret_cast<uint2 *>(take((size_t)8 * n_chunks));
    b.chunk0 = reinterpret_cast<uint32_t *>(take((size_t)4 * (C + 1)));
    b.total = off;
    return b;
}

// Field by source component at points (self == false) or of every body (self == true); labels already checked.
// The host sorts the members, packs their order and cuts the chunks; every shard packs the same source array once per
// call, then runs its targets in batches: [sum S][4][cap] partial rows, summed per component into [cap][C][3] and
// [cap][C] rows.
static int component_run(b200nb_ctx *c, const uint32_t *comp, uint32_t C, bool self, uint64_t m, const float *const pts[3],
                         float *acc, float *phi)
{
    const uint32_t n = (uint32_t)c->n;
    std::vector<uint32_t> cnt(C, 0);
    for (uint32_t i = 0; i < n; ++i)
        if (comp[i] != B200NB_NO_GROUP) cnt[comp[i]]++;
    // component h: packed blocks [blk0[h], blk0[h] + nblk_h), chunks [chunk0[h], chunk0[h + 1]) cut as field_kernel cuts
    std::vector<uint32_t> blk0(C), chunk0(C + 1);
    std::vector<uint2> chunk;
    uint32_t nb = 0, max_chunk = 0;
    for (uint32_t h = 0; h < C; ++h) {
        const uint32_t nblk = (cnt[h] + BLK - 1) / BLK, S = cnt[h] ? field_chunks(cnt[h]) : 0;
        blk0[h] = nb;
        chunk0[h] = (uint32_t)chunk.size();
        for (uint32_t k = 0; k < S; ++k) {
            const uint2 r = make_uint2(nb + (uint32_t)((uint64_t)nblk * k / S), nb + (uint32_t)((uint64_t)nblk * (k + 1) / S));
            max_chunk = std::max(max_chunk, r.y - r.x);
            chunk.push_back(r);
        }
        nb += nblk;
    }
    const uint32_t n_chunks = (uint32_t)chunk.size();
    chunk0[C] = n_chunks;
    const uint32_t T = nb * BLK;
    // the stable (component, index) order: map[packed position] = body (padding: COMP_PAD | h's last member), pos = its inverse
    std::vector<uint32_t> map(T), pos(self ? n : 0), next(C);
    for (uint32_t h = 0; h < C; ++h) next[h] = blk0[h] * BLK;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t h = comp[i];
        if (h == B200NB_NO_GROUP) {
            if (self) pos[i] = COMP_NONE;
            continue;
        }
        map[next[h]] = i;
        if (self) pos[i] = next[h];
        next[h]++;
    }
    for (uint32_t h = 0; h < C; ++h)
        for (uint32_t p = next[h]; p < (blk0[h] + (cnt[h] + BLK - 1) / BLK) * BLK; ++p) map[p] = map[next[h] - 1] | COMP_PAD;

    const uint32_t batch = std::min<uint32_t>(FIELD_BATCH, std::max<uint32_t>(1, COMP_PARTIAL_FLOATS / 4 / std::max(n_chunks, 1u) / FIELD_TI) * FIELD_TI);
    const std::vector<TargetOut> outs = {{acc, 12 * (size_t)C}, {phi, 4 * (size_t)C}};
    auto work = [&](uint32_t cap) { return comp_carve(nullptr, n_chunks, cap, T, (uint32_t)pos.size(), C).total; };
    std::vector<char> packed(c->shards.size(), 0);
    auto launch = [&](Shard &s, uint64_t base, uint32_t cnt_, uint32_t cap, unsigned char *wk, const float *dpts,
                      unsigned char *dout) -> int {
        const CompBufs b = comp_carve(wk, n_chunks, cap, T, (uint32_t)pos.size(), C);
        char &done = packed[&s - c->shards.data()];
        if (!done) { // once per shard and call: the tables and the packed sources
            if (T) CU(c, cudaMemcpyAsync(b.map, map.data(), (size_t)4 * T, cudaMemcpyHostToDevice, s.s_compute));
            if (self) CU(c, cudaMemcpyAsync(b.pos, pos.data(), (size_t)4 * n, cudaMemcpyHostToDevice, s.s_compute));
            if (n_chunks) CU(c, cudaMemcpyAsync(b.chunk, chunk.data(), (size_t)8 * n_chunks, cudaMemcpyHostToDevice, s.s_compute));
            CU(c, cudaMemcpyAsync(b.chunk0, chunk0.data(), (size_t)4 * (C + 1), cudaMemcpyHostToDevice, s.s_compute));
            if (T) {
                component_pack_kernel<<<(T + 255) / 256, 256, 0, s.s_compute>>>(s.bodies, b.map, T, b.src);
                c->launches++;
            }
            done = 1;
        }
        float *dacc = reinterpret_cast<float *>(dout), *dphi = dacc + (size_t)3 * C * cap;
        if (n_chunks) {
            CompArgs a{};
            a.src = b.src;
            a.chunk = b.chunk;
            a.partial = b.partial;
            a.stride = cap;
            a.count = cnt_;
            a.soft2 = c->soft2;
            const dim3 grid((cnt_ + FIELD_TI - 1) / FIELD_TI, n_chunks);
            if (self) {
                a.bodies = s.bodies;
                a.pos = b.pos;
                a.self0 = base;
                component_field_kernel<true><<<grid, FIELD_THREADS, comp_smem_bytes(max_chunk), s.s_compute>>>(a);
            } else {
                a.px = dpts; a.py = dpts + cap; a.pz = dpts + 2 * (size_t)cap;
                component_field_kernel<false><<<grid, FIELD_THREADS, field_smem_bytes(), s.s_compute>>>(a);
            }
            c->launches++;
        }
        component_reduce_kernel<<<dim3((cnt_ + 255) / 256, C), 256, 0, s.s_compute>>>(b.partial, b.chunk0, cap, cnt_, C, dacc, dphi);
        c->launches++;
        return B200NB_OK;
    };
    return run_targets(c, self, m, pts, FIELD_TI, batch, outs, work, launch);
}

// B200NB_EINVAL unless comp is non-NULL, n_comp is in [1, COMP_MAX] and every label is < n_comp or B200NB_NO_GROUP
static int component_labels(b200nb_ctx *c, const char *what, const uint32_t *comp, uint32_t n_comp)
{
    if (!comp) return fail(c, B200NB_EINVAL, "%s: comp is NULL", what);
    if (n_comp < 1 || n_comp > COMP_MAX) return fail(c, B200NB_EINVAL, "%s: n_comp = %u outside [1, %u]", what, n_comp, COMP_MAX);
    for (uint64_t i = 0; i < c->n; ++i)
        if (comp[i] >= n_comp && comp[i] != B200NB_NO_GROUP)
            return fail(c, B200NB_EINVAL, "%s: comp[%llu] = %u is neither < n_comp nor B200NB_NO_GROUP", what, (unsigned long long)i, comp[i]);
    return B200NB_OK;
}

int b200nb_component_field(b200nb_ctx *c, const uint32_t *comp, uint32_t n_comp, uint64_t n_points, const float *px,
                           const float *py, const float *pz, float *acc, float *phi)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "component_field before upload");
    if (n_points == 0) return B200NB_OK;
    if (int rc = component_labels(c, "component_field", comp, n_comp)) return rc;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "component_field: NULL point array");
    const float *pts[3] = {px, py, pz};
    return component_run(c, comp, n_comp, false, n_points, pts, acc, phi);
}

int b200nb_component_field_bodies(b200nb_ctx *c, const uint32_t *comp, uint32_t n_comp, float *acc, float *phi)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "component_field_bodies before upload");
    if (int rc = component_labels(c, "component_field_bodies", comp, n_comp)) return rc;
    return component_run(c, comp, n_comp, true, c->n, nullptr, acc, phi);
}

// k nearest bodies of the points (self == false) or of every body (self == true): [S][KB][cap] candidate d2 bits and
// indices, merged into [cap][k] index and distance rows.
static int neighbors_run(b200nb_ctx *c, bool self, uint64_t m, const float *const pts[3], uint32_t k, uint32_t *idx, float *dist)
{
    const int kb = nb_bucket((int)k);
    const uint32_t src_nblk = (uint32_t)((c->n + BLK - 1) / BLK);
    std::vector<TargetOut> outs = {{idx, 4 * (size_t)k}, {dist, 4 * (size_t)k}};
    auto work = [&](uint32_t cap) { return (size_t)nb_max_chunks(kb, cap) * kb * cap * 8; };
    auto launch = [&](Shard &s, uint64_t base, uint32_t cnt, uint32_t cap, unsigned char *wk, const float *dpts,
                      unsigned char *dout) -> int {
        NbArgs a{};
        a.src = s.bodies;
        a.self0 = self ? base : 0; // a multiple of BLK: slices and batches are
        a.px = dpts; a.py = dpts + cap; a.pz = dpts + 2 * (size_t)cap;
        a.n_chunks = nb_chunks(kb, cnt, cap, src_nblk, (uint32_t)s.n_sms * NB_MINB);
        a.cd2 = reinterpret_cast<uint32_t *>(wk);
        a.cidx = a.cd2 + (size_t)a.n_chunks * kb * cap;
        a.stride = cap;
        a.count = cnt;
        a.n = (uint32_t)c->n;
        a.src_nblk = src_nblk;
        uint32_t *didx = reinterpret_cast<uint32_t *>(dout);
        float *ddist = reinterpret_cast<float *>(dout + 4 * (size_t)k * cap);
        switch (kb) {
        case 1: nb_launch<1>(self, a, k, didx, ddist, s.s_compute); break;
        case 8: nb_launch<8>(self, a, k, didx, ddist, s.s_compute); break;
        case 16: nb_launch<16>(self, a, k, didx, ddist, s.s_compute); break;
        default: nb_launch<32>(self, a, k, didx, ddist, s.s_compute); break;
        }
        c->launches += 2;
        return B200NB_OK;
    };
    return run_targets(c, self, m, pts, nb_tile(kb), nb_batch(kb), outs, work, launch);
}

int b200nb_neighbors(b200nb_ctx *c, uint32_t k, uint32_t *idx, float *dist)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "neighbors before upload");
    if (k < 1 || k > (uint32_t)NB_K_MAX) return fail(c, B200NB_EINVAL, "neighbors: k = %u is outside [1, %d]", k, NB_K_MAX);
    return neighbors_run(c, true, c->n, nullptr, k, idx, dist);
}

int b200nb_neighbors_at(b200nb_ctx *c, uint64_t n_points, const float *px, const float *py, const float *pz, uint32_t k,
                        uint32_t *idx, float *dist)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "neighbors_at before upload");
    if (k < 1 || k > (uint32_t)NB_K_MAX) return fail(c, B200NB_EINVAL, "neighbors_at: k = %u is outside [1, %d]", k, NB_K_MAX);
    if (n_points == 0) return B200NB_OK;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "neighbors_at: NULL point array");
    const float *pts[3] = {px, py, pz};
    return neighbors_run(c, false, n_points, pts, k, idx, dist);
}

} // extern "C"

namespace {

// Scratch bytes of the friends-of-friends forests of shard i, from byte `off` of its query scratch: P forests of F =
// total_pad entries on the shard that merges (every rank when each rank is its own process), one on every other shard.
size_t fof_scratch_bytes(const b200nb_ctx *c, size_t i, size_t off)
{
    const bool gather = c->shards.size() != (size_t)c->n_ranks;
    return off + 4 * c->total_pad * (gather || i == 0 ? (size_t)c->n_ranks : 1);
}

// The host side shared by the friends-of-friends calls (b200nb_fof, b200nb_fof_phase).  Every shard links its own bodies
// against all bodies into a forest of F = total_pad entries at byte `off` of its query scratch (fof_sm100.cuh):
// link(s, forest) enqueues that pass on s.s_compute when the shard has bodies.  In-process shards copy their forests to
// shard 0, one rank per process all-gathers them; then shard 0, or every rank, folds forests 1..P-1 into forest 0,
// finalizes it to labels and downloads them.  Reads only the body array and the scratch: state and cached step graphs
// are untouched.
template <class Link>
int fof_forests(b200nb_ctx *c, size_t off, uint32_t *group, Link link)
{
    DeviceGuard guard;
    const bool gather = c->shards.size() != (size_t)c->n_ranks;
    const size_t F = c->total_pad;
    const uint32_t P = (uint32_t)c->n_ranks, n = (uint32_t)c->n;
    for (size_t i = 0; i < c->shards.size(); ++i)
        if (int rc = query_scratch(c, c->shards[i], fof_scratch_bytes(c, i, off))) return rc;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        // an asynchronous step may still be exchanging positions: the whole body array is read
        if (c->n_ranks > 1)
            if (int rc = wait_remote_positions(c, s)) return rc;
        uint32_t *forest = reinterpret_cast<uint32_t *>(s.query_buf + off) + (gather ? s.rank * F : 0);
        fof_init_kernel<<<(unsigned)((F + 255) / 256), 256, 0, s.s_compute>>>(forest, (uint32_t)F);
        c->launches++;
        if (s.n_local > 0) {
            link(s, forest);
            c->launches++;
        }
        CU(c, cudaGetLastError());
    }
    Shard &m = c->shards[0];
    uint32_t *forests = reinterpret_cast<uint32_t *>(m.query_buf + off);
    if (gather) {
        CU(c, cudaSetDevice(m.device));
        NC(c, g_nccl.AllGather(forests + m.rank * F, forests, F, ncclUint32, m.comm, m.s_compute));
    } else {
        for (size_t i = 1; i < c->shards.size(); ++i) {
            Shard &s = c->shards[i];
            CU(c, cudaSetDevice(s.device));
            CU(c, cudaMemcpyPeerAsync(forests + (size_t)s.rank * F, m.device, s.query_buf + off, s.device, 4 * F, s.s_compute));
            CU(c, cudaStreamSynchronize(s.s_compute)); // the merge on shard 0 reads the copy
        }
    }
    CU(c, cudaSetDevice(m.device));
    if (P > 1) {
        fof_merge_kernel<<<(n + 255) / 256, 256, 0, m.s_compute>>>(forests, P, F, n);
        c->launches++;
    }
    fof_finalize_kernel<<<(n + 255) / 256, 256, 0, m.s_compute>>>(forests, n);
    c->launches++;
    CU(c, cudaGetLastError());
    CU(c, cudaMemcpyAsync(group, forests, (size_t)n * 4, cudaMemcpyDeviceToHost, m.s_compute));
    return sync_all(c);
}

} // namespace

extern "C" {

int b200nb_fof(b200nb_ctx *c, float b, uint32_t *group)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "fof before upload");
    if (!group) return fail(c, B200NB_EINVAL, "fof: group is NULL");
    const float b2 = b * b;
    if (!(b >= 0.f) || !(b2 <= FLT_MAX)) return fail(c, B200NB_EINVAL, "fof: b = %g must be >= 0 with b * b finite in fp32", (double)b);
    uint32_t b2u;
    memcpy(&b2u, &b2, 4);
    const uint32_t n = (uint32_t)c->n, nb = (n + BLK - 1) / BLK, stream = std::min<uint32_t>(nb / 2 + FOF_R, nb);
    return fof_forests(c, 0, group, [&](Shard &s, uint32_t *forest) {
        FofArgs a{};
        a.src = s.bodies;
        a.parent = forest;
        a.first = (uint32_t)((uint64_t)s.rank * c->L);
        a.count = s.n_local;
        a.n = n;
        a.nb = nb;
        a.stream = stream;
        a.thr = b2u + 1;
        const uint32_t tiles = (s.n_local + FOF_TI - 1) / FOF_TI;
        a.n_chunks = fof_chunks(tiles, stream, (uint32_t)s.n_sms * FOF_MINB);
        fof_link_kernel<<<dim3(tiles, a.n_chunks), FOF_THREADS, fof_smem_bytes(), s.s_compute>>>(a);
    });
}

} // extern "C"

namespace {

// Phase-space friends-of-friends labels (b200nb_fof_phase; phase_fof_sm100.cuh).  Scratch per shard: the 6-float array of
// all N_pad = total_pad bodies (24 N_pad bytes), then fof_forests' forests.  Each shard packs its own slice from its
// blocked positions and its own velocities; the slices are then replicated: in-process shards copy every slice to every
// other shard (a plain copy when both share a device), one rank per process all-gathers them in place.  Each shard then
// links its own bodies against all of them.
int phase_fof_run(b200nb_ctx *c, float sx, float sv, uint32_t *group)
{
    DeviceGuard guard;
    const bool gather = c->shards.size() != (size_t)c->n_ranks;
    const size_t off = 24 * c->total_pad, slice = (size_t)6 * c->L; // floats of one shard's slice
    const uint32_t L = (uint32_t)c->L, n = (uint32_t)c->n;
    for (size_t i = 0; i < c->shards.size(); ++i)
        if (int rc = query_scratch(c, c->shards[i], fof_scratch_bytes(c, i, off))) return rc;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        if (c->n_ranks > 1) // an asynchronous step may still be exchanging positions
            if (int rc = wait_remote_positions(c, s)) return rc;
        float *mine = reinterpret_cast<float *>(s.query_buf);
        phase_fof_pack_kernel<<<(L + 255) / 256, 256, 0, s.s_compute>>>(s.bodies, s.vel, mine, (uint32_t)(s.rank * c->L), L,
                                                                        s.n_local, sx, sv);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    if (gather) {
        Shard &s = c->shards[0];
        float *arr = reinterpret_cast<float *>(s.query_buf);
        CU(c, cudaSetDevice(s.device));
        NC(c, g_nccl.AllGather(arr + (size_t)s.rank * slice, arr, slice, ncclFloat, s.comm, s.s_compute));
    } else if (c->n_ranks > 1) {
        if (int rc = sync_all(c)) return rc; // every slice is packed
        for (auto &o : c->shards) { // into o, on o's stream: its link pass follows in stream order
            CU(c, cudaSetDevice(o.device));
            for (auto &s : c->shards) {
                if (&s == &o) continue;
                float *dst = reinterpret_cast<float *>(o.query_buf) + (size_t)s.rank * slice;
                const float *src = reinterpret_cast<const float *>(s.query_buf) + (size_t)s.rank * slice;
                if (s.device == o.device)
                    CU(c, cudaMemcpyAsync(dst, src, slice * 4, cudaMemcpyDeviceToDevice, o.s_compute));
                else
                    CU(c, cudaMemcpyPeerAsync(dst, o.device, src, s.device, slice * 4, o.s_compute));
            }
        }
    }
    const uint32_t nb = (n + BLK - 1) / BLK, stream = std::min<uint32_t>(nb / 2 + PF_R, nb);
    return fof_forests(c, off, group, [&](Shard &s, uint32_t *forest) {
        PhaseFofArgs a{};
        a.src = reinterpret_cast<const float *>(s.query_buf);
        a.parent = forest;
        a.first = (uint32_t)((uint64_t)s.rank * c->L);
        a.count = s.n_local;
        a.n = n;
        a.nb = nb;
        a.stream = stream;
        const uint32_t tiles = (s.n_local + PF_TI - 1) / PF_TI;
        a.n_chunks = fof_chunks(tiles, stream, (uint32_t)s.n_sms * PF_MINB);
        phase_fof_link_kernel<<<dim3(tiles, a.n_chunks), PF_THREADS, phase_fof_smem_bytes(), s.s_compute>>>(a);
    });
}

} // namespace

extern "C" {

int b200nb_fof_phase(b200nb_ctx *c, float b_x, float b_v, uint32_t *group)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "fof_phase before upload");
    if (!group) return fail(c, B200NB_EINVAL, "fof_phase: group is NULL");
    if (!(b_x > 0.f) || !(b_v > 0.f))
        return fail(c, B200NB_EINVAL, "fof_phase: b_x = %g and b_v = %g must be > 0 (+inf allowed)", (double)b_x, (double)b_v);
    // correctly rounded fp32 divisions (no fast-math here); 1 / +inf = 0 switches that part of the metric off
    const float one = 1.0f, sx = one / b_x, sv = one / b_v;
    return phase_fof_run(c, sx, sv, group);
}

int b200nb_set_tracers(b200nb_ctx *c, uint64_t n_tracers, const float *qx, const float *qy, const float *qz, const float *vx,
                       const float *vy, const float *vz)
{
    if (!c) return B200NB_EINVAL;
    if (n_tracers > 0 && (!qx || !qy || !qz || !vx || !vy || !vz)) return fail(c, B200NB_EINVAL, "set_tracers: NULL array");
    const uint64_t per = (n_tracers + c->n_ranks - 1) / c->n_ranks;
    const uint64_t T = (per + FIELD_TI - 1) / FIELD_TI * FIELD_TI;
    if (T >= (1ull << 31))
        return fail(c, B200NB_EINVAL, "set_tracers: %llu tracers per shard; the field kernel counts targets in 32 bits",
                    (unsigned long long)T);
    DeviceGuard guard;
    // steps in flight read the old tracers, and captured step graphs hold their buffers and count
    if (int rc = sync_all(c)) return rc;
    for (auto &g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
    free_tracers(c);
    if (n_tracers == 0) return B200NB_OK;
    const uint32_t S = field_chunks(c->n), cap = (uint32_t)std::min<uint64_t>(FIELD_BATCH, T);
    const uint64_t bytes = tracer_bytes(T, cap, S);
    // a set that cannot fit fails before it takes any memory (shards may share a device)
    for (auto &s : c->shards) {
        uint64_t need = 0;
        for (auto &o : c->shards) need += o.device == s.device ? bytes : 0;
        size_t free_b = 0, total_b = 0;
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaMemGetInfo(&free_b, &total_b));
        if (need > free_b)
            return fail(c, B200NB_ECUDA, "set_tracers: %llu tracers need %llu bytes on device %d, %llu are free",
                        (unsigned long long)n_tracers, (unsigned long long)need, s.device, (unsigned long long)free_b);
    }
    for (auto &s : c->shards) {
        cudaError_t e = cudaSetDevice(s.device);
        if (e == cudaSuccess) e = cudaMalloc((void **)&s.tr, 9 * T * 4);
        if (e == cudaSuccess) e = cudaMalloc((void **)&s.tr_part, (size_t)S * 4 * cap * 4);
        if (e != cudaSuccess) { // never half set: no tracers at all
            (void)cudaGetLastError();
            free_tracers(c);
            return fail(c, B200NB_ECUDA, "set_tracers: %s", cudaGetErrorString(e));
        }
        s.tr_bytes = bytes;
        s.bytes += bytes;
    }
    const float *src[6] = {qx, qy, qz, vx, vy, vz};
    for (auto &s : c->shards) {
        const uint64_t first = (uint64_t)s.rank * T;
        s.tr_local = first >= n_tracers ? 0u : (uint32_t)std::min<uint64_t>(T, n_tracers - first);
        cudaError_t e = cudaSetDevice(s.device);
        for (int k = 0; k < 6 && s.tr_local > 0 && e == cudaSuccess; ++k)
            e = cudaMemcpyAsync(s.tr + k * T, src[k] + first, (size_t)s.tr_local * 4, cudaMemcpyHostToDevice, s.s_compute);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            sync_all(c);
            free_tracers(c);
            return fail(c, B200NB_ECUDA, "set_tracers: %s", cudaGetErrorString(e));
        }
    }
    // host pointers are only borrowed for the call (see upload)
    if (int rc = sync_all(c)) { free_tracers(c); return rc; }
    c->m_tracers = n_tracers;
    c->tr_T = T;
    c->tr_cap = cap;
    if (c->scf.on) { // the expansion's tracer rows; without them, no tracers at all
        const cudaError_t e = alloc_ext_tracers(c);
        if (e != cudaSuccess) {
            free_tracers(c);
            return fail(c, B200NB_ECUDA, "set_tracers: %s", cudaGetErrorString(e));
        }
    }
    return B200NB_OK;
}

// ------------------------------------------------------------------------------------------------ external potential
// A term is valid when its parameters obey the rules of include/b200nb.h, "external potential".
static bool external_term_ok(const b200nb_external_term &t, char *why, size_t n)
{
    const bool finite = std::isfinite(t.gm) && std::isfinite(t.a) && std::isfinite(t.b) && std::isfinite(t.centre[0]) &&
                        std::isfinite(t.centre[1]) && std::isfinite(t.centre[2]);
    const char *bad = nullptr;
    if (t.kind < B200NB_EXT_PLUMMER || t.kind > B200NB_EXT_LOGARITHMIC) bad = "unknown kind";
    else if (t.reserved != 0) bad = "reserved must be 0";
    else if (!finite) bad = "non-finite parameter";
    else if (!(t.gm >= 0.0)) bad = "gm must be >= 0";
    else if (t.kind == B200NB_EXT_PLUMMER && !(t.a >= 0.0)) bad = "Plummer needs a >= 0";
    else if ((t.kind == B200NB_EXT_HERNQUIST || t.kind == B200NB_EXT_NFW) && !(t.a > 0.0)) bad = "needs a > 0";
    else if (t.kind <= B200NB_EXT_NFW && t.b != 0.0) bad = "b must be 0 for this kind";
    else if (t.kind == B200NB_EXT_MIYAMOTO_NAGAI && !(t.a >= 0.0 && t.b > 0.0)) bad = "Miyamoto-Nagai needs a >= 0, b > 0";
    else if (t.kind == B200NB_EXT_LOGARITHMIC && !(t.a > 0.0 && t.b > 0.0)) bad = "logarithmic needs r_c = a > 0, q = b > 0";
    if (bad) snprintf(why, n, "%s", bad);
    return bad == nullptr;
}

int b200nb_set_external(b200nb_ctx *c, uint32_t n_terms, const b200nb_external_term *terms)
{
    if (!c) return B200NB_EINVAL;
    if (n_terms > B200NB_EXTERNAL_MAX)
        return fail(c, B200NB_EINVAL, "set_external: %u terms, at most %d", n_terms, B200NB_EXTERNAL_MAX);
    if (n_terms > 0 && !terms) return fail(c, B200NB_EINVAL, "set_external: NULL terms");
    for (uint32_t k = 0; k < n_terms; ++k) {
        char why[96];
        if (!external_term_ok(terms[k], why, sizeof why))
            return fail(c, B200NB_EINVAL, "set_external: term %u (kind %d): %s", k, terms[k].kind, why);
    }
    DeviceGuard guard;
    // steps in flight read the old terms, and captured step graphs bake them in
    if (int rc = sync_all(c)) return rc;
    for (auto &g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
    ExtTerms e{};
    for (uint32_t k = 0; k < n_terms; ++k) e.t[k] = terms[k];
    e.n = n_terms;
    c->ext = e;
    c->acc_valid = false; // the leapfrog's a(x_n) and a(p) were taken under the old terms
    c->tr_acc_valid = false;
    return B200NB_OK;
}

int b200nb_get_external(const b200nb_ctx *c, b200nb_external_term *out, uint32_t *n_terms)
{
    if (!c || !out || !n_terms) return B200NB_EINVAL;
    for (uint32_t k = 0; k < c->ext.n; ++k) out[k] = c->ext.t[k];
    *n_terms = c->ext.n;
    return B200NB_OK;
}

constexpr uint32_t EXTERNAL_BATCH = 1u << 20; // points per launch of b200nb_external_field: 44 MiB of scratch

int b200nb_external_field(b200nb_ctx *c, uint64_t n_points, const float *px, const float *py, const float *pz, double *ax,
                          double *ay, double *az, double *phi)
{
    if (!c) return B200NB_EINVAL;
    if (n_points == 0) return B200NB_OK;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "external_field: NULL point array");
    DeviceGuard guard;
    Shard &s = c->shards[0];
    const uint32_t cap = (uint32_t)std::min<uint64_t>(EXTERNAL_BATCH, (n_points + 255) / 256 * 256);
    if (int rc = query_scratch(c, s, (size_t)cap * (3 * 4 + 4 * 8))) return rc;
    CU(c, cudaSetDevice(s.device));
    double *dout = reinterpret_cast<double *>(s.query_buf);
    float *dpts = reinterpret_cast<float *>(dout + 4 * (size_t)cap);
    const float *pts[3] = {px, py, pz};
    double *out[4] = {ax, ay, az, phi};
    for (uint64_t base = 0; base < n_points; base += cap) {
        const uint32_t cnt = (uint32_t)std::min<uint64_t>(cap, n_points - base);
        for (int k = 0; k < 3; ++k)
            CU(c, cudaMemcpyAsync(dpts + (size_t)k * cap, pts[k] + base, (size_t)cnt * 4, cudaMemcpyHostToDevice, s.s_compute));
        if (c->scf.on) {
            if (int rc = enqueue_ext_total(c, s, SoaPoints{dpts, dpts + cap, dpts + 2 * (size_t)cap}, cnt, cap, dout)) return rc;
        } else {
            external_field_kernel<<<(cnt + 255) / 256, 256, 0, s.s_compute>>>(c->ext, dpts, dpts + cap, dpts + 2 * (size_t)cap,
                                                                              cnt, cap, dout);
            c->launches++;
            CU(c, cudaGetLastError());
        }
        for (int k = 0; k < 4; ++k)
            if (out[k])
                CU(c, cudaMemcpyAsync(out[k] + base, dout + (size_t)k * cap, (size_t)cnt * 8, cudaMemcpyDeviceToHost, s.s_compute));
    }
    CU(c, cudaStreamSynchronize(s.s_compute));
    return B200NB_OK;
}

int b200nb_download_tracers(b200nb_ctx *c, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz)
{
    if (!c) return B200NB_EINVAL;
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    const uint64_t M = c->m_tracers, T = c->tr_T;
    float *dst[6] = {qx, qy, qz, vx, vy, vz};
    if (M == 0) return B200NB_OK;
    if (c->shards.size() == (size_t)c->n_ranks) { // every shard is local: each one returns its own slice
        for (auto &s : c->shards) {
            if (s.tr_local == 0) continue;
            CU(c, cudaSetDevice(s.device));
            for (int k = 0; k < 6; ++k)
                if (dst[k])
                    CU(c, cudaMemcpyAsync(dst[k] + (size_t)s.rank * T, s.tr + k * T, (size_t)s.tr_local * 4, cudaMemcpyDeviceToHost,
                                          s.s_compute));
        }
        return sync_all(c);
    }
    // one rank per process: all-gather the [6][T] slices through a temporary [P][6][T] device buffer (download_sliced)
    Shard &s = c->shards[0];
    CU(c, cudaSetDevice(s.device));
    struct Scratch { // freed on every exit path
        float *p = nullptr;
        ~Scratch() { if (p) cudaFree(p); }
    } tmp;
    const size_t count = 6 * (size_t)T;
    CU(c, cudaMalloc((void **)&tmp.p, count * c->n_ranks * 4));
    NC(c, g_nccl.AllGather(s.tr, tmp.p, count, ncclFloat, s.comm, s.s_compute));
    for (int rk = 0; rk < c->n_ranks; ++rk) {
        const uint64_t first = (uint64_t)rk * T;
        if (first >= M) break;
        const size_t cnt = (size_t)std::min<uint64_t>(T, M - first);
        for (int k = 0; k < 6; ++k)
            if (dst[k])
                CU(c, cudaMemcpyAsync(dst[k] + first, tmp.p + (size_t)rk * count + (size_t)k * T, cnt * 4, cudaMemcpyDeviceToHost,
                                      s.s_compute));
    }
    CU(c, cudaStreamSynchronize(s.s_compute));
    return B200NB_OK;
}

uint64_t b200nb_n_tracers(const b200nb_ctx *c) { return c ? c->m_tracers : 0; }

} // extern "C"

// ------------------------------------------------------------------------------------------------ basis-function expansion
namespace {

// The recurrence tables of scf_sm100.cuh, in long double, each entry rounded once.
void scf_tables(ScfTables &t)
{
    memset(&t, 0, sizeof t);
    for (int l = 0; l <= SCF_LMAX; ++l) {
        const long double alpha = 2.0L * l + 1.5L;
        for (int n = 1; n <= SCF_NMAX; ++n) {
            t.ga[l][n] = (double)(2.0L * (n + alpha - 1.0L) / n);
            t.gb[l][n] = (double)((n + 2.0L * alpha - 2.0L) / n);
        }
    }
    long double dfact = 1.0L; // (2m - 1)!!
    for (int m = 0; m <= SCF_LMAX + 1; ++m) {
        if (m > 0) dfact *= 2.0L * m - 1.0L;
        t.qs[m] = (double)(m % 2 ? -dfact : dfact);
        for (int l = m + 1; l <= SCF_LMAX + 1; ++l) {
            t.qa[l][m] = (double)((2.0L * l - 1.0L) / (l - m));
            t.qb[l][m] = (double)((l + m - 1.0L) / (l - m));
        }
    }
}

// F_nlm = (2 - delta_m0) A~_nl N_lm / a, packed as the coefficients (include/b200nb.h), in long double
void scf_norms(uint32_t nmax, uint32_t lmax, double a, std::vector<double> &F)
{
    const uint32_t LM = (lmax + 1) * (lmax + 2) / 2;
    F.assign((size_t)(nmax + 1) * LM, 0.0);
    for (uint32_t n = 0; n <= nmax; ++n)
        for (uint32_t l = 0; l <= lmax; ++l) {
            const long double K = 0.5L * n * (n + 4.0L * l + 3.0L) + (l + 1.0L) * (2.0L * l + 1.0L);
            const long double lg = (8.0L * l + 6.0L) * logl(2.0L) + lgammal(n + 1.0L) + logl(n + 2.0L * l + 1.5L) +
                                   2.0L * lgammal(2.0L * l + 1.5L) - logl(4.0L * 3.14159265358979323846264338327950288L * K) -
                                   lgammal(n + 4.0L * l + 3.0L);
            const long double At = -expl(lg);
            long double ratio = 1.0L; // (l - m)! / (l + m)!
            for (uint32_t m = 0; m <= l; ++m) {
                if (m > 0) ratio /= (long double)(l + m) * (long double)(l - m + 1);
                F[(size_t)n * LM + l * (l + 1) / 2 + m] = (double)((m ? 2.0L : 1.0L) * At * (2.0L * l + 1.0L) * ratio / a);
            }
        }
}

int scf_check(b200nb_ctx *c, const char *what, uint32_t nmax, uint32_t lmax, double a, const double *centre)
{
    if (nmax > (uint32_t)SCF_NMAX || lmax > (uint32_t)SCF_LMAX)
        return fail(c, B200NB_EINVAL, "%s: nmax = %u and lmax = %u must lie in [0, %d] and [0, %d]", what, nmax, lmax, SCF_NMAX,
                    SCF_LMAX);
    if (!(std::isfinite(a) && a > 0.0)) return fail(c, B200NB_EINVAL, "%s: a = %g must be finite and > 0", what, a);
    if (!centre) return fail(c, B200NB_EINVAL, "%s: centre is NULL", what);
    if (!(std::isfinite(centre[0]) && std::isfinite(centre[1]) && std::isfinite(centre[2])))
        return fail(c, B200NB_EINVAL, "%s: non-finite centre", what);
    return B200NB_OK;
}

} // namespace

extern "C" {

int b200nb_scf_coefficients(b200nb_ctx *c, uint32_t nmax, uint32_t lmax, double a, const double centre[3], const uint32_t *group,
                            uint32_t label, double *S, double *T)
{
    if (!c) return B200NB_EINVAL;
    if (int rc = scf_check(c, "scf_coefficients", nmax, lmax, a, centre)) return rc;
    if (!S || !T) return fail(c, B200NB_EINVAL, "scf_coefficients: S or T is NULL");
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "scf_coefficients before upload");
    DeviceGuard guard;
    Shard &s = c->shards[0];
    const uint32_t n = (uint32_t)c->n, K = (nmax + 1) * (lmax + 1) * (lmax + 2) / 2, n_chunks = scf_chunks(n);
    ScfTables tab;
    scf_tables(tab);
    std::vector<double> F;
    scf_norms(nmax, lmax, a, F);
    // scratch: tables | F | [S | T] | partial rows | labels
    const size_t o_f = round256(sizeof(ScfTables)), o_out = o_f + round256(8 * (size_t)K), o_part = o_out + round256(16 * (size_t)K),
                 o_grp = o_part + round256((size_t)n_chunks * 16 * K), bytes = o_grp + (group ? round256(4 * (size_t)n) : 0);
    if (int rc = query_scratch(c, s, bytes)) return rc;
    CU(c, cudaSetDevice(s.device));
    if (c->n_ranks > 1) // an asynchronous step may still be exchanging positions: the whole body array is read
        if (int rc = wait_remote_positions(c, s)) return rc;
    unsigned char *buf = s.query_buf;
    CU(c, cudaMemcpyAsync(buf, &tab, sizeof tab, cudaMemcpyHostToDevice, s.s_compute));
    CU(c, cudaMemcpyAsync(buf + o_f, F.data(), 8 * (size_t)K, cudaMemcpyHostToDevice, s.s_compute));
    if (group) CU(c, cudaMemcpyAsync(buf + o_grp, group, 4 * (size_t)n, cudaMemcpyHostToDevice, s.s_compute));
    ScfArgs A{};
    A.bodies = s.bodies;
    A.group = group ? reinterpret_cast<const uint32_t *>(buf + o_grp) : nullptr;
    A.tab = reinterpret_cast<const ScfTables *>(buf);
    A.partial = reinterpret_cast<double *>(buf + o_part);
    A.label = label;
    A.n = n;
    A.chunk = (n + n_chunks - 1) / n_chunks;
    A.nmax = nmax;
    A.lmax = lmax;
    A.K = K;
    A.cx = centre[0]; A.cy = centre[1]; A.cz = centre[2];
    A.a = a;
    const size_t smem = scf_coef_smem(nmax, lmax);
    CU(c, cudaFuncSetAttribute(scf_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    scf_coef_kernel<<<n_chunks, SCF_THREADS, smem, s.s_compute>>>(A);
    c->launches++;
    CU(c, cudaGetLastError());
    double *dout = reinterpret_cast<double *>(buf + o_out);
    scf_reduce_kernel<<<(2 * K + 255) / 256, 256, 0, s.s_compute>>>(A.partial, reinterpret_cast<const double *>(buf + o_f), n_chunks,
                                                                    K, lmax, dout);
    c->launches++;
    CU(c, cudaGetLastError());
    CU(c, cudaMemcpyAsync(S, dout, 8 * (size_t)K, cudaMemcpyDeviceToHost, s.s_compute));
    CU(c, cudaMemcpyAsync(T, dout + K, 8 * (size_t)K, cudaMemcpyDeviceToHost, s.s_compute));
    CU(c, cudaStreamSynchronize(s.s_compute));
    return B200NB_OK;
}

int b200nb_scf_field(b200nb_ctx *c, uint32_t nmax, uint32_t lmax, double a, const double centre[3], const double *S, const double *T,
                     uint64_t n_points, const float *px, const float *py, const float *pz, double *ax, double *ay, double *az,
                     double *phi)
{
    if (!c) return B200NB_EINVAL;
    if (int rc = scf_check(c, "scf_field", nmax, lmax, a, centre)) return rc;
    if (!S || !T) return fail(c, B200NB_EINVAL, "scf_field: S or T is NULL");
    if (n_points == 0) return B200NB_OK;
    if (!px || !py || !pz) return fail(c, B200NB_EINVAL, "scf_field: NULL point array");
    DeviceGuard guard;
    Shard &s = c->shards[0];
    const uint32_t K = (nmax + 1) * (lmax + 1) * (lmax + 2) / 2;
    const uint32_t cap = (uint32_t)std::min<uint64_t>(SCF_BATCH, (n_points + 255) / 256 * 256);
    ScfTables tab;
    scf_tables(tab);
    // scratch: tables | [S | T] | [4][cap] outputs | [3][cap] points
    const size_t o_coef = round256(sizeof(ScfTables)), o_out = o_coef + round256(16 * (size_t)K), o_pts = o_out + 32 * (size_t)cap;
    if (int rc = query_scratch(c, s, o_pts + 12 * (size_t)cap)) return rc;
    CU(c, cudaSetDevice(s.device));
    unsigned char *buf = s.query_buf;
    CU(c, cudaMemcpyAsync(buf, &tab, sizeof tab, cudaMemcpyHostToDevice, s.s_compute));
    CU(c, cudaMemcpyAsync(buf + o_coef, S, 8 * (size_t)K, cudaMemcpyHostToDevice, s.s_compute));
    CU(c, cudaMemcpyAsync(buf + o_coef + 8 * (size_t)K, T, 8 * (size_t)K, cudaMemcpyHostToDevice, s.s_compute));
    double *dout = reinterpret_cast<double *>(buf + o_out);
    float *dpts = reinterpret_cast<float *>(buf + o_pts);
    const size_t smem = scf_field_smem(K);
    CU(c, cudaFuncSetAttribute(scf_field_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const float *pts[3] = {px, py, pz};
    double *out[4] = {ax, ay, az, phi};
    for (uint64_t base = 0; base < n_points; base += cap) {
        const uint32_t cnt = (uint32_t)std::min<uint64_t>(cap, n_points - base);
        for (int k = 0; k < 3; ++k)
            CU(c, cudaMemcpyAsync(dpts + (size_t)k * cap, pts[k] + base, (size_t)cnt * 4, cudaMemcpyHostToDevice, s.s_compute));
        ScfFieldArgs A{};
        A.coef = reinterpret_cast<const double *>(buf + o_coef);
        A.tab = reinterpret_cast<const ScfTables *>(buf);
        A.px = dpts; A.py = dpts + cap; A.pz = dpts + 2 * (size_t)cap;
        A.out = dout;
        A.count = cnt; A.stride = cap; A.nmax = nmax; A.lmax = lmax; A.K = K;
        A.cx = centre[0]; A.cy = centre[1]; A.cz = centre[2];
        A.a = a;
        scf_field_kernel<<<(cnt + SCF_EVAL_THREADS - 1) / SCF_EVAL_THREADS, SCF_EVAL_THREADS, smem, s.s_compute>>>(A);
        c->launches++;
        CU(c, cudaGetLastError());
        for (int k = 0; k < 4; ++k)
            if (out[k])
                CU(c, cudaMemcpyAsync(out[k] + base, dout + (size_t)k * cap, (size_t)cnt * 8, cudaMemcpyDeviceToHost, s.s_compute));
    }
    CU(c, cudaStreamSynchronize(s.s_compute));
    return B200NB_OK;
}

// ------------------------------------------------------------------------------------------------ external expansion
int b200nb_set_external_scf(b200nb_ctx *c, uint32_t nmax, uint32_t lmax, double a, const double centre[3], const double *S,
                            const double *T)
{
    if (!c) return B200NB_EINVAL;
    const bool remove = !S && !T;
    uint32_t K = 0;
    if (!remove) {
        if (!S || !T) return fail(c, B200NB_EINVAL, "set_external_scf: one of S and T is NULL");
        if (int rc = scf_check(c, "set_external_scf", nmax, lmax, a, centre)) return rc;
        const uint32_t LM = (lmax + 1) * (lmax + 2) / 2;
        K = (nmax + 1) * LM;
        for (uint32_t k = 0; k < K; ++k)
            if (!std::isfinite(S[k]) || !std::isfinite(T[k]))
                return fail(c, B200NB_EINVAL, "set_external_scf: non-finite S or T entry at packed index %u", k);
        for (uint32_t n = 0; n <= nmax; ++n)
            for (uint32_t l = 0; l <= lmax; ++l)
                if (T[n * LM + l * (l + 1) / 2] != 0.0)
                    return fail(c, B200NB_EINVAL, "set_external_scf: T[n=%u, l=%u, m=0] = %g must be 0", n, l,
                                T[n * LM + l * (l + 1) / 2]);
    }
    DeviceGuard guard;
    // steps in flight read the old coefficients, and captured step graphs bake in their buffers
    if (int rc = sync_all(c)) return rc;
    for (auto &g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
    c->acc_valid = false; // the leapfrog's a(x_n) and a(p) were taken in the old field
    c->tr_acc_valid = false;
    if (remove) {
        free_ext_scf(c);
        return B200NB_OK;
    }
    ScfTables tab;
    scf_tables(tab);
    const size_t o_coef = round256(sizeof(ScfTables)), need = o_coef + round256(16 * (size_t)K);
    const int smem_max = (int)scf_field_smem((SCF_NMAX + 1) * (SCF_LMAX + 1) * (SCF_LMAX + 2) / 2);
    for (auto &s : c->shards) {
        cudaError_t e = cudaSetDevice(s.device);
        if (e == cudaSuccess && s.ext_coef_bytes < need) { // grow-only
            cudaFree(s.ext_coef);
            s.bytes -= s.ext_coef_bytes;
            s.ext_coef = nullptr;
            s.ext_coef_bytes = 0;
            e = cudaMalloc((void **)&s.ext_coef, need);
            if (e == cudaSuccess) { s.ext_coef_bytes = need; s.bytes += need; } else s.ext_coef = nullptr;
        }
        if (e == cudaSuccess && !s.ext_body) {
            e = cudaMalloc((void **)&s.ext_body, 32 * c->L);
            if (e == cudaSuccess) s.bytes += 32 * c->L; else s.ext_body = nullptr;
        }
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(ext_total_kernel<BlockedPoints>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(ext_total_kernel<SoaPoints>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s.ext_coef, &tab, sizeof tab, cudaMemcpyHostToDevice, s.s_compute);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s.ext_coef + o_coef, S, 8 * (size_t)K, cudaMemcpyHostToDevice, s.s_compute);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s.ext_coef + o_coef + 8 * (size_t)K, T, 8 * (size_t)K, cudaMemcpyHostToDevice, s.s_compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s.s_compute); // S and T are borrowed for the call
        if (e == cudaSuccess && c->m_tracers > 0) e = alloc_ext_tracers(c);
        if (e != cudaSuccess) { // never half set: no expansion at all
            (void)cudaGetLastError();
            sync_all(c);
            free_ext_scf(c);
            return fail(c, B200NB_ECUDA, "set_external_scf: %s", cudaGetErrorString(e));
        }
    }
    c->scf.on = true;
    c->scf.nmax = nmax; c->scf.lmax = lmax; c->scf.K = K;
    c->scf.a = a;
    for (int k = 0; k < 3; ++k) c->scf.centre[k] = centre[k];
    c->scf.coef.assign(S, S + K);
    c->scf.coef.insert(c->scf.coef.end(), T, T + K);
    return B200NB_OK;
}

int b200nb_get_external_scf(const b200nb_ctx *c, uint32_t *present, uint32_t *nmax, uint32_t *lmax, double *a, double centre[3],
                            double *S, double *T)
{
    if (!c || !present) return B200NB_EINVAL;
    *present = c->scf.on ? 1u : 0u;
    if (!c->scf.on) return B200NB_OK;
    const uint32_t K = c->scf.K;
    if (nmax) *nmax = c->scf.nmax;
    if (lmax) *lmax = c->scf.lmax;
    if (a) *a = c->scf.a;
    if (centre) for (int k = 0; k < 3; ++k) centre[k] = c->scf.centre[k];
    if (S) memcpy(S, c->scf.coef.data(), 8 * (size_t)K);
    if (T) memcpy(T, c->scf.coef.data() + K, 8 * (size_t)K);
    return B200NB_OK;
}

} // extern "C"

namespace {

// Carving of the group calls' scratch (groups_sm100.cuh), the same on every shard.  The sort buffers alias `piece`,
// which is first written after the sort.
struct GpBufs {
    uint32_t *key[2], *val[2];
    uint64_t *mem[2];
    unsigned char *flags;
    float *src, *phi, *vm, *phi_out, *partial;
    uint32_t *lo, *hi, *bound, *info;
    GpSum *piece;
    void *temp;
    size_t temp_bytes, total;
};

GpBufs gp_carve(unsigned char *base, uint64_t n, uint64_t n_pad, uint32_t P, uint32_t cap, size_t temp_bytes)
{
    GpBufs b{};
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char *p = base ? base + off : nullptr; off += (bytes + 255) / 256 * 256; return p; };
    b.piece = reinterpret_cast<GpSum *>(take(sizeof(GpSum) * n));
    for (int i = 0; i < 2; ++i) {
        b.key[i] = reinterpret_cast<uint32_t *>(base ? reinterpret_cast<unsigned char *>(b.piece) + 8 * n * i : nullptr);
        b.val[i] = reinterpret_cast<uint32_t *>(base ? reinterpret_cast<unsigned char *>(b.piece) + 8 * n * i + 4 * n : nullptr);
    }
    for (int i = 0; i < 2; ++i) b.mem[i] = reinterpret_cast<uint64_t *>(take(8 * n));
    b.flags = take(n);
    b.src = reinterpret_cast<float *>(take(16 * ((n + BLK - 1) / BLK * BLK)));
    b.lo = reinterpret_cast<uint32_t *>(take(4 * n));
    b.hi = reinterpret_cast<uint32_t *>(take(4 * n));
    b.phi = reinterpret_cast<float *>(take(4 * n));
    b.vm = reinterpret_cast<float *>(take(16 * n_pad));
    b.bound = reinterpret_cast<uint32_t *>(take(4 * n));
    b.phi_out = reinterpret_cast<float *>(take(4 * n));
    b.partial = reinterpret_cast<float *>(take((size_t)4 * GP_MAX_CHUNKS * cap));
    b.info = reinterpret_cast<uint32_t *>(take(4 * ((size_t)P + 2)));
    b.temp = take(temp_bytes);
    b.temp_bytes = temp_bytes;
    b.total = off;
    return b;
}

// Group potential (max_iter == 0) or unbinding (max_iter passes at most) of the labels `group`; see include/b200nb.h.
// Every shard sorts and packs the same members and runs the same O(N) unbinding step; the potential pass is split over
// the shards by tile cost.  The host reads the member count and the split once per pass.
int groups_run(b200nb_ctx *c, const uint32_t *group, uint32_t max_iter, uint32_t *bound, float *phi, uint32_t *n_iter,
               int *converged)
{
    DeviceGuard guard;
    // ordered after a preceding asynchronous step: positions exchanged, velocities final
    if (int rc = sync_all(c)) return rc;
    const bool gather = c->shards.size() != (size_t)c->n_ranks;
    const bool unbind = max_iter > 0;
    const uint32_t n = (uint32_t)c->n, P = (uint32_t)c->n_ranks, L = (uint32_t)c->L;
    const uint32_t cap = (uint32_t)std::min<uint64_t>(GP_BATCH, (c->n + GP_TI - 1) / GP_TI * GP_TI);
    std::vector<GpBufs> bufs;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        size_t sort_bytes = 0, sel_bytes = 0;
        CU(c, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                              (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n));
        CU(c, cub::DeviceSelect::Flagged(nullptr, sel_bytes, (const uint64_t *)nullptr, (const unsigned char *)nullptr,
                                         (uint64_t *)nullptr, (uint32_t *)nullptr, (int)n));
        const size_t temp = std::max(sort_bytes, sel_bytes);
        if (int rc = query_scratch(c, s, gp_carve(nullptr, n, c->total_pad, P, cap, temp).total)) return rc;
        bufs.push_back(gp_carve(s.query_buf, n, c->total_pad, P, cap, temp));
    }
    const unsigned g256 = (n + 255) / 256;
    // members of the current set, packed sources, label ranges and (P > 1) the cost split, from info[0] = M <= bound
    auto prepare = [&](Shard &s, GpBufs &b, int cur, uint32_t bound_m) -> int {
        const uint32_t span = (bound_m + BLK - 1) / BLK * BLK;
        gp_pack_kernel<<<(span + 255) / 256, 256, 0, s.s_compute>>>(s.bodies, b.mem[cur], b.info, span, b.src, b.lo, b.hi);
        c->launches++;
        if (P > 1) {
            gp_split_kernel<<<1, GP_SPLIT_THREADS, 0, s.s_compute>>>(b.lo, b.hi, b.info, P);
            c->launches++;
        }
        CU(c, cudaGetLastError());
        return B200NB_OK;
    };
    for (size_t k = 0; k < c->shards.size(); ++k) {
        Shard &s = c->shards[k];
        GpBufs &b = bufs[k];
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaMemcpyAsync(b.key[0], group, (size_t)n * 4, cudaMemcpyHostToDevice, s.s_compute));
        gp_iota_kernel<<<g256, 256, 0, s.s_compute>>>(b.val[0], n);
        CU(c, cudaMemsetAsync(b.info, 0, 4 * ((size_t)P + 2), s.s_compute));
        CU(c, cub::DeviceRadixSort::SortPairs(b.temp, b.temp_bytes, b.key[0], b.key[1], b.val[0], b.val[1], (int)n, 0, 32,
                                              s.s_compute));
        gp_members_kernel<<<g256, 256, 0, s.s_compute>>>(b.key[1], b.val[1], n, b.mem[0], b.info);
        c->launches += 3; // iota, the sort (counted once), members
        CU(c, cudaMemsetAsync(b.phi_out, 0, (size_t)n * 4, s.s_compute));
        CU(c, cudaMemsetAsync(b.bound, 0xFF, (size_t)n * 4, s.s_compute));
        if (unbind && !gather) // velocities and masses of every shard, [P][4][L]: vx, vy, vz, m
            for (auto &o : c->shards) {
                CU(c, cudaMemcpyPeerAsync(b.vm + (size_t)o.rank * 4 * L, s.device, o.vel, o.device, (size_t)12 * L, s.s_compute));
                CU(c, cudaMemcpyPeerAsync(b.vm + ((size_t)o.rank * 4 + 3) * L, s.device, o.mass, o.device, (size_t)4 * L, s.s_compute));
            }
        if (unbind && gather) {
            float *mine = b.vm + (size_t)s.rank * 4 * L;
            CU(c, cudaMemcpyAsync(mine, s.vel, (size_t)12 * L, cudaMemcpyDeviceToDevice, s.s_compute));
            CU(c, cudaMemcpyAsync(mine + (size_t)3 * L, s.mass, (size_t)4 * L, cudaMemcpyDeviceToDevice, s.s_compute));
            NC(c, g_nccl.AllGather(mine, b.vm, (size_t)4 * L, ncclFloat, s.comm, s.s_compute));
        }
        if (int rc = prepare(s, b, 0, n)) return rc;
    }
    std::vector<uint32_t> info(P + 2);
    auto read_info = [&]() -> int {
        Shard &s = c->shards[0];
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaMemcpyAsync(info.data(), bufs[0].info, 4 * info.size(), cudaMemcpyDeviceToHost, s.s_compute));
        return sync_all(c);
    };
    if (int rc = read_info()) return rc;
    uint32_t M = info[0], t = 0;
    int cur = 0;
    bool conv = false;
    const float soft2 = c->soft2;
    for (;;) {
        if (M == 0) { // S_0 empty: no pass.  Later: a pass over the empty set removes nobody.
            if (t > 0) {
                ++t;
                for (size_t k = 0; k < c->shards.size(); ++k) {
                    CU(c, cudaSetDevice(c->shards[k].device));
                    CU(c, cudaMemsetAsync(bufs[k].phi_out, 0, (size_t)n * 4, c->shards[k].s_compute));
                }
            }
            conv = true;
            break;
        }
        // ---- the potential pass: this shard's tiles [split[rank], split[rank + 1]) in batches of `cap` targets
        const uint32_t T = (M + GP_TI - 1) / GP_TI, cb = gp_chunk_blks(M);
        const uint32_t n_chunks = ((M + BLK - 1) / BLK + cb - 1) / cb;
        auto range = [&](int rank, uint32_t &a, uint32_t &e) {
            const uint32_t ta = P > 1 ? info[1 + rank] : 0, tb = P > 1 ? info[2 + rank] : T;
            a = std::min(ta * GP_TI, M);
            e = std::min(tb * GP_TI, M);
        };
        for (size_t k = 0; k < c->shards.size(); ++k) {
            Shard &s = c->shards[k];
            GpBufs &b = bufs[k];
            CU(c, cudaSetDevice(s.device));
            if (gather) CU(c, cudaMemsetAsync(b.phi, 0, (size_t)M * 4, s.s_compute)); // summed over the ranks below
            uint32_t a, e;
            range(s.rank, a, e);
            for (uint32_t t0 = a; t0 < e; t0 += cap) {
                GpArgs g{};
                g.src = b.src; g.lo = b.lo; g.hi = b.hi; g.partial = b.partial;
                g.stride = cap; g.t0 = t0; g.count = std::min(cap, e - t0); g.cb = cb; g.soft2 = soft2;
                group_potential_kernel<<<dim3((g.count + GP_TI - 1) / GP_TI, n_chunks), GP_THREADS, gp_smem_bytes(), s.s_compute>>>(g);
                group_reduce_kernel<<<(g.count + 255) / 256, 256, 0, s.s_compute>>>(b.partial, cap, t0, g.count, cb, b.lo, b.hi, b.phi);
                c->launches += 2;
                CU(c, cudaGetLastError());
            }
        }
        if (P > 1 && gather) {
            Shard &s = c->shards[0];
            CU(c, cudaSetDevice(s.device));
            // every other rank's entries are +0 here, and x + 0 == x for every value phi takes (never -0)
            NC(c, g_nccl.AllReduce(bufs[0].phi, bufs[0].phi, M, ncclFloat, ncclSum, s.comm, s.s_compute));
        } else if (P > 1) {
            for (size_t k = 0; k < c->shards.size(); ++k) {
                Shard &s = c->shards[k];
                uint32_t a, e;
                range(s.rank, a, e);
                if (a >= e) continue;
                CU(c, cudaSetDevice(s.device));
                for (size_t o = 0; o < c->shards.size(); ++o)
                    if (o != k)
                        CU(c, cudaMemcpyPeerAsync(bufs[o].phi + a, c->shards[o].device, bufs[k].phi + a, s.device, (size_t)(e - a) * 4,
                                                  s.s_compute));
            }
            if (int rc = sync_all(c)) return rc; // every shard's phi is complete
        }
        ++t;
        // ---- the unbinding step, the same on every shard: frame velocities, energies, flags, compaction, next set
        for (size_t k = 0; k < c->shards.size(); ++k) {
            Shard &s = c->shards[k];
            GpBufs &b = bufs[k];
            CU(c, cudaSetDevice(s.device));
            const unsigned gm = (M + 255) / 256;
            if (unbind) {
                CU(c, cudaMemsetAsync(b.phi_out, 0, (size_t)n * 4, s.s_compute));
                const uint32_t pieces = (M + GP_PIECE - 1) / GP_PIECE;
                gp_piece_kernel<<<(pieces + 255) / 256, 256, 0, s.s_compute>>>(b.mem[cur], b.info, b.vm, L, b.piece);
                gp_frame_kernel<<<gm, 256, 0, s.s_compute>>>(b.lo, b.hi, b.info, b.piece);
                c->launches += 2;
            }
            gp_finish_kernel<<<gm, 256, 0, s.s_compute>>>(b.mem[cur], b.info, b.lo, unbind ? b.vm : nullptr, L, b.piece, b.phi,
                                                          b.flags, b.bound, b.phi_out);
            c->launches++;
            CU(c, cudaGetLastError());
            if (!unbind) continue;
            CU(c, cub::DeviceSelect::Flagged(b.temp, b.temp_bytes, b.mem[cur], b.flags, b.mem[cur ^ 1], b.info, (int)M, s.s_compute));
            c->launches++; // the compaction (counted once)
            if (t < max_iter)
                if (int rc = prepare(s, b, cur ^ 1, M)) return rc;
        }
        if (!unbind) break;
        cur ^= 1;
        if (int rc = read_info()) return rc;
        if (info[0] == M) { conv = true; break; }
        M = info[0];
        if (t == max_iter) break;
    }
    Shard &s = c->shards[0];
    CU(c, cudaSetDevice(s.device));
    if (phi) CU(c, cudaMemcpyAsync(phi, bufs[0].phi_out, (size_t)n * 4, cudaMemcpyDeviceToHost, s.s_compute));
    if (bound) CU(c, cudaMemcpyAsync(bound, bufs[0].bound, (size_t)n * 4, cudaMemcpyDeviceToHost, s.s_compute));
    if (int rc = sync_all(c)) return rc;
    if (n_iter) *n_iter = t;
    if (converged) *converged = conv ? 1 : 0;
    return B200NB_OK;
}

} // namespace

extern "C" {

int b200nb_group_potential(b200nb_ctx *c, const uint32_t *group, float *phi)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "group_potential before upload");
    if (!group || !phi) return fail(c, B200NB_EINVAL, "group_potential: group or phi is NULL");
    return groups_run(c, group, 0, nullptr, phi, nullptr, nullptr);
}

int b200nb_unbind(b200nb_ctx *c, const uint32_t *group, uint32_t max_iter, uint32_t *bound, float *phi, uint32_t *n_iter,
                  int *converged)
{
    if (!c) return B200NB_EINVAL;
    if (!c->uploaded) return fail(c, B200NB_ESTATE, "unbind before upload");
    if (!group || !bound) return fail(c, B200NB_EINVAL, "unbind: group or bound is NULL");
    if (max_iter == 0) return fail(c, B200NB_EINVAL, "unbind: max_iter must be >= 1");
    return groups_run(c, group, max_iter, bound, phi, n_iter, converged);
}

int b200nb_sync(b200nb_ctx *c)
{
    if (!c) return B200NB_EINVAL;
    DeviceGuard guard;
    return sync_all(c);
}

uint64_t b200nb_slice_length(uint64_t n_bodies, int n_ranks)
{
    if (n_ranks < 1) return 0;
    const uint64_t per = (n_bodies + n_ranks - 1) / n_ranks;
    return (per + SLICE_ALIGN - 1) / SLICE_ALIGN * SLICE_ALIGN;
}
uint64_t b200nb_n_bodies(const b200nb_ctx *c) { return c ? c->n : 0; }
int b200nb_n_local_gpus(const b200nb_ctx *c) { return c ? (int)c->shards.size() : 0; }
uint64_t b200nb_allocated_bytes(const b200nb_ctx *c)
{
    uint64_t b = 0;
    if (c) for (auto &s : c->shards) b += s.bytes;
    return b;
}
uint64_t b200nb_launch_count(const b200nb_ctx *c) { return c ? c->launches : 0; }
const char *b200nb_kernel_name(const b200nb_ctx *c) { return c ? c->kname.c_str() : ""; }
const char *b200nb_exchange_name(const b200nb_ctx *c)
{
    if (!c) return "";
    return c->n_ranks == 1 ? "none" : (c->p2p ? "p2p-push" : "nccl-allgather");
}

int b200nb_event_record(b200nb_ctx *c, int slot)
{
    if (!c || slot < 0 || slot >= N_TIMER_SLOTS) return B200NB_EINVAL;
    DeviceGuard guard;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaEventRecord(s.timer[slot], s.s_compute));
    }
    return B200NB_OK;
}

int b200nb_event_elapsed_ms(b200nb_ctx *c, int a, int b, float *ms)
{
    if (!c || !ms || a < 0 || b < 0 || a >= N_TIMER_SLOTS || b >= N_TIMER_SLOTS) return B200NB_EINVAL;
    DeviceGuard guard;
    float mx = 0.f;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        CU(c, cudaEventSynchronize(s.timer[b]));
        float t = 0.f;
        CU(c, cudaEventElapsedTime(&t, s.timer[a], s.timer[b]));
        mx = std::max(mx, t);
    }
    *ms = mx;
    return B200NB_OK;
}

int b200nb_profile_enable(b200nb_ctx *c, int on)
{
    if (!c) return B200NB_EINVAL;
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    for (auto &s : c->shards) { // pending pairs are dropped, their events kept for reuse
        s.prof_free.insert(s.prof_free.end(), s.prof.begin(), s.prof.end());
        s.prof.clear();
        s.prof_ms = 0.0;
        s.prof_n = 0;
    }
    c->profiling = on != 0;
    return B200NB_OK;
}

int b200nb_profile_get(b200nb_ctx *c, double *force_ms_total, uint64_t *force_launches)
{
    if (!c) return B200NB_EINVAL;
    DeviceGuard guard;
    if (int rc = sync_all(c)) return rc;
    double mx = 0.0;
    uint64_t n = 0;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        if (int rc = prof_drain(c, s)) return rc;
        mx = std::max(mx, s.prof_ms);
        n = std::max<uint64_t>(n, s.prof_n);
    }
    if (force_ms_total) *force_ms_total = mx;
    if (force_launches) *force_launches = n;
    return B200NB_OK;
}

int b200nb_flush_l2(b200nb_ctx *c)
{
    if (!c) return B200NB_EINVAL;
    DeviceGuard guard;
    constexpr size_t bytes = 256ull << 20;
    for (auto &s : c->shards) {
        CU(c, cudaSetDevice(s.device));
        if (!s.l2_scratch) CU(c, cudaMalloc(&s.l2_scratch, bytes));
        CU(c, cudaMemsetAsync(s.l2_scratch, 0x5a, bytes, s.s_compute));
    }
    return B200NB_OK;
}

int b200nb_host_alloc(void **ptr, uint64_t bytes)
{
    if (!ptr) return B200NB_EINVAL;
    cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(nullptr, B200NB_ECUDA, "cudaHostAlloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return B200NB_OK;
}

int b200nb_host_free(void *ptr)
{
    if (!ptr) return B200NB_OK;
    return cudaFreeHost(ptr) == cudaSuccess ? B200NB_OK : B200NB_ECUDA;
}

} // extern "C"
