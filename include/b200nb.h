/* b200nb.h — C ABI of libb200nb: the B200-native all-pairs gravity engine behind MUrB's `--im gpu+b200`.
 *
 * The reference (albtad01/NBody-EuroHPC) has no FFI; its seam is the C++ virtual class
 * SimulationNBodyInterface<T> (src/common/core/SimulationNBodyInterface.hpp:15-88) selected by the `--im` string in
 * createImplem() (src/murb/main.cpp:205-270).  The glue class SimulationNBodyB200 (nbody-eurohpc_b200/glue/) derives
 * from that interface and forwards to the functions below; see INTEGRATION.md for the one-branch patch a maintainer
 * adds to main.cpp.  Every entry point names the reference code it replaces.
 *
 * Conventions
 *  - plain C, plain pointers and sizes, no C++/torch types, no exceptions across the boundary;
 *  - return 0 (B200NB_OK) on success, a B200NB_E* code otherwise; b200nb_last_error() gives the text.  The library
 *    never calls exit() (the reference's CUDA_CHECK does: SimulationNBodyCUDATileFullDevice.cu:10-17) — the glue maps a
 *    failure onto the reference convention (print + exit);
 *  - host pointers are borrowed for the duration of the call; the context owns all device memory, streams, events
 *    and NCCL communicators; the caller's current CUDA device is restored before returning;
 *  - a context is used from one host thread at a time (the reference never calls an implementation from more than
 *    one thread); several contexts may exist one after another or side by side;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with B200NB_ECUDA.
 *
 * Units follow the reference: SI, fp32 state, G = 6.67384e-11f (SimulationNBodyInterface.hpp:18).
 */
#ifndef B200NB_H_
#define B200NB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200NB_VERSION 100

enum {
    B200NB_OK = 0,
    B200NB_EINVAL = 1, /* bad argument */
    B200NB_ECUDA = 2,  /* CUDA runtime / driver error, or no device */
    B200NB_ENCCL = 3,  /* NCCL missing or failed */
    B200NB_ESTATE = 4  /* call not valid in the current state (e.g. step before upload) */
};

/* Integrators.  0 is MUrB's scheme, Bodies<T>::updatePositionAndVelocity (src/common/core/Bodies.cpp:259-278) ==
 * devUpdatePositionsAndVelocities (src/common/core/CUDABodies.cu:125-153):  q += (v + a*dt/2)*dt ; v += a*dt.
 * 1 is the kick-drift-kick leapfrog the reference documents but does not implement correctly
 * (spec: src/common/core/CUDABodies.cu:172-211):  v+ = v + a(x)*dt/2 ; x' = x + v+*dt ; v' = v+ + a(x')*dt/2. */
enum { B200NB_INTEGRATOR_MURB = 0, B200NB_INTEGRATOR_LEAPFROG = 1 };

typedef struct b200nb_ctx b200nb_ctx;

/* ---- lifetime ------------------------------------------------------------------------------------------------
 * Replaces: CUDABodies ctor/dtor (src/common/core/CUDABodies.cu:3-49,379-399) + SimulationNBodyCUDATileFullDevice
 * ctor/dtor (src/murb/implem/SimulationNBodyCUDATileFullDevice.cu:155-201,238-244). */

/* One process driving n_gpus devices (0 = every visible device, 1 = the current device).  Targets are sharded
 * contiguously over the devices; for n_gpus > 1 positions are exchanged with ncclAllGather each step. */
int b200nb_create(b200nb_ctx **out, uint64_t n_bodies, int n_gpus, float G, float soft);

/* One process driving n_shards shards with an explicit placement: shard i (targets [i*L, (i+1)*L)) lives on CUDA device
 * devices[i].  A device may be listed more than once ("virtual shards"): the slice arithmetic, chunk rotation, double
 * buffering and exchange of the multi-GPU path then run on a single GPU, which is how the sharded path is tested on a
 * one-GPU box.  Shards that share a device exchange positions with the p2p-push path (see b200nb_exchange_name; NCCL
 * cannot hold the same GPU twice in a communicator).  n_shards <= 16.
 * Replaces: the rank layout of SimulationNBodyMultiNode.cpp:62-91 (MPI ranks -> shards). */
int b200nb_create_sharded(b200nb_ctx **out, uint64_t n_bodies, int n_shards, const int *devices, float G, float soft);

/* One process per GPU (torchrun style): this process owns shard `rank` of `n_ranks` on CUDA device `device`.
 * nccl_id is the 128-byte ncclUniqueId made by b200nb_comm_unique_id() on rank 0 and broadcast by the caller
 * (ignored, may be NULL, when n_ranks == 1); like any ncclUniqueId it is good for ONE context — make a fresh one
 * for every b200nb_create_rank.  Collective over all ranks when n_ranks > 1.
 * Replaces: MPI_Init + buildCountsDispls in SimulationNBodyMultiNode.cpp:62-91. */
int b200nb_create_rank(b200nb_ctx **out, uint64_t n_bodies, float G, float soft, int rank, int n_ranks, int device,
                       const void *nccl_id);
int b200nb_comm_unique_id(void *id128);

void b200nb_destroy(b200nb_ctx *ctx);
const char *b200nb_last_error(const b200nb_ctx *ctx); /* ctx may be NULL: error of the last failed create */

/* ---- state ---------------------------------------------------------------------------------------------------
 * Host SoA arrays of n_bodies floats, the layout of dataSoA_t (src/common/core/Bodies.hpp:15-24).
 * upload replaces CUDABodies::memcpyBuffersOnDevice (CUDABodies.cu:31-49) and devInitializeDevGM
 * (SimulationNBodyCUDATileFullDevice.cu:41-45): G*m is folded into the device layout once.  Every rank passes the
 * full arrays (the reference's MPI variant replicates state the same way, SimulationNBodyMultiNode.cpp:93-117), but
 * each shard copies only its own slice (and reads the last body, where the padding sits) across the host link; the
 * position exchange of the step path then replicates the slices on every GPU.  Collective when n_ranks > 1. */
int b200nb_upload(b200nb_ctx *ctx, const float *qx, const float *qy, const float *qz, const float *m, const float *vx,
                  const float *vy, const float *vz);

/* Joins all devices, then copies positions and velocities of all n_bodies back (any pointer may be NULL).
 * Replaces the lazy D2H in CUDABodies::getDataSoA (CUDABodies.cu:63-93).  Collective when n_ranks > 1. */
int b200nb_download_state(b200nb_ctx *ctx, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz);

/* The same for the local shards' own bodies only: entries [first, first + count) of each array are written (global
 * indexing, see b200nb_slice_bounds), the rest is left untouched.  With one rank per process this is the D2H side of
 * a sharded driver (every rank keeps the host copy of its own targets, the analogue of the send buffers of
 * SimulationNBodyMultiNode.cpp:119-148) and moves 24 B per local body instead of 24 B per body per rank.  Not
 * collective. */
int b200nb_download_slice(b200nb_ctx *ctx, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz);

/* Accelerations of the last force pass (b200nb_accel or the last step).  Replaces getAccSoA()
 * (SimulationNBodyCUDAPropertyTracking.cu:308-319).  Collective when n_ranks > 1. */
int b200nb_download_accel(b200nb_ctx *ctx, float *ax, float *ay, float *az);

/* ---- the hot path ---------------------------------------------------------------------------------------------
 * b200nb_step == n_steps x computeOneIteration() (SimulationNBodyCUDATileFullDevice.cu:203-236; oracle:
 * SimulationNBodyNaive.cpp:56-61): force pass over all N^2 ordered pairs, self included, then the integrator.
 * Asynchronous: returns after enqueueing; b200nb_sync / download_* join. */
int b200nb_step(b200nb_ctx *ctx, float dt, int integrator, int n_steps);

/* Force pass only: computeBodiesAcceleration() (SimulationNBodyNaive.cpp:34-53) on the current positions. */
int b200nb_accel(b200nb_ctx *ctx);

/* Integrator only, with caller-supplied accelerations (host SoA, n_bodies each): the shape of
 * Bodies<T>::updatePositionsAndVelocities(const accSoA_t&, T&) (Bodies.cpp:280-288; CUDABodies.cu:353-371), which
 * test_CUDABodies.cpp:42-75 exercises.  MUrB integrator only. */
int b200nb_integrate_host_accel(b200nb_ctx *ctx, const float *ax, const float *ay, const float *az, float dt);

/* Total energy  sum_i [ m_i |v_i|^2 / 2  -  (1/2) sum_{j != i} G m_i m_j / sqrt(|r_ij|^2 + soft^2) ],  accumulated in
 * fp64.  Definition: devComputeBodiesMetrics (SimulationNBodyCUDAPropertyTracking.cu:217-304), which subtracts the
 * self term the same way.  Joins the devices.  Collective when n_ranks > 1. */
int b200nb_energy(b200nb_ctx *ctx, double *total);

/* Every per-iteration metric of the reference's history in one pass (SimulationHistory.hpp:12-15; CSV columns
 * "iteration,energy,ang_momentum,density_center_x,density_center_y,density_center_z", SimulationHistory.hpp:45 and
 * SimulationHistory.cpp:103-122).  Upstream only ever fills in the energy (SimulationNBodyCUDAPropertyTracking.cu:
 * 217-304); the angular momentum and density centre are declared and exported but never computed, so their
 * definitions are fixed here:  L = sum_i m_i (r_i x v_i) about the origin (ang_momentum = |L|);  centre of mass;
 * density centre = sum_i w_i r_i / sum_i w_i with w_i = m_i * sum_{j != i} G m_j / sqrt(|r_ij|^2 + soft^2), the
 * potential-weighted centre.  out[B200NB_N_METRICS], fp64.  Joins the devices.  Collective when n_ranks > 1. */
enum {
    B200NB_METRIC_ENERGY = 0,
    B200NB_METRIC_ANG_X = 1, B200NB_METRIC_ANG_Y = 2, B200NB_METRIC_ANG_Z = 3,
    B200NB_METRIC_MASS = 4,
    B200NB_METRIC_COM_X = 5, B200NB_METRIC_COM_Y = 6, B200NB_METRIC_COM_Z = 7,
    B200NB_METRIC_DENSITY_X = 8, B200NB_METRIC_DENSITY_Y = 9, B200NB_METRIC_DENSITY_Z = 10,
    B200NB_N_METRICS = 11
};
int b200nb_metrics(b200nb_ctx *ctx, double *out);

/* ---- the gravitational field ----------------------------------------------------------------------------------
 * The reference has no counterpart: it only ever asks for the acceleration of each body.  Same G, softening and G*m
 * fold as the force pass:
 *   field at a point p, over ALL bodies:  a(p) = sum_j G m_j (q_j - p) / (|q_j - p|^2 + soft^2)^(3/2),
 *                                         phi(p) = -sum_j G m_j / (|q_j - p|^2 + soft^2)^(1/2);
 *   per-body potential, self pair excluded by INDEX (a body at the same position as another still counts it):
 *                                         phi_i = -sum_{j != i} G m_j / (|r_ij|^2 + soft^2)^(1/2),
 * so b200nb_energy == sum_i m_i |v_i|^2 / 2 + (1/2) sum_i m_i phi_i, and the density-centre weight of b200nb_metrics is
 * w_i = -m_i phi_i.  fp32 pair terms, hierarchical sums finished in fp64 (same accuracy design as the force pass).
 * A result depends only on its point (or body) and the current bodies: bit-identical whatever the other points of
 * the call, their number, the shard or rank count, and on reruns.  Neither call changes the simulation state
 * (positions, velocities, the accelerations of b200nb_download_accel, the leapfrog's stored a(x_n), cached step graphs);
 * both are ordered after a preceding asynchronous b200nb_step and join the devices before returning.  Device scratch is
 * bounded (points go through in fixed-size batches), grow-only, owned by the context and counted in
 * b200nb_allocated_bytes. */

/* Acceleration and potential at n_points arbitrary points (host SoA).  Any output pointer may be NULL.  Joins the
 * devices.  Collective when n_ranks > 1: every rank passes the same points and receives every result.
 * n_points == 0 is a no-op; NULL point arrays otherwise give B200NB_EINVAL; B200NB_ESTATE before an upload. */
int b200nb_field(b200nb_ctx *ctx, uint64_t n_points, const float *px, const float *py, const float *pz,
                 float *ax, float *ay, float *az, float *phi);
/* Per-body potential of the current positions, self pair excluded, all n_bodies values.  Collective when n_ranks > 1. */
int b200nb_potential(b200nb_ctx *ctx, float *phi);

/* ---- the tidal tensor -----------------------------------------------------------------------------------------
 * The derivative of the field above, T_ab = d a_a / d p_b = -d^2 phi / dp_a dp_b: the input of tidal and Jacobi radii,
 * tidal-field histories along orbits, tidal-environment classification by eigenvalue signs and |lambda|^(-1/2)
 * time-step criteria.  The reference has no counterpart.  Same G, softening and G*m fold as b200nb_field; with
 * d = q_j - p and s^2 = |d|^2 + soft^2:
 *   at a point p, over ALL bodies:         T_ab(p) = sum_j G m_j [ 3 d_a d_b / s^5 - delta_ab / s^3 ],
 *   per body, self pair excluded by INDEX: T_ab,i  = sum_{j != i} (the same term with p = q_i),
 * exactly d a_a / d p_b of the softened a(p) of b200nb_field.  One body at distance r with soft = 0 gives
 * G m / r^3 * diag(2, -1, -1) in a frame whose x axis points at it; the trace is -3 soft^2 sum_j G m_j / s^5 (0 for
 * soft = 0 away from bodies).  Output: six fp32 components per target, rows t[i][6] in the order xx, yy, zz, xy, xz, yz.
 * Accuracy: fp32 pair terms whose every intermediate stays in fp32's normal range, sums finished in fp64; every entry is
 * within 5e-6 * A_ab of fp64, A_ab = sum_j G m_j (3 |d_a d_b| / s^5 + delta_ab / s^3) (the cancellation-free scale).
 * Same calling contract as the field section: a result depends only on its point (or body) and the current bodies,
 * bit-identical whatever the other points of the call, the batching, the shard or rank count, and on reruns; ordered after
 * a preceding asynchronous b200nb_step; joins the devices; collective when n_ranks > 1 (every rank passes the same points
 * and receives every row); no change to the simulation state, the stored accelerations, the tracers or cached step
 * graphs.  Padding bodies add nothing.  Non-finite results occur exactly where b200nb_field gives them (a point on a body,
 * or coincident bodies, when soft = 0).  Device scratch is grow-only, owned by the context and counted in
 * b200nb_allocated_bytes; targets go through in batches of B = min(32768, Q rounded up to a multiple of 256), Q = the
 * points or bodies of one rank, and a call needs 28 * S * B + 36 * B bytes per GPU (at most 56 MiB + 1.125 MiB), plus
 * 24 * B * n_ranks for the gathered rows when each rank is its own process, S = min(64, max(1, ceil(ceil(n_bodies / 128)
 * / 32))).  The buffer is shared with the field, neighbour and friends-of-friends calls: it grows to the largest need.
 * Errors: B200NB_ESTATE before an upload; B200NB_EINVAL for NULL point arrays or a NULL t.  n_points == 0 is a no-op. */

/* Tidal tensor at n_points arbitrary points (host SoA); t[n_points][6]. */
int b200nb_tidal(b200nb_ctx *ctx, uint64_t n_points, const float *px, const float *py, const float *pz, float *t);
/* Tidal tensor of every body, self pair excluded; t[n_bodies][6]. */
int b200nb_tidal_bodies(b200nb_ctx *ctx, float *t);

/* ---- field by component ---------------------------------------------------------------------------------------
 * Who pulls on whom in a run with several structures (the galaxies of a merger, a disk, bulge and halo, a satellite):
 * the field of b200nb_field split by source component, the input of rotation-curve decompositions, the self and
 * interaction energies of a merger, and the force and torque between components (dynamical friction, angular-momentum
 * exchange).  The reference has no counterpart.  Labels comp[n_bodies] (uint32) and n_comp in [1, 64]: a body with
 * comp[j] = h < n_comp is a source of component h; a body labelled B200NB_NO_GROUP is a source of nothing but is still a
 * target in bodies mode.  Same law, G, softening and G*m fold as b200nb_field; with d = q_j - p:
 *   at a point p:  a^h(p)   = sum_{j: comp[j] = h} G m_j d / (|d|^2 + soft^2)^(3/2),
 *                  phi^h(p) = -sum_{j: comp[j] = h} G m_j / (|d|^2 + soft^2)^(1/2);
 *   per body i:    the same sums at p = q_i, self pair excluded by INDEX (it matters only for h = comp[i]).
 * A component without members gives a = 0 and phi = -0.  Rows: acc[m][n_comp][3], phi[m][n_comp].
 * Promises:
 *  1. bit-identity with the field: with one component holding every body (n_comp = 1, every label 0),
 *     b200nb_component_field returns b200nb_field's ax, ay, az and phi, and b200nb_component_field_bodies returns
 *     b200nb_potential's phi, bit for bit;
 *  2. locality: the value for (target, h) depends only on the target (its point, or its index in bodies mode) and on the
 *     positions and masses of h's members in index order.  It is bit-identical when other bodies are relabelled, merged,
 *     split or set to NO_GROUP, when n_comp changes and when h is renumbered, and across reruns, batching, the other
 *     points of the call, and the shard and rank count;
 *  3. accuracy: per component, the field's bound: |a - a64| <= 1e-6 * sum_{j in h} |a_ij| and |phi - phi64| <= 1e-6 *
 *     |phi64| (galaxy and random schemes, soft 2e8 and 1e4).
 * Calling contract of the field section: ordered after a preceding asynchronous b200nb_step; joins the devices;
 * collective when n_ranks > 1 (every rank passes the same labels and points and receives every row); no change to the
 * simulation state, the stored accelerations, the leapfrog's a(x_n), the tracers or cached step graphs.  acc or phi may be
 * NULL.  n_points == 0 is a no-op.  Errors: B200NB_ESTATE before an upload; B200NB_EINVAL for a NULL comp, n_comp outside
 * [1, 64], a label that is neither < n_comp nor B200NB_NO_GROUP, or NULL point arrays.
 * Cost: one field pass whatever n_comp, plus at most 127 padding sources per component.  Device scratch is grow-only,
 * owned by the context, counted in b200nb_allocated_bytes and shared with the field, tidal, neighbour and friends-of-
 * friends calls.  With M_h the members of h, T = sum_h 128 * ceil(M_h / 128) packed sources, S_h = 0 for M_h = 0 and
 * min(64, max(1, ceil(ceil(M_h / 128) / 32))) otherwise, S = sum_h S_h (<= ceil(n_bodies / 4096) + n_comp), and targets in
 * batches of B = min(Q rounded up to a multiple of 512, 65536, max(1, floor(2^22 / (512 * max(S, 1)))) * 512), Q = the
 * points or bodies of one rank, a call needs per GPU
 *     r(16 * S * B) + r(16 * T) + r(4 * T) + r(4 * n_bodies) [bodies mode only] + r(8 * S) + r(4 * (n_comp + 1))
 *     + 12 * B + 16 * n_comp * B,     r(x) = x rounded up to a multiple of 256,
 * plus 16 * n_comp * B * n_ranks for the gathered rows when each rank is its own process: at most 64 MiB of partial rows
 * and 64 MiB of result rows, plus 20 B per packed source.  Kernel launches per call: one packing kernel per GPU when some
 * component has members, and per batch the field kernel (when some component has members) and one reduction. */

/* a^h and phi^h at n_points arbitrary points (host SoA): acc[n_points][n_comp][3], phi[n_points][n_comp] */
int b200nb_component_field(b200nb_ctx *ctx, const uint32_t *comp, uint32_t n_comp, uint64_t n_points, const float *px,
                           const float *py, const float *pz, float *acc, float *phi);
/* a^h and phi^h of every body, self pair excluded: acc[n_bodies][n_comp][3], phi[n_bodies][n_comp] */
int b200nb_component_field_bodies(b200nb_ctx *ctx, const uint32_t *comp, uint32_t n_comp, float *acc, float *phi);

/* ---- nearest neighbours ---------------------------------------------------------------------------------------
 * The k nearest bodies of every body, or of arbitrary points (close encounters, bound pairs, Casertano-Hut densities
 * from the 6th neighbour, nearest-distance time-step criteria).  The reference has no counterpart.  Definition, for a
 * target p and a body j at q_j (fp32, round to nearest, no softening, no flush to zero):
 *   dx = xj - px, dy = yj - py, dz = zj - pz;   d2 = dx*dx;  d2 = fmaf(dy, dy, d2);  d2 = fmaf(dz, dz, d2);
 * Candidates are ordered by the key (d2, j) lexicographically, a strict total order, so the k smallest keys are unique
 * and the result is a pure function of the fp32 positions: it does not depend on batching, shard or rank count, and
 * the answer for k is the first k columns of the answer for any larger k.  Reported distance: sqrtf(d2), correctly
 * rounded.  Bodies mode excludes the self pair by INDEX (a coincident body is a neighbour at distance 0); points mode
 * takes every body (a point on a body has it at distance 0).  Mass plays no part: zero-mass bodies are neighbours too.
 * Padding bodies (index >= n_bodies) are never candidates.  Slots that cannot be filled (k > n_bodies - 1 for bodies,
 * k > n_bodies for points) hold idx = 0xFFFFFFFF, dist = +inf.  d2 overflows to +inf for separations above ~1.8e19 m
 * (the force pass forms the same fp32 d2, so the library already assumes smaller systems); such pairs still come in
 * (d2, j) order, after every finite one.  Bodies at non-finite positions are never neighbours.
 * k ranges over [1, 32].  Same calling contract as the field section: ordered after a preceding asynchronous
 * b200nb_step, joins the devices, collective when n_ranks > 1 (every rank receives every row), no change to the
 * simulation state.  Device scratch is grow-only, owned by the context, counted in b200nb_allocated_bytes and bounded
 * independently of n_bodies and n_points: each launch's batch is sized from k so that its candidate rows stay within
 * 2^23 entries (64 MiB); with the staged points and result rows it stays within 84 MiB per GPU, plus 16 MiB per rank
 * for the gathered rows when each rank is its own process.  Errors: B200NB_ESTATE before an upload, B200NB_EINVAL for k outside
 * [1, 32] or NULL point arrays. */

/* k nearest other bodies of every body; idx/dist are [n_bodies][k] row-major; either may be NULL. */
int b200nb_neighbors(b200nb_ctx *ctx, uint32_t k, uint32_t *idx, float *dist);
/* k nearest bodies of n_points arbitrary points (host SoA); outputs [n_points][k].  n_points == 0 is a no-op. */
int b200nb_neighbors_at(b200nb_ctx *ctx, uint64_t n_points, const float *px, const float *py, const float *pz,
                        uint32_t k, uint32_t *idx, float *dist);

/* ---- friends-of-friends groups --------------------------------------------------------------------------------
 * Which bodies form a structure together (the galaxies of a merger, tidal tails, satellites, clumps): the standard
 * friends-of-friends group finder of N-body work.  The reference has no counterpart.  Definition, for bodies i != j
 * (fp32, round to nearest, no flush to zero, the operation sequence of the nearest-neighbour section):
 *   dx = xj - xi, dy = yj - yi, dz = zj - zi;   d2 = dx*dx;  d2 = fmaf(dy, dy, d2);  d2 = fmaf(dz, dz, d2);
 * i and j are linked iff d2 <= b2, where b2 = b*b rounded to fp32.  fp32 subtraction is exactly antisymmetric, so d2(i, j)
 * and d2(j, i) are bitwise equal: the relation is symmetric and the library visits each unordered pair from one side
 * only.  Groups are the connected components of the link graph; group[i] is the SMALLEST body index in i's group, so a
 * body without friends has group[i] = i.  The result is a pure function of the fp32 positions and b: it does not depend
 * on shard or rank count, chunking, reruns or the order in which the device's atomics land.  Mass plays no part
 * (zero-mass bodies link like any other); padding bodies (index >= n_bodies) are never linked; a body at a non-finite
 * position has d2 NaN or +inf with everyone and is always alone.  b must be >= 0 with b*b finite in fp32 (b <= ~1.84e19);
 * b = 0 links exactly the coincident bodies.  Same calling contract as the field section: ordered after a preceding
 * asynchronous b200nb_step, joins the devices, collective when n_ranks > 1 (every rank receives all n_bodies labels), no
 * change to the simulation state.  Device scratch is grow-only, owned by the context and counted in
 * b200nb_allocated_bytes: with N_pad = n_ranks * b200nb_slice_length(n_bodies, n_ranks) and P = n_ranks, one forest of
 * 4 * N_pad bytes per shard; the shard that merges (the first, when the shards are in one process), or every rank when
 * each rank is its own process, holds P forests, 4 * N_pad * P bytes, instead.  O(N), independent of the number of
 * links.  Errors: B200NB_ESTATE before an upload, B200NB_EINVAL for a NULL group or a b outside the range above. */

/* friends-of-friends groups of linking length b; group[n_bodies] = smallest body index of each body's group */
int b200nb_fof(b200nb_ctx *ctx, float b, uint32_t *group);

/* ---- phase-space friends-of-friends ---------------------------------------------------------------------------
 * Friends-of-friends in positions AND velocities (6D FoF, Diemand et al. 2006; the first stage of Rockstar).  When two
 * systems overlap in space, in a collision or a fly-by, position-only groups merge them into one; their bodies are close
 * in space but far apart in velocity, so in phase space they stay apart.  Definition (fp32, round to nearest, no flush to
 * zero): the scales are s_x = 1.0f / b_x and s_v = 1.0f / b_v, each a correctly rounded fp32 division (b = +inf gives 0,
 * which switches that part of the metric off).  The scaled coordinates of body i are
 *   X = x*s_x, Y = y*s_x, Z = z*s_x, U = vx*s_v, V = vy*s_v, W = vz*s_v   (each product rounded to fp32)
 * of the current state, as b200nb_download_state returns it.  For bodies i != j, with dX = Xj - Xi, ..., dW = Wj - Wi:
 *   d2 = dX*dX;  d2 = fmaf(dY, dY, d2);  d2 = fmaf(dZ, dZ, d2);  d2 = fmaf(dU, dU, d2);  d2 = fmaf(dV, dV, d2);
 *   d2 = fmaf(dW, dW, d2);
 * i and j are linked iff d2 <= 1.0f.  fp32 subtraction is exactly antisymmetric, so d2(i, j) and d2(j, i) are bitwise
 * equal and the library visits each unordered pair from one side only.  Groups are the connected components; group[i] is
 * the SMALLEST body index in i's group: a pure function of the fp32 state and the two scales, independent of shard or
 * rank count, chunking, reruns and the order of the device's atomics.  Mass plays no part; padding bodies are never
 * linked; a non-finite scaled coordinate (a NaN or inf position or velocity, or an overflow for a tiny b) gives d2 NaN
 * or +inf with everyone, so that body is alone.  If both b are +inf every body links to every other.
 * If b_x is a power of two and b_v = +inf, the scaling is exact (away from subnormals and overflow, velocities finite)
 * and the labels are b200nb_fof(b_x)'s: scaling by a power of two commutes with every rounding, so d2 is b200nb_fof's d2
 * times s_x*s_x, and the velocity terms add exact zeros.
 * b_x and b_v must be > 0 (+inf allowed); 0, negative values and NaN are B200NB_EINVAL.  The result feeds
 * b200nb_unbind and b200nb.fof_groups like b200nb_fof's labels.  Same calling contract as b200nb_fof: ordered after a
 * preceding asynchronous b200nb_step, joins the devices, collective when n_ranks > 1 (every rank receives all n_bodies
 * labels), no change to the simulation state.  Device scratch is grow-only, owned by the context and counted in
 * b200nb_allocated_bytes: with N_pad and P as in the friends-of-friends section, every shard holds the scaled array of
 * all bodies, 24 * N_pad bytes, followed by b200nb_fof's forests (4 * N_pad bytes, or 4 * N_pad * P on the shard that
 * merges and on every rank when each rank is its own process).  Errors: B200NB_ESTATE before an upload, B200NB_EINVAL
 * for a NULL group or a b outside the range above. */

/* phase-space friends-of-friends groups of linking lengths b_x (positions) and b_v (velocities); group[n_bodies] =
 * smallest body index of each body's group */
int b200nb_fof_phase(b200nb_ctx *ctx, float b_x, float b_v, uint32_t *group);

/* ---- group potential and unbinding ----------------------------------------------------------------------------
 * Which bodies of a group are held together by gravity: the unbinding step of every halo or structure finder, whose
 * result (the bound mass of each structure) is the diagnostic of a merger or of tidal stripping.  The reference has no
 * counterpart.  Labels group[n_bodies] are arbitrary uint32 values (friends-of-friends roots of b200nb_fof, galaxy or
 * component ids, halo ids from elsewhere); a body labelled B200NB_NO_GROUP takes no part in anything.
 * Group potential, for a body i whose label g != B200NB_NO_GROUP:
 *   phi^g_i = -sum_{j != i, group[j] = g} G m_j / (|r_ij|^2 + soft^2)^(1/2),
 * self pair excluded by index, with the G, softening, G*m fold, fp32 pair terms and fp64 second-level sums of
 * b200nb_potential; with a single label it agrees with b200nb_potential to about 1e-6 relative, not bitwise.  phi = +0
 * for NO_GROUP bodies and for bodies alone in their label.  Padding bodies never contribute; zero-mass bodies feel the
 * potential but add nothing to it; a body at a non-finite position makes its group's values NaN (b200nb_fof puts such
 * bodies alone).  The result is a pure function of the positions, the masses and the whole label array: bit-identical
 * on reruns, for any shard or rank count and straight after an asynchronous step.  It is not promised to be bitwise
 * invariant under a relabelling, which may move rounding in the last bits.
 * Unbinding: S_0 = {i : group[i] != NO_GROUP}.  Pass t = 1, 2, ..., max_iter takes phi_i, the group potential over
 * S_(t-1), and for each label g the frame velocity V_g = sum m_j v_j / sum m_j over g's members in S_(t-1) (fp64 sums of
 * the fp32 masses and velocities in a fixed order; V_g = 0 when their mass is 0), evaluates
 * E_i = |v_i - V_g|^2 / 2 + phi_i in fp64 and keeps body i iff E_i < 0 (NaN leaves; a lone body, phi = 0, leaves).
 * S_t is the bodies kept.  The loop stops after the first pass that removes nobody (converged) or after max_iter passes.
 * Outputs: bound[i] = group[i] for i in the final set, NO_GROUP otherwise; phi (may be NULL) = phi of the last pass for
 * the bodies of the set it was computed over, +0 for the others (on convergence: the group potential of the final
 * set); n_iter = passes run (0 when S_0 is empty); converged.  n_iter and converged may be NULL.  It follows that
 * unbind(unbind(g, 1).bound, 1) returns bound and phi bit-identical to unbind(g, 2).
 * Same calling contract as the field section: ordered after a preceding asynchronous b200nb_step, joins the devices,
 * collective when n_ranks > 1 (every rank passes the same labels and receives every result), no change to the
 * simulation state or cached step graphs.  Device scratch is grow-only, owned by the context, counted in
 * b200nb_allocated_bytes and O(N) whatever the group sizes: on every shard, with N = n_bodies and N_pad = n_ranks *
 * b200nb_slice_length(n_bodies, n_ranks), at most 102 N + 16 N_pad bytes (rounded up to 256 B per array) plus 64 MiB of
 * partial sums (less when N < 262144) plus CUB's temporary storage for sorting N (key, value) pairs.
 * Errors: B200NB_ESTATE before an upload; B200NB_EINVAL for a NULL group, a NULL phi (group potential), a NULL bound or
 * max_iter == 0 (unbinding). */
#define B200NB_NO_GROUP 0xFFFFFFFFu

/* phi[n_bodies] = the group potential of the labels group[n_bodies] */
int b200nb_group_potential(b200nb_ctx *ctx, const uint32_t *group, float *phi);
/* unbinding of the labels group[n_bodies], at most max_iter passes; bound[n_bodies], phi[n_bodies] (may be NULL) */
int b200nb_unbind(b200nb_ctx *ctx, const uint32_t *group, uint32_t max_iter, uint32_t *bound, float *phi,
                  uint32_t *n_iter, int *converged);

/* ---- test particles -------------------------------------------------------------------------------------------
 * Massless test particles ("tracers") moving in the field of the bodies: the restricted N-body method (Toomre & Toomre)
 * that resolves tidal tails, bridges and stripped material at N*M instead of (N+M)^2 interactions per step.  The
 * reference has no counterpart.  A context holds M >= 0 tracers, each an fp32 position p and velocity w.  Tracers have
 * no mass: they never act on the bodies or on each other, and the bodies move exactly as without them.
 * Every b200nb_step iteration advances them with the bodies' integrator and dt.  A tracer's acceleration a(p) is the
 * b200nb_field acceleration at p over all bodies, bit for bit (same kernel, same chunking, same fixed-order fp64
 * reduction, rounded once to fp32), taken at the body positions of the same instant:
 *  - MUrB:      a = a(p_n; q_n), the positions before the update; then p and w are updated with the operation sequence of
 *               the bodies' MUrB update:  adt = a*dt (fp32);  p' = fp32(p + (w + adt*0.5)*dt) evaluated in fp64;
 *               w' = w + adt (fp32);
 *  - leapfrog:  w+ = fmaf(a(p_n; q_n), dt*0.5f, w);  p' = fp32(fma((double)w+, dt, (double)p));
 *               w' = fmaf(a(p'; q_{n+1}), dt*0.5f, w+),  the bodies' kick-drift-kick; a(p_n; q_n) is kept between steps
 *               as the bodies keep a(x_n).
 * It follows that a tracer's trajectory depends only on its own initial state and on the body trajectory: not on the
 * other tracers, on M, on the shard or rank count, on whether a step went through a captured graph, or on reruns.
 * Non-finite tracer states, and a tracer exactly on a body when soft = 0, give what b200nb_field gives there.
 * Body uploads: tracers persist across b200nb_upload; an upload invalidates their stored acceleration, as it does the
 * bodies' a(x_0), so the next leapfrog step evaluates a(p; q) anew.  b200nb_integrate_host_accel moves the bodies but not
 * the tracers, and invalidates their stored acceleration likewise.  b200nb_accel, the field / neighbour / group calls,
 * b200nb_energy and b200nb_metrics neither read nor change tracers.  With M = 0 a context behaves exactly as one that
 * never had tracers: the same launches, the same step graphs, the same state and the same b200nb_allocated_bytes.
 * Placement: tracers are split contiguously over the ranks, T = ceil(M / n_ranks) rounded up to a multiple of 512 per
 * shard (rank r owns tracers [r*T, min((r+1)*T, M)); later shards may own none); a shard keeps its slice as device SoA
 * and never exchanges it.  Device bytes, counted in b200nb_allocated_bytes and freed with the tracer set (replacement,
 * removal or b200nb_destroy), on every local shard when M > 0:
 *     36 * T + 16 * S * min(T, 65536),     S = min(64, max(1, ceil(ceil(n_bodies / 128) / 32)))
 * (positions, velocities and the stored acceleration, plus the partial sums of the field pass, at most 64 MiB).
 * Both calls are collective when n_ranks > 1: every rank passes the full arrays and keeps only its own slice, or
 * receives every tracer.  Host pointers are borrowed for the duration of the call.  b200nb_set_tracers is allowed before
 * the first b200nb_upload (a step still needs one); it joins the devices and drops the cached step graphs.
 * Errors: B200NB_EINVAL for NULL arrays with n_tracers > 0 or a per-shard slice T >= 2^31; B200NB_ECUDA when the device
 * memory cannot be allocated (a set larger than a device's free memory fails before anything is allocated).  Any error
 * leaves the context with no tracers at all, never half set. */

/* replaces the context's tracers; n_tracers == 0 removes them (pointers ignored); SoA host arrays of n_tracers floats */
int b200nb_set_tracers(b200nb_ctx *ctx, uint64_t n_tracers, const float *qx, const float *qy, const float *qz,
                       const float *vx, const float *vy, const float *vz);
/* joins the devices, copies back all tracers (any pointer may be NULL) */
int b200nb_download_tracers(b200nb_ctx *ctx, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz);
uint64_t b200nb_n_tracers(const b200nb_ctx *ctx);

/* ---- external potential --------------------------------------------------------------------------------------
 * A static analytic host potential acting on the bodies and the tracers: the galaxy, halo or cluster that strips a
 * satellite, at O(N) per step instead of the millions of live bodies it would take.  The reference has no counterpart.
 * A context holds 0 to B200NB_EXTERNAL_MAX terms; Phi_ext is their sum and a_ext = -grad Phi_ext.  SI units, fp64
 * parameters.  With d = p - centre evaluated in fp64 from the fp32 position p, r = |d| and R^2 = dx^2 + dy^2:
 *   Plummer         Phi = -gm / sqrt(r^2 + a^2)                      a >= 0 (a = 0: a point mass)
 *   Hernquist       Phi = -gm / (r + a)                              a > 0; a_ext = 0 exactly at r = 0
 *   NFW             Phi = -gm ln(1 + r/a) / r  (-gm/a at r = 0)      a = r_s > 0; gm = G M_s = 4 pi G rho_0 r_s^3;
 *                   a_ext = -gm mu(r/a) d / r^3, mu(x) = ln(1+x) - x/(1+x); a_ext = 0 exactly at r = 0
 *   Miyamoto-Nagai  Phi = -gm / sqrt(R^2 + (a + sqrt(z^2 + b^2))^2) a >= 0, b > 0
 *   logarithmic     Phi = gm/2 ln(R^2 + z^2/q^2 + r_c^2)             gm = v_0^2, a = r_c > 0, b = q > 0
 * Every parameter must be finite, gm >= 0, reserved = 0, and b = 0 for Plummer, Hernquist and NFW.  The terms are summed
 * in the order given, starting from +0, in explicitly rounded fp64 arithmetic whose operation order
 * csrc/external_sm100.cuh states: a host restatement of that order compiled without contraction matches bit for bit
 * wherever no log is involved (every Phi and a_ext of Plummer, Hernquist and Miyamoto-Nagai, the logarithmic a_ext),
 * and within 1e-14 relative otherwise.  NFW's mu(x) uses a positive series below x = 0.1, so Phi and |a_ext| are within
 * 1e-12 relative of exact for every x >= 0.
 * Where the terms act, with e = a_ext in fp64 at the current fp32 position:
 *  - bodies: the step rounds S + e to fp32, S the fp64 sum of the self-gravity partials (MUrB at q_n; leapfrog at the
 *    positions of the force pass, a(x_0) and the closing kick at x_{n+1}).  The stored accelerations include e:
 *    b200nb_download_accel, b200nb_accel and the leapfrog's a(x_n).  b200nb_integrate_host_accel adds nothing;
 *  - tracers: a(p) = fp32(a_field(p) sums + e(p)), at the same instants as without terms;
 *  - b200nb_energy and METRIC_ENERGY add sum_i m_i Phi_ext(q_i) in fp64; the other metrics are unchanged;
 *  - b200nb_field, potential, tidal, component_field*, neighbors*, fof, group_potential and unbind keep describing the
 *    bodies' own field; add b200nb_external_field for the total.
 * With no terms a context makes the same launches and graphs, holds the same b200nb_allocated_bytes and gives
 * bit-identical results to one that never had terms; with terms the step makes no extra launches.  The terms are
 * kernel arguments, no device memory is set aside for them.
 * b200nb_set_external replaces the set (n_terms = 0 removes it).  It is allowed before the first upload, joins the
 * devices, drops the cached step graphs and invalidates the leapfrog's stored a(x_n) and tracer a(p), so the next
 * leapfrog step evaluates them under the new terms.  Every rank must pass the same terms.  Not collective.
 * Errors (B200NB_EINVAL; the previous terms stay in place): n_terms > B200NB_EXTERNAL_MAX, NULL terms with n_terms > 0,
 * an unknown kind, reserved != 0, a parameter outside the rules above. */
#define B200NB_EXTERNAL_MAX 8
enum {
    B200NB_EXT_PLUMMER = 0, B200NB_EXT_HERNQUIST = 1, B200NB_EXT_NFW = 2,
    B200NB_EXT_MIYAMOTO_NAGAI = 3, B200NB_EXT_LOGARITHMIC = 4
};
typedef struct b200nb_external_term { /* 56 bytes */
    int32_t kind, reserved; /* reserved must be 0 */
    double gm;              /* G*M [m^3 s^-2]; NFW: G*M_s = 4 pi G rho_0 r_s^3; logarithmic: v_0^2 [m^2 s^-2] */
    double a;               /* Plummer a | Hernquist a | NFW r_s | MN a | logarithmic r_c   [m] */
    double b;               /* MN b [m] | logarithmic q (flattening); must be 0 for the other kinds */
    double centre[3];       /* [m] */
} b200nb_external_term;

int b200nb_set_external(b200nb_ctx *ctx, uint32_t n_terms, const b200nb_external_term *terms);
/* the current terms into out[0 .. *n_terms) (out has room for B200NB_EXTERNAL_MAX) */
int b200nb_get_external(const b200nb_ctx *ctx, b200nb_external_term *out, uint32_t *n_terms);
/* a_ext and Phi_ext in fp64 at n_points fp32 points (host SoA): bit for bit the e and Phi_ext the step uses there (the
 * same device evaluator).  Any output may be NULL; n_points == 0 is a no-op.  Allowed before an upload; not collective
 * (each rank evaluates all its points).  Points go through the context's grow-only query scratch in batches of at most
 * 2^20, 44 B each (at most 44 MiB per call, counted in b200nb_allocated_bytes and shared with the field calls).  Joins
 * the device of the first local shard.  Errors: B200NB_EINVAL for NULL point arrays with n_points > 0. */
int b200nb_external_field(b200nb_ctx *ctx, uint64_t n_points, const float *px, const float *py, const float *pz,
                          double *ax, double *ay, double *az, double *phi);

/* ---- basis-function expansion ---------------------------------------------------------------------------------
 * The mean field of a structure in a few hundred numbers: the self-consistent-field (SCF) expansion of Hernquist &
 * Ostriker (1992, ApJ 386, 375) in the normalisation of Lowing et al. (2011, MNRAS 416, 2697), the basis gala, AGAMA and
 * galpy provide.  Uses: l = 2 / m = 2 power (triaxiality, bars), l = 1 lopsidedness and monopole drift over time; a
 * potential without sqrt(N) sampling noise and without softening (rotation curves, escape speeds, tracer orbits).  The
 * reference has no counterpart.  Inputs: scale radius a > 0 [m], centre c (fp64 [3]), nmax in [0, 31], lmax in [0, 15].
 * For a body or point p, with d = p - c in fp64 (from the fp32 coordinates): r = |d|, s = r / a, xi = (s - 1)/(s + 1),
 * cos theta = d_z / r, phi the azimuth of (d_x, d_y).
 *   Phi~_nl(s) = - s^l (1+s)^-(2l+1) C_n^(2l+3/2)(xi)                      (Gegenbauer polynomial)
 *   K_nl       = n(n+4l+3)/2 + (l+1)(2l+1)
 *   A~_nl      = - 2^(8l+6) n! (n+2l+3/2) Gamma(2l+3/2)^2 / (4 pi K_nl Gamma(n+4l+3))
 *   N_lm       = (2l+1) (l-m)! / (l+m)!
 *   S_nlm      = (2 - delta_m0) A~_nl N_lm (1/a) sum_k (G m_k) Phi~_nl(s_k) P_l^m(cos theta_k) cos(m phi_k)
 *   T_nlm      = the same with sin(m phi_k)                                 (T_nl0 = 0)
 *   Phi(p)     = sum_{n<=nmax, l<=lmax, m<=l} Phi~_nl(s) P_l^m(cos theta) [S_nlm cos(m phi) + T_nlm sin(m phi)]
 *   a(p)       = -grad Phi(p)
 * P_l^m carries the Condon-Shortley phase (as scipy.special.lpmv); it cancels between coefficients and evaluation.  G m_k
 * is the fp32 G*m fold of the force pass, so S and T are in m^2/s^2.  A Hernquist sphere of mass M and scale a has
 * S_000 = GM/a and every other coefficient 0, and then Phi = -GM/(r + a).  Members: the bodies k < n_bodies with
 * group[k] == label (group == NULL: every body); padding bodies never take part.  A body at r = 0 adds to l = 0 only
 * (s^l = 0), without a NaN from its undefined angles.  A member at a non-finite position, or with a non-finite G*m,
 * makes every S and every T with m > 0 NaN (T_nl0 stays 0); nothing is filtered.  Layout of S and T: packed
 * [nmax+1][(lmax+1)(lmax+2)/2], index n*(lmax+1)(lmax+2)/2 + l(l+1)/2 + m.
 * Evaluation: at r = 0 (the centre itself) Phi is the l = 0 sum and a = 0, since the l = 0 term has a cusp there whose
 * direction is undefined; everywhere else, the z axis included, Phi and a are the formulas above, finite.
 * Promises:
 *  1. pure function: the coefficients depend only on the fp32 positions and G*m of the members, the member mask, nmax,
 *     lmax, a and c.  Bit-identical on reruns, for any shard or rank count, straight after an asynchronous step of
 *     either integrator or a graph-replayed one, and when non-members are relabelled; group == NULL is bit-identical to
 *     a label array that puts every body in `label`;
 *  2. truncation: the coefficients of (nmax', lmax') <= (nmax, lmax) are the matching entries of the larger call, bit
 *     for bit (the summation order of a coefficient does not depend on nmax or lmax);
 *  3. locality: Phi and a at a point depend only on the point, the coefficients, nmax, lmax, a and c: bit-identical
 *     under any batching and whatever the other points of the call;
 *  4. accuracy: fp64 recurrences (Gegenbauer in n, reduced associated Legendre in l) with host tables rounded once from
 *     long double; every coefficient is within 1e-12 of its cancellation-free scale sum_k |term_k| of an exact
 *     evaluation, and Phi and each component of a within 1e-12 of sum |term| at the point.
 * Calling contract of the field section: both calls are ordered after a preceding asynchronous b200nb_step, join the
 * device of the first local shard and change nothing in the state (positions, velocities, the stored accelerations, the
 * leapfrog's a(x_n), the tracers, the external terms, cached step graphs).  Neither is collective:
 * b200nb_scf_coefficients runs on the first local shard over its replicated body array, so every rank computes the same
 * result on its own device; b200nb_scf_field is allowed before an upload.  Device scratch is grow-only, owned by the
 * context, counted in b200nb_allocated_bytes and shared with the field calls.  With K = (nmax+1)(lmax+1)(lmax+2)/2
 * (at most 4352), C = min(512, ceil(n_bodies / 64)) chunks and r(x) = x rounded up to a multiple of 256:
 *   coefficients  r(12952) + r(8 K) + r(16 K) + r(16 K C) + r(4 n_bodies) [only with group]  bytes: at most 34 MiB of
 *                 partial rows;
 *   field         r(12952) + r(16 K) + 44 B per point of a batch of B = min(2^20, n_points rounded up to 256): at most
 *                 44 MiB + 81 KiB.
 * Kernel launches: two per coefficient call; one per batch of the field call.
 * Errors: B200NB_ESTATE for coefficients before an upload; B200NB_EINVAL for nmax or lmax out of range, a not finite or
 * <= 0, a NULL or non-finite centre, NULL S or T, and NULL point arrays with n_points > 0 (n_points == 0 is a no-op). */
#define B200NB_SCF_NMAX 31
#define B200NB_SCF_LMAX 15

/* coefficients of the bodies with group[i] == label (group == NULL: all bodies); S, T packed [nmax+1][(lmax+1)(lmax+2)/2],
 * index n*(lmax+1)(lmax+2)/2 + l(l+1)/2 + m */
int b200nb_scf_coefficients(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3],
                            const uint32_t *group, uint32_t label, double *S, double *T);
/* Phi and a of an expansion at n_points fp32 points (host SoA), fp64 outputs, any output may be NULL */
int b200nb_scf_field(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3], const double *S,
                     const double *T, uint64_t n_points, const float *px, const float *py, const float *pz,
                     double *ax, double *ay, double *az, double *phi);

/* ---- frozen expansion as an external potential -------------------------------------------------------------------
 * A host taken from a simulation (triaxial, lopsided, barred) expanded once and frozen: the satellite, stream or tracers
 * then move in it at O(N) per step, as gala, AGAMA and galpy run orbits in simulated haloes.  A context holds at most one
 * expansion (nmax, lmax, a, centre, S, T) next to its 0 to B200NB_EXTERNAL_MAX analytic terms, with exactly the meaning,
 * packed layout and limits of b200nb_scf_field; its Phi_scf and a_scf at an fp32 point are bit for bit what
 * b200nb_scf_field returns there.  With an expansion the external field is, per component, in fp64:
 *   e = fl(e_terms + a_scf),  Phi_ext = fl(Phi_terms + Phi_scf)
 * where e_terms and Phi_terms are the sums of the analytic terms above (+0 without terms); the expansion is added last.
 * Everything "external potential" states for the terms holds with this e and Phi_ext: the bodies' step rounds S + e once
 * to fp32 (MUrB at q_n, the leapfrog's a(x_0) and closing kick at x_{n+1}); the stored accelerations include it;
 * b200nb_integrate_host_accel adds nothing; tracers take a(p) = fp32(field sums + e(p)) at the same instants;
 * b200nb_energy and METRIC_ENERGY add sum_i m_i Phi_ext(q_i); b200nb_external_field returns the total e and Phi_ext, bit
 * for bit what the step uses.  The field, tidal, component, neighbour, friends-of-friends, group and SCF calls keep
 * describing the bodies' own field.
 * b200nb_set_external_scf installs or replaces the expansion; S == NULL and T == NULL removes it (the other arguments
 * are then ignored).  Lifecycle as b200nb_set_external: allowed before the first upload, not collective (every rank
 * passes the same expansion), joins the devices, drops the cached step graphs and invalidates the leapfrog's stored
 * a(x_n) and tracer a(p).  b200nb_set_external and b200nb_set_external_scf do not affect each other.
 * Cost: one extra kernel launch per local shard for every evaluation of e (each force pass of a step, each tracer pass
 * of a shard with tracers, each energy or metrics call).  Without an expansion, whether or not one was ever set, a
 * context makes the same launches and step graphs, holds the same b200nb_allocated_bytes and gives bit-identical results.
 * Device memory, per local shard, counted in b200nb_allocated_bytes and freed on removal or b200nb_destroy, with
 * K = (nmax+1)(lmax+1)(lmax+2)/2, r(x) = x rounded up to a multiple of 256, L = b200nb_slice_length and T the tracer
 * slots per shard of "test particles":
 *   r(12952) + r(16 K_max)   the tables and S | T, K_max the largest K set since the expansion was last removed
 *                            (grow-only while an expansion is set; at most 82 688 bytes);
 *   32 L                     fp64 (ax, ay, az, Phi) of each slot of the shard's body slice;
 *   32 T                     with tracers, fp64 (ax, ay, az, Phi) of each tracer slot, allocated by whichever of
 *                            b200nb_set_tracers and b200nb_set_external_scf comes second and freed by either.
 * A failed allocation leaves the context with no expansion (B200NB_ECUDA), never with half of one; one in
 * b200nb_set_tracers leaves it with no tracers.
 * Errors (B200NB_EINVAL; the previous expansion stays in place): nmax or lmax out of range, a not finite or <= 0, a NULL
 * or non-finite centre, exactly one of S and T NULL, a non-finite S or T entry, a T_nl0 != 0 (b200nb_scf_coefficients
 * always returns +0 there). */
int b200nb_set_external_scf(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3],
                            const double *S, const double *T);
/* *present = 0 or 1; when 1, fills nmax, lmax, a, centre and S and T (packed, K entries each), each where non-NULL */
int b200nb_get_external_scf(const b200nb_ctx *ctx, uint32_t *present, uint32_t *nmax, uint32_t *lmax, double *a,
                            double centre[3], double *S, double *T);

/* Joins every device and communication stream.  main.cpp:353-371 only synchronises the current device, so the glue
 * calls this when more than one device is in use. */
int b200nb_sync(b200nb_ctx *ctx);

/* ---- introspection / measurement ------------------------------------------------------------------------------ */
/* Targets per rank L (host only): rank r owns global bodies [r*L, min((r+1)*L, n)).  Contiguous, balanced to the
 * 256-body granularity (two 128-body AoSoA blocks; the launch rounds up to whole target tiles on its own); the
 * analogue of buildCountsDispls (SimulationNBodyMultiNode.cpp:76-91). */
uint64_t b200nb_slice_length(uint64_t n_bodies, int n_ranks);
/* Global body range [first, first + count) owned by the local_shard-th shard of this context (0 <= local_shard <
 * b200nb_n_local_gpus); count is 0 for a shard that holds only padding. */
int b200nb_slice_bounds(const b200nb_ctx *ctx, int local_shard, uint64_t *first, uint64_t *count);
uint64_t b200nb_n_bodies(const b200nb_ctx *ctx);
int b200nb_n_local_gpus(const b200nb_ctx *ctx);
uint64_t b200nb_allocated_bytes(const b200nb_ctx *ctx); /* device bytes, all local GPUs */
uint64_t b200nb_launch_count(const b200nb_ctx *ctx);    /* kernels of this library launched so far */
const char *b200nb_kernel_name(const b200nb_ctx *ctx);  /* force-kernel variant in use */
/* How positions travel between GPUs each step (the role of the MPI_Allgatherv calls of
 * SimulationNBodyMultiNode.cpp:93-148): "none" (one GPU); "nccl-allgather" (default) - in-place ncclAllGather on a
 * communication stream, overlapped with the own-slice force launch; "p2p-push" - in-process multi-GPU with NVLink peer
 * access, chosen with B200NB_EXCHANGE=p2p or when libnccl cannot be loaded: the integrator kernel stores the new
 * positions of its slice into every GPU's double-buffered body array, one event per GPU is the only synchronisation.
 * The two produce bit-identical results. */
const char *b200nb_exchange_name(const b200nb_ctx *ctx);

/* CUDA-event stopwatch on the library's own compute stream(s) (torch.cuda.Event cannot see them).
 * slot in [0,8); elapsed is the max over the local devices. */
int b200nb_event_record(b200nb_ctx *ctx, int slot);
int b200nb_event_elapsed_ms(b200nb_ctx *ctx, int slot_start, int slot_stop, float *ms);

/* When enabled every force-kernel launch is bracketed by events; get returns the accumulated device time of the
 * force kernels and their launch count since the last enable (joins the devices). */
int b200nb_profile_enable(b200nb_ctx *ctx, int on);
int b200nb_profile_get(b200nb_ctx *ctx, double *force_ms_total, uint64_t *force_launches);

/* Evicts the L2 between timed steps: overwrites a 256 MiB scratch buffer (larger than the 126 MB L2) on the compute
 * stream(s) with cudaMemsetAsync.  Measurement hygiene only; the hot path never calls it. */
int b200nb_flush_l2(b200nb_ctx *ctx);

/* Page-locked host buffers for the end-to-end path (cudaHostAlloc / cudaFreeHost). */
int b200nb_host_alloc(void **ptr, uint64_t bytes);
int b200nb_host_free(void *ptr);

/* ---- initial conditions (host only, no GPU needed) ------------------------------------------------------------
 * Bit-identical restatement of Bodies<float>::initGalaxy / initRandomly (src/common/core/Bodies.cpp:158-257) for
 * drivers that do not link the reference (bench.py).  scheme: 0 = "galaxy", 1 = "random"; arrays of n floats;
 * uses glibc srand(seed)/rand() in the reference's call order.  Not thread-safe (libc rand state). */
int b200nb_init_bodies(int scheme, uint64_t n, unsigned seed, float *qx, float *qy, float *qz, float *vx, float *vy,
                       float *vz, float *m, float *r);

/* The reference's file-based scheme, Bodies<T>::initMilkyWayAndromeda (src/common/core/Bodies.cpp:82-153): a text file
 * with one body per non-empty line, "mass x y z vx vy vz" in galaxy units, rescaled per galaxy component.  Count the
 * bodies first, then load into arrays of that many floats.  Host only. */
int b200nb_tab_count(const char *path, uint64_t *n_bodies);
int b200nb_tab_load(const char *path, uint64_t n, float *qx, float *qy, float *qz, float *vx, float *vy, float *vz,
                    float *m, float *r);

#ifdef __cplusplus
}
#endif
#endif /* B200NB_H_ */
