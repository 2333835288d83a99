// Basis-function (self-consistent-field) expansion of the bodies' potential in the Hernquist-Ostriker basis, for sm_100a:
// the coefficients S_nlm, T_nlm of b200nb_scf_coefficients and the evaluator of b200nb_scf_field.  Definition and
// normalisation: include/b200nb.h, "basis-function expansion".
//
// Basis values, per body or point with d = p - c (fp64 from the fp32 coordinates), r = |d|, s = r / a:
//   radial   Phi~_nl(s) = -P_l(s) C_n^(2l+3/2)(xi),  P_l = (s/(1+s))^l (1+s)^-(l+1) = q t^l with q = 1/(1+s), t = s q^2,
//            xi = (s-1)/(s+1), C_n by the three-term recurrence C_n = ga[l][n] xi C_(n-1) - gb[l][n] C_(n-2) (host table);
//   angular  P_l^m(cos th) {cos, sin}(m ph) = Q_l^m(x) {Re, Im} w^m,  x = d_z / r, w = (d_x + i d_y) / r,
//            Q_l^m = P_l^m / sin^m th the reduced polynomial (Q_m^m = (-1)^m (2m-1)!!, Q_l^m = qa x Q_(l-1)^m - qb Q_(l-2)^m).
// No atan2, sin or cos; exact on the z axis.  At r = 0 the kernels take x = 0 and w = 0, so only l = 0 terms survive
// (P_l(0) = 0 for l > 0) and nothing is NaN.  A non-finite d makes s NaN, so every basis value of that body is NaN.
//
// Coefficients (scf_coef_kernel + scf_reduce_kernel): the body range is cut into n_chunks contiguous chunks, a function
// of n_bodies alone (scf_chunks).  One CTA per chunk stages SCF_SB bodies at a time in shared memory: Gm_k Phi~_nl(s_k)
// as R[k][l][n] (one thread per (body, l) runs the n recurrence) and Q_l^m {Re, Im} w^m as A[k][l][2m + part] (one thread
// per (body, m) runs the l recurrence).  Non-members, padding and bodies past the chunk stage exact zeros.  Each thread
// then owns up to SCF_TILES register tiles of 4 n x (2 m x {Re, Im}) accumulators of one l: per l the chunk's part of
// R_l^T A_l.  Every accumulator is its own fma chain over the chunk's bodies in index order starting from +0, so a
// coefficient's partial sum does not depend on nmax, lmax or which thread holds it (x + (+-0) leaves x unchanged, and an
// accumulator that starts at +0 never becomes -0).  The reduce kernel sums the rows in chunk order and multiplies by
// F_nlm = (2 - delta_m0) A~_nl N_lm / a from the host.  Hence the "sub-block" promise: (nmax', lmax') <= (nmax, lmax) gives
// the matching entries bit for bit.
//
// Evaluation (scf_eval, called by scf_field_kernel and by external_sm100.cuh's ext_total_kernel): one thread per point,
// S, T and the tables in shared memory.  For each m it runs the l
// recurrences of Q_l^m and Q_l^(m+1), for each (l, m) the n recurrence of C_n and of dC_n/dxi (the recurrence
// differentiated), and dots them with S and T.  The gradient is assembled in Cartesian form:
//   grad Phi = (dPhi/ds / a) u + (V - u (u . V)) / r,  u = d / r,
// where V is the gradient of the angular factors in u taken as free variables: d/du_x Q w^m = m Q w^(m-1),
// d/du_y = i m Q w^(m-1), d/du_z = Q' w^m with Q_l^m' = -Q_l^(m+1).  No 1/sin th anywhere; a = 0 at r = 0.
#pragma once
#include <cstdint>

namespace b200nb {

constexpr int SCF_NMAX = 31, SCF_LMAX = 15;
constexpr int SCF_THREADS = 256;
constexpr int SCF_SB = 8;        // bodies staged per round: SCF_SB * (lmax + 1) <= 128 radial and as many angular threads
constexpr int SCF_TILES = 3;     // register tiles per thread: 3 * 256 >= 576, the tile count at nmax = 31, lmax = 15
constexpr uint32_t SCF_MAX_CHUNKS = 512, SCF_MIN_CHUNK = 64;
constexpr uint32_t SCF_EVAL_THREADS = 128;
constexpr uint32_t SCF_BATCH = 1u << 20; // points per scf_field_kernel launch

// Recurrence coefficients, computed on the host in long double and rounded once (the same table for every call).
struct ScfTables {
    double ga[SCF_LMAX + 1][SCF_NMAX + 1]; // 2 (n + alpha - 1) / n,  alpha = 2l + 3/2   (n >= 1)
    double gb[SCF_LMAX + 1][SCF_NMAX + 1]; // (n + 2 alpha - 2) / n
    double qa[SCF_LMAX + 2][SCF_LMAX + 2]; // (2l - 1) / (l - m)   (l > m)
    double qb[SCF_LMAX + 2][SCF_LMAX + 2]; // (l + m - 1) / (l - m)
    double qs[SCF_LMAX + 2];               // (-1)^m (2m - 1)!!
};

struct ScfArgs {
    const float *bodies;     // the replicated AoSoA-128 body array: x | y | z | G*m per block
    const uint32_t *group;   // labels (nullptr: every body is a member)
    const ScfTables *tab;
    double *partial;         // [n_chunks][2][K] rows: S sums then T sums
    uint32_t label, n, chunk, nmax, lmax, K;
    double cx, cy, cz, a;
};

// Chunks of the coefficient pass: a function of n_bodies alone.  min(512, ceil(n / 64)), each ceil(n / n_chunks) long.
__host__ __device__ inline uint32_t scf_chunks(uint32_t n)
{
    const uint32_t c = (n + SCF_MIN_CHUNK - 1) / SCF_MIN_CHUNK;
    return c < 1 ? 1 : (c > SCF_MAX_CHUNKS ? SCF_MAX_CHUNKS : c);
}
__host__ __device__ inline uint32_t scf_npad(uint32_t nmax) { return (nmax + 4) / 4 * 4; }        // n rows, in 4s
__host__ __device__ inline uint32_t scf_apad(uint32_t lmax) { return 2 * ((lmax + 2) / 2 * 2); } // 2 x m columns, m in 2s
__host__ __device__ inline size_t scf_coef_smem(uint32_t nmax, uint32_t lmax)
{
    return (size_t)SCF_SB * (lmax + 1) * (scf_npad(nmax) + scf_apad(lmax)) * sizeof(double);
}
__host__ __device__ inline size_t scf_field_smem(uint32_t K) { return sizeof(ScfTables) + 2 * (size_t)K * sizeof(double); }

// s, xi, x = cos th and w = (wr, wi) of the point p relative to the centre
struct ScfGeom {
    double r, s, xi, x, wr, wi;
};
__device__ __forceinline__ ScfGeom scf_geom(float px, float py, float pz, double cx, double cy, double cz, double a)
{
    ScfGeom g;
    const double dx = (double)px - cx, dy = (double)py - cy, dz = (double)pz - cz;
    g.r = sqrt(dx * dx + dy * dy + dz * dz);
    const bool pos = g.r > 0.0;
    g.s = g.r <= 1.79769313486231570e308 ? g.r / a : __longlong_as_double(0x7ff8000000000000ll); // non-finite d: NaN
    g.xi = (g.s - 1.0) / (g.s + 1.0);
    g.x = pos ? dz / g.r : 0.0;
    g.wr = pos ? dx / g.r : 0.0;
    g.wi = pos ? dy / g.r : 0.0;
    return g;
}

__device__ __forceinline__ void scf_body(const float *__restrict__ bodies, uint32_t i, float &x, float &y, float &z, float &gm)
{
    const float *b = bodies + (size_t)(i / 128) * 512 + (i % 128);
    x = b[0]; y = b[128]; z = b[256]; gm = b[384];
}

__global__ void __launch_bounds__(SCF_THREADS) scf_coef_kernel(const ScfArgs A)
{
    extern __shared__ double smem[];
    const uint32_t L1 = A.lmax + 1, NP = scf_npad(A.nmax), AP = scf_apad(A.lmax), NB = NP / 4;
    double *R = smem;                                  // [SB][L1][NP]
    double *Ang = smem + (size_t)SCF_SB * L1 * NP;     // [SB][L1][AP]
    const uint32_t tid = threadIdx.x;
    const uint32_t lo = blockIdx.x * A.chunk, hi = min(lo + A.chunk, A.n);

    // this thread's tiles: (l, n block, column block of 2 m values x {Re, Im})
    uint32_t tl[SCF_TILES], tn[SCF_TILES], tc[SCF_TILES];
    bool tv[SCF_TILES];
#pragma unroll
    for (int j = 0; j < SCF_TILES; ++j) {
        uint32_t t = tid + j * SCF_THREADS, l = 0;
        tv[j] = false; tl[j] = 0; tn[j] = 0; tc[j] = 0;
        for (; l < L1; ++l) {
            const uint32_t cb = (l + 2) / 2, cnt = NB * cb;
            if (t < cnt) { tv[j] = true; tl[j] = l; tn[j] = t / cb; tc[j] = t % cb; break; }
            t -= cnt;
        }
    }
    double acc[SCF_TILES][16];
#pragma unroll
    for (int j = 0; j < SCF_TILES; ++j)
#pragma unroll
        for (int e = 0; e < 16; ++e) acc[j][e] = 0.0;

    for (uint32_t base = lo; base < hi; base += SCF_SB) {
        __syncthreads(); // the previous round's tiles have read the stage
        if (tid < SCF_SB * L1) { // radial: body k, degree l, the n recurrence
            const uint32_t k = tid / L1, l = tid % L1, i = base + k;
            double *row = R + ((size_t)k * L1 + l) * NP;
            double w = 0.0, xi = 0.0;
            if (i < hi) {
                float x, y, z, gm;
                scf_body(A.bodies, i, x, y, z, gm);
                if (!A.group || A.group[i] == A.label) {
                    const ScfGeom g = scf_geom(x, y, z, A.cx, A.cy, A.cz, A.a);
                    const double q = 1.0 / (1.0 + g.s), t = g.s * q * q;
                    double P = q;
                    for (uint32_t e = 0; e < l; ++e) P *= t;
                    w = -(P * (double)gm);
                    xi = g.xi;
                }
            }
            double cp = 0.0, c = 1.0;
            row[0] = w;
            for (uint32_t n = 1; n < NP; ++n) {
                double v = 0.0;
                if (n <= A.nmax) {
                    const double cn = A.tab->ga[l][n] * xi * c - A.tab->gb[l][n] * cp;
                    cp = c; c = cn;
                    v = w * cn;
                }
                row[n] = v;
            }
        } else if (tid >= 128 && tid < 128 + SCF_SB * L1) { // angular: body k, order m, the l recurrence
            const uint32_t k = (tid - 128) / L1, m = (tid - 128) % L1, i = base + k;
            double x = 0.0, cm = 0.0, sm = 0.0;
            bool mem = false;
            if (i < hi) {
                float px, py, pz, gm;
                scf_body(A.bodies, i, px, py, pz, gm);
                if (!A.group || A.group[i] == A.label) {
                    const ScfGeom g = scf_geom(px, py, pz, A.cx, A.cy, A.cz, A.a);
                    x = g.x; cm = 1.0; sm = 0.0;
                    for (uint32_t e = 0; e < m; ++e) {
                        const double c2 = cm * g.wr - sm * g.wi;
                        sm = cm * g.wi + sm * g.wr;
                        cm = c2;
                    }
                    mem = true;
                }
            }
            double qp = 0.0, qv = mem ? A.tab->qs[m] : 0.0;
            for (uint32_t l = m; l < L1; ++l) {
                if (l > m) {
                    const double qn = A.tab->qa[l][m] * x * qv - A.tab->qb[l][m] * qp;
                    qp = qv; qv = qn;
                }
                double *row = Ang + ((size_t)k * L1 + l) * AP;
                row[2 * m] = qv * cm;
                row[2 * m + 1] = qv * sm;
            }
        }
        __syncthreads();
        const uint32_t nk = min((uint32_t)SCF_SB, hi - base);
#pragma unroll
        for (int j = 0; j < SCF_TILES; ++j) {
            if (!tv[j]) continue;
            const double *rp = R + (size_t)tl[j] * NP + 4 * tn[j];
            const double *ap = Ang + (size_t)tl[j] * AP + 4 * tc[j];
            for (uint32_t k = 0; k < nk; ++k) {
                const double2 r01 = *reinterpret_cast<const double2 *>(rp + (size_t)k * L1 * NP);
                const double2 r23 = *reinterpret_cast<const double2 *>(rp + (size_t)k * L1 * NP + 2);
                const double2 a01 = *reinterpret_cast<const double2 *>(ap + (size_t)k * L1 * AP);
                const double2 a23 = *reinterpret_cast<const double2 *>(ap + (size_t)k * L1 * AP + 2);
                const double rv[4] = {r01.x, r01.y, r23.x, r23.y}, av[4] = {a01.x, a01.y, a23.x, a23.y};
#pragma unroll
                for (int u = 0; u < 4; ++u)
#pragma unroll
                    for (int v = 0; v < 4; ++v) acc[j][u * 4 + v] = __fma_rn(rv[u], av[v], acc[j][u * 4 + v]);
            }
        }
    }
    double *row = A.partial + (size_t)blockIdx.x * 2 * A.K;
    const uint32_t LM = L1 * (L1 + 1) / 2;
#pragma unroll
    for (int j = 0; j < SCF_TILES; ++j) {
        if (!tv[j]) continue;
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const uint32_t n = 4 * tn[j] + u, m = 2 * tc[j] + v / 2;
                if (n <= A.nmax && m <= tl[j]) row[(v % 2) * A.K + n * LM + tl[j] * (tl[j] + 1) / 2 + m] = acc[j][u * 4 + v];
            }
    }
}

// out = [S | T] (K each): the chunk rows summed in chunk order from +0, times F; T_nl0 = +0
__global__ void __launch_bounds__(256) scf_reduce_kernel(const double *__restrict__ partial, const double *__restrict__ F,
                                                         uint32_t n_chunks, uint32_t K, uint32_t lmax, double *__restrict__ out)
{
    const uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= 2 * K) return;
    const uint32_t idx = o % K, LM = (lmax + 1) * (lmax + 2) / 2, lm = idx % LM;
    uint32_t l = 0;
    while ((l + 1) * (l + 2) / 2 <= lm) ++l;
    if (o >= K && lm == l * (l + 1) / 2) { out[o] = 0.0; return; } // m = 0: T_nl0 = 0
    double s = 0.0;
    for (uint32_t c = 0; c < n_chunks; ++c) s = __dadd_rn(s, partial[(size_t)c * 2 * K + o]);
    out[o] = __dmul_rn(s, F[idx]);
}

struct ScfFieldArgs {
    const double *coef;     // [S | T], K each, packed n (l (l+1)/2 + m)
    const ScfTables *tab;
    const float *px, *py, *pz;
    double *out;            // [4][stride]: ax, ay, az, phi
    uint32_t count, stride, nmax, lmax, K;
    double cx, cy, cz, a;
};

// Phi and a = -grad Phi of the expansion (S, T packed, tab the tables) at the fp32 point p: the one evaluator of
// b200nb_scf_field and of the step's external expansion (ext_total_kernel), so both give the same bits at a point.
// E is the kernel's argument struct (nmax, lmax, a, cx, cy, cz), read where the arithmetic uses it as scf_field_kernel
// always did.  Where ptxas would be free to fuse either product of a two-product sum and has been seen to choose
// differently between callers, the operation is written out: those are the choices scf_field_kernel compiled to
// before scf_eval existed, so b200nb_scf_field keeps its bits.
template <class E>
__device__ __forceinline__ void scf_eval(const ScfTables &tab, const double *S, const double *T, const E &A, float px, float py,
                                         float pz, double acc[3], double *phi_out)
{
    const ScfGeom g = scf_geom(px, py, pz, A.cx, A.cy, A.cz, A.a);
    const uint32_t L1 = A.lmax + 1, LM = L1 * (L1 + 1) / 2;
    const double q = 1.0 / (1.0 + g.s), t = g.s * q * q, dxi = 2.0 * q * q; // dxi / ds
    double phi = 0.0, gs = 0.0, vx = 0.0, vy = 0.0, vz = 0.0;
    double cm1 = 0.0, sm1 = 0.0, cm = 1.0, sm = 0.0; // w^(m-1), w^m
    double Pm = q;                                   // P_m = q t^m
    for (uint32_t m = 0; m < L1; ++m) {
        double qap = 0.0, qa = tab.qs[m], qbp = 0.0, qb = 0.0; // Q_l^m, Q_l^(m+1) (0 for l = m)
        double P = Pm;
        for (uint32_t l = m; l < L1; ++l) {
            if (l > m) {
                const double qn = tab.qa[l][m] * g.x * qa - tab.qb[l][m] * qap;
                qap = qa; qa = qn;
                if (l == m + 1) {
                    qb = tab.qs[m + 1];
                } else {
                    const double qn2 = tab.qa[l][m + 1] * g.x * qb - tab.qb[l][m + 1] * qbp;
                    qbp = qb; qb = qn2;
                }
                P *= t;
            }
            const double dP = P * ((double)l - (double)(l + 1) * g.s) * q / g.s; // dP_l / ds
            double cs = 0.0, ct = 0.0, ds = 0.0, dt = 0.0, cp = 0.0, c = 1.0, dp = 0.0, d = 0.0;
            const double *Sp = S + l * (l + 1) / 2 + m, *Tp = T + l * (l + 1) / 2 + m;
            for (uint32_t n = 0; n <= A.nmax; ++n) {
                if (n > 0) {
                    const double ga = tab.ga[l][n], gb = tab.gb[l][n];
                    const double cn = ga * g.xi * c - gb * cp, dn = ga * (c + g.xi * d) - gb * dp;
                    cp = c; c = cn; dp = d; d = dn;
                }
                const double sv = Sp[n * LM], tv = Tp[n * LM];
                cs += c * sv; ct += c * tv; ds += d * sv; dt += d * tv;
            }
            const double rs = -P * cs, rt = -P * ct;
            const double rds = -(dP * cs + P * dxi * ds), rdt = -(dP * ct + P * dxi * dt);
            const double re = qa * cm, im = qa * sm;
            phi += rs * re + rt * im;
            gs += rds * re + rdt * im;
            const double mq = (double)m * qa;
            vx += mq * (rs * cm1 + rt * sm1);
            vy += mq * (rt * cm1 - rs * sm1);
            vz -= qb * (rs * cm + rt * sm);
        }
        cm1 = cm; sm1 = sm;
        const double c2 = __fma_rn(cm, g.wr, -__dmul_rn(sm, g.wi));
        sm = __fma_rn(sm, g.wr, __dmul_rn(cm, g.wi));
        cm = c2;
        Pm *= t;
    }
    double ax = 0.0, ay = 0.0, az = 0.0;
    if (!(g.r == 0.0)) { // a = -grad Phi;  u = (wr, wi, x)
        const double uv = g.wr * vx + g.wi * vy + g.x * vz, k = gs / A.a;
        ax = -(k * g.wr + (vx - g.wr * uv) / g.r);
        ay = -(k * g.wi + (vy - g.wi * uv) / g.r);
        az = -(k * g.x + (vz - g.x * uv) / g.r);
    }
    acc[0] = ax; acc[1] = ay; acc[2] = az;
    *phi_out = phi;
}

__global__ void __launch_bounds__(SCF_EVAL_THREADS) scf_field_kernel(const ScfFieldArgs A)
{
    extern __shared__ double smem[];
    ScfTables &tab = *reinterpret_cast<ScfTables *>(smem);
    double *S = smem + sizeof(ScfTables) / sizeof(double), *T = S + A.K;
    {
        const double *src = reinterpret_cast<const double *>(A.tab);
        for (uint32_t e = threadIdx.x; e < sizeof(ScfTables) / sizeof(double); e += blockDim.x) smem[e] = src[e];
        for (uint32_t e = threadIdx.x; e < 2 * A.K; e += blockDim.x) S[e] = A.coef[e];
    }
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.count) return;
    double acc[3], phi;
    scf_eval(tab, S, T, A, A.px[i], A.py[i], A.pz[i], acc, &phi);
    A.out[i] = acc[0]; A.out[A.stride + i] = acc[1]; A.out[2 * (size_t)A.stride + i] = acc[2]; A.out[3 * (size_t)A.stride + i] = phi;
}

} // namespace b200nb
