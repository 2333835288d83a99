// Static analytic external potential (b200nb_set_external): the one __device__ evaluator of the terms, for sm_100a.
//
// Every kernel that applies the terms (integrate_kernel, tracer_update_kernel, energy_kernel, external_field_kernel)
// calls ext_eval, so the e and Phi_ext a step uses at an fp32 point are exactly what b200nb_external_field returns there.
// With a frozen expansion (b200nb_set_external_scf) ext_total_kernel below adds scf_eval's field to ext_eval's, and the
// <true, true> forms of those kernels read its output instead of calling ext_eval.
// The terms travel by value as a __grid_constant__ kernel parameter: no device memory, and a captured step graph bakes
// them in like any other argument (b200nb_set_external drops the cached graphs).
//
// Arithmetic: fp64, every operation explicitly rounded (__dadd_rn, __dmul_rn, __ddiv_rn, __dsqrt_rn), no contraction,
// in the order written below.  A host restatement compiled with -ffp-contract=off that performs the same operations in
// the same order (tests/external_oracle.c) matches bit for bit wherever no log / log1p is involved.  With
// d = p - centre (fp64 differences of the fp32 coordinates and the fp64 centre), x*x etc. rounded products:
//   R2 = dx*dx + dy*dy;  r2 = R2 + dz*dz;  r = sqrt(r2)
//   Plummer     s2 = r2 + a*a; s = sqrt(s2); Phi = -(gm / s); k = gm / (s2 * s); a_i = -(k * d_i)
//   Hernquist   u = r + a; Phi = -(gm / u); k = r > 0 ? gm / ((r * u) * u) : 0; a_i = -(k * d_i)
//   NFW         x = r / a; Phi = r > 0 ? -((gm * log1p(x)) / r) : -(gm / a);
//               mu = x < 0.1 ? the series below : log1p(x) - x / (1 + x);  k = r > 0 ? (gm * mu) / (r2 * r) : 0;
//               a_i = -(k * d_i).  Series: y = x / (1 + x), mu = sum_{j >= 2} y^j / j = y*y * P(y) with
//               P(y) = 1/2 + y*(1/3 + y*(1/4 + ... + y*(1/17 + y/18))) (Horner, coefficients 1.0 / j rounded);
//               truncation below 2e-18 relative for x < 0.1, and no cancellation: every term is positive.  Above the
//               cutoff the log1p form loses at most log1p(x)/mu <= 22 units of its own rounding.
//   Miyamoto-Nagai   zeta = sqrt(dz*dz + b*b); w = a + zeta; D2 = R2 + w*w; D = sqrt(D2); Phi = -(gm / D);
//               k = gm / (D2 * D); a_x = -(k * dx); a_y = -(k * dy); a_z = -(((k * w) / zeta) * dz)
//   logarithmic q2 = b*b; S = (R2 + (dz*dz) / q2) + a*a; Phi = (0.5 * gm) * log(S); k = gm / S;
//               a_x = -(k * dx); a_y = -(k * dy); a_z = -((k * dz) / q2)
// The terms are summed in the order given, starting from +0: a = a + a_term, Phi = Phi + Phi_term.
#pragma once
#include <cstddef>
#include <cstdint>
#include "../../include/b200nb.h"
#include "scf_sm100.cuh"

static_assert(sizeof(b200nb_external_term) == 56, "b200nb_external_term is 56 bytes");
static_assert(offsetof(b200nb_external_term, gm) == 8 && offsetof(b200nb_external_term, a) == 16 &&
                  offsetof(b200nb_external_term, b) == 24 && offsetof(b200nb_external_term, centre) == 32,
              "b200nb_external_term layout");

namespace b200nb {

// the context's terms, passed to the kernels by value; n == 0 means none (the kernels are then their <false> forms)
struct ExtTerms {
    b200nb_external_term t[B200NB_EXTERNAL_MAX];
    uint32_t n;
};

constexpr double NFW_SERIES_CUTOFF = 0.1;

// Phi_ext and a_ext = -grad Phi_ext at the fp32 point (px, py, pz)
__device__ __forceinline__ void ext_eval(const ExtTerms &e, float px, float py, float pz, double acc[3], double *phi)
{
    double ax = 0.0, ay = 0.0, az = 0.0, ph = 0.0;
    for (uint32_t n = 0; n < e.n; ++n) {
        const b200nb_external_term &t = e.t[n];
        const double dx = __dsub_rn((double)px, t.centre[0]);
        const double dy = __dsub_rn((double)py, t.centre[1]);
        const double dz = __dsub_rn((double)pz, t.centre[2]);
        const double R2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        const double dz2 = __dmul_rn(dz, dz);
        double p, k, tz; // term potential; a_x = -(k dx), a_y = -(k dy), a_z = tz
        if (t.kind == B200NB_EXT_PLUMMER) {
            const double s2 = __dadd_rn(__dadd_rn(R2, dz2), __dmul_rn(t.a, t.a));
            const double s = __dsqrt_rn(s2);
            p = -__ddiv_rn(t.gm, s);
            k = __ddiv_rn(t.gm, __dmul_rn(s2, s));
            tz = -__dmul_rn(k, dz);
        } else if (t.kind == B200NB_EXT_HERNQUIST) {
            const double r = __dsqrt_rn(__dadd_rn(R2, dz2));
            const double u = __dadd_rn(r, t.a);
            p = -__ddiv_rn(t.gm, u);
            k = r > 0.0 ? __ddiv_rn(t.gm, __dmul_rn(__dmul_rn(r, u), u)) : 0.0;
            tz = -__dmul_rn(k, dz);
        } else if (t.kind == B200NB_EXT_NFW) {
            const double r2 = __dadd_rn(R2, dz2);
            const double r = __dsqrt_rn(r2);
            const double x = __ddiv_rn(r, t.a);
            const double l = log1p(x);
            const double xp1 = __dadd_rn(1.0, x);
            double mu;
            if (x < NFW_SERIES_CUTOFF) {
                const double y = __ddiv_rn(x, xp1);
                double s = 1.0 / 18;
#pragma unroll
                for (int j = 17; j >= 2; --j) s = __dadd_rn(1.0 / j, __dmul_rn(y, s));
                mu = __dmul_rn(__dmul_rn(y, y), s);
            } else {
                mu = __dsub_rn(l, __ddiv_rn(x, xp1));
            }
            p = r > 0.0 ? -__ddiv_rn(__dmul_rn(t.gm, l), r) : -__ddiv_rn(t.gm, t.a);
            k = r > 0.0 ? __ddiv_rn(__dmul_rn(t.gm, mu), __dmul_rn(r2, r)) : 0.0;
            tz = -__dmul_rn(k, dz);
        } else if (t.kind == B200NB_EXT_MIYAMOTO_NAGAI) {
            const double zeta = __dsqrt_rn(__dadd_rn(dz2, __dmul_rn(t.b, t.b)));
            const double w = __dadd_rn(t.a, zeta);
            const double D2 = __dadd_rn(R2, __dmul_rn(w, w));
            const double D = __dsqrt_rn(D2);
            p = -__ddiv_rn(t.gm, D);
            k = __ddiv_rn(t.gm, __dmul_rn(D2, D));
            tz = -__dmul_rn(__ddiv_rn(__dmul_rn(k, w), zeta), dz);
        } else { // B200NB_EXT_LOGARITHMIC (b200nb_set_external admits no other kind)
            const double q2 = __dmul_rn(t.b, t.b);
            const double S = __dadd_rn(__dadd_rn(R2, __ddiv_rn(dz2, q2)), __dmul_rn(t.a, t.a));
            p = __dmul_rn(__dmul_rn(0.5, t.gm), log(S));
            k = __ddiv_rn(t.gm, S);
            tz = -__ddiv_rn(__dmul_rn(k, dz), q2);
        }
        ax = __dadd_rn(ax, -__dmul_rn(k, dx));
        ay = __dadd_rn(ay, -__dmul_rn(k, dy));
        az = __dadd_rn(az, tz);
        ph = __dadd_rn(ph, p);
    }
    acc[0] = ax; acc[1] = ay; acc[2] = az;
    *phi = ph;
}

// b200nb_external_field: e and Phi_ext at `count` fp32 points; out = [4][stride] doubles (ax, ay, az, phi)
__global__ void __launch_bounds__(256) external_field_kernel(const __grid_constant__ ExtTerms e, const float *__restrict__ px,
                                                            const float *__restrict__ py, const float *__restrict__ pz,
                                                            uint32_t count, uint32_t stride, double *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double a[3], phi;
    ext_eval(e, px[i], py[i], pz[i], a, &phi);
    out[i] = a[0]; out[stride + i] = a[1]; out[2 * (size_t)stride + i] = a[2]; out[3 * (size_t)stride + i] = phi;
}

// ---------------------------------------------------------------------------------------------- external expansion
// The context's frozen basis-function expansion (b200nb_set_external_scf) on the device: the tables and [S | T] packed
// as b200nb_scf_field reads them, in the shard's coefficient block.
struct ExtScf {
    const ScfTables *tab;
    const double *coef;
    uint32_t nmax, lmax, K;
    double cx, cy, cz, a;
};

// Point loaders of ext_total_kernel: bodies [first, first + count) of the blocked body array, or SoA coordinate arrays.
struct BlockedPoints {
    const float *bodies;
    uint64_t first;
    __device__ __forceinline__ void operator()(uint32_t i, float &x, float &y, float &z) const
    {
        const uint64_t g = first + i; // AoSoA-128: x | y | z | G*m per block of 128 bodies
        const float *b = bodies + g / 128 * 512 + g % 128;
        x = b[0]; y = b[128]; z = b[256];
    }
};
struct SoaPoints {
    const float *px, *py, *pz;
    __device__ __forceinline__ void operator()(uint32_t i, float &x, float &y, float &z) const
    {
        x = px[i]; y = py[i]; z = pz[i];
    }
};

// The total external field with an expansion: e = fl(e_terms + a_scf), Phi_ext = fl(Phi_terms + Phi_scf), per component,
// e_terms and Phi_terms from ext_eval (+0 without terms), a_scf and Phi_scf from scf_eval.  out = [4][stride] doubles
// (ax, ay, az, phi), read by b200nb_external_field and by the <true, true> forms of the step's consumers.  The tables
// and [S | T] are staged in shared memory as scf_field_kernel stages them: scf_field_smem(K) bytes.
template <class Points>
__global__ void __launch_bounds__(SCF_EVAL_THREADS) ext_total_kernel(const __grid_constant__ ExtTerms ext, const ExtScf E,
                                                                     const Points pts, uint32_t count, uint32_t stride,
                                                                     double *__restrict__ out)
{
    extern __shared__ double smem[];
    ScfTables &tab = *reinterpret_cast<ScfTables *>(smem);
    double *S = smem + sizeof(ScfTables) / sizeof(double), *T = S + E.K;
    {
        const double *src = reinterpret_cast<const double *>(E.tab);
        for (uint32_t e = threadIdx.x; e < sizeof(ScfTables) / sizeof(double); e += blockDim.x) smem[e] = src[e];
        for (uint32_t e = threadIdx.x; e < 2 * E.K; e += blockDim.x) S[e] = E.coef[e];
    }
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float x, y, z;
    pts(i, x, y, z);
    double e[3], phi, s[3], sphi;
    ext_eval(ext, x, y, z, e, &phi);
    scf_eval(tab, S, T, E, x, y, z, s, &sphi);
    out[i] = __dadd_rn(e[0], s[0]);
    out[stride + i] = __dadd_rn(e[1], s[1]);
    out[2 * (size_t)stride + i] = __dadd_rn(e[2], s[2]);
    out[3 * (size_t)stride + i] = __dadd_rn(phi, sphi);
}

} // namespace b200nb
