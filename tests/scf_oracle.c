/* Long-double restatement of the basis-function expansion (include/b200nb.h, "basis-function expansion").  TEST
 * INFRASTRUCTURE ONLY: the GPU coefficients and field are checked against it, and it is checked against an independent
 * scipy restatement (tests/test_scf_cpu.py).
 *
 * It follows the definition directly: Gegenbauer polynomials by their recurrence, P_l^m(cos theta) by the standard
 * recurrence in l with the Condon-Shortley phase, cos(m phi) and sin(m phi) from atan2, powl for s^l (1+s)^-(2l+1) and the
 * normalisation from lgammal.  Every coefficient and value comes with its cancellation-free scale sum |term|.  The field
 * uses the reduced polynomials Q_l^m = P_l^m / sin^m theta for its gradient, so it is finite on the z axis. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

typedef long double R;

static R gegenbauer(int n, R alpha, R x) /* C_n^alpha(x) */
{
    R c0 = 1.0L, c1 = 2.0L * alpha * x;
    if (n == 0) return c0;
    for (int k = 2; k <= n; ++k) {
        const R c2 = (2.0L * (k + alpha - 1.0L) * x * c1 - (k + 2.0L * alpha - 2.0L) * c0) / k;
        c0 = c1; c1 = c2;
    }
    return c1;
}

static R norm_f(int n, int l, int m, R a) /* (2 - delta_m0) A~_nl N_lm / a */
{
    const R K = 0.5L * n * (n + 4.0L * l + 3.0L) + (l + 1.0L) * (2.0L * l + 1.0L);
    const R lg = (8.0L * l + 6.0L) * logl(2.0L) + lgammal(n + 1.0L) + logl(n + 2.0L * l + 1.5L) + 2.0L * lgammal(2.0L * l + 1.5L) -
                 logl(4.0L * 3.14159265358979323846264338327950288L * K) - lgammal(n + 4.0L * l + 3.0L);
    R ratio = 1.0L;
    for (int k = l - m + 1; k <= l + m; ++k) ratio /= k;
    return (m ? 2.0L : 1.0L) * -expl(lg) * (2.0L * l + 1.0L) * ratio / a;
}

/* P_l^m(x) for all l <= lmax, m <= l, Condon-Shortley phase: p[l*(l+1)/2 + m] */
static void legendre(int lmax, R x, R *p)
{
    const R sn = sqrtl(fmaxl(0.0L, 1.0L - x * x));
    R pmm = 1.0L;
    for (int m = 0; m <= lmax; ++m) {
        if (m > 0) pmm *= -(2.0L * m - 1.0L) * sn;
        p[m * (m + 1) / 2 + m] = pmm;
        R a = 0.0L, b = pmm;
        for (int l = m + 1; l <= lmax; ++l) {
            const R c = ((2.0L * l - 1.0L) * x * b - (l + m - 1.0L) * a) / (l - m);
            a = b; b = c;
            p[l * (l + 1) / 2 + m] = c;
        }
    }
}

/* Coefficients of the bodies with member[k] != 0; gm = the fp32 G*m.  S, T, Ss, Ts: [nmax+1][LM], packed as the ABI. */
void oracle_scf_coefficients(uint64_t nb, const float *qx, const float *qy, const float *qz, const float *gm, const uint8_t *member,
                             int nmax, int lmax, double a, const double *c, double *S, double *T, double *Ss, double *Ts)
{
    const int LM = (lmax + 1) * (lmax + 2) / 2, K = (nmax + 1) * LM;
    R s_acc[32 * 136], t_acc[32 * 136], s_sc[32 * 136], t_sc[32 * 136], F[32 * 136], p[136], rad[16][32];
    for (int e = 0; e < K; ++e) s_acc[e] = t_acc[e] = s_sc[e] = t_sc[e] = 0.0L;
    for (int n = 0; n <= nmax; ++n)
        for (int l = 0; l <= lmax; ++l)
            for (int m = 0; m <= l; ++m) F[n * LM + l * (l + 1) / 2 + m] = norm_f(n, l, m, a);
    for (uint64_t k = 0; k < nb; ++k) {
        if (!member[k]) continue;
        const R dx = (R)((double)qx[k] - c[0]), dy = (R)((double)qy[k] - c[1]), dz = (R)((double)qz[k] - c[2]);
        const R r = sqrtl(dx * dx + dy * dy + dz * dz), s = r / a, xi = (s - 1.0L) / (s + 1.0L);
        const R ct = r > 0 ? dz / r : 0.0L, ph = r > 0 ? atan2l(dy, dx) : 0.0L;
        legendre(lmax, ct, p);
        for (int l = 0; l <= lmax; ++l)
            for (int n = 0; n <= nmax; ++n)
                rad[l][n] = -(R)gm[k] * powl(s, l) * powl(1.0L + s, -(2.0L * l + 1.0L)) * gegenbauer(n, 2.0L * l + 1.5L, xi);
        for (int m = 0; m <= lmax; ++m) {
            const R cm = cosl(m * ph), sm = m ? sinl(m * ph) : 0.0L;
            for (int l = m; l <= lmax; ++l)
                for (int n = 0; n <= nmax; ++n) {
                    const int i = n * LM + l * (l + 1) / 2 + m;
                    const R base = F[i] * rad[l][n] * p[l * (l + 1) / 2 + m];
                    s_acc[i] += base * cm;
                    t_acc[i] += base * sm;
                    s_sc[i] += fabsl(base);
                    t_sc[i] += m ? fabsl(base) : 0.0L;
                }
        }
    }
    for (int e = 0; e < K; ++e) {
        S[e] = (double)s_acc[e]; T[e] = (double)t_acc[e];
        Ss[e] = (double)s_sc[e]; Ts[e] = (double)t_sc[e];
    }
}

/* Phi and a of an expansion at fp32 points, with scales: sphi = sum |Phi term|, sa[3][m] = sum |a_i term| per component. */
void oracle_scf_field(int nmax, int lmax, double a, const double *c, const double *S, const double *T, uint64_t np, const float *px,
                      const float *py, const float *pz, double *acc, double *phi, double *sphi, double *sa)
{
    const int LM = (lmax + 1) * (lmax + 2) / 2;
#pragma omp parallel for schedule(dynamic, 16)
    for (uint64_t i = 0; i < np; ++i) {
        const R dx = (R)((double)px[i] - c[0]), dy = (R)((double)py[i] - c[1]), dz = (R)((double)pz[i] - c[2]);
        const R r = sqrtl(dx * dx + dy * dy + dz * dz), s = r / a, xi = (s - 1.0L) / (s + 1.0L);
        const R ux = r > 0 ? dx / r : 0.0L, uy = r > 0 ? dy / r : 0.0L, uz = r > 0 ? dz / r : 0.0L;
        /* Q_l^m for m <= l + 1 (Q_l^(l+1) = 0), Q_l^m = (-1)^m d^m P_l / dx^m */
        R Q[16][18];
        for (int l = 0; l <= lmax; ++l)
            for (int m = 0; m <= 17; ++m) Q[l][m] = 0.0L;
        R qmm = 1.0L;
        for (int m = 0; m <= lmax; ++m) {
            if (m > 0) qmm *= -(2.0L * m - 1.0L);
            Q[m][m] = qmm;
            R qa = 0.0L, qb = qmm;
            for (int l = m + 1; l <= lmax; ++l) {
                const R qc = ((2.0L * l - 1.0L) * uz * qb - (l + m - 1.0L) * qa) / (l - m);
                qa = qb; qb = qc;
                Q[l][m] = qc;
            }
        }
        R wr[18], wi[18]; /* w^m */
        wr[0] = 1.0L; wi[0] = 0.0L;
        for (int m = 1; m <= lmax + 1; ++m) {
            wr[m] = wr[m - 1] * ux - wi[m - 1] * uy;
            wi[m] = wr[m - 1] * uy + wi[m - 1] * ux;
        }
        R P = 0, g[3] = {0, 0, 0}, sp = 0, sg[3] = {0, 0, 0};
        for (int l = 0; l <= lmax; ++l) {
            const R pl = powl(s, l) * powl(1.0L + s, -(2.0L * l + 1.0L));
            const R dpl = r > 0 ? pl * (l / s - (2.0L * l + 1.0L) / (1.0L + s)) : 0.0L; /* d pl / ds */
            for (int n = 0; n <= nmax; ++n) {
                const R alpha = 2.0L * l + 1.5L;
                const R cn = gegenbauer(n, alpha, xi);
                const R dcn = n ? 2.0L * alpha * gegenbauer(n - 1, alpha + 1.0L, xi) : 0.0L; /* dC_n^alpha / dxi */
                const R rad = -pl * cn;
                const R drad = -(dpl * cn + pl * dcn * 2.0L / ((1.0L + s) * (1.0L + s))); /* d rad / ds */
                for (int m = 0; m <= l; ++m) {
                    const int idx = n * LM + l * (l + 1) / 2 + m;
                    for (int part = 0; part < 2; ++part) {
                        const R coef = part ? T[idx] : S[idx];
                        if (coef == 0.0L) continue;
                        const R ang = Q[l][m] * (part ? wi[m] : wr[m]);
                        /* gradient of the angular factor in u as free variables */
                        const R cm1 = m ? (part ? wi[m - 1] : wr[m - 1]) : 0.0L, sm1 = m ? (part ? -wr[m - 1] : wi[m - 1]) : 0.0L;
                        const R gu[3] = {m * Q[l][m] * cm1, -m * Q[l][m] * sm1, -Q[l][m + 1] * (part ? wi[m] : wr[m])};
                        const R ug = ux * gu[0] + uy * gu[1] + uz * gu[2];
                        const R u[3] = {ux, uy, uz};
                        const R term = coef * rad * ang;
                        P += term;
                        sp += fabsl(term);
                        if (r > 0)
                            for (int k = 0; k < 3; ++k) {
                                const R tk = coef * (drad / a * ang * u[k] + rad / r * (gu[k] - u[k] * ug));
                                g[k] += tk;
                                sg[k] += fabsl(coef * drad / a * ang * u[k]) + fabsl(coef * rad / r * gu[k]) +
                                         fabsl(coef * rad / r * u[k] * ug);
                            }
                    }
                }
            }
        }
        for (int k = 0; k < 3; ++k) {
            acc[k * np + i] = (double)-g[k];
            sa[k * np + i] = (double)sg[k];
        }
        phi[i] = (double)P;
        sphi[i] = (double)sp;
    }
}
