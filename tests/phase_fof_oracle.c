/* phase_fof_oracle.c — brute-force CPU restatement of b200nb_fof_phase.  TEST INFRASTRUCTURE ONLY.
 *
 * The definition of include/b200nb.h word for word: s_x = 1.0f / b_x, s_v = 1.0f / b_v (fp32 divisions), scaled
 * coordinates X = x * s_x, ..., W = vz * s_v (fp32 products), and for i < j with d = scaled j - scaled i
 *   d2 = fmaf(dW, dW, fmaf(dV, dV, fmaf(dU, dU, fmaf(dZ, dZ, fmaf(dY, dY, dX * dX)))))
 * linked iff d2 <= 1.0f; group[i] = the smallest index of i's connected component.  Every pair i < j is visited and
 * linked pairs are joined on the fly in a union-find whose pointers only go to smaller indices (as tests/fof_oracle.c).
 * OpenMP threads take rows i into forests of their own, folded into one at the end.
 * Build: gcc -O3 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target phase_fof_oracle).  With -ffp-contract=off no
 * product or sum is fused except the explicit fmaf; the FMA clone only makes those single instructions. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static uint32_t find(uint32_t *p, uint32_t x)
{
    while (p[x] != x) {
        p[x] = p[p[x]];
        x = p[x];
    }
    return x;
}

static uint32_t unite(uint32_t *p, uint32_t a, uint32_t b)
{
    a = find(p, a);
    b = find(p, b);
    if (a < b) p[b] = a;
    else p[a] = b;
    return a < b ? a : b;
}

#define CHUNK 256

/* row i of the pair triangle into forest p: s[6][n] scaled coordinates, sources j > i in chunks, d2 first, links after */
__attribute__((target_clones("fma", "default"))) static void link_row(uint64_t n, const float *s, uint64_t i, uint32_t *p)
{
    float t[6], d2[CHUNK];
    for (int k = 0; k < 6; k++) t[k] = s[k * n + i];
    uint32_t ri = find(p, (uint32_t)i);
    for (uint64_t j0 = i + 1; j0 < n; j0 += CHUNK) {
        const uint64_t m = n - j0 < CHUNK ? n - j0 : CHUNK;
        for (uint64_t q = 0; q < m; q++) {
            const uint64_t j = j0 + q;
            const float dX = s[j] - t[0], dY = s[n + j] - t[1], dZ = s[2 * n + j] - t[2];
            const float dU = s[3 * n + j] - t[3], dV = s[4 * n + j] - t[4], dW = s[5 * n + j] - t[5];
            float d = dX * dX;
            d = fmaf(dY, dY, d);
            d = fmaf(dZ, dZ, d);
            d = fmaf(dU, dU, d);
            d = fmaf(dV, dV, d);
            d = fmaf(dW, dW, d);
            d2[q] = d;
        }
        for (uint64_t q = 0; q < m; q++)
            if (d2[q] <= 1.0f) {
                const uint32_t rj = find(p, (uint32_t)(j0 + q));
                if (rj != ri) ri = unite(p, ri, rj);
            }
    }
}

/* group[n]: the smallest body index of each body's phase-space friends-of-friends group of linking lengths b_x, b_v */
void oracle_fof_phase(uint64_t n, const float *qx, const float *qy, const float *qz, const float *vx, const float *vy,
                      const float *vz, float b_x, float b_v, uint32_t *group)
{
    const float sx = 1.0f / b_x, sv = 1.0f / b_v;
    float *s = (float *)malloc(6 * n * sizeof(float));
    const float *in[6] = {qx, qy, qz, vx, vy, vz};
    for (int k = 0; k < 6; k++)
        for (uint64_t i = 0; i < n; i++) s[k * n + i] = in[k][i] * (k < 3 ? sx : sv);
    for (uint64_t x = 0; x < n; x++) group[x] = (uint32_t)x;
#pragma omp parallel
    {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        uint32_t *p = t == 0 ? group : (uint32_t *)malloc(n * sizeof(uint32_t));
        if (t != 0)
            for (uint64_t x = 0; x < n; x++) p[x] = (uint32_t)x;
#pragma omp for schedule(dynamic, 8)
        for (int64_t i = 0; i < (int64_t)n; i++) link_row(n, s, (uint64_t)i, p);
        if (t != 0) {
#pragma omp critical
            for (uint64_t x = 0; x < n; x++)
                if (p[x] != x) unite(group, (uint32_t)x, p[x]);
            free(p);
        }
    }
    for (uint64_t x = 0; x < n; x++) group[x] = find(group, (uint32_t)x);
    free(s);
}
