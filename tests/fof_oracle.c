/* fof_oracle.c — brute-force CPU restatement of b200nb_fof.  TEST INFRASTRUCTURE ONLY.
 *
 * The definition of include/b200nb.h word for word: for i < j, fp32 d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) with
 * d = q_j - q_i, linked iff d2 <= b2 = b * b (fp32); group[i] = the smallest index of i's connected component.  Every
 * pair i < j is visited and linked pairs are joined on the fly (no edge list) in a union-find whose pointers only go to
 * smaller indices, so each root is its tree's minimum.  OpenMP threads take rows i into forests of their own, folded into
 * one at the end.  Non-finite positions give d2 NaN or +inf, never <= a finite b2.
 * Build: gcc -O3 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target fof_oracle).  With -ffp-contract=off no
 * product or sum is fused except the two explicit fmaf; the FMA clone only makes those two single instructions. */
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

/* rows [i] of the pair triangle into forest p: sources j > i in chunks, d2 first (vectorisable), links after */
__attribute__((target_clones("fma", "default"))) static void link_row(uint64_t n, const float *qx, const float *qy,
                                                                      const float *qz, float b2, uint64_t i, uint32_t *p)
{
    const float x = qx[i], y = qy[i], z = qz[i];
    float d2[CHUNK];
    uint32_t ri = find(p, (uint32_t)i);
    for (uint64_t j0 = i + 1; j0 < n; j0 += CHUNK) {
        const uint64_t m = n - j0 < CHUNK ? n - j0 : CHUNK;
        for (uint64_t k = 0; k < m; k++) {
            const float dx = qx[j0 + k] - x, dy = qy[j0 + k] - y, dz = qz[j0 + k] - z;
            float d = dx * dx;
            d = fmaf(dy, dy, d);
            d = fmaf(dz, dz, d);
            d2[k] = d;
        }
        for (uint64_t k = 0; k < m; k++)
            if (d2[k] <= b2) {
                const uint32_t rj = find(p, (uint32_t)(j0 + k));
                if (rj != ri) ri = unite(p, ri, rj);
            }
    }
}

/* group[n]: the smallest body index of each body's friends-of-friends group of linking length b */
void oracle_fof(uint64_t n, const float *qx, const float *qy, const float *qz, float b, uint32_t *group)
{
    const float b2 = b * b;
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
        for (int64_t i = 0; i < (int64_t)n; i++) link_row(n, qx, qy, qz, b2, (uint64_t)i, p);
        if (t != 0) {
#pragma omp critical
            for (uint64_t x = 0; x < n; x++)
                if (p[x] != x) unite(group, (uint32_t)x, p[x]);
            free(p);
        }
    }
    for (uint64_t x = 0; x < n; x++) group[x] = find(group, (uint32_t)x);
}
