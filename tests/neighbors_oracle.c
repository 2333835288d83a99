/* neighbors_oracle.c — brute-force CPU restatement of b200nb_neighbors / b200nb_neighbors_at.  TEST INFRASTRUCTURE ONLY.
 *
 * The definition of include/b200nb.h word for word: fp32 d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) with d = q_j - p,
 * key (d2, j) lexicographic, dist = sqrtf(d2), self pair excluded by index in bodies mode, empty slots
 * (0xFFFFFFFF, +inf).  Bodies at non-finite positions (d2 NaN) are never neighbours.  OpenMP over targets.
 * Build: gcc -O2 -ffp-contract=off -fopenmp -fPIC -shared (Makefile target neighbors_oracle). */
#include <math.h>
#include <stdint.h>

#define NONE 0xFFFFFFFFu

/* k nearest bodies of n_t targets, rows idx[t][k], dist[t][k].  Targets are bodies tgt[t] (self != 0; tgt == NULL:
 * bodies 0..n_t-1) or the points px/py/pz[t] (self == 0). */
void oracle_neighbors(uint64_t n, const float *qx, const float *qy, const float *qz, int self, const uint64_t *tgt,
                      const float *px, const float *py, const float *pz, uint64_t n_t, uint32_t k, uint32_t *idx,
                      float *dist)
{
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t t = 0; t < (int64_t)n_t; t++) {
        const uint64_t i = self ? (tgt ? tgt[t] : (uint64_t)t) : 0;
        const float x = self ? qx[i] : px[t], y = self ? qy[i] : py[t], z = self ? qz[i] : pz[t];
        float kd[32];
        uint32_t kj[32];
        uint32_t filled = 0;
        for (uint64_t j = 0; j < n; j++) {
            if (self && j == i) continue;
            const float dx = qx[j] - x, dy = qy[j] - y, dz = qz[j] - z;
            float d2 = dx * dx;
            d2 = fmaf(dy, dy, d2);
            d2 = fmaf(dz, dz, d2);
            if (isnan(d2)) continue;
            /* j grows, so (d2, j) goes after every stored key of equal d2 */
            if (filled == k && !(d2 < kd[k - 1])) continue;
            uint32_t p = filled < k ? filled++ : k - 1;
            while (p > 0 && kd[p - 1] > d2) {
                kd[p] = kd[p - 1];
                kj[p] = kj[p - 1];
                p--;
            }
            kd[p] = d2;
            kj[p] = (uint32_t)j;
        }
        for (uint32_t p = 0; p < k; p++) {
            idx[(uint64_t)t * k + p] = p < filled ? kj[p] : NONE;
            dist[(uint64_t)t * k + p] = p < filled ? sqrtf(kd[p]) : INFINITY;
        }
    }
}
