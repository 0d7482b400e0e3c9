/* Exposed-point masks of the CPU oracle (test infrastructure): the per-point decision of the oracle's atom_count_l
 * (oracle/sasa_oracle.c, the reference's AtomSasaKernel::with_simd) over the oracle's own neighbour lists
 * (oracle_neighbor_lists: CSR offsets, neighbour indices and thresholds (r_j + probe)^2).
 *   body points [0, lanes * floor(n / lanes)): fma-nested dot, occluded iff dot <  limit
 *   tail points:                               unfused dot,    occluded iff dot <= limit
 *   atoms of equal id never occlude each other.
 * atom_count_l's early exit of a chunk fires only once every point of the chunk is occluded, so testing the whole list
 * gives the same decision per point.  Built with -ffp-contract=off like the oracle, so nothing is fused but the fmaf calls.
 * out[n * W], W = ceil(n_points / 32): bit p % 32 of word p / 32 of row i set when point p of atom i is exposed. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>

static inline uint64_t atom_id(const uint64_t *ids, size_t i) { return ids ? ids[i] : (uint64_t)i; }

__attribute__((visibility("default"))) void mask_oracle_exposed(const float *xyzr, const uint64_t *ids, size_t n, float probe,
                                                                 size_t n_points, int lanes, const float *sx, const float *sy,
                                                                 const float *sz, const uint32_t *off, const uint32_t *idx,
                                                                 const float *thr, uint32_t *out) {
    const size_t W = (n_points + 31) / 32;
    const size_t n_body = (n_points / (size_t)lanes) * (size_t)lanes;
    memset(out, 0, n * W * sizeof(uint32_t));
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 64)
#endif
    for (size_t i = 0; i < n; ++i) {
        const float *ci = &xyzr[4 * i];
        const float r = ci[3] + probe;
        const float r2 = r * r;
        const uint64_t id_i = atom_id(ids, i);
        uint32_t *row = out + i * W;
        for (size_t p = 0; p < n_points; ++p) {
            int occluded = 0;
            for (uint32_t q = off[i]; q < off[i + 1] && !occluded; ++q) {
                const size_t j = idx[q];
                if (atom_id(ids, j) == id_i) continue;
                const float vx = ci[0] - xyzr[4 * j + 0];
                const float vy = ci[1] - xyzr[4 * j + 1];
                const float vz = ci[2] - xyzr[4 * j + 2];
                const float vmag = vx * vx + vy * vy + vz * vz;
                const float limit = (thr[q] - vmag - r2) / (2.0f * r);
                if (p < n_body) occluded = fmaf(sx[p], vx, fmaf(sy[p], vy, sz[p] * vz)) < limit;
                else occluded = sx[p] * vx + sy[p] * vy + sz[p] * vz <= limit;
            }
            if (!occluded) row[p >> 5] |= 1u << (p & 31);
        }
    }
}
