// sasa_pair_sums.cuh -- level sums of the partner slots of a pairwise buried-area run (sasa_b200_batch_run_group_pairs_frames_host).
//
// Both kernels read the slot rows of the pairs kernels (PairParams: k slots per atom in batch order, partner label and area) and
// the batch's group labels, and sum in float64 in atom order -- the order of engine.group_pair_table's np.add.at -- so their
// results equal the host reduction bit for bit.  A slot not in use holds partner UINT32_MAX and area 0.0f; skipping it leaves a
// float64 sum of non-negative terms unchanged, so only partners below n_labels are added.  A structure with non-finite input has
// area NaN in every slot (pair_blank_rows): its block and its segment rows come out NaN.
#pragma once
#include "sasa_device.cuh"

namespace sasa {

constexpr uint32_t kPairSumsMaxLabels = 17;   // k = n_labels - 1 <= 16 slots, the pairs kernels' limit
constexpr int kPairSumsRegs = (kPairSumsMaxLabels * (kPairSumsMaxLabels - 1) + 31) / 32;   // accumulators per lane
static_assert(kPairSumsRegs == 9, "pair_sums_kernel adds through nine explicit cases");

// pair_area[(s * L + g) * L + h]: the area of group g that group h buries in structure s, for s in [s0, s1); one warp per structure.
// The L (L - 1) off-diagonal (g, h) cells are numbered p = g (L - 1) + h - (h > g); lane p % 32 owns cell p in register p / 32.
// The warp reads 32 slots at a time, coalesced, and steps through the slots in use in batch order with shuffles; the owner adds,
// so every cell is one sequential chain in atom order with no atomics and no shared memory.
__global__ void __launch_bounds__(128) pair_sums_kernel(const uint32_t *__restrict__ struct_off, const uint32_t *__restrict__ grp,
                                                        const uint32_t *__restrict__ partner, const float *__restrict__ area, uint32_t k,
                                                        uint32_t L, uint32_t s0, uint32_t s1, double *__restrict__ pair_area) {
    const int lane = lane_id();
    const uint32_t s = s0 + (blockIdx.x * blockDim.x + threadIdx.x) / kWarp;
    if (s >= s1) return;
    const size_t e0 = (size_t)struct_off[s] * k, e1 = (size_t)struct_off[s + 1] * k;   // slot range of the structure
    double acc[kPairSumsRegs];
#pragma unroll
    for (int r = 0; r < kPairSumsRegs; ++r) acc[r] = 0.0;
    bool bad = false;
    for (size_t b = e0; b < e1; b += kWarp) {
        const size_t e = b + (size_t)lane;
        int cell = -1;
        float a = 0.0f;
        if (e < e1) {
            const uint32_t h = __ldg(partner + e);
            a = __ldg(area + e);
            bad |= isnan(a);
            if (h < L) {
                const uint32_t g = __ldg(grp + e / k);
                cell = (int)(g * (L - 1) + h - (h > g ? 1u : 0u));
            }
        }
        unsigned used = __ballot_sync(kFull, cell >= 0);
        while (used) {
            const int t = __ffs(used) - 1;
            used &= used - 1;
            const int c = __shfl_sync(kFull, cell, t);
            const float v = __shfl_sync(kFull, a, t);
            if ((c & (kWarp - 1)) == lane) {
                const double dv = (double)v;
                switch (c >> 5) {   // explicit cases keep acc in registers (an indexed add puts the array on the stack)
                    case 0: acc[0] = __dadd_rn(acc[0], dv); break;
                    case 1: acc[1] = __dadd_rn(acc[1], dv); break;
                    case 2: acc[2] = __dadd_rn(acc[2], dv); break;
                    case 3: acc[3] = __dadd_rn(acc[3], dv); break;
                    case 4: acc[4] = __dadd_rn(acc[4], dv); break;
                    case 5: acc[5] = __dadd_rn(acc[5], dv); break;
                    case 6: acc[6] = __dadd_rn(acc[6], dv); break;
                    case 7: acc[7] = __dadd_rn(acc[7], dv); break;
                    default: acc[8] = __dadd_rn(acc[8], dv); break;
                }
            }
        }
    }
    bad = __any_sync(kFull, bad);
    const double qn = __longlong_as_double(0x7ff8000000000000ll);
    double *out = pair_area + (size_t)s * L * L;
#pragma unroll
    for (int r = 0; r < kPairSumsRegs; ++r) {
        const uint32_t p = (uint32_t)(lane + kWarp * r);
        if (p < L * (L - 1)) {
            const uint32_t g = p / (L - 1), hh = p % (L - 1), h = hh + (hh >= g ? 1u : 0u);
            out[g * L + h] = bad ? qn : acc[r];
        }
    }
    if ((uint32_t)lane < L) out[lane * L + lane] = bad ? qn : 0.0;
}

// seg_pair_area[q * L + h]: the area of segment q that group h buries, for the segments [q0, q1) of structures [s0, s1); one
// thread per (segment, h), summing the segment's slots in atom order.  The segment's structure is non-finite when its pair_area
// diagonal -- written by pair_sums_kernel before this kernel runs -- is NaN.
__global__ void __launch_bounds__(256) seg_pair_sums_kernel(const uint32_t *__restrict__ struct_off, const uint32_t *__restrict__ struct_seg_off,
                                                            const uint2 *__restrict__ seg_be, const uint32_t *__restrict__ partner,
                                                            const float *__restrict__ area, uint32_t k, uint32_t L, uint32_t s0, uint32_t s1,
                                                            uint32_t q0, uint32_t q1, const double *__restrict__ pair_area,
                                                            double *__restrict__ seg_pair_area) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)(q1 - q0) * L) return;
    const uint32_t q = q0 + (uint32_t)(t / L), h = (uint32_t)(t % L);
    uint32_t lo = s0, hi = s1;   // the structure s with struct_seg_off[s] <= q < struct_seg_off[s + 1]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (__ldg(struct_seg_off + mid) <= q) lo = mid;
        else hi = mid;
    }
    const uint32_t s = lo;
    const uint2 be = __ldg(seg_be + q);
    const size_t a0 = struct_off[s];
    double sum = 0.0;
    for (size_t i = a0 + be.x; i < a0 + be.y; ++i)
        for (uint32_t r = 0; r < k; ++r)
            if (__ldg(partner + i * k + r) == h) sum = __dadd_rn(sum, (double)__ldg(area + i * k + r));
    const double d = pair_area[(size_t)s * L * L];
    seg_pair_area[(size_t)q * L + h] = isnan(d) ? d : sum;
}

}  // namespace sasa
