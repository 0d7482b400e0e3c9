// sasa_tight.cuh -- the fused per-structure kernel for n_points <= 128 (the reference's default, 100 points,
// is the headline configuration).  Same stages as the generic kernel of sasa_small.cuh, but the per-atom
// pipeline is written for a SMALL INSTRUCTION FOOTPRINT: the generic kernel's hot code spans ~45 KB of SASS,
// more than the SM's 32 KB L1.5 instruction cache, and ncu showed 37 % of its stall cycles as "no instruction"
// (profiles/r01a_baseline.txt).  Here every stage is one short rolled loop, the cell's candidate list lives in
// shared memory instead of unrolled register windows, the tile routine takes its shape at run time, and the
// never-taken fallbacks (dense clusters) sit behind one __noinline__ call.
//
// Per cell (warps claim runs of the cell-sorted atom order, snapped to whole cells):
//   list     the (2e+1)^2 cell rows around the cell are contiguous ranges of the cell-sorted atom array; their
//            positions are flattened once into a per-warp u16 list, padded to a multiple of 32 with the
//            far-away sentinel atom
// Per atom of the cell:
//   gather   32 listed candidates per step: distance test, ballot, compaction into a u16 neighbour list
//   cap      the cap-table occlusion of sasa_cap.cuh (default): one lane per neighbour, table masks, exact ring tests
// or, with -DSASA_OPT_CAP=0, the earlier two-phase point tests:
//   entries  (vx, vy, vz, limit) per neighbour with the reference's arithmetic, "near" neighbours first
//   phase 1  all body points (3 slots per lane for n = 100) against the first m entries:
//            one broadcast LDS.128 + 3 x (FMUL, 2 FFMA, FSETP.LT.OR) per entry
//   phase 2  the surviving points against the remaining entries as a G x (32/G) tile of (survivor, entry) pairs
//   tail     the n mod lanes tail points (unfused dot, <=) against all entries, same tile form
// Between structures: warp 0 claims the CTA's next structure early and prefetches its atoms into L2.
#pragma once
#include "sasa_cap.cuh"
#include "sasa_small.cuh"

namespace sasa {

#ifndef SASA_CELL_FETCH
#define SASA_CELL_FETCH 4
#endif
// tuning switches (tools/variants.py builds A/B libraries with -D overrides)
#ifndef SASA_OPT_FILL4
#define SASA_OPT_FILL4 1      // fill_list: four positions per trip
#endif
#ifndef SASA_OPT_FILLP
#define SASA_OPT_FILLP 1      // fill_list: the four stores of a trip predicated (inline PTX) instead of branched: 487.2 -> 477.5 warp
                              // instructions per atom, 1,863 -> 1,912 M atoms/s (gpurun_out r04f)
#endif
#ifndef SASA_OPT_HDR
#define SASA_OPT_HDR 1        // fill_list header: lane / w by multiplication (nvcc emitted the 30-instruction integer division per claim),
                              // inclusive scan with the shuffle's own predicate on the add: 454.0 -> 449.1 warp instructions per atom,
                              // 1,986 -> 2,012 M atoms/s (gpurun_out r04h)
#endif
#ifndef SASA_OPT_P1U
#define SASA_OPT_P1U 4        // phase 1: entries per unrolled trip
#endif
#ifndef SASA_OPT_TAILX
#define SASA_OPT_TAILX 0      // tail tiles: nearest N entries tested on their own first (0: one pass over all entries).
                              // Measured (gpurun_out v1/v2, cfg2): 16 costs ~30 warp instructions per atom more than it saves.
#endif
#ifndef SASA_OPT_CAP
#define SASA_OPT_CAP 1        // cap-table occlusion (sasa_cap.cuh) instead of phase 1 / tile point tests
#endif
#ifndef SASA_OPT_NSLT
#define SASA_OPT_NSLT 1       // launch the kernel compiled for 3 body slots when it applies
#endif
#ifndef SASA_OPT_GU
#define SASA_OPT_GU 2         // gather: 32-candidate steps per unrolled trip
#endif
#ifndef SASA_OPT_G2
#define SASA_OPT_G2 2         // gather: explicit G-step trips with the loads of all G steps ahead of the stores (0: plain loop)
#endif
#ifndef SASA_OPT_AREA
#define SASA_OPT_AREA 0       // 1: the per-atom phase stores areas (and writes counts straight to global memory) so that the
                              // output stage needs no second read of the radii -- measured 1 % slower (lane-0 work), off
#endif
#ifndef SASA_OPT_ACLAIM
#define SASA_OPT_ACLAIM 4     // > 0: warps claim runs of ATOMS (at least this many) of the cell-sorted order instead of runs
                              // of cells -- finer tail at the price of some cells' candidate lists being built twice
#endif
#ifndef SASA_OPT_SNAP
#define SASA_OPT_SNAP 1       // atom-granular claims are snapped to whole cells: a cell is worked by the warp whose claim holds
                              // the cell's first atom, so no candidate list is built twice
#endif
#ifndef SASA_OPT_GRIDLD
#define SASA_OPT_GRIDLD 0     // 1: the grid is re-read from shared memory at every cell instead of living in registers (-1 %)
#endif
#ifndef SASA_OPT_PAIR
#define SASA_OPT_PAIR 1       // pairs of atoms of a cell share one pass over the cell's candidate list: each candidate is loaded once
                              // and tested against both (VERDICT r01's per-cell gather in the form that paid).  Measured on cfg2
                              // (gpurun_out r02w-r02z): off 1,635 M atoms/s / 560.6 warp instructions per atom; pairs 1,684 / 539.0;
                              // groups of up to 3 or 4 atoms with the occlusion unrolled per atom 1,022 / 670 (three more copies of
                              // cap_atom push the hot code out of the instruction cache: issue utilisation 49 % / 32 %); the same
                              // groups with ONE rolled occlusion loop 1,523-1,591 (the bookkeeping costs more than the loads saved)
#endif
#ifndef SASA_OPT_UWARP
#define SASA_OPT_UWARP 1      // 1: the warp index goes through a warp reduction (REDUX writes a uniform register), so that the per-warp
#endif                        // scratch addresses live on the uniform datapath; ptxas otherwise re-derives them from SR_TID.X wherever
                              // the 64 vector registers run out.  Measured together with SASA_OPT_UGRID (gpurun_out r04a/r04b, cfg2):
                              // either one alone changes nothing, both together 539.0 -> 512 warp instructions per atom, and with
                              // SASA_OPT_NOGUARD + SASA_CAP_FULLX 487.2 (1,683 -> 1,867 M atoms/s); the spills of the per-atom loop
                              // (five LDL per cell) are gone
#ifndef SASA_OPT_UGRID
#define SASA_OPT_UGRID 1      // 1: the structure's cell grid (eight CTA-uniform values) is held in uniform registers
#endif
#ifndef SASA_OPT_UCLAIM
#define SASA_OPT_UCLAIM 0     // 1: the claimed atom range and the list length come out of warp reductions (uniform registers) instead of
                              // shuffles -- measured neutral (r04c: 1,868 vs 1,867), off
#endif
#ifndef SASA_OPT_USTRUCT
#define SASA_OPT_USTRUCT 0    // 1: the structure's id, first atom and atom count in uniform registers -- measured neutral (1,859), off
#endif
#ifndef SASA_OPT_UCELL
#define SASA_OPT_UCELL 0      // 1: the end of the cell's atom run in a uniform register -- one more REDUX per cell: 495 instructions, 1,848; off
#endif
#ifndef SASA_OPT_NOGUARD
#define SASA_OPT_NOGUARD 1    // 1: the neighbour lists of the cap path live in the idle entry strip with room for every listed
#endif                        // candidate, so the gather needs no capacity test on its stores
#define SASA_NOGUARD_ON (SASA_OPT_NOGUARD && SASA_OPT_CAP)   // (the two-phase build keeps its 128-entry lists and their capacity test)
#ifndef SASA_OPT_NEXT
#define SASA_OPT_NEXT 1       // warp 0 claims the CTA's next structure and prefetches its atoms into L2 while the other
                              // warps already work on the current one (hides the claim / first-touch latency of the setup)
#endif

// Flatten the candidate rows of cell (cx, cy, cz) into list[0, total) (positions in the sorted atom array),
// padded with `sentinel` up to the next multiple of 32.  Returns total, or -1 when it exceeds kListCap.
__device__ __forceinline__ int tight_fill_list(const Grid &g, const uint16_t *cell, int cx, int cy, int cz,
                                               uint16_t *list, int sentinel) {
    const int lane = lane_id();
    const int w = 2 * g.e + 1;
#if SASA_OPT_HDR
    // lane / w without the integer-division sequence: the search extent e is 1 or 2, so w is 3 or 5 (exact for lane < 32)
    const int q = g.e == 2 ? (lane * 13) >> 6 : (lane * 11) >> 5;
    const int dy = lane - q * w - g.e, dz = q - g.e;
#else
    const int dy = lane % w - g.e, dz = lane / w - g.e;
#endif
    const int y = cy + dy, z = cz + dz;
    int start = 0, len = 0;
    if (lane < w * w && y >= 0 && y < g.ny && z >= 0 && z < g.nz) {
        const int x0 = max(cx - g.e, 0), x1 = min(cx + g.e, g.nx - 1);
        const int base = (z * g.ny + y) * g.nx;
        start = (int)cell[base + x0];
        len = (int)cell[base + x1 + 1] - start;
    }
    int incl = len;
#if SASA_OPT_HDR
    // inclusive scan, two instructions per step: the shuffle's own predicate (source lane in range) guards the addition
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
        asm volatile("{\n .reg .pred p;\n .reg .b32 t;\n shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n @p add.s32 %0, %0, t;\n}"
                     : "+r"(incl) : "r"(d));
#else
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += t;
    }
#endif
#if SASA_OPT_UCLAIM
    const int total = (int)__reduce_max_sync(kFull, (unsigned)incl);   // the inclusive scan is non-decreasing: lane 31 holds the maximum
#else
    const int total = __shfl_sync(kFull, incl, 31);
#endif
    if (total > kListCap) return -1;
    const int maxlen = __reduce_max_sync(kFull, len);
    // row expansion, four positions per trip (the longest row of a protein-density cell block holds ~13 atoms)
#if SASA_OPT_FILLP
    // the same with four PREDICATED stores per trip (nvcc turns the monotone conditions below into a chain of divergent
    // branches: 22 instructions per trip with a reconvergence point; this form is 15)
    uint32_t dsts = (uint32_t)__cvta_generic_to_shared(list + (incl - len));
    int v = start, left = len;
#pragma unroll 1
    for (int t = 0; t < maxlen; t += 4) {
        asm volatile("{\n .reg .pred p0, p1, p2, p3;\n"
                     " setp.gt.s32 p0, %2, 0;\n setp.gt.s32 p1, %2, 1;\n setp.gt.s32 p2, %2, 2;\n setp.gt.s32 p3, %2, 3;\n"
                     " @p0 st.shared.u16 [%0], %1;\n"
                     " @p1 st.shared.u16 [%0+2], %3;\n"
                     " @p2 st.shared.u16 [%0+4], %4;\n"
                     " @p3 st.shared.u16 [%0+6], %5;\n}"
                     :: "r"(dsts), "h"((uint16_t)v), "r"(left), "h"((uint16_t)(v + 1)), "h"((uint16_t)(v + 2)), "h"((uint16_t)(v + 3))
                     : "memory");
        dsts += 8; v += 4; left -= 4;
    }
#elif SASA_OPT_FILL4
    uint16_t *dst = list + (incl - len);
    int v = start, left = len;
#pragma unroll 1
    for (int t = 0; t < maxlen; t += 4) {
        if (left > 0) dst[0] = (uint16_t)v;
        if (left > 1) dst[1] = (uint16_t)(v + 1);
        if (left > 2) dst[2] = (uint16_t)(v + 2);
        if (left > 3) dst[3] = (uint16_t)(v + 3);
        dst += 4; v += 4; left -= 4;
    }
#else
    uint16_t *dst = list + (incl - len);
#pragma unroll 1
    for (int t = 0; t < maxlen; ++t)
        if (t < len) dst[t] = (uint16_t)(start + t);
#endif
    const int pad = total + lane;
    if (pad < ((total + 31) & ~31)) list[pad] = (uint16_t)sentinel;
    __syncwarp();
    return total;
}

// Neighbours of atom `pos` among the listed candidates: positions of all atoms within r_i + r_j + 2*probe
// (+ slack) go to cand[0, k).  Membership is result-neutral (any superset of the overlapping pairs gives the
// same counts), so this test may use contracted arithmetic; the 1e-3 A slack absorbs its rounding.
template <bool HAS_CLS>
__device__ __forceinline__ int tight_gather(const float4 *s_atom, const uint32_t *s_cls, const uint16_t *list, int total,
                                            int pos, const float4 ai, float reach_i, uint16_t *cand) {
    const int lane = lane_id();
    const unsigned lt = lanemask_lt();
    const uint32_t cls_i = HAS_CLS ? s_cls[pos] : 0u;
    int k = 0;
#if SASA_OPT_G2
    // G steps per trip with every load ahead of the first store, so that the dependent shared-memory round trips
    // (list entry -> atom) of all G steps overlap
    constexpr int G = SASA_OPT_G2 < 2 ? 2 : SASA_OPT_G2;
    int w0 = 0;
#pragma unroll 1
    for (; w0 + 32 * (G - 1) < total; w0 += 32 * G) {
        int j[G];
        float4 b[G];
        bool acc[G];
        unsigned m[G];
#pragma unroll
        for (int g = 0; g < G; ++g) j[g] = (int)list[w0 + 32 * g + lane];
#pragma unroll
        for (int g = 0; g < G; ++g) b[g] = s_atom[j[g]];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const float dx = ai.x - b[g].x, dy = ai.y - b[g].y, dz = ai.z - b[g].z;
            const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            const float cut = reach_i + b[g].w;
            acc[g] = (d2 <= cut * cut) & (j[g] != pos);          // sentinel pads fail the distance test
            if (HAS_CLS) acc[g] = acc[g] && (s_cls[j[g]] != cls_i);   // (the sentinel slot of s_cls is never read)
        }
#pragma unroll
        for (int g = 0; g < G; ++g) m[g] = __ballot_sync(kFull, acc[g]);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int at = k + __popc(m[g] & lt);
            if (SASA_NOGUARD_ON ? acc[g] : (acc[g] & (at < kQueueCap))) cand[at] = (uint16_t)j[g];
            k += __popc(m[g]);
        }
    }
#pragma unroll 1
    for (; w0 < total; w0 += 32) {
        const int j = (int)list[w0 + lane];
        const float4 aj = s_atom[j];
        const float dx = ai.x - aj.x, dy = ai.y - aj.y, dz = ai.z - aj.z;
        const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
        const float cut = reach_i + aj.w;
        bool acc = (d2 <= cut * cut) & (j != pos);
        if (HAS_CLS) acc = acc && (s_cls[j] != cls_i);
        const unsigned m = __ballot_sync(kFull, acc);
        const int at = k + __popc(m & lt);
        if (SASA_NOGUARD_ON ? acc : (acc & (at < kQueueCap))) cand[at] = (uint16_t)j;
        k += __popc(m);
    }
#else
    constexpr int kGU = SASA_OPT_GU;
#pragma unroll kGU
    for (int w0 = 0; w0 < total; w0 += 32) {
        const int j = (int)list[w0 + lane];
        const float4 aj = s_atom[j];
        const float dx = ai.x - aj.x, dy = ai.y - aj.y, dz = ai.z - aj.z;
        const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
        const float cut = reach_i + aj.w;
        bool acc = (d2 <= cut * cut) & (j != pos);          // sentinel pads fail the distance test
        if (HAS_CLS) acc = acc && (s_cls[j] != cls_i);       // (the sentinel slot of s_cls is never read: && short-circuits)
        const unsigned m = __ballot_sync(kFull, acc);
        const int at = k + __popc(m & lt);
        if (acc & (at < kQueueCap)) cand[at] = (uint16_t)j;
        k += __popc(m);
    }
#endif
    __syncwarp();
    return k;
}

// Two atoms of one cell against the listed candidates in ONE pass: every candidate is loaded once and tested against both.
__device__ __forceinline__ void tight_gather2(const float4 *s_atom, const uint16_t *list, int total, int pos_a, int pos_b,
                                              const float4 aa, const float4 ab, float reach_a, float reach_b, uint16_t *cand_a,
                                              uint16_t *cand_b, int &ka, int &kb) {
    const int lane = lane_id();
    const unsigned lt = lanemask_lt();
    int k0 = 0, k1 = 0;
#ifndef SASA_OPT_PAIR_U
#define SASA_OPT_PAIR_U 1
#endif
    constexpr int kPairUnroll = SASA_OPT_PAIR_U;
#pragma unroll kPairUnroll
    for (int w0 = 0; w0 < total; w0 += 32) {
        const int j = (int)list[w0 + lane];
        const float4 b = s_atom[j];
        const float dxa = aa.x - b.x, dya = aa.y - b.y, dza = aa.z - b.z;
        const float dxb = ab.x - b.x, dyb = ab.y - b.y, dzb = ab.z - b.z;
        const float d2a = fmaf(dxa, dxa, fmaf(dya, dya, dza * dza)), d2b = fmaf(dxb, dxb, fmaf(dyb, dyb, dzb * dzb));
        const float ca = reach_a + b.w, cb = reach_b + b.w;
        const bool acc_a = (d2a <= ca * ca) & (j != pos_a), acc_b = (d2b <= cb * cb) & (j != pos_b);   // sentinel pads fail both
        const unsigned ma = __ballot_sync(kFull, acc_a), mb = __ballot_sync(kFull, acc_b);
        const int at_a = k0 + __popc(ma & lt), at_b = k1 + __popc(mb & lt);
        if (SASA_NOGUARD_ON ? acc_a : (acc_a & (at_a < kQueueCap))) cand_a[at_a] = (uint16_t)j;
        if (SASA_NOGUARD_ON ? acc_b : (acc_b & (at_b < kQueueCap))) cand_b[at_b] = (uint16_t)j;
        k0 += __popc(ma);
        k1 += __popc(mb);
    }
    __syncwarp();
    ka = k0;
    kb = k1;
}

// (vx, vy, vz, limit) per neighbour -- the per-pair setup of src/lib.rs:128-136 -- with the "near" neighbours
// (centre distance^2 < near2) packed at the front and the rest at the back.  Returns the number of near entries.
__device__ __forceinline__ int tight_entries(const float4 *s_atom, const float4 ai, float probe, float r2, float two_r,
                                             float near2, const uint16_t *cand, int k, float4 *ent) {
    const int lane = lane_id();
    const unsigned lt = lanemask_lt();
    int nfront = 0, nback = k - 1;
#pragma unroll 1
    for (int q0 = 0; q0 < k; q0 += 32) {
        const int q = q0 + lane;
        const bool valid = q < k;
        const float4 aj = s_atom[valid ? (int)cand[q] : 0];
        float vmag;
        const float4 e = make_entry(ai, aj, probe, r2, two_r, &vmag);
        const bool near = valid & (vmag < near2);
        const unsigned mn = __ballot_sync(kFull, near);
        const unsigned mv = __ballot_sync(kFull, valid);
        const unsigned mf = mv & ~mn;
        const int at = near ? nfront + __popc(mn & lt) : nback - __popc(mf & lt);
        if (valid) ent[at] = e;
        nfront += __popc(mn);
        nback -= __popc(mf);
    }
    __syncwarp();
    return nfront;
}

// Phase 1: NSL slots of body points per lane against entries [0, m).  Returns the per-slot "still exposed" ballots.
template <int NSL>
__device__ __forceinline__ void tight_phase1(const float4 *ent, int m, const float4 *pts, int nbody, unsigned (&live)[4]) {
    const int lane = lane_id();
    float4 p0 = pts[lane], p1, p2, p3;
    if (NSL > 1) p1 = pts[32 + lane];
    if (NSL > 2) p2 = pts[64 + lane];
    if (NSL > 3) p3 = pts[96 + lane];
    // scalar flags so that ptxas keeps them in predicate registers: FSETP.LT.OR P, dot, limit, P
    bool o0 = lane >= nbody, o1 = 32 + lane >= nbody, o2 = 64 + lane >= nbody, o3 = 96 + lane >= nbody;
    const float4 *const eend = ent + m;
    constexpr int kUnroll = SASA_OPT_P1U;
#pragma unroll kUnroll
    for (const float4 *ep = ent; ep < eend; ++ep) {
        const float4 e = *ep;
        o0 = o0 || (dot_body(p0.x, p0.y, p0.z, e) < e.w);
        if (NSL > 1) o1 = o1 || (dot_body(p1.x, p1.y, p1.z, e) < e.w);
        if (NSL > 2) o2 = o2 || (dot_body(p2.x, p2.y, p2.z, e) < e.w);
        if (NSL > 3) o3 = o3 || (dot_body(p3.x, p3.y, p3.z, e) < e.w);
    }
    live[0] = __ballot_sync(kFull, !o0);
    live[1] = NSL > 1 ? __ballot_sync(kFull, !o1) : 0u;
    live[2] = NSL > 2 ? __ballot_sync(kFull, !o2) : 0u;
    live[3] = NSL > 3 ? __ballot_sync(kFull, !o3) : 0u;
}

// Shape of a (point x entry) tile for ns (1..32) points: G = 2^sh is the power of two >= ns; lane l owns point
// (l mod G) and entry offset (l div G), so one step tests 32/G entries against every point.
__device__ __forceinline__ int tile_shift(int ns) { return 32 - __clz(ns - 1); }   // ns = 1 -> clz(0) = 32 -> 0

// `pt` (this lane's point of the tile) against entries [q0, k).  Returns the mask of occluded points (bit g = point g
// of the tile, g < 2^sh).  Every lane runs the same number of full steps (unrollable); the ragged last step is predicated.
template <bool TAIL>
__device__ __forceinline__ unsigned tight_tile(const float4 *ent, int q0, int k, const float4 pt, int sh) {
    const int lane = lane_id();
    const int kstep = 32 >> sh;
    const float4 *ep = ent + q0 + (lane >> sh);
    const float4 *const eend = ent + k;
    const int full = (k - q0) >> (5 - sh);
    // A point is occluded iff some entry has dot < limit (tail: dot <= limit), i.e. iff the largest margin
    // limit - dot is > 0 (tail: >= 0): with gradual underflow (nvcc's default, -ftz=false) an IEEE subtraction of two
    // floats is zero exactly when they are equal, so the sign of the rounded margin is the exact comparison.  The
    // running FMNMX keeps the loop free of predicates and loop-carried branches (NaN margins are ignored by fmaxf,
    // matching a false comparison).
    float best = -INFINITY;
#pragma unroll 2
    for (int t = 0; t < full; ++t) {
        const float4 e = *ep;
        ep += kstep;
        best = fmaxf(best, __fsub_rn(e.w, TAIL ? dot_tail(pt.x, pt.y, pt.z, e) : dot_body(pt.x, pt.y, pt.z, e)));
    }
    if (ep < eend) {
        const float4 e = *ep;
        best = fmaxf(best, __fsub_rn(e.w, TAIL ? dot_tail(pt.x, pt.y, pt.z, e) : dot_body(pt.x, pt.y, pt.z, e)));
    }
    const bool hit = TAIL ? (best >= 0.0f) : (best > 0.0f);
    // OR over the lanes that share a point: one REDUX.OR of per-point bits
    return __reduce_or_sync(kFull, hit ? (1u << (lane & ((1 << sh) - 1))) : 0u);
}

// The first ns (1..32) bits set.
__device__ __forceinline__ unsigned low_bits(int ns) { return 0xffffffffu >> (32 - ns); }

// Optional staging of tail tiles (off by default): test the kTailFirst nearest entries on their own and the rest only
// while some tail point is still exposed.
constexpr int kTailFirst = SASA_OPT_TAILX;

// One atom with its complete neighbour list in ent[0, k), nfront near entries first.  nbody = body points
// (index < n_body), the tail points are [nbody, n_points); tail_sh = tile_shift(min(32, ntail)).
// Returns the exposed-point count.
template <int NSL>
__device__ __forceinline__ int tight_atom(const KParams &p, const float4 *ent, int k, int nfront, const float4 *pts,
                                          uint16_t *queue, int nbody, int tail_sh) {
    const int lane = lane_id();
    const unsigned lt = lanemask_lt();
    const int m = min(k, min(max(nfront, p.m_min), p.m_max));
    unsigned live[4];
    tight_phase1<NSL>(ent, m, pts, nbody, live);
    int exposed = 0;
    const int ns = __popc(live[0]) + __popc(live[1]) + __popc(live[2]) + __popc(live[3]);
    if (m == k) {
        exposed = ns;
    } else if (ns) {
        int at = 0;     // survivors -> queue, slot-major
#pragma unroll
        for (int s = 0; s < NSL; ++s) {
            if ((live[s] >> lane) & 1u) queue[at + __popc(live[s] & lt)] = (uint16_t)(32 * s + lane);
            at += __popc(live[s]);
        }
        __syncwarp();
#pragma unroll 1
        for (int b = 0; b < ns; b += 32) {
            const int nb = min(32, ns - b);
            const int sh = tile_shift(nb);
            const int sidx = lane & ((1 << sh) - 1);
            exposed += __popc(~tight_tile<false>(ent, m, k, pts[sidx < nb ? (int)queue[b + sidx] : 0], sh) & low_bits(nb));
        }
        __syncwarp();
    }
    const int ntail = (int)p.n_points - nbody;
    if (ntail) {
        if (k == 0) {
            exposed += ntail;
        } else {
            const int sidx = lane & ((1 << tail_sh) - 1);
#pragma unroll 1
            for (int t0 = 0; t0 < ntail; t0 += 32) {
                const int nt = min(32, ntail - t0);
                // the last batch of a long tail may be narrower than the tile: its surplus lanes re-test point 0
                const float4 pt = pts[nbody + t0 + (sidx < nt ? sidx : 0)];
                const unsigned valid = low_bits(nt);
                unsigned hm = 0u;
                int q0 = 0, q1 = kTailFirst > 0 ? min(k, kTailFirst) : k;
                do {   // the nearest entries first; the rest only while some tail point is still exposed
                    hm |= tight_tile<true>(ent, q0, q1, pt, tail_sh);
                    q0 = q1;
                    q1 = k;
                } while (q0 < k && (~hm & valid) != 0u);
                exposed += __popc(~hm & valid);
            }
        }
    }
    return exposed;
}

// Cold path, out of line on purpose.  Cells with more than kListCap candidates (structures whose bounding box
// forced a coarser grid) take the generic per-atom gather and the generic chunked evaluation; atoms with more
// than kNbCap neighbours (denser than any protein) the list-free streaming routine.  Returns the exposed-point
// count and adds the atom's list length to misc[6] (pairs), or 1 to misc[7] (streamed atoms).
// HAS_MASK: every cold atom streams (atom_fast keeps no per-point result) and writes its mask row `mrow`.
template <bool HAS_CLS, class Atoms, bool HAS_MASK = false>
__device__ __forceinline__ int tight_cold_eval(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                               float probe, float near2, int m_min, int m_max, Grid g, const Atoms &atoms,
                                               const uint16_t *s_cell, const uint32_t *s_cls, const float4 *s_pts, int pos,
                                               float4 *ent, uint16_t *cand, int *misc, uint32_t *mrow = nullptr) {
    KParams q;
    q.px = px; q.py = py; q.pz = pz;
    q.n_points = n_points; q.n_body = n_body; q.probe = probe;
    q.near2 = near2; q.m_min = m_min; q.m_max = m_max; q.bcast_min = 16;
    const uint32_t *cls = HAS_CLS ? s_cls : nullptr;
    if (!HAS_MASK) {
        const float4 ai = atoms(pos);
        const int k = gather_candidates(q, g, atoms, s_cell, cls, pos, ai, cand);
        if (k >= 0) {
            const float r = __fadd_rn(ai.w, probe);
            const int nfront = build_entries(q, atoms, ai, __fmul_rn(r, r), __fmul_rn(2.0f, r), cand, k, ent);
            if (lane_id() == 0) atomicAdd(&misc[6], k);
            return (int)atom_fast(q, ent, k, nfront, cand, s_pts);
        }
    }
    if (lane_id() == 0) atomicAdd(&misc[7], 1);
    return (int)atom_streaming<Atoms, uint16_t, false, HAS_MASK>(q, g, atoms, s_cell, cls, pos, ent, nullptr, mrow);
}
template <bool HAS_CLS>
__device__ __noinline__ int tight_cold_atom(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                            float probe, float near2, int m_min, int m_max, Grid g, const float4 *s_atom,
                                            const uint16_t *s_cell, const uint32_t *s_cls, const float4 *s_pts, int pos,
                                            float4 *ent, uint16_t *cand, int *misc) {
    return tight_cold_eval<HAS_CLS>(px, py, pz, n_points, n_body, probe, near2, m_min, m_max, g, SmemAtoms{s_atom}, s_cell, s_cls,
                                    s_pts, pos, ent, cand, misc);
}
// The same for the masked kernel: the atom streams and writes its mask row.
template <bool HAS_CLS>
__device__ __noinline__ int tight_cold_atom_mask(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                                 float probe, Grid g, const float4 *s_atom, const uint16_t *s_cell, const uint32_t *s_cls,
                                                 int pos, float4 *ent, int *misc, uint32_t *mrow) {
    return tight_cold_eval<HAS_CLS, SmemAtoms, true>(px, py, pz, n_points, n_body, probe, 0.0f, 0, 0, g, SmemAtoms{s_atom}, s_cell, s_cls,
                                                     nullptr, pos, ent, nullptr, misc, mrow);
}
// The same with the atom's group standing alone (grouped runs): atoms of other groups are invisible.
template <bool HAS_CLS>
__device__ __noinline__ int tight_cold_atom_iso(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                                float probe, float near2, int m_min, int m_max, Grid g, const float4 *s_atom,
                                                const uint32_t *s_grp, const uint16_t *s_cell, const uint32_t *s_cls,
                                                const float4 *s_pts, int pos, float4 *ent, uint16_t *cand, int *misc) {
    return tight_cold_eval<HAS_CLS>(px, py, pz, n_points, n_body, probe, near2, m_min, m_max, g, GroupAtoms<false>{s_atom, s_grp, s_grp[pos]},
                                    s_cell, s_cls, s_pts, pos, ent, cand, misc);
}

// NSLT: number of 32-point body slots the kernel is compiled for (3 = the reference's default of 100 points on 8- and
// 16-lane builds, 96 body points), or 0 to choose per launch among 1..4.
// HAS_GRP: grouped run -- every atom is evaluated in the complex and with its group standing alone (the cap path in one pass,
// cap_atom_groups; the cold path twice), and the output stage runs once per value array.
// HAS_MASK: every atom also writes its exposed-point mask row (mp); cold atoms stream.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX, int NSLT, bool HAS_GRP, bool HAS_MASK = false>
__device__ __forceinline__ void tight_kernel_body(const KParams &p, const GroupParams &gp, const MaskParams &mp = MaskParams{}) {
    static_assert(!(HAS_GRP && HAS_MASK), "grouped runs write no masks");
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int NW = NT / 32;
    constexpr uint32_t NMAX = max_atoms(NT, MINB, CMAX, HAS_CLS, HAS_GRP);
    const SmemView V = smem_view<NT, HAS_CLS, NMAX, CMAX, HAS_GRP>(smem);
#if SASA_OPT_UWARP
    const int lane = lane_id(), warp = uniform_i32((int)(threadIdx.x >> 5));
#else
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#endif
    unsigned char *const wblock = smem + kOffWarpBlocks + (size_t)warp * kWarpBlockBytes;
    float4 *const w_ent = reinterpret_cast<float4 *>(wblock);
    uint16_t *const w_cand = reinterpret_cast<uint16_t *>(wblock + kWarpOffCand);
    uint16_t *const w_list = reinterpret_cast<uint16_t *>(wblock + kWarpOffList);
#if SASA_OPT_NOGUARD && SASA_OPT_CAP
    // neighbour lists of the cap path: two strips of kListCap positions inside the (idle) entry strip
    static_assert(2 * (size_t)kListCap * 2 <= (size_t)kNbCap * 16, "entry strip too small for two full candidate lists");
    uint16_t *const w_nba = reinterpret_cast<uint16_t *>(wblock), *const w_nbb = w_nba + kListCap;
#else
    uint16_t *const w_nba = w_cand, *const w_nbb = reinterpret_cast<uint16_t *>(w_ent);
#endif
    stage_points(p, V.ptab);
    const int nbody = (int)min(p.n_points, p.n_body), nsl = (nbody + 31) >> 5;
    (void)nsl;
    const int tail_sh = tile_shift(max(1, min(32, (int)p.n_points - nbody)));
    const float reach0 = 2.0f * p.probe + kCutSlack;

    uint32_t sid, a0;
    int N;
#if SASA_OPT_NEXT
    bool first = true;
    while (first ? claim_structure(p, V.misc, sid, a0, N) : claim_prefetched(p, V.misc, sid, a0, N)) {
        first = false;
#else
    while (claim_structure(p, V.misc, sid, a0, N)) {
#endif
        Grid g0;   // also parked in V.misc by the setup (load_grid)
        int ncell;
        const bool ok = structure_setup<NT, HAS_CLS, CMAX, HAS_GRP>(p, V, sid, a0, N, g0, ncell, gp);
#if SASA_OPT_NEXT
        if (warp == 0) claim_next_and_prefetch(p, V.misc);   // every structure, also after a rejected one
#endif
        if (!ok) {
            if (HAS_MASK) mask_zero_rows(mp, p.n_points, a0, (size_t)N, threadIdx.x, NT);
            continue;
        }
#if SASA_OPT_USTRUCT
        sid = uniform_u32(sid); a0 = uniform_u32(a0); N = uniform_i32(N);
#endif
#if SASA_OPT_UGRID
        g0.minx = uniform_f32(g0.minx); g0.miny = uniform_f32(g0.miny); g0.minz = uniform_f32(g0.minz);
        g0.inv_c = uniform_f32(g0.inv_c);
        g0.nx = uniform_i32(g0.nx); g0.ny = uniform_i32(g0.ny); g0.nz = uniform_i32(g0.nz); g0.e = uniform_i32(g0.e);
#endif

        // ---- per-atom work: warps claim runs of the cell-sorted atom order, whole cells at a time; the atoms of a cell
        // share its candidate list ----
        unsigned pairs = 0;   // neighbour pairs seen by this warp (statistics; the cold path counts into misc[6] itself)
        for (;;) {
            // guided self-scheduling: long runs while plenty remain, short ones near the end of the structure
            // (any positive increment partitions the range, so the stale read of the counter is harmless)
            int c0 = 0, take = 0;
#if SASA_OPT_ACLAIM > 0
            if (lane == 0) {
                const int left = N - *(volatile int *)&V.misc[1];
                take = max(SASA_OPT_ACLAIM, min(16 * SASA_OPT_ACLAIM, left / (4 * NW)));
                c0 = atomicAdd(&V.misc[1], take);
            }
#if SASA_OPT_UCLAIM
            c0 = uniform_i32(c0);       // lanes 1..31 hold 0
            take = uniform_i32(take);
#else
            c0 = __shfl_sync(kFull, c0, 0);
            take = __shfl_sync(kFull, take, 0);
#endif
            if (c0 >= N) break;
            int pos = c0;
            const int pos_end = min(c0 + take, N);
#else
            if (lane == 0) {
                const int left = ncell - *(volatile int *)&V.misc[1];
                take = max(SASA_CELL_FETCH, min(8 * SASA_CELL_FETCH, left / (4 * NW)));
                c0 = atomicAdd(&V.misc[1], take);
            }
            c0 = __shfl_sync(kFull, c0, 0);
            take = __shfl_sync(kFull, take, 0);
            if (c0 >= ncell) break;
            const int c1 = min(c0 + take, ncell);
            int pos = (int)V.cell[c0];
            const int pos_end = (int)V.cell[c1];
#endif
#if SASA_OPT_ACLAIM > 0 && SASA_OPT_SNAP
            {   // the cell that holds the first claimed atom started in an earlier claim: its owner finishes it
#if SASA_OPT_GRIDLD
                const Grid g = load_grid(V.misc);
#else
                const Grid g = g0;
#endif
                const float4 a = V.atom[pos];
                const int c = (cell_coord(a.z, g.minz, g.inv_c, g.nz) * g.ny + cell_coord(a.y, g.miny, g.inv_c, g.ny)) * g.nx +
                              cell_coord(a.x, g.minx, g.inv_c, g.nx);
                if ((int)V.cell[c] < pos) pos = (int)V.cell[c + 1];
            }
#endif
            while (pos < pos_end) {
                // the cell of atom `pos` and the end of its run in the sorted array (SASA_OPT_GRIDLD: the grid re-read from
                // shared memory at every cell instead of held in registers -- measured 1 % slower, off)
#if SASA_OPT_GRIDLD
                const Grid g = load_grid(V.misc);
#else
                const Grid g = g0;
#endif
                const float4 a_first = V.atom[pos];
                const int cx = cell_coord(a_first.x, g.minx, g.inv_c, g.nx), cy = cell_coord(a_first.y, g.miny, g.inv_c, g.ny),
                          cz = cell_coord(a_first.z, g.minz, g.inv_c, g.nz);
#if SASA_OPT_ACLAIM > 0 && SASA_OPT_SNAP && SASA_OPT_UCELL
                const int cell_end = uniform_i32((int)V.cell[(cz * g.ny + cy) * g.nx + cx + 1]);
#elif SASA_OPT_ACLAIM > 0 && SASA_OPT_SNAP
                const int cell_end = (int)V.cell[(cz * g.ny + cy) * g.nx + cx + 1];   // whole cells, past pos_end if need be
#else
                const int cell_end = min((int)V.cell[(cz * g.ny + cy) * g.nx + cx + 1], pos_end);
#endif
                const int total = tight_fill_list(g, V.cell, cx, cy, cz, w_list, N);
#if SASA_OPT_PAIR && SASA_OPT_CAP
                if (!HAS_CLS && !HAS_GRP && total >= 0) {
                    uint16_t *const w_cand2 = w_nbb;   // the entry strip is idle on the cap path
                    uint16_t *const w_cand = w_nba;
                    while (pos + 1 < cell_end) {
                        const float4 aa = V.atom[pos], ab = V.atom[pos + 1];
                        int ka, kb;
                        tight_gather2(V.atom, w_list, total, pos, pos + 1, aa, ab, aa.w + reach0, ab.w + reach0, w_cand, w_cand2, ka, kb);
                        if (ka > kNbCap || kb > kNbCap) break;   // dense neighbourhood: the one-atom path below sorts it out
                        uint32_t *const ra = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos]) : nullptr;
                        uint32_t *const rb = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos + 1]) : nullptr;
                        const int ca = cap_atom<SASA_CAP_TEX != 0, HAS_MASK>(p.cap, SmemAtoms{V.atom}, aa, p.probe, w_cand, ka, V.ptab, (int)p.n_points, nbody, p.cap_tex, ra);
                        const int cb = cap_atom<SASA_CAP_TEX != 0, HAS_MASK>(p.cap, SmemAtoms{V.atom}, ab, p.probe, w_cand2, kb, V.ptab, (int)p.n_points, nbody, p.cap_tex, rb);
                        pairs += (unsigned)(ka + kb);
                        if (lane < 2) V.val[(int)V.orig[pos + lane]] = (float)(lane ? cb : ca);
                        __syncwarp();
                        pos += 2;
                    }
                }
#endif
                for (; pos < cell_end; ++pos) {
                    const float4 ai = V.atom[pos];
                    int cnt;
#if SASA_OPT_CAP
                    uint16_t *const w_nb = w_nba;
#else
                    uint16_t *const w_nb = w_cand;
#endif
                    int k = total >= 0 ? tight_gather<HAS_CLS>(V.atom, V.cls, w_list, total, pos, ai, ai.w + reach0, w_nb)
                                       : kNbCap + 1;
                    int cnt_iso = 0;
                    uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos]) : nullptr;
                    if (k <= kNbCap) {
#if SASA_OPT_CAP
                        if (HAS_GRP)
                            cnt = cap_atom_groups<SASA_CAP_TEX != 0>(p.cap, SmemAtoms{V.atom}, ai, p.probe, w_nb, k, V.grp, V.grp[pos], V.ptab,
                                                                     (int)p.n_points, nbody, p.cap_tex, &cnt_iso);
                        else
                            cnt = cap_atom<SASA_CAP_TEX != 0, HAS_MASK>(p.cap, SmemAtoms{V.atom}, ai, p.probe, w_nb, k, V.ptab, (int)p.n_points, nbody,
                                                                        p.cap_tex, mrow);
#else
                        static_assert(!HAS_GRP, "grouped runs need the cap path");
                        const float r = __fadd_rn(ai.w, p.probe);
                        const int nfront = tight_entries(V.atom, ai, p.probe, __fmul_rn(r, r), __fmul_rn(2.0f, r), p.near2,
                                                         w_nb, k, w_ent);
                        if (NSLT > 0) cnt = tight_atom<NSLT ? NSLT : 1>(p, w_ent, k, nfront, V.ptab, w_cand, nbody, tail_sh);
                        else if (nsl == 3) cnt = tight_atom<3>(p, w_ent, k, nfront, V.ptab, w_cand, nbody, tail_sh);
                        else if (nsl == 4) cnt = tight_atom<4>(p, w_ent, k, nfront, V.ptab, w_cand, nbody, tail_sh);
                        else if (nsl == 2) cnt = tight_atom<2>(p, w_ent, k, nfront, V.ptab, w_cand, nbody, tail_sh);
                        else cnt = tight_atom<1>(p, w_ent, k, nfront, V.ptab, w_cand, nbody, tail_sh);
#endif
                        pairs += (unsigned)k;
                    } else if (HAS_MASK) {
                        cnt = tight_cold_atom_mask<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, g, V.atom, V.cell, V.cls, pos,
                                                            w_ent, V.misc, mrow);
                    } else {
                        cnt = tight_cold_atom<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, p.near2, p.m_min, p.m_max,
                                                       g, V.atom, V.cell, V.cls, V.ptab, pos, w_ent, w_cand, V.misc);
                        if (HAS_GRP)
                            cnt_iso = tight_cold_atom_iso<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, p.near2, p.m_min,
                                                                   p.m_max, g, V.atom, V.grp, V.cell, V.cls, V.ptab, pos, w_ent, w_cand, V.misc);
                    }
                    if (lane == 0) {
                        const int oi = (int)V.orig[pos];
                        if (HAS_GRP) V.val2[oi] = (float)cnt_iso;
#if SASA_OPT_AREA
                        V.val[oi] = atom_area(ai.w, p.probe, (float)cnt, p.inv_n);
                        if (p.out_counts) p.out_counts[a0 + oi] = (uint32_t)cnt;
#else
                        V.val[oi] = (float)cnt;
#endif
                    }
                    __syncwarp();
                }
            }
        }
        if (lane == 0 && pairs) atomicAdd(&V.misc[6], (int)pairs);
        __syncthreads();
        if (threadIdx.x == 0 && p.stat) {
            if (V.misc[6]) atomicAdd(p.stat + 1, (unsigned long long)(unsigned)V.misc[6]);
            if (V.misc[7]) atomicAdd(p.stat + 2, (unsigned long long)(unsigned)V.misc[7]);
        }
        structure_outputs<NT, SASA_OPT_AREA != 0>(p, V, sid, a0, N, smem + kOffWarpBlocks);
        if (HAS_GRP) {
            static_assert(!HAS_GRP || !SASA_OPT_AREA, "grouped runs store counts");
            SmemView W = V;
            W.val = V.val2;
            __syncthreads();   // the output stage's scratch is refilled
            structure_outputs<NT>(iso_outputs(p, gp), W, sid, a0, N, smem + kOffWarpBlocks);
        }
    }
}

template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX, int NSLT>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_kernel(const KParams p) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, NSLT, false>(p, GroupParams{});
}

// Exposed-point masks (n_points <= 128): the plain run's outputs plus every atom's mask row.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_masks_kernel(const KParams p, const MaskParams mp) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, 0, false, true>(p, GroupParams{}, mp);
}

// Grouped runs (n_points <= 128): complex and isolated outputs of every structure in one pass.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_groups_kernel(const KParams p, const GroupParams gp) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, 0, true>(p, gp);
}

}  // namespace sasa
