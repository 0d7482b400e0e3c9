// sasa_tight.cuh -- the fused per-structure kernel for n_points <= 128 (the reference's default, 100 points,
// is the headline configuration).  Same stages as the generic kernel of sasa_small.cuh, but the per-atom
// pipeline is written for a SMALL INSTRUCTION FOOTPRINT: the generic kernel's hot code spans ~45 KB of SASS,
// more than the SM's 32 KB L1.5 instruction cache, and ncu showed 37 % of its stall cycles as "no instruction"
// (profiles/r01a_baseline.txt).  Here every stage is one short rolled loop, the cell's candidate list lives in
// shared memory instead of unrolled register windows, and the never-taken fallbacks (dense clusters) sit behind one __noinline__ call.
//
// Per cell (warps claim runs of the cell-sorted atom order, snapped to whole cells):
//   list     the (2e+1)^2 cell rows around the cell are contiguous ranges of the cell-sorted atom array; their
//            positions are flattened once into a per-warp u16 list, padded to a multiple of 32 with the
//            far-away sentinel atom
// Per atom of the cell:
//   gather   32 listed candidates per step: distance test, ballot, compaction into a u16 neighbour list
//   cap      the cap-table occlusion of sasa_cap.cuh: one lane per neighbour, table masks, exact ring tests
// Between structures: warp 0 claims the CTA's next structure early and prefetches its atoms into L2 while the other warps
// already work on the current one (hides the claim / first-touch latency of the setup).
#pragma once
#include "sasa_cap.cuh"
#include "sasa_small.cuh"

namespace sasa {

// Flatten the candidate rows of cell (cx, cy, cz) into list[0, total) (positions in the sorted atom array),
// padded with `sentinel` up to the next multiple of 32.  Returns total, or -1 when it exceeds kListCap.
// The header (lane / w by multiplication, the scan with the shuffle's own predicate) took 454.0 -> 449.1 warp instructions per
// atom, 1,986 -> 2,012 M atoms/s (run r04h); the predicated row stores 487.2 -> 477.5, 1,863 -> 1,912 (r04f).
__device__ __forceinline__ int tight_fill_list(const Grid &g, const uint16_t *cell, int cx, int cy, int cz,
                                               uint16_t *list, int sentinel) {
    const int lane = lane_id();
    const int w = 2 * g.e + 1;
    // lane / w without the integer-division sequence: the search extent e is 1 or 2, so w is 3 or 5 (exact for lane < 32)
    const int q = g.e == 2 ? (lane * 13) >> 6 : (lane * 11) >> 5;
    const int dy = lane - q * w - g.e, dz = q - g.e;
    const int y = cy + dy, z = cz + dz;
    int start = 0, len = 0;
    if (lane < w * w && y >= 0 && y < g.ny && z >= 0 && z < g.nz) {
        const int x0 = max(cx - g.e, 0), x1 = min(cx + g.e, g.nx - 1);
        const int base = (z * g.ny + y) * g.nx;
        start = (int)cell[base + x0];
        len = (int)cell[base + x1 + 1] - start;
    }
    int incl = len;
    // inclusive scan, two instructions per step: the shuffle's own predicate (source lane in range) guards the addition
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
        asm volatile("{\n .reg .pred p;\n .reg .b32 t;\n shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n @p add.s32 %0, %0, t;\n}"
                     : "+r"(incl) : "r"(d));
    const int total = __shfl_sync(kFull, incl, 31);
    if (total > kListCap) return -1;
    const int maxlen = __reduce_max_sync(kFull, len);
    // row expansion, four positions per trip (the longest row of a protein-density cell block holds ~13 atoms), with four
    // PREDICATED stores per trip (nvcc turns plain monotone conditions into a chain of divergent branches: 22 instructions per
    // trip with a reconvergence point; this form is 15)
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
    // G steps per trip with every load ahead of the first store, so that the dependent shared-memory round trips
    // (list entry -> atom) of all G steps overlap.  The neighbour list has room for every listed candidate (kListCap), so the
    // stores need no capacity test.
    constexpr int G = 2;
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
            if (acc[g] != 0) cand[at] = (uint16_t)j[g];
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
        if (acc != 0) cand[at] = (uint16_t)j;
        k += __popc(m);
    }
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
#pragma unroll 1
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
        if (acc_a) cand_a[at_a] = (uint16_t)j;
        if (acc_b) cand_b[at_b] = (uint16_t)j;
        k0 += __popc(ma);
        k1 += __popc(mb);
    }
    __syncwarp();
    ka = k0;
    kb = k1;
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
// The same with only the atom's group and partner group gh present (pairwise buried area).
template <bool HAS_CLS>
__device__ __noinline__ int tight_cold_atom_pair(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                                 float probe, float near2, int m_min, int m_max, Grid g, const float4 *s_atom,
                                                 const uint32_t *s_grp, uint32_t gh, const uint16_t *s_cell, const uint32_t *s_cls,
                                                 const float4 *s_pts, int pos, float4 *ent, uint16_t *cand, int *misc) {
    return tight_cold_eval<HAS_CLS>(px, py, pz, n_points, n_body, probe, near2, m_min, m_max, g,
                                    PairAtoms<false>{s_atom, s_grp, s_grp[pos], gh}, s_cell, s_cls, s_pts, pos, ent, cand, misc);
}
// The isolated evaluation of a masked grouped run: the atom streams with its group standing alone and writes its isolated row.
template <bool HAS_CLS>
__device__ __noinline__ int tight_cold_atom_iso_mask(const float *px, const float *py, const float *pz, uint32_t n_points, uint32_t n_body,
                                                     float probe, Grid g, const float4 *s_atom, const uint32_t *s_grp, const uint16_t *s_cell,
                                                     const uint32_t *s_cls, int pos, float4 *ent, int *misc, uint32_t *irow) {
    return tight_cold_eval<HAS_CLS, GroupAtoms<false>, true>(px, py, pz, n_points, n_body, probe, 0.0f, 0, 0, g,
                                                             GroupAtoms<false>{s_atom, s_grp, s_grp[pos]}, s_cell, s_cls, nullptr, pos, ent,
                                                             nullptr, misc, irow);
}

// HAS_GRP: grouped run -- every atom is evaluated in the complex and with its group standing alone (the cap path in one pass,
// cap_atom_groups; the cold path twice), and the output stage runs once per value array.
// HAS_MASK: every atom also writes its exposed-point mask row (mp); cold atoms stream.  With HAS_GRP also its isolated row (mpi).
// HAS_PAIRS (with HAS_GRP): every atom also writes its partner slots (pp).  Cap-path atoms get them from cap_atom_groups; a cold
// atom enumerates its partners over the cell rows and is evaluated once more per partner with only its group and the partner's.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX, bool HAS_GRP, bool HAS_MASK = false, bool HAS_PAIRS = false>
__device__ __forceinline__ void tight_kernel_body(const KParams &p, const GroupParams &gp, const MaskParams &mp = MaskParams{},
                                                  const MaskParams &mpi = MaskParams{}, const PairParams &pp = PairParams{}) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int NW = NT / 32;
    constexpr uint32_t NMAX = max_atoms(NT, MINB, CMAX, HAS_CLS, HAS_GRP);
    const SmemView V = smem_view<NT, HAS_CLS, NMAX, CMAX, HAS_GRP>(smem);
    // The warp index goes through a warp reduction (REDUX writes a uniform register), so that the per-warp scratch addresses live
    // on the uniform datapath; ptxas otherwise re-derives them from SR_TID.X wherever the 64 vector registers run out.  Measured
    // together with the uniform cell grid below (run r04a/r04b, cfg2): either one alone changes nothing, both together
    // 539.0 -> 512 warp instructions per atom, and with the unguarded neighbour lists and the full-coverage exit of cap_atom 487.2
    // (1,683 -> 1,867 M atoms/s); the spills of the per-atom loop (five LDL per cell) are gone.
    const int lane = lane_id(), warp = uniform_i32((int)(threadIdx.x >> 5));
    unsigned char *const wblock = smem + kOffWarpBlocks + (size_t)warp * kWarpBlockBytes;
    float4 *const w_ent = reinterpret_cast<float4 *>(wblock);
    uint16_t *const w_cand = reinterpret_cast<uint16_t *>(wblock + kWarpOffCand);
    uint16_t *const w_list = reinterpret_cast<uint16_t *>(wblock + kWarpOffList);
    // neighbour lists of the cap path: two strips of kListCap positions inside the entry strip (idle on the cap path), with room
    // for every listed candidate, so the gather needs no capacity test on its stores
    static_assert(2 * (size_t)kListCap * 2 <= (size_t)kNbCap * 16, "entry strip too small for two full candidate lists");
    uint16_t *const w_nba = reinterpret_cast<uint16_t *>(wblock), *const w_nbb = w_nba + kListCap;
    stage_points(p, V.ptab);
    const int nbody = (int)min(p.n_points, p.n_body);
    const float reach0 = 2.0f * p.probe + kCutSlack;

    uint32_t sid, a0;
    int N;
    bool first = true;
    while (first ? claim_structure(p, V.misc, sid, a0, N) : claim_prefetched(p, V.misc, sid, a0, N)) {
        first = false;
        Grid g;
        int ncell;
        const bool ok = structure_setup<NT, HAS_CLS, CMAX, HAS_GRP>(p, V, sid, a0, N, g, ncell, gp);
        if (warp == 0) claim_next_and_prefetch(p, V.misc);   // every structure, also after a rejected one
        if (!ok) {
            if (HAS_MASK) mask_zero_rows(mp, p.n_points, a0, (size_t)N, threadIdx.x, NT);
            if (HAS_GRP && HAS_MASK) mask_zero_rows(mpi, p.n_points, a0, (size_t)N, threadIdx.x, NT);
            if (HAS_PAIRS) pair_blank_rows(pp, a0, (size_t)N, threadIdx.x, NT);
            continue;
        }
        // the structure's cell grid (eight CTA-uniform values) in uniform registers
        g.minx = uniform_f32(g.minx); g.miny = uniform_f32(g.miny); g.minz = uniform_f32(g.minz);
        g.inv_c = uniform_f32(g.inv_c);
        g.nx = uniform_i32(g.nx); g.ny = uniform_i32(g.ny); g.nz = uniform_i32(g.nz); g.e = uniform_i32(g.e);

        // ---- per-atom work: warps claim runs of at least kAtomClaim atoms of the cell-sorted order (a finer tail than runs of
        // cells), snapped to whole cells: a cell is worked by the warp whose claim holds the cell's first atom, so no candidate
        // list is built twice; the atoms of a cell share its candidate list ----
        constexpr int kAtomClaim = 4;
        unsigned pairs = 0;   // neighbour pairs seen by this warp (statistics; the cold path counts into misc[6] itself)
        for (;;) {
            // guided self-scheduling: long runs while plenty remain, short ones near the end of the structure
            // (any positive increment partitions the range, so the stale read of the counter is harmless)
            int c0 = 0, take = 0;
            if (lane == 0) {
                const int left = N - *(volatile int *)&V.misc[1];
                take = max(kAtomClaim, min(16 * kAtomClaim, left / (4 * NW)));
                c0 = atomicAdd(&V.misc[1], take);
            }
            c0 = __shfl_sync(kFull, c0, 0);
            take = __shfl_sync(kFull, take, 0);
            if (c0 >= N) break;
            int pos = c0;
            const int pos_end = min(c0 + take, N);
            {   // the cell that holds the first claimed atom started in an earlier claim: its owner finishes it
                const float4 a = V.atom[pos];
                const int c = (cell_coord(a.z, g.minz, g.inv_c, g.nz) * g.ny + cell_coord(a.y, g.miny, g.inv_c, g.ny)) * g.nx +
                              cell_coord(a.x, g.minx, g.inv_c, g.nx);
                if ((int)V.cell[c] < pos) pos = (int)V.cell[c + 1];
            }
            while (pos < pos_end) {
                // the cell of atom `pos` and the end of its run in the sorted array
                const float4 a_first = V.atom[pos];
                const int cx = cell_coord(a_first.x, g.minx, g.inv_c, g.nx), cy = cell_coord(a_first.y, g.miny, g.inv_c, g.ny),
                          cz = cell_coord(a_first.z, g.minz, g.inv_c, g.nz);
                const int cell_end = (int)V.cell[(cz * g.ny + cy) * g.nx + cx + 1];   // whole cells, past pos_end if need be
                const int total = tight_fill_list(g, V.cell, cx, cy, cz, w_list, N);
                // Pairs of atoms of a cell share one pass over the cell's candidate list: each candidate is loaded once and tested
                // against both.  Measured on cfg2 (run r02w-r02z): one atom at a time 1,635 M atoms/s / 560.6 warp
                // instructions per atom; pairs 1,684 / 539.0; groups of up to 3 or 4 atoms with the occlusion unrolled per atom
                // 1,022 / 670 (three more copies of cap_atom push the hot code out of the instruction cache: issue utilisation
                // 49 % / 32 %); the same groups with ONE rolled occlusion loop 1,523-1,591 (the bookkeeping costs more than the
                // loads saved).
                if (!HAS_CLS && !HAS_GRP && total >= 0) {
                    while (pos + 1 < cell_end) {
                        const float4 aa = V.atom[pos], ab = V.atom[pos + 1];
                        int ka, kb;
                        tight_gather2(V.atom, w_list, total, pos, pos + 1, aa, ab, aa.w + reach0, ab.w + reach0, w_nba, w_nbb, ka, kb);
                        if (ka > kNbCap || kb > kNbCap) break;   // dense neighbourhood: the one-atom path below sorts it out
                        uint32_t *const ra = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos]) : nullptr;
                        uint32_t *const rb = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos + 1]) : nullptr;
                        const int ca = cap_atom<true, HAS_MASK>(p.cap, SmemAtoms{V.atom}, aa, p.probe, w_nba, ka, V.ptab, (int)p.n_points, nbody, p.cap_tex, ra);
                        const int cb = cap_atom<true, HAS_MASK>(p.cap, SmemAtoms{V.atom}, ab, p.probe, w_nbb, kb, V.ptab, (int)p.n_points, nbody, p.cap_tex, rb);
                        pairs += (unsigned)(ka + kb);
                        if (lane < 2) V.val[(int)V.orig[pos + lane]] = (float)(lane ? cb : ca);
                        __syncwarp();
                        pos += 2;
                    }
                }
                for (; pos < cell_end; ++pos) {
                    const float4 ai = V.atom[pos];
                    int cnt;
                    int k = total >= 0 ? tight_gather<HAS_CLS>(V.atom, V.cls, w_list, total, pos, ai, ai.w + reach0, w_nba)
                                       : kNbCap + 1;
                    int cnt_iso = 0;
                    uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos]) : nullptr;
                    uint32_t *const irow = HAS_GRP && HAS_MASK ? mask_row(mpi, p.n_points, a0 + V.orig[pos]) : nullptr;
                    if (k <= kNbCap) {
                        if (HAS_PAIRS) {
                            PairSlot ps;
                            cnt = cap_atom_groups<true, false, true>(p.cap, SmemAtoms{V.atom}, ai, p.probe, w_nba, k, V.grp, V.grp[pos],
                                                                     V.ptab, (int)p.n_points, nbody, p.cap_tex, &cnt_iso, nullptr, nullptr, &ps);
                            pair_store(pp, a0 + V.orig[pos], ps, ai.w, p.probe, p.inv_n, p.err_flag);
                        } else if (HAS_GRP)
                            cnt = cap_atom_groups<true, HAS_MASK>(p.cap, SmemAtoms{V.atom}, ai, p.probe, w_nba, k, V.grp, V.grp[pos], V.ptab,
                                                                  (int)p.n_points, nbody, p.cap_tex, &cnt_iso, mrow, irow);
                        else
                            cnt = cap_atom<true, HAS_MASK>(p.cap, SmemAtoms{V.atom}, ai, p.probe, w_nba, k, V.ptab, (int)p.n_points, nbody,
                                                           p.cap_tex, mrow);
                        pairs += (unsigned)k;
                    } else if (HAS_MASK) {
                        cnt = tight_cold_atom_mask<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, g, V.atom, V.cell, V.cls, pos,
                                                            w_ent, V.misc, mrow);
                        if (HAS_GRP)
                            cnt_iso = tight_cold_atom_iso_mask<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, g, V.atom, V.grp,
                                                                        V.cell, V.cls, pos, w_ent, V.misc, irow);
                    } else {
                        cnt = tight_cold_atom<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, p.near2, p.m_min, p.m_max,
                                                       g, V.atom, V.cell, V.cls, V.ptab, pos, w_ent, w_cand, V.misc);
                        if (HAS_GRP)
                            cnt_iso = tight_cold_atom_iso<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, p.near2, p.m_min,
                                                                   p.m_max, g, V.atom, V.grp, V.cell, V.cls, V.ptab, pos, w_ent, w_cand, V.misc);
                        if (HAS_PAIRS) {
                            PairSlot ps = pair_empty();
                            const uint32_t gi = V.grp[pos];
                            bool first = true;
                            uint32_t h = 0u;
                            while (cnt_iso > 0 && pair_next_scan(g, V.cell, SmemAtoms{V.atom}, V.grp, pos, ai, ai.w + reach0, gi, first, h, h)) {
                                first = false;
                                const int cp = tight_cold_atom_pair<HAS_CLS>(p.px, p.py, p.pz, p.n_points, p.n_body, p.probe, p.near2,
                                                                             p.m_min, p.m_max, g, V.atom, V.grp, h, V.cell, V.cls, V.ptab,
                                                                             pos, w_ent, w_cand, V.misc);
                                pair_take(ps, h, cnt_iso - cp);
                            }
                            pair_store(pp, a0 + V.orig[pos], ps, ai.w, p.probe, p.inv_n, p.err_flag);
                        }
                    }
                    if (lane == 0) {
                        const int oi = (int)V.orig[pos];
                        if (HAS_GRP) V.val2[oi] = (float)cnt_iso;
                        V.val[oi] = (float)cnt;
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
        structure_outputs<NT>(p, V, sid, a0, N, smem + kOffWarpBlocks);
        if (HAS_GRP) {
            SmemView W = V;
            W.val = V.val2;
            __syncthreads();   // the output stage's scratch is refilled
            structure_outputs<NT>(iso_outputs(p, gp), W, sid, a0, N, smem + kOffWarpBlocks);
        }
    }
}

template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_kernel(const KParams p) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, false>(p, GroupParams{});
}

// Exposed-point masks (n_points <= 128): the plain run's outputs plus every atom's mask row.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_masks_kernel(const KParams p, const MaskParams mp) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, false, true>(p, GroupParams{}, mp);
}

// Grouped runs (n_points <= 128): complex and isolated outputs of every structure in one pass.
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_groups_kernel(const KParams p, const GroupParams gp) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, true>(p, gp);
}

// Pairwise buried area (n_points <= 128): the grouped run's outputs plus every atom's partner slots (pp).
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_group_pairs_kernel(const KParams p, const GroupParams gp, const PairParams pp) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, true, false, true>(p, gp, MaskParams{}, MaskParams{}, pp);
}

// Grouped runs with exposed-point masks (n_points <= 128): the grouped run's outputs plus every atom's mask row in the complex
// (mp) and with its group standing alone (mpi).
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_tight_groups_masks_kernel(const KParams p, const GroupParams gp, const MaskParams mp,
                                                                           const MaskParams mpi) {
    tight_kernel_body<NT, MINB, HAS_CLS, CMAX, true, true>(p, gp, mp, mpi);
}

}  // namespace sasa
