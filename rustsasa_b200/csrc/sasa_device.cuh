// sasa_device.cuh -- device-side building blocks of the B200 Shrake-Rupley engine.
//
// Arithmetic contract (what makes per-atom exposed-point counts bit-identical to the
// reference's CPU path, /root/reference/src/lib.rs:94-224):
//   v      = c_i - c_j                       three IEEE subtractions           (:129-131)
//   vmag   = (vx*vx + vy*vy) + vz*vz         unfused, left to right            (:132-133)
//   limit  = ((t_j - vmag) - r2) / (2*r)     IEEE division                     (:135-136)
//   body   : dot = fma(sx,vx, fma(sy,vy, sz*vz)),  occluded iff dot <  limit   (:143-147)
//   tail   : dot = (sx*vx + sy*vy) + sz*vz,        occluded iff dot <= limit   (:185-186)
// Every operation on that path is written with an explicit round-to-nearest intrinsic so
// that nvcc can neither contract nor re-associate it, whatever -fmad says.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sasa {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kNbCap = 96;            // neighbour entries staged per warp (protein lists peak around 75)
constexpr int kQueueCap = 128;        // survivor queue of one 128-point chunk (u16 per warp; aliases the candidate list)
constexpr int kCandSlots = kQueueCap;       // u16 slots of the per-warp candidate list
constexpr int kListCap = 320;         // cell candidate positions cached per warp by the tight kernel (10 windows of 32)
constexpr float kCutSlack = 1.0e-3f;  // Angstrom; keeps exactly-tangent pairs in the list (SURVEY.md 8a, row A2)
constexpr float kCellSafety = 1.0002f;
constexpr double kBoundaryTol = 1.0e-5;

// Dimensions of a chunked cap table (sasa_cap.cuh, 128 < n_points <= 1024).
struct CapDims {
    float half, scale;      // direction: iu = floor(u * scale + half)
    float lhalf;            // level:     l  = clamp(floor(c * lhalf + lhalf + 1), 0, levels - 1)
    int n, levels, nchp_shift;
    unsigned bin_degenerate, bin_empty;
};

struct KParams {
    // batch (device pointers)
    const float4 *xyzr;
    const float *xyz3, *radii;    // MD form (fused kernels only): 3 floats per atom + per-frame-index radii; else null
    const uint8_t *ridx;          // indexed form: 3 floats per atom (xyz3) + one byte per atom into the palette `radii`; else null
    const uint32_t *cls;          // nullable
    const uint32_t *struct_off;   // S+1
    const uint32_t *order;        // structures handled by this launch
    uint32_t n_work;
    uint32_t *work_counter;
    const uint32_t *ready;        // gate of the single-launch host pipeline (sasa_api.cu): the number of input chunks that have arrived in
    const uint32_t *need;         // device memory -- the copy stream raises it after every chunk -- and, per queue position, how many
                                  // chunks that position's structure needs.  null: everything is there
    const uint2 *seg_be;          // nullable
    const uint32_t *struct_seg_off;
    const uint8_t *seg_polar;     // nullable
    // outputs (nullable)
    uint32_t *out_counts;
    float *out_atom;
    float *out_seg;
    float *out_protein;
    // atom-range split with peer writes: the per-atom outputs of this rank's share go straight into every rank's vectors
    // (pointers valid on THIS device: the local vector and the peers' over NVLink); n_peers = 0: out_counts / out_atom only
    uint32_t *peer_counts[8];
    float *peer_atom[8];
    int n_peers;
    // sphere points (SoA) and run parameters
    const float *px, *py, *pz;
    const uint4 *cap;             // cap table of this point set (sasa_cap.cuh), n_points <= 128 only; else null
    unsigned long long cap_tex;   // the same table as a linear texture of uint4 (the fused kernel fetches its bins through the
                                  // texture pipe, off the LSU data pipe that carries the shared-memory traffic); 0: none
    const uint4 *capm_in, *capm_rg;   // chunked cap table (inner / ring masks), 128 < n_points <= 1024; else null
    const float4 *pts4;           // the points as float4 (chunked cap path)
    CapDims capd;
    uint32_t n_points, n_body;
    float inv_n, probe;
    float near2;                  // squared centre distance below which a neighbour is "near"
    int bcast_min;                // survivors needed for the broadcast form of phase 2
    int m_min, m_max;             // bounds on the number of entries phase 1 tests against every point
    // shared-memory capacities of this launch
    uint32_t nmax, cmax;
    uint32_t flags;
    int *err_flag;
    unsigned long long *stat;     // [0] boundary points, [1] neighbour pairs, [2] streamed atoms
};

// Grouped runs (sasa_b200_batch_run_groups_*), a kernel argument of their own next to KParams: one group label per atom and the
// outputs of every atom with its group standing alone (nullable each).
struct GroupParams {
    const uint32_t *grp;
    uint32_t *counts;
    float *atom, *seg, *protein;
};

// The run parameters with the isolated outputs in place of the complex ones (the output stages of grouped runs).
__host__ __device__ __forceinline__ KParams iso_outputs(const KParams &p, const GroupParams &gp) {
    KParams q = p;
    q.out_counts = gp.counts;
    q.out_atom = gp.atom;
    q.out_seg = gp.seg;
    q.out_protein = gp.protein;
    return q;
}

// Atom accessor of an isolated evaluation: an atom of another group than `gi` reads as a far-away sentinel, so it fails every
// distance test and never occludes -- the neighbour search and occlusion routines run unchanged on the group standing alone.
template <bool GLOBAL>
struct GroupAtoms {
    const float4 *a;
    const uint32_t *grp;
    uint32_t gi;
    __device__ __forceinline__ float4 operator()(int j) const {
        const uint32_t gj = GLOBAL ? __ldg(grp + j) : grp[j];
        return gj == gi ? (GLOBAL ? __ldg(a + j) : a[j]) : make_float4(1.0e18f, 1.0e18f, 1.0e18f, 0.0f);
    }
};

// Pairwise buried area (sasa_b200_batch_run_group_pairs_*), a kernel argument of its own next to GroupParams: k slots per atom in
// batch order (slot s of atom i at i * k + s) holding the partner groups that bury a point of the atom, in ascending label order.
// needed: two words, the largest number of partners of an atom in this run [0] and since the last sasa_b200_batch_sync [1].
struct PairParams {
    uint32_t *partner;
    uint32_t *counts;   // nullable
    float *area;        // nullable
    uint32_t *needed;
    uint32_t k;
};

// The evaluation of atom i (group gi) with only the atoms of gi and gh present: every other atom reads as the far-away sentinel.
template <bool GLOBAL>
struct PairAtoms {
    const float4 *a;
    const uint32_t *grp;
    uint32_t gi, gh;
    __device__ __forceinline__ float4 operator()(int j) const {
        const uint32_t gj = GLOBAL ? __ldg(grp + j) : grp[j];
        return (gj == gi || gj == gh) ? (GLOBAL ? __ldg(a + j) : a[j]) : make_float4(1.0e18f, 1.0e18f, 1.0e18f, 0.0f);
    }
};

// Exposed-point masks (sasa_b200_batch_run_masks_*), a kernel argument of its own next to KParams: mask_words(n_points) u32 per
// atom in batch order, bit b of word w set when point 32 w + b is exposed.  Every routine writes an atom's whole row with the
// lanes w < W of its warp (one coalesced store), so no row is left unwritten and the buffer needs no zero-fill.
struct MaskParams {
    uint32_t *exposed;
};
__host__ __device__ constexpr uint32_t mask_words(uint32_t n_points) { return (n_points + 31u) / 32u; }
__device__ __forceinline__ uint32_t *mask_row(const MaskParams &mp, uint32_t n_points, size_t atom) {
    return mp.exposed + atom * mask_words(n_points);
}

struct Grid {
    float minx, miny, minz, inv_c;
    int nx, ny, nz, e;
};

// threadIdx.x & 31 rather than %laneid: the special register saves 6 instructions per atom where ptxas rematerialises the
// lane index but measured 1 % slower (r04b: 1,848 vs 1,868 M atoms/s)
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
// A warp-uniform value routed through a warp reduction: REDUX writes a UNIFORM register, so ptxas may keep the value (and
// what is computed from it) on the uniform datapath instead of in one of the 64 vector registers of every thread.
__device__ __forceinline__ unsigned uniform_u32(unsigned v) { return __reduce_max_sync(kFull, v); }
__device__ __forceinline__ int uniform_i32(int v) { return (int)__reduce_max_sync(kFull, (unsigned)v); }
__device__ __forceinline__ float uniform_f32(float v) { return __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(v))); }
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Bits of the points that exist in word w of a mask row.
__device__ __forceinline__ unsigned mask_valid(int n_points, int w) {
    const int left = n_points - 32 * w;
    return left >= 32 ? 0xffffffffu : (left > 0 ? (0xffffffffu >> (32 - left)) : 0u);
}
// Mask row of a point set of at most 128 points from the warp-uniform coverage words c0..c3 (all ones: a covered atom, zeros).
__device__ __forceinline__ void mask_store4(uint32_t *row, int n_points, unsigned c0, unsigned c1, unsigned c2, unsigned c3) {
    const int lane = lane_id();
    if (lane < (int)mask_words((uint32_t)n_points))
        row[lane] = mask_valid(n_points, lane) & ~(lane == 0 ? c0 : lane == 1 ? c1 : lane == 2 ? c2 : c3);
}
// A mask row of zeros (every point occluded).
__device__ __forceinline__ void mask_zero(uint32_t *row, int n_points) {
    const int W = (int)mask_words((uint32_t)n_points);
    for (int w = lane_id(); w < W; w += 32) row[w] = 0u;
}
// The mask rows of atoms [a0, a0 + N) zeroed by the threads of a block (a structure with non-finite input).
__device__ __forceinline__ void mask_zero_rows(const MaskParams &mp, uint32_t n_points, size_t a0, size_t N, size_t tid, size_t nth) {
    const size_t W = mask_words(n_points);
    for (size_t i = tid; i < N * W; i += nth) mp.exposed[a0 * W + i] = 0u;
}

__device__ __forceinline__ int cell_coord(float x, float mn, float inv_c, int n) {
    int c = (int)(__fmul_rn(__fsub_rn(x, mn), inv_c));
    return min(max(c, 0), n - 1);
}

// (vx, vy, vz, limit) of neighbour j as seen from atom i -- the per-pair setup of lib.rs:128-136.
__device__ __forceinline__ float4 make_entry(const float4 ai, const float4 aj, float probe, float r2, float two_r,
                                             float *vmag_out) {
    const float vx = __fsub_rn(ai.x, aj.x), vy = __fsub_rn(ai.y, aj.y), vz = __fsub_rn(ai.z, aj.z);
    const float vmag = __fadd_rn(__fadd_rn(__fmul_rn(vx, vx), __fmul_rn(vy, vy)), __fmul_rn(vz, vz));
    const float tj = __fadd_rn(aj.w, probe);
    const float t = __fmul_rn(tj, tj);
    const float limit = __fdiv_rn(__fsub_rn(__fsub_rn(t, vmag), r2), two_r);
    *vmag_out = vmag;
    return make_float4(vx, vy, vz, limit);
}

__device__ __forceinline__ float dot_body(float sx, float sy, float sz, const float4 e) {
    return __fmaf_rn(sx, e.x, __fmaf_rn(sy, e.y, __fmul_rn(sz, e.z)));
}
__device__ __forceinline__ float dot_tail(float sx, float sy, float sz, const float4 e) {
    return __fadd_rn(__fadd_rn(__fmul_rn(sx, e.x), __fmul_rn(sy, e.y)), __fmul_rn(sz, e.z));
}
__device__ __forceinline__ bool occl(float sx, float sy, float sz, bool tail, const float4 e) {
    return tail ? (dot_tail(sx, sy, sz, e) <= e.w) : (dot_body(sx, sy, sz, e) < e.w);
}

// Area expression of lib.rs:220-222: ((4*pi_f32 * r2) * count) * (1/n).
__device__ __forceinline__ float atom_area(float radius, float probe, float count, float inv_n) {
    const float r = __fadd_rn(radius, probe);
    const float r2 = __fmul_rn(r, r);
    const float sa = __fmul_rn(12.566370614359172f, r2);
    return __fmul_rn(__fmul_rn(sa, count), inv_n);
}

// ---------------------------------------------------------------------------------------
// Candidate enumeration around one atom: the (2e+1)^2 cell rows that can hold a neighbour,
// each a contiguous range of the cell-sorted atom array, flattened into one index space so
// that all 32 lanes test a candidate per step.
// ---------------------------------------------------------------------------------------
struct Rows {
    int start, incl, excl, total;  // per lane (= per row) range start, inclusive/exclusive prefix; warp total
};

template <typename CellT>
__device__ __forceinline__ Rows rows_of(const Grid &g, const CellT *cell, int cx, int cy, int cz) {
    const int lane = lane_id();
    const int w = 2 * g.e + 1;
    const int dy = lane % w - g.e, dz = lane / w - g.e;
    const int y = cy + dy, z = cz + dz;
    const bool ok = lane < w * w && y >= 0 && y < g.ny && z >= 0 && z < g.nz;
    int start = 0, len = 0;
    if (ok) {
        const int x0 = max(cx - g.e, 0), x1 = min(cx + g.e, g.nx - 1);
        const int base = (z * g.ny + y) * g.nx;
        start = (int)cell[base + x0];
        len = (int)cell[base + x1 + 1] - start;
    }
    int incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += t;
    }
    Rows r;
    r.start = start;
    r.incl = incl;
    r.excl = incl - len;
    r.total = __shfl_sync(kFull, incl, 31);
    return r;
}

// Flat candidate index -> position in the sorted atom array (valid only when idx < rows.total).
__device__ __forceinline__ int row_lookup(const Rows &r, int idx) {
    int lo = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(kFull, r.incl, lo + step - 1);
        if (v <= idx) lo += step;
    }
    lo = min(lo, 31);
    const int rs = __shfl_sync(kFull, r.start, lo);
    const int re = __shfl_sync(kFull, r.excl, lo);
    return rs + (idx - re);
}

// ---------------------------------------------------------------------------------------
// Streaming (list-free) evaluation of one atom: always correct for any density, used when
// the neighbour list would overflow the per-warp staging area, when boundary statistics
// are requested and as the in-kernel cross-check of the fast path.
// Returns the exposed-point count; all lanes receive it.  HAS_MASK: the per-slot ballots are the
// words of the atom's mask row `mrow`, stored by lanes 0-3 after every 128-point chunk.
// ---------------------------------------------------------------------------------------
template <typename AtomAcc, typename CellT, bool STATS, bool HAS_MASK = false>
__device__ float atom_streaming(const KParams &p, const Grid &g, const AtomAcc &atoms, const CellT *cell,
                                const uint32_t *cls_sorted, int pos, float4 *ent, unsigned long long *boundary,
                                uint32_t *mrow = nullptr) {
    const int lane = lane_id();
    const float4 ai = atoms(pos);
    const float r = __fadd_rn(ai.w, p.probe);
    const float r2 = __fmul_rn(r, r);
    const float two_r = __fmul_rn(2.0f, r);
    const float reach_i = ai.w + 2.0f * p.probe + kCutSlack;
    const uint32_t cls_i = cls_sorted ? cls_sorted[pos] : 0u;
    const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
              cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
    const Rows rows = rows_of(g, cell, cx, cy, cz);
    float exposed = 0.0f;
    unsigned nbnd = 0;
    for (uint32_t p0 = 0; p0 < p.n_points; p0 += 128) {
        float sx[4], sy[4], sz[4];
        bool occ[4], tail[4], bnd[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const uint32_t pi = p0 + 32u * s + lane;
            const bool valid = pi < p.n_points;
            sx[s] = valid ? __ldg(p.px + pi) : 0.0f;
            sy[s] = valid ? __ldg(p.py + pi) : 0.0f;
            sz[s] = valid ? __ldg(p.pz + pi) : 0.0f;
            occ[s] = !valid;
            bnd[s] = false;
            tail[s] = pi >= p.n_body;
        }
        for (int t0 = 0; t0 < rows.total; t0 += 32) {
            const int idx = t0 + lane;
            const int j = row_lookup(rows, idx);
            bool acc = false;
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
            if (idx < rows.total && j != pos) {
                const float4 aj = atoms(j);
                float vmag;
                e = make_entry(ai, aj, p.probe, r2, two_r, &vmag);
                const float cut = reach_i + aj.w;
                acc = vmag <= cut * cut && !(cls_sorted && cls_sorted[j] == cls_i);
            }
            const unsigned m = __ballot_sync(kFull, acc);
            if (acc) ent[__popc(m & lanemask_lt())] = e;
            __syncwarp();
            const int cnt = __popc(m);
            for (int q = 0; q < cnt; ++q) {
                const float4 eq = ent[q];
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float d = tail[s] ? dot_tail(sx[s], sy[s], sz[s], eq) : dot_body(sx[s], sy[s], sz[s], eq);
                    occ[s] = occ[s] || (tail[s] ? (d <= eq.w) : (d < eq.w));
                    if (STATS) bnd[s] = bnd[s] || (fabs(2.0 * (double)r * ((double)d - (double)eq.w)) <= kBoundaryTol);
                }
            }
            __syncwarp();
        }
        unsigned word = 0u;   // HAS_MASK: lane s keeps the ballot of slot s
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const unsigned live = __ballot_sync(kFull, !occ[s]);
            exposed += (float)__popc(live);
            if (HAS_MASK && lane == s) word = live;
            if (STATS) nbnd += __popc(__ballot_sync(kFull, bnd[s] && (p0 + 32u * s + lane < p.n_points)));
        }
        if (HAS_MASK && lane < 4 && p0 / 32u + lane < mask_words(p.n_points)) mrow[p0 / 32u + lane] = word;
    }
    if (STATS && lane == 0 && nbnd) atomicAdd(boundary, (unsigned long long)nbnd);
    return exposed;
}

// ---------------------------------------------------------------------------------------
// Fast path pieces.
// ---------------------------------------------------------------------------------------

// Pass 1: positions (in the sorted array) of all atoms within r_i + r_j + 2*probe (+slack) of
// atom `pos`.  Returns the count, or -1 if it exceeds kNbCap (caller falls back to streaming).
template <typename AtomAcc, typename CellT, typename IdxT>
__device__ __forceinline__ int gather_candidates(const KParams &p, const Grid &g, const AtomAcc &atoms,
                                                 const CellT *cell, const uint32_t *cls_sorted, int pos,
                                                 const float4 ai, IdxT *cand) {
    const int lane = lane_id();
    const float reach_i = ai.w + 2.0f * p.probe + kCutSlack;
    const uint32_t cls_i = cls_sorted ? cls_sorted[pos] : 0u;
    const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
              cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
    const Rows rows = rows_of(g, cell, cx, cy, cz);
    int k = 0;
    for (int t0 = 0; t0 < rows.total; t0 += 32) {
        const int idx = t0 + lane;
        const int j = row_lookup(rows, idx);
        bool acc = false;
        if (idx < rows.total && j != pos) {
            const float4 aj = atoms(j);
            const float dx = ai.x - aj.x, dy = ai.y - aj.y, dz = ai.z - aj.z;
            const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            const float cut = reach_i + aj.w;
            // membership is result-neutral (a superset of the overlapping pairs is all that is needed), so this
            // test may use contracted arithmetic; the slack absorbs its rounding.
            acc = d2 <= cut * cut && !(cls_sorted && cls_sorted[j] == cls_i);
        }
        const unsigned m = __ballot_sync(kFull, acc);
        if (m) {
            const int at = k + __popc(m & lanemask_lt());
            if (acc && at < kNbCap) cand[at] = (IdxT)j;
            k += __popc(m);
        }
    }
    __syncwarp();
    return k <= kNbCap ? k : -1;
}

// Register cache of the flattened candidate list of one cell: window w of lane l is candidate 32*w + l.
// All atoms of a cell share it, so consecutive atoms of the same cell skip rows_of / row_lookup altogether.
constexpr int kCacheWin = 12;   // 384 candidates; denser neighbourhoods use the uncached gather
template <typename IdxT>
struct CandCache {
    static constexpr int kPer = sizeof(IdxT) == 2 ? 2 : 1;
    uint32_t v[kCacheWin / kPer];
    int total;   // < 0: not cacheable (too many candidates)
    int cell;
    __device__ __forceinline__ void set(int w, int j) {
        if (kPer == 2) v[w >> 1] = (w & 1) ? ((v[w >> 1] & 0xffffu) | ((uint32_t)j << 16)) : ((uint32_t)j & 0xffffu);
        else v[w] = (uint32_t)j;
    }
    __device__ __forceinline__ int get(int w) const {
        if (kPer == 2) return (int)((w & 1) ? (v[w >> 1] >> 16) : (v[w >> 1] & 0xffffu));
        return (int)v[w];
    }
};

template <typename CellT, typename IdxT>
__device__ __forceinline__ void fill_cache(const Grid &g, const CellT *cell, int cx, int cy, int cz, int cell_id,
                                           CandCache<IdxT> &cc) {
    const Rows rows = rows_of(g, cell, cx, cy, cz);
    cc.cell = cell_id;
    cc.total = rows.total <= 32 * kCacheWin ? rows.total : -1;
    if (cc.total < 0) return;
#pragma unroll
    for (int w = 0; w < kCacheWin; ++w)
        if (32 * w < rows.total) {
            const int idx = 32 * w + lane_id();
            const int j = row_lookup(rows, idx);
            cc.set(w, idx < rows.total ? j : 0);   // slots past the end hold a harmless in-range position
        }
}

// Pass 1 through the cache: same result as gather_candidates.
template <typename AtomAcc, typename IdxT>
__device__ __forceinline__ int gather_cached(const KParams &p, const AtomAcc &atoms, const uint32_t *cls_sorted, int pos,
                                             const float4 ai, const CandCache<IdxT> &cc, IdxT *cand) {
    const int lane = lane_id();
    const float reach_i = ai.w + 2.0f * p.probe + kCutSlack;
    const uint32_t cls_i = cls_sorted ? cls_sorted[pos] : 0u;
    int k = 0;
#pragma unroll
    for (int w = 0; w < kCacheWin; ++w) {
        if (32 * w >= cc.total) break;
        const int j = cc.get(w);
        bool acc = false;
        if (32 * w + lane < cc.total && j != pos) {
            const float4 aj = atoms(j);
            const float dx = ai.x - aj.x, dy = ai.y - aj.y, dz = ai.z - aj.z;
            const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            const float cut = reach_i + aj.w;
            acc = d2 <= cut * cut && !(cls_sorted && cls_sorted[j] == cls_i);
        }
        const unsigned m = __ballot_sync(kFull, acc);
        if (m) {
            const int at = k + __popc(m & lanemask_lt());
            if (acc && at < kNbCap) cand[at] = (IdxT)j;
            k += __popc(m);
        }
    }
    __syncwarp();
    return k <= kNbCap ? k : -1;
}

// Pass 2: turn candidate positions into (v, limit) entries; "near" neighbours (centre distance^2 < near2) are
// packed at the front, the rest at the back.  Returns the number of near entries.
template <typename AtomAcc, typename IdxT>
__device__ __forceinline__ int build_entries(const KParams &p, const AtomAcc &atoms, const float4 ai, float r2,
                                             float two_r, const IdxT *cand, int k, float4 *ent) {
    const int lane = lane_id();
    int nfront = 0, nback = 0;
    for (int q0 = 0; q0 < k; q0 += 32) {
        const int q = q0 + lane;
        const bool valid = q < k;
        float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
        float vmag = 0.0f;
        if (valid) e = make_entry(ai, atoms((int)cand[q]), p.probe, r2, two_r, &vmag);
        const bool near = valid && vmag < p.near2;
        const unsigned mn = __ballot_sync(kFull, near);
        const unsigned mf = __ballot_sync(kFull, valid && !near);
        if (valid) {
            const int at = near ? nfront + __popc(mn & lanemask_lt()) : (k - 1) - (nback + __popc(mf & lanemask_lt()));
            ent[at] = e;
        }
        nfront += __popc(mn);
        nback += __popc(mf);
    }
    __syncwarp();
    return nfront;
}

// One 128-point chunk of sphere points held in registers: slot s of a lane is point p0 + 32*s + lane.
struct PointChunk {
    float sx[4], sy[4], sz[4];
};

__device__ __forceinline__ void load_chunk(const KParams &p, const float4 *s_pts, uint32_t p0, PointChunk &c) {
    const int lane = lane_id();
    if (s_pts) {   // whole point set (<= 128 points) staged as float4 in shared memory
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const float4 q = s_pts[32 * s + lane];
            c.sx[s] = q.x; c.sy[s] = q.y; c.sz[s] = q.z;
        }
        return;
    }
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const uint32_t pi = p0 + 32u * s + lane;
        const bool valid = pi < p.n_points;
        c.sx[s] = valid ? __ldg(p.px + pi) : 0.0f;
        c.sy[s] = valid ? __ldg(p.py + pi) : 0.0f;
        c.sz[s] = valid ? __ldg(p.pz + pi) : 0.0f;
    }
}

// A single sphere point by index: from the per-CTA float4 table when the whole point set fits it
// (n_points <= 128), else from the global SoA arrays through L1.
__device__ __forceinline__ float4 point_at(const KParams &p, const float4 *s_pts, uint32_t pi) {
    if (s_pts) return s_pts[pi];
    return make_float4(__ldg(p.px + pi), __ldg(p.py + pi), __ldg(p.pz + pi), 0.0f);
}

// Phase 1: the body points of one 128-point chunk (NS slots per lane) against entries [0, m): one broadcast
// LDS.128 per neighbour, 4 FP32-pipe instructions per point-neighbour test.
template <int NS>
__device__ __forceinline__ void phase1(const float4 *ent, int m, const PointChunk &c, bool (&occ)[4]) {
    // scalar flags (not an array) so that ptxas keeps them in predicate registers: FSETP.LT.OR P, dot, limit, P
    bool o0 = occ[0], o1 = occ[1], o2 = occ[2], o3 = occ[3];
#pragma unroll 2
    for (int q = 0; q < m; ++q) {
        const float4 e = ent[q];
        if (NS > 0) o0 = o0 || (dot_body(c.sx[0], c.sy[0], c.sz[0], e) < e.w);
        if (NS > 1) o1 = o1 || (dot_body(c.sx[1], c.sy[1], c.sz[1], e) < e.w);
        if (NS > 2) o2 = o2 || (dot_body(c.sx[2], c.sy[2], c.sz[2], e) < e.w);
        if (NS > 3) o3 = o3 || (dot_body(c.sx[3], c.sy[3], c.sz[3], e) < e.w);
    }
    occ[0] = o0; occ[1] = o1; occ[2] = o2; occ[3] = o3;
}

// Phase 2: `ns` (<= 32) surviving points, listed in queue[0, ns), against entries [q0, k) as a 2-D tile:
// with G = the power of two >= ns, lane l owns survivor (l mod G) and entry offset (l div G), so one
// step tests 32/G entries against every survivor (ns = 32: one entry broadcast per step; ns = 1: 32 entries
// per step for the single survivor).  Returns the number of survivors no entry occludes.
template <bool TAIL>
__device__ __forceinline__ int phase2_tile(const KParams &p, const float4 *s_pts, const float4 *ent, int q0, int k,
                                           const uint16_t *queue, int ns, uint32_t p0) {
    const int lane = lane_id();
    int g = 1, sh = 0;
    while (g < ns) { g <<= 1; ++sh; }
    const int sidx = lane & (g - 1), eoff = lane >> sh, estep = 32 >> sh;
    const bool have = sidx < ns;
    const float4 pt = point_at(p, s_pts, p0 + (have ? (uint32_t)queue[sidx] : 0u));
    bool hit = false;
    for (int q = q0 + eoff; q < k; q += estep) {
        const float4 e = ent[q];
        hit = hit || (TAIL ? (dot_tail(pt.x, pt.y, pt.z, e) <= e.w) : (dot_body(pt.x, pt.y, pt.z, e) < e.w));
    }
    unsigned mk = __ballot_sync(kFull, hit);
    for (int st = 16; st >= g; st >>= 1) mk |= mk >> st;     // OR over the lanes that share a survivor
    const unsigned valid = ns >= 32 ? 0xffffffffu : ((1u << ns) - 1u);
    return __popc(~mk & valid);
}

// Broadcast form with early exit for many survivors (G = 32): leaves as soon as every survivor is occluded.
__device__ __forceinline__ int phase2_bcast(const KParams &p, const float4 *s_pts, const float4 *ent, int q0, int k,
                                            const uint16_t *queue, int ns, uint32_t p0) {
    const int lane = lane_id();
    const bool have = lane < ns;
    const float4 pt = point_at(p, s_pts, p0 + (have ? (uint32_t)queue[lane] : 0u));
    bool dead = !have;
    int q = q0;
    for (; q + 4 <= k; q += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float4 e = ent[q + u];
            dead = dead || (dot_body(pt.x, pt.y, pt.z, e) < e.w);
        }
        if (__all_sync(kFull, dead)) return 0;
    }
    for (; q < k; ++q) {
        const float4 e = ent[q];
        dead = dead || (dot_body(pt.x, pt.y, pt.z, e) < e.w);
    }
    return __popc(__ballot_sync(kFull, !dead));
}

// Fast evaluation of one atom whose complete neighbour list sits in ent[0, k) with nfront near entries first.
// `queue` is per-warp scratch for point indices (kQueueCap u16, may alias the candidate list).
// Body points (index < n_body) go through phase 1 (first m entries, all points) and phase 2 (survivors, the
// remaining entries); the few tail points skip phase 1 and are tested against all entries by the tile routine.
__device__ __forceinline__ float atom_fast(const KParams &p, const float4 *ent, int k, int nfront, uint16_t *queue,
                                           const float4 *s_pts, const PointChunk *pre = nullptr) {
    const int lane = lane_id();
    int exposed = 0;
    const int m = min(k, min(max(nfront, p.m_min), p.m_max));
    for (uint32_t p0 = 0; p0 < p.n_points; p0 += 128) {
        PointChunk c;
        if (pre) c = *pre;
        else load_chunk(p, s_pts, p0, c);
        const uint32_t pend = min(p0 + 128u, p.n_points);
        const uint32_t bend = min(pend, max(p.n_body, p0));      // body points of the chunk: [p0, bend)
        const int nsl = (int)((bend - p0 + 31u) >> 5);           // slots holding at least one body point
        bool occ[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) occ[s] = p0 + 32u * s + lane >= bend;
        if (nsl == 4) phase1<4>(ent, m, c, occ);
        else if (nsl == 3) phase1<3>(ent, m, c, occ);
        else if (nsl == 2) phase1<2>(ent, m, c, occ);
        else if (nsl == 1) phase1<1>(ent, m, c, occ);
        if (m == k) {
#pragma unroll
            for (int s = 0; s < 4; ++s) exposed += __popc(__ballot_sync(kFull, !occ[s]));
        } else {
            int ns = 0;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const unsigned mb = __ballot_sync(kFull, !occ[s]);
                if (!occ[s]) queue[ns + __popc(mb & lanemask_lt())] = (uint16_t)(32 * s + lane);
                ns += __popc(mb);
            }
            __syncwarp();
            for (int b = 0; b < ns; b += 32) {
                const int nb = min(32, ns - b);
                exposed += nb > p.bcast_min ? phase2_bcast(p, s_pts, ent, m, k, queue + b, nb, p0)
                                            : phase2_tile<false>(p, s_pts, ent, m, k, queue + b, nb, p0);
            }
            __syncwarp();
        }
        // tail points [bend, pend) of this chunk against every entry
        for (uint32_t t0 = bend; t0 < pend; t0 += 32) {
            const int nt = (int)min(32u, pend - t0);
            if (lane < nt) queue[lane] = (uint16_t)(t0 - p0 + lane);
            __syncwarp();
            exposed += k ? phase2_tile<true>(p, s_pts, ent, 0, k, queue, nt, p0) : nt;
            __syncwarp();
        }
    }
    return (float)exposed;
}

// ---------------------------------------------------------------------------------------
// Pairwise buried area: the slot row of one atom.  Partners are enumerated warp-uniformly in ascending label order; one with a
// non-zero buried count takes the next slot, held by lane n (so lane s < k ends up holding slot s).  n counts every partner with a
// non-zero count, also past the k slots.
// ---------------------------------------------------------------------------------------
struct PairSlot {
    uint32_t label, count;   // this lane's slot
    int n;                   // partners with a non-zero count (warp-uniform)
};

__device__ __forceinline__ PairSlot pair_empty() { return PairSlot{0xffffffffu, 0u, 0}; }

__device__ __forceinline__ void pair_take(PairSlot &ps, uint32_t h, int buried) {
    if (buried <= 0) return;
    if (lane_id() == ps.n) {
        ps.label = h;
        ps.count = (uint32_t)buried;
    }
    ++ps.n;
}

// The atom's row (one coalesced store per array from lanes s < k), and the number of partners into both `needed` words.  More
// partners than slots raise SASA_B200_ERR_INVALID_ARGUMENT (1) in the error flag unless an error is already there, so a
// non-finite structure (4, written by exchange) always wins.
__device__ __forceinline__ void pair_store(const PairParams &pp, size_t atom, const PairSlot &ps, float radius, float probe, float inv_n,
                                           int *err_flag) {
    const int lane = lane_id();
    if (lane < (int)pp.k) {
        const bool used = lane < ps.n;
        const size_t o = atom * pp.k + (size_t)lane;
        pp.partner[o] = used ? ps.label : 0xffffffffu;
        if (pp.counts) pp.counts[o] = used ? ps.count : 0u;
        if (pp.area) pp.area[o] = used ? atom_area(radius, probe, (float)ps.count, inv_n) : 0.0f;
    }
    if (lane == 0 && ps.n > 0) {
        atomicMax(pp.needed, (unsigned)ps.n);
        atomicMax(pp.needed + 1, (unsigned)ps.n);
        if (ps.n > (int)pp.k) atomicCAS(err_flag, 0, 1);
    }
}

// The slot rows of atoms [a0, a0 + N) of a structure with non-finite input: no partner, count 0, area NaN.
__device__ __forceinline__ void pair_blank_rows(const PairParams &pp, size_t a0, size_t N, size_t tid, size_t nth) {
    const float qn = __int_as_float(0x7fc00000);
    for (size_t i = tid; i < N * pp.k; i += nth) {
        pp.partner[a0 * pp.k + i] = 0xffffffffu;
        if (pp.counts) pp.counts[a0 * pp.k + i] = 0u;
        if (pp.area) pp.area[a0 * pp.k + i] = qn;
    }
}

// Partner enumeration of an atom without a candidate list (the cold paths): the smallest label above `prev` (any label when
// `first`) other than gi among the atoms within reach of atom `pos` in the cell rows around it -- the rows the streaming routine
// scans.  Returns false when there is none.  A superset of the partners is harmless: one that buries nothing is dropped.
template <typename AtomAcc, typename CellT>
__device__ __forceinline__ bool pair_next_scan(const Grid &g, const CellT *cell, const AtomAcc &atoms, const uint32_t *grp, int pos,
                                               const float4 ai, float reach_i, uint32_t gi, bool first, uint32_t prev, uint32_t &next) {
    const int lane = lane_id();
    const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
              cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
    const Rows rows = rows_of(g, cell, cx, cy, cz);
    bool any = false;
    uint32_t lo = 0xffffffffu;
    for (int t0 = 0; t0 < rows.total; t0 += 32) {
        const int idx = t0 + lane;
        const int j = row_lookup(rows, idx);
        if (idx < rows.total && j != pos) {
            const uint32_t gj = grp[j];
            if (gj != gi && (first || gj > prev)) {
                const float4 aj = atoms(j);
                const float dx = ai.x - aj.x, dy = ai.y - aj.y, dz = ai.z - aj.z;
                const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
                const float cut = reach_i + aj.w;
                if (d2 <= cut * cut) {
                    any = true;
                    lo = min(lo, gj);
                }
            }
        }
    }
    if (!__any_sync(kFull, any)) return false;
    next = __reduce_min_sync(kFull, lo);
    return true;
}

}  // namespace sasa
