// sasa_small.cuh -- the fused per-structure kernel: one CTA owns one structure at a time and keeps
// it entirely in shared memory from the raw float4 atoms to the residue / chain / protein sums:
//
//   bounds -> cell grid -> counting sort (shared-memory atomics) -> per-atom neighbour gather ->
//   occlusion test -> per-atom counts/areas -> segment sums
//
// replacing, for structures of up to `nmax` atoms, the reference's SpatialGrid::new +
// build_all_neighbor_lists (src/structures/spatial_grid.rs:28-465), AtomSasaKernel::with_simd
// (src/lib.rs:94-224), the driver loop (src/lib.rs:249-298) and the numeric part of process_atoms
// (src/options.rs:195-232, :292-315, :370-410).  CTAs are persistent and pull structures from an
// atomic queue ordered largest-first by the host.
//
// Two kernels share the per-structure setup and output stages defined here: the generic one below (any
// n_points, boundary statistics, forced streaming) and the tight one of sasa_tight.cuh (n_points <= 128, the
// headline configuration).  Template parameters: NT threads, MINB resident CTAs per SM, HAS_CLS (Atom.id
// equality classes present).
#pragma once
#include "sasa_cap.cuh"
#include "sasa_device.cuh"

namespace sasa {

struct SmemAtoms {
    const float4 *a;
    __device__ __forceinline__ float4 operator()(int j) const { return a[j]; }
};

// Shared-memory layout.  Everything the per-atom loops touch sits at compile-time offsets (given the warp
// count), so no base pointer has to stay in a register: point table | per-warp entries | per-warp index
// lists | per-warp cell candidate lists | reduction scratch | misc | atoms (+1 sentinel) | per-atom values |
// [isolated values] | [classes] | [groups] | original indices | cell table.
struct SmallLayout {
    size_t pts, ent, cand, list, red, misc, atom, val, val2, cls, grp, orig, cellw, total;
};

// Per-warp scratch is ONE contiguous block per warp -- entries | candidate lists | cell candidate list -- so that a single
// warp base address serves all three with immediate offsets (three separate arrays cost three re-derived addresses
// wherever the 64-register budget makes ptxas rematerialise them).
constexpr size_t kWarpOffCand = (size_t)kNbCap * 16, kWarpOffList = kWarpOffCand + (size_t)kCandSlots * 2,
                 kWarpBlockBytes = (kWarpOffList + (size_t)kListCap * 2 + 15) & ~(size_t)15;
constexpr size_t kOffWarpBlocks = 128 * 16;

__host__ __device__ constexpr size_t small_fixed_bytes(int nwarps) {
    return kOffWarpBlocks + (size_t)nwarps * kWarpBlockBytes + 32 * 8 * 4 + 64;
}

// has_grp: grouped runs add the isolated values and the group labels (8 B per atom).
__host__ __device__ constexpr SmallLayout small_layout(uint32_t nmax, uint32_t cmax, int nwarps, bool has_cls, bool has_grp = false) {
    SmallLayout L{};
    size_t o = 0;
    L.pts = o;   o += 128 * 16;
    L.ent = o;                                  // warp w: ent at L.ent + w * kWarpBlockBytes,
    L.cand = o + kWarpOffCand;                  //         cand at + kWarpOffCand, list at + kWarpOffList
    L.list = o + kWarpOffList;
    o += (size_t)nwarps * kWarpBlockBytes;
    L.red = o;   o += 32 * 8 * 4;
    L.misc = o;  o += 64;
    L.atom = o;  o += ((size_t)nmax + 1) * 16;   // +1: the far-away sentinel atom the tight kernel pads its lists with
    L.val = o;   o += (size_t)nmax * 4;
    L.val2 = o;  o += has_grp ? (size_t)nmax * 4 : 0;   // 16-byte aligned like val (seq_sum): nmax is a multiple of 16
    L.cls = o;   o += has_cls ? (size_t)nmax * 4 : 0;
    L.grp = o;   o += has_grp ? (size_t)nmax * 4 : 0;
    L.orig = o;  o += (size_t)nmax * 2;
    o = (o + 3) & ~(size_t)3;
    L.cellw = o; o += (((size_t)cmax + 2 + 1) / 2) * 4;
    L.total = (o + 15) & ~(size_t)15;
    return L;
}

// Capacities are compile-time constants of a configuration (threads, CTAs per SM, cell-table size): B200 has 228 KB of
// shared memory per SM, 1 KB of it reserved per resident CTA, and at most 227 KB per CTA.  With constant capacities
// every region of the layout sits at an immediate offset, which frees the registers a run-time layout would pin.
constexpr size_t kSmemPerSM = 228 * 1024, kSmemPerCtaMax = 227 * 1024, kSmemCtaReserve = 1024;
__host__ __device__ constexpr size_t cta_budget(int minb) {
    return kSmemPerSM / (size_t)minb - kSmemCtaReserve < kSmemPerCtaMax ? kSmemPerSM / (size_t)minb - kSmemCtaReserve : kSmemPerCtaMax;
}
// Largest atom capacity (multiple of 16, < 65520 for the u16 indices) whose layout fits the budget of the configuration.
__host__ __device__ constexpr uint32_t max_atoms(int nt, int minb, uint32_t cmax, bool has_cls, bool has_grp = false) {
    uint32_t lo = 0, hi = 65520 / 16 - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) / 2;
        if (small_layout(mid * 16, cmax, nt / 32, has_cls, has_grp).total <= cta_budget(minb)) lo = mid;
        else hi = mid - 1;
    }
    return lo * 16;
}

// min or max of 8 per-thread values over the block; result valid in every thread.
template <int NT>
__device__ __forceinline__ void block_minmax8(float (&v)[8], float *red) {
    const int lane = lane_id(), w = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1)
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = fmaxf(v[k], __shfl_xor_sync(kFull, v[k], d));
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 8; ++k) red[w * 8 + k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float r = red[k];
        for (int i = 1; i < NT / 32; ++i) r = fmaxf(r, red[i * 8 + k]);
        v[k] = r;
    }
    __syncthreads();
}

// Radius of atom i of the structure that starts at a0 in the two 12-byte forms: the frame-shared radius table (MD), or a
// palette indexed by one byte per atom (13 B/atom on the wire: what proteins with ProtOr radii need).
__device__ __forceinline__ float load_radius3(const KParams &p, uint32_t a0, int i) {
    return p.ridx ? __ldg(p.radii + __ldg(p.ridx + (size_t)a0 + (size_t)i)) : __ldg(p.radii + i);
}

// Atom i of the structure that starts at a0: packed float4, or -- MD-trajectory / indexed form -- 12-byte coordinates plus
// the radius table (what sasa_b200_batch_run_frames_host / _run_indexed_host upload; no intermediate float4 copy).
__device__ __forceinline__ float4 load_atom(const KParams &p, uint32_t a0, int i) {
    if (p.xyz3) {
        const float *q = p.xyz3 + 3 * ((size_t)a0 + (size_t)i);
        return make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), load_radius3(p, a0, i));
    }
    return __ldg(p.xyzr + a0 + i);
}

// Views of the dynamic shared memory of one CTA (see small_layout).
struct SmemView {
    float4 *ptab;       // 128 sphere points as float4 (n_points <= 128), else unused
    float4 *atom;       // cell-sorted atoms; atom[N] is the far-away sentinel of the tight kernel
    float *red;         // block reduction scratch
    int *misc;          // [0] structure claimed by the CTA, [1] work counter of the per-atom loop, [2..5] the next structure
                        // (claim_next_and_prefetch), [6..7] statistics, [8..15] the cell grid (store_grid)
    float *val;         // per-atom exposed-point count, then area, by ORIGINAL index
    uint16_t *cellid, *rank;   // alias val during the counting sort
    uint32_t *cls;      // id classes in sorted order (HAS_CLS)
    float *val2;        // grouped runs: per-atom values with the atom's group standing alone, by ORIGINAL index
    uint32_t *grp;      // grouped runs: group labels in sorted order
    uint16_t *orig;     // sorted position -> original index
    uint32_t *cellw;    // cell table as u32 words (pairs of u16 counters) during counting
    uint16_t *cell;     // cell table: start position of every cell, cell[ncell] = N
};

template <int NT, bool HAS_CLS, uint32_t NMAX, uint32_t CMAX, bool HAS_GRP = false>
__device__ __forceinline__ SmemView smem_view(unsigned char *smem) {
    constexpr int NW = NT / 32;
    constexpr SmallLayout L = small_layout(NMAX, CMAX, NW, HAS_CLS, HAS_GRP);
    SmemView v;
    v.ptab = reinterpret_cast<float4 *>(smem);
    v.atom = reinterpret_cast<float4 *>(smem + small_fixed_bytes(NW));
    v.red = reinterpret_cast<float *>(smem + L.red);
    v.misc = reinterpret_cast<int *>(smem + L.misc);
    v.val = reinterpret_cast<float *>(smem + L.val);
    v.cellid = reinterpret_cast<uint16_t *>(smem + L.val);
    v.rank = v.cellid + NMAX;
    v.cls = HAS_CLS ? reinterpret_cast<uint32_t *>(smem + L.cls) : nullptr;
    v.val2 = HAS_GRP ? reinterpret_cast<float *>(smem + L.val2) : nullptr;
    v.grp = HAS_GRP ? reinterpret_cast<uint32_t *>(smem + L.grp) : nullptr;
    v.orig = reinterpret_cast<uint16_t *>(smem + L.orig);
    v.cellw = reinterpret_cast<uint32_t *>(smem + L.cellw);
    v.cell = reinterpret_cast<uint16_t *>(smem + L.cellw);
    return v;
}

// The whole point set as a float4 table when it fits (n_points <= 128).
__device__ __forceinline__ void stage_points(const KParams &p, float4 *ptab) {
    if (threadIdx.x < 128) {
        const int t = threadIdx.x;
        const bool v = (uint32_t)t < p.n_points;
        ptab[t] = make_float4(v ? __ldg(p.px + t) : 0.f, v ? __ldg(p.py + t) : 0.f, v ? __ldg(p.pz + t) : 0.f, 0.f);
    }
}

// The structure's cell grid parked in misc[8..15].  Nothing reads it back any more; the stores stay because dropping them
// changes the SASS of every fused kernel, which wants a measurement of its own.
__device__ __forceinline__ void store_grid(int *misc, const Grid &g) {
    misc[8] = __float_as_int(g.minx); misc[9] = __float_as_int(g.miny); misc[10] = __float_as_int(g.minz);
    misc[11] = __float_as_int(g.inv_c); misc[12] = g.nx; misc[13] = g.ny; misc[14] = g.nz; misc[15] = g.e;
}

// One structure from raw float4 atoms to a cell-sorted shared-memory copy: bounds / r_max / finiteness (one fused
// block reduction), the cell grid, a counting sort with shared-memory atomics and the exclusive scan of the
// cell counts.  Replaces SpatialGrid::new (src/structures/spatial_grid.rs:28-106).  Returns false when the
// structure holds a non-finite value (outputs are then NaN-filled and the error flag raised).
template <int NT, bool HAS_CLS, uint32_t CMAX, bool HAS_GRP = false>
__device__ __forceinline__ bool structure_setup(const KParams &p, const SmemView &V, uint32_t sid, uint32_t a0, int N,
                                                Grid &g, int &ncell, const GroupParams &gp = GroupParams{}) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // ---- bounds, r_max, finiteness (maxima of {-min, max, r, bad}) -------------------------------------
    float red8[8] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY, 0.0f, 0.0f};
    for (int i = tid; i < N; i += NT) {
        const float4 a = load_atom(p, a0, i);
        const bool fin = isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w);
        red8[0] = fmaxf(red8[0], -a.x); red8[1] = fmaxf(red8[1], -a.y); red8[2] = fmaxf(red8[2], -a.z);
        red8[3] = fmaxf(red8[3], a.x);  red8[4] = fmaxf(red8[4], a.y);  red8[5] = fmaxf(red8[5], a.z);
        red8[6] = fmaxf(red8[6], a.w);
        if (!fin) red8[7] = 1.0f;
    }
    block_minmax8<NT>(red8, V.red);
    const float mnx = -red8[0], mny = -red8[1], mnz = -red8[2], mxx = red8[3], mxy = red8[4], mxz = red8[5],
                rmax = red8[6];
    if (red8[7] != 0.0f) {
        // the reference panics on non-finite input; report it and emit NaN for this structure
        if (tid == 0) atomicExch(p.err_flag, 4);
        const float qn = __int_as_float(0x7fc00000);
        for (int i = tid; i < N; i += NT) {
            if (p.out_counts) p.out_counts[a0 + i] = 0u;
            if (p.out_atom) p.out_atom[a0 + i] = qn;
        }
        if (p.seg_be && p.out_seg)
            for (uint32_t k = p.struct_seg_off[sid] + tid; k < p.struct_seg_off[sid + 1]; k += NT) p.out_seg[k] = qn;
        if (p.out_protein && tid < 3) p.out_protein[3 * (size_t)sid + tid] = qn;
        if (HAS_GRP) {   // grouped run: the isolated outputs alike
            for (int i = tid; i < N; i += NT) {
                if (gp.counts) gp.counts[a0 + i] = 0u;
                if (gp.atom) gp.atom[a0 + i] = qn;
            }
            if (p.seg_be && gp.seg)
                for (uint32_t k = p.struct_seg_off[sid] + tid; k < p.struct_seg_off[sid + 1]; k += NT) gp.seg[k] = qn;
            if (gp.protein && tid < 3) gp.protein[3 * (size_t)sid + tid] = qn;
        }
        return false;
    }
    // ---- cell grid: cell edge >= half the largest possible pair cutoff, grown until it fits ----------------
    {
        const float cutoff = (2.0f * rmax + 2.0f * p.probe + kCutSlack) * kCellSafety;
        float c = 0.5f * cutoff;
        const float ex = fmaxf(mxx - mnx, 0.0f), ey = fmaxf(mxy - mny, 0.0f), ez = fmaxf(mxz - mnz, 0.0f);
        float fx, fy, fz;
        for (int it = 0; it < 64; ++it) {
            fx = floorf(ex / c) + 1.0f; fy = floorf(ey / c) + 1.0f; fz = floorf(ez / c) + 1.0f;
            const float nc = fx * fy * fz;
            if (nc <= (float)CMAX) break;
            c *= fmaxf(1.05f, cbrtf(nc / (float)CMAX));
        }
        g.minx = mnx; g.miny = mny; g.minz = mnz;
        g.inv_c = 1.0f / c;
        g.nx = (int)fx; g.ny = (int)fy; g.nz = (int)fz;
        g.e = (c >= cutoff) ? 1 : 2;
    }
    ncell = g.nx * g.ny * g.nz;
    // ---- counting sort into cells ---------------------------------------------------------------------
    for (int i = tid; i < (ncell + 2 + 1) / 2; i += NT) V.cellw[i] = 0u;
    __syncthreads();
    for (int i = tid; i < N; i += NT) {
        const float4 a = load_atom(p, a0, i);
        const int c = (cell_coord(a.z, g.minz, g.inv_c, g.nz) * g.ny + cell_coord(a.y, g.miny, g.inv_c, g.ny)) * g.nx +
                      cell_coord(a.x, g.minx, g.inv_c, g.nx);
        const uint32_t old = atomicAdd(&V.cellw[c >> 1], (c & 1) ? 0x10000u : 1u);
        V.cellid[i] = (uint16_t)c;
        V.rank[i] = (uint16_t)((c & 1) ? (old >> 16) : (old & 0xffffu));
    }
    __syncthreads();
    {   // exclusive scan of the u16 counts -> cell starts; cell[ncell] = N
        const int per = (ncell + NT - 1) / NT;
        const int b = min(tid * per, ncell), e = min(b + per, ncell);
        int sum = 0;
        for (int c = b; c < e; ++c) sum += V.cell[c];
        int incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += t;
        }
        int *s_wsum = reinterpret_cast<int *>(V.red);
        if (lane == 31) s_wsum[warp] = incl;
        __syncthreads();
        int base = 0;
        for (int i = 0; i < warp; ++i) base += s_wsum[i];
        int run = base + incl - sum;
        for (int c = b; c < e; ++c) {
            const int cnt = V.cell[c];
            V.cell[c] = (uint16_t)run;
            run += cnt;
        }
        if (tid == 0) V.cell[ncell] = (uint16_t)N;
        __syncthreads();
    }
    for (int i = tid; i < N; i += NT) {
        const int at = (int)V.cell[V.cellid[i]] + (int)V.rank[i];
        V.atom[at] = load_atom(p, a0, i);
        V.orig[at] = (uint16_t)i;
        if (HAS_CLS) V.cls[at] = p.cls[a0 + i];
        if (HAS_GRP) V.grp[at] = gp.grp[a0 + i];
    }
    if (tid == 0) {
        V.misc[1] = 0;
        V.misc[6] = 0;   // neighbour pairs / streamed atoms of this structure (tight kernel)
        V.misc[7] = 0;
        store_grid(V.misc, g);
        V.atom[N] = make_float4(1.0e18f, 1.0e18f, 1.0e18f, 0.0f);   // sentinel: farther than any cutoff from everything
    }
    __syncthreads();   // cellid / rank are dead from here on: val may be written
    return true;
}

// Sequential f32 sum of v[0, n) in index order (simd_sum, src/utils.rs:14-22) by ONE thread, starting from `t`.  The
// additions form a dependent chain (4 cycles each) that no reordering may shorten, but the loads need not sit on it:
// sixteen values are fetched ahead of every sixteen additions (a plain `t += v[i]` loop costs a shared-memory round
// trip per element: 190 us per 5,000-atom structure, the barrier stall of profiles/r02a_cfg3_tight.txt).
__device__ __forceinline__ float seq_sum(const float *v, int n, float t) {
    int i = 0;
    // v is 16-byte aligned (SmallLayout: the atom region in front of it is a multiple of 16 bytes)
    const float4 *v4 = reinterpret_cast<const float4 *>(v);
    for (; i + 16 <= n; i += 16) {
        const float4 a = v4[(i >> 2) + 0], b = v4[(i >> 2) + 1], c = v4[(i >> 2) + 2], d = v4[(i >> 2) + 3];
        t = __fadd_rn(t, a.x); t = __fadd_rn(t, a.y); t = __fadd_rn(t, a.z); t = __fadd_rn(t, a.w);
        t = __fadd_rn(t, b.x); t = __fadd_rn(t, b.y); t = __fadd_rn(t, b.z); t = __fadd_rn(t, b.w);
        t = __fadd_rn(t, c.x); t = __fadd_rn(t, c.y); t = __fadd_rn(t, c.z); t = __fadd_rn(t, c.w);
        t = __fadd_rn(t, d.x); t = __fadd_rn(t, d.y); t = __fadd_rn(t, d.z); t = __fadd_rn(t, d.w);
    }
    for (; i < n; ++i) t = __fadd_rn(t, v[i]);
    return t;
}

// Per-atom counts -> areas (coalesced stores), then the level sums in the reference's order: replaces the
// numeric part of process_atoms (src/options.rs:195-232, :292-315, :370-410) and simd_sum (src/utils.rs:14-22).
// Every sum keeps the reference's order (bit-identical results) but only the two chains that ARE sequential run on a
// single thread: residue / chain sums are one thread each; the ProteinLevel polar / non-polar totals -- running sums of
// the residue sums in residue order (src/options.rs:376-403) -- take the residue sums from a shared-memory scratch
// (`scratch`: the per-warp blocks, idle between structures) instead of recomputing them with dependent loads; the global
// total (src/options.rs:404) is seq_sum over all atoms.  The two chains run concurrently on threads 0 and 32.
template <int NT>
__device__ __forceinline__ void structure_outputs(const KParams &p, const SmemView &V, uint32_t sid, uint32_t a0, int N,
                                                  unsigned char *scratch) {
    const int tid = threadIdx.x;
    constexpr int kScratch = (int)(((size_t)(NT / 32) * kWarpBlockBytes / 5) & ~(size_t)3);   // 4 B sum + 1 B polar flag each
    float *const s_sum = reinterpret_cast<float *>(scratch);
    uint8_t *const s_pol = scratch + (size_t)kScratch * 4;
    for (int i = tid; i < N; i += NT) {
        const float cnt = V.val[i];
        const float area = atom_area(p.xyz3 ? load_radius3(p, a0, i) : __ldg(p.xyzr + a0 + i).w, p.probe, cnt, p.inv_n);
        if (p.out_counts) p.out_counts[a0 + i] = (uint32_t)cnt;
        if (p.out_atom) p.out_atom[a0 + i] = area;
        V.val[i] = area;
    }
    __syncthreads();
    if (p.seg_be) {
        const uint32_t g0 = p.struct_seg_off[sid], g1 = p.struct_seg_off[sid + 1];
        if (p.out_protein) {
            float polar = 0.0f, nonpolar = 0.0f;
            for (uint32_t base = g0; base < g1; base += (uint32_t)kScratch) {
                const uint32_t gend = min(g1, base + (uint32_t)kScratch);
                // sequential f32 sum in atom order, one thread per segment
                for (uint32_t k = base + tid; k < gend; k += NT) {
                    const uint2 be = p.seg_be[k];
                    float t = 0.0f;
                    for (uint32_t i = be.x; i < be.y && i < (uint32_t)N; ++i) t = __fadd_rn(t, V.val[i]);
                    if (p.out_seg) p.out_seg[k] = t;
                    s_sum[k - base] = t;
                    s_pol[k - base] = p.seg_polar ? p.seg_polar[k] : (uint8_t)0;
                }
                __syncthreads();
                if (tid == 32 % NT) {
                    const int n = (int)(gend - base);
                    int k = 0;
                    for (; k + 8 <= n; k += 8) {   // loads ahead of the dependent additions
                        float t[8];
                        uint8_t f[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) { t[u] = s_sum[k + u]; f[u] = s_pol[k + u]; }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            if (f[u]) polar = __fadd_rn(polar, t[u]);
                            else nonpolar = __fadd_rn(nonpolar, t[u]);
                        }
                    }
                    for (; k < n; ++k) {
                        if (s_pol[k]) polar = __fadd_rn(polar, s_sum[k]);
                        else nonpolar = __fadd_rn(nonpolar, s_sum[k]);
                    }
                }
                if (gend < g1) __syncthreads();   // the scratch is refilled by the next round
            }
            if (tid == 32 % NT) {
                p.out_protein[3 * (size_t)sid + 1] = polar;
                p.out_protein[3 * (size_t)sid + 2] = nonpolar;
            }
        } else if (p.out_seg) {
            for (uint32_t k = g0 + tid; k < g1; k += NT) {
                const uint2 be = p.seg_be[k];
                float t = 0.0f;
                for (uint32_t i = be.x; i < be.y && i < (uint32_t)N; ++i) t = __fadd_rn(t, V.val[i]);
                p.out_seg[k] = t;
            }
        }
    }
    if (p.out_protein && tid == 0) {
        const float t = seq_sum(V.val, N, 0.0f);   // global_total = simd_sum(atom_sasa), src/options.rs:404
        p.out_protein[3 * (size_t)sid + 0] = t;
        if (!p.seg_be) { p.out_protein[3 * (size_t)sid + 1] = 0.0f; p.out_protein[3 * (size_t)sid + 2] = t; }
    }
}

// Gate of the single-launch host pipeline: queue position w may be worked on once the copy stream has raised *p.ready to
// p.need[w], the number of input chunks its structure needs (the counter is copied after the data, in stream order).  One thread
// polls with an acquire load at system scope; the caller's barrier publishes the result to the CTA.  The wait is bounded: a
// copy that never arrives raises the error flag instead of hanging the device.
__device__ __forceinline__ void wait_ready(const KParams &p, uint32_t w) {
    if (!p.ready) return;
    const uint32_t need = __ldg(p.need + w);
    const long long t0 = clock64();
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p.ready) : "memory");
        if (v >= need) return;
        __nanosleep(200);
        if (clock64() - t0 > (1ll << 36)) {   // about half a minute: far beyond any copy, short of a driver time-out
            atomicExch(p.err_flag, 2);
            return;
        }
    }
}

// Claim the next structure of this launch for the CTA (largest-first order prepared by the host).
__device__ __forceinline__ bool claim_structure(const KParams &p, int *misc, uint32_t &sid, uint32_t &a0, int &N) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t w = atomicAdd(p.work_counter, 1u);
        misc[0] = (int)w;
        if (w < p.n_work) wait_ready(p, w);
    }
    __syncthreads();
    const uint32_t w = (uint32_t)misc[0];
    if (w >= p.n_work) return false;
    sid = p.order[w];
    a0 = p.struct_off[sid];
    N = (int)(p.struct_off[sid + 1] - a0);
    return true;
}

// The same with the claim taken early: warp 0 of the CTA calls claim_next_and_prefetch while the other warps already
// work on the current structure -- it takes the next queue position, reads that structure's range into misc[2..5] and
// prefetches its atoms into L2, so that
// neither the atomic's round trip nor the first touch of the input sits on the CTA's critical path.
__device__ __forceinline__ void claim_next_and_prefetch(const KParams &p, int *misc) {
    const int lane = lane_id();
    uint32_t na0 = 0, nN = 0;
    if (lane == 0) {
        const uint32_t w = atomicAdd(p.work_counter, 1u);
        misc[0] = (int)w;   // claim_prefetched waits for this queue position's data (wait_ready)
        uint32_t nsid = 0;
        if (w < p.n_work) {
            nsid = p.order[w];
            na0 = p.struct_off[nsid];
            nN = p.struct_off[nsid + 1] - na0;
        }
        misc[2] = (int)(w < p.n_work);
        misc[3] = (int)nsid;
        misc[4] = (int)na0;
        misc[5] = (int)nN;
    }
    na0 = __shfl_sync(kFull, na0, 0);
    nN = __shfl_sync(kFull, nN, 0);
    const char *base = p.xyz3 ? reinterpret_cast<const char *>(p.xyz3 + 3 * (size_t)na0) : reinterpret_cast<const char *>(p.xyzr + na0);
    const size_t bytes = (size_t)nN * (p.xyz3 ? 12 : 16);
    for (size_t o = (size_t)lane * 128; o < bytes; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + o));
}

__device__ __forceinline__ bool claim_prefetched(const KParams &p, int *misc, uint32_t &sid, uint32_t &a0, int &N) {
    __syncthreads();
    if (p.ready) {   // (uniform) the prefetch may have run ahead of the copy; the loads of the setup must not
        if (threadIdx.x == 0 && misc[2]) wait_ready(p, (uint32_t)misc[0]);
        __syncthreads();
    }
    const int have = misc[2];
    sid = (uint32_t)misc[3];
    a0 = (uint32_t)misc[4];
    N = misc[5];
    return have != 0;
}

// ---------------------------------------------------------------------------------------------------------
// Generic fused kernel: any n_points (128-point chunks), boundary statistics, forced streaming.
// HAS_MASK: every atom also writes its exposed-point mask row (mp); atoms that would take atom_fast (n_points > 1024) stream.
// ---------------------------------------------------------------------------------------------------------
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX, bool HAS_MASK>
__device__ __forceinline__ void small_kernel_body(const KParams &p, const MaskParams &mp) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr uint32_t NMAX = max_atoms(NT, MINB, CMAX, HAS_CLS);
    const SmemView V = smem_view<NT, HAS_CLS, NMAX, CMAX>(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char *const wblock = smem + kOffWarpBlocks + (size_t)warp * kWarpBlockBytes;
    float4 *const w_ent = reinterpret_cast<float4 *>(wblock);
    uint16_t *const w_cand = reinterpret_cast<uint16_t *>(wblock + kWarpOffCand);
    const bool force_stream = (p.flags & 2u) != 0, stats = (p.flags & 1u) != 0;
    const float4 *s_pts = p.n_points <= 128 ? V.ptab : nullptr;
    stage_points(p, V.ptab);

    uint32_t sid, a0;
    int N;
    while (claim_structure(p, V.misc, sid, a0, N)) {
        Grid g;
        int ncell;
        if (!structure_setup<NT, HAS_CLS, CMAX>(p, V, sid, a0, N, g, ncell)) {
            if (HAS_MASK) mask_zero_rows(mp, p.n_points, a0, (size_t)N, threadIdx.x, NT);
            continue;
        }

        // ---- per-atom work: warps pull runs of consecutive cell-sorted atoms from a shared counter ----------
        const SmemAtoms atoms{V.atom};
        unsigned pairs = 0, streamed = 0;
        constexpr int kFetch = 4;   // atoms per claim
        CandCache<uint16_t> cc;
        for (;;) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&V.misc[1], kFetch);
            base = __shfl_sync(kFull, base, 0);
            if (base >= N) break;
            int cell_end = -1;   // atoms [.., cell_end) share the cached candidate list
            cc.total = -1;
            const int pend = min(base + kFetch, N);
            for (int pos = base; pos < pend; ++pos) {
                const float4 ai = V.atom[pos];
                int cnt;
                int k = -1;
                uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + V.orig[pos]) : nullptr;
                if (!force_stream && !stats && (!HAS_MASK || p.capm_in)) {
                    if (pos >= cell_end) {
                        const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
                                  cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
                        const int cid = (cz * g.ny + cy) * g.nx + cx;
                        cell_end = (int)V.cell[cid + 1];
                        fill_cache(g, V.cell, cx, cy, cz, cid, cc);
                    }
                    k = cc.total >= 0 ? gather_cached(p, atoms, V.cls, pos, ai, cc, w_cand)
                                      : gather_candidates(p, g, atoms, V.cell, V.cls, pos, ai, w_cand);
                }
                if (k >= 0 && p.capm_in) {
                    // 128 < n_points <= 1024: the chunked cap table (sasa_cap.cuh) on the shared-memory atoms; the entry strip
                    // serves as the packed (bin, index) scratch
                    cnt = capm_atom<8, 13, HAS_MASK>(p.capm_in, p.capm_rg, p.capd, atoms, ai, p.probe, w_cand, k, reinterpret_cast<uint32_t *>(w_ent),
                                                     p.pts4, (int)p.n_points, (int)min(p.n_points, p.n_body), mrow);
                    pairs += (unsigned)k;
                } else if (k >= 0) {
                    const float r = __fadd_rn(ai.w, p.probe);
                    const int nfront = build_entries(p, atoms, ai, __fmul_rn(r, r), __fmul_rn(2.0f, r), w_cand, k, w_ent);
                    cnt = (int)atom_fast(p, w_ent, k, nfront, w_cand, s_pts);
                    pairs += (unsigned)k;
                } else {
                    cnt = (int)(stats ? atom_streaming<SmemAtoms, uint16_t, true, HAS_MASK>(p, g, atoms, V.cell, V.cls, pos, w_ent, p.stat, mrow)
                                      : atom_streaming<SmemAtoms, uint16_t, false, HAS_MASK>(p, g, atoms, V.cell, V.cls, pos, w_ent, p.stat, mrow));
                    streamed += 1;
                }
                if (lane == 0) V.val[V.orig[pos]] = (float)cnt;
                __syncwarp();
            }
        }
        if (lane == 0 && p.stat) {
            if (pairs) atomicAdd(p.stat + 1, (unsigned long long)pairs);
            if (streamed) atomicAdd(p.stat + 2, (unsigned long long)streamed);
        }
        __syncthreads();
        structure_outputs<NT>(p, V, sid, a0, N, smem + kOffWarpBlocks);
    }
}

template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_small_kernel(const KParams p) {
    small_kernel_body<NT, MINB, HAS_CLS, CMAX, false>(p, MaskParams{});
}

// Exposed-point masks: the plain run's outputs plus every atom's mask row (n_points > 128, statistics, forced streaming).
template <int NT, int MINB, bool HAS_CLS, uint32_t CMAX>
__global__ void __launch_bounds__(NT, MINB) sasa_small_masks_kernel(const KParams p, const MaskParams mp) {
    small_kernel_body<NT, MINB, HAS_CLS, CMAX, true>(p, mp);
}

}  // namespace sasa
