// sasa_large.cuh -- structures too large for the fused shared-memory kernel (ribosome / capsid scale).
//
// Same algorithm as sasa_small.cuh with the cell list in global memory: bounds -> dense cell grid ->
// counting sort by cell (global atomics + three-kernel exclusive scan) -> one warp per atom gathers its
// neighbours from the cell-sorted float4 array through L1/L2 and runs the same occlusion routines.
// Replaces SpatialGrid::new / build_all_neighbor_lists (src/structures/spatial_grid.rs:28-465), which the
// reference runs serially, for N up to 2^32 / 16 atoms.
#pragma once
#include "sasa_cap.cuh"
#include "sasa_device.cuh"

namespace sasa {

struct GlobalAtoms {
    const float4 *a;
    __device__ __forceinline__ float4 operator()(int j) const { return __ldg(a + j); }
};

// Everything the pipeline keeps between its kernels.  One cudaMemsetAsync zeroes the header, the cell counters and the
// scan's tile states together (LargeWorkspace::zero_block), so all running values below are MAXIMA that start at 0.
struct LargeHeader {
    unsigned enc[8];        // maxima of order-preserving encodings: -min xyz [0..2], max xyz [3..5], r_max [6]; [7] = non-finite flag
    unsigned next_block;    // work counter of the atoms kernels: next owned work block
    unsigned tile_counter;  // scan kernel: next tile
    int err;                // error flag / statistics of runs that own their workspace (the one-structure calls): zeroed with the
    unsigned pad;           // rest of the header, copied back with the results
    unsigned long long stat[4];
    Grid grid;              // written by the count kernel (every block derives the same grid from enc[])
    int ncell;              // 0: non-finite input, nothing to evaluate
    unsigned pad2[3];
};
static_assert(sizeof(LargeHeader) % 16 == 0, "header is followed by 16-byte aligned arrays");

constexpr int kScanItems = 2048;   // cells per scan tile (256 threads x 8)
constexpr int kLBlock = 8;         // most atoms per work block of the atoms kernels (blocks are cut at cell boundaries); structures too
                                   // small to give every resident warp such a block use smaller ones (large_block_atoms)
constexpr int kLGroup = 4;         // consecutive work blocks owned by one rank in the atom-range split

struct LargeWorkspace {
    uint32_t cap_atoms = 0, cap_cells = 0;
    float4 *sorted = nullptr;
    uint32_t *orig = nullptr, *cellid = nullptr, *rank = nullptr, *cls_sorted = nullptr, *bstart = nullptr;
    float *val = nullptr;
    uint32_t *grp_sorted = nullptr;   // grouped runs: group labels in cell-sorted order, per-atom areas with the group standing alone
    float *val_iso = nullptr;
    // one allocation, zeroed by one memset per structure: header | tile states (u64) | cell counters
    unsigned char *zero_block = nullptr;
    LargeHeader *hdr = nullptr;
    unsigned long long *tiles = nullptr;
    uint32_t *cells = nullptr;
};

__device__ __forceinline__ unsigned enc_f(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// Bounds, r_max and finiteness: per-thread running values, warp shuffle, one shared-memory round per block and seven
// atomics per BLOCK (one per warp made the 4,700 warps of a 150k-atom launch queue on seven addresses: 24 us).
__global__ void __launch_bounds__(256) large_bounds_kernel(const float4 *__restrict__ at, int N, LargeHeader *h) {
    float v[7] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY, 0.0f};
    bool finite = true;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const float4 a = __ldg(at + i);
        finite = finite && isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w);
        v[0] = fmaxf(v[0], -a.x); v[1] = fmaxf(v[1], -a.y); v[2] = fmaxf(v[2], -a.z);
        v[3] = fmaxf(v[3], a.x);  v[4] = fmaxf(v[4], a.y);  v[5] = fmaxf(v[5], a.z);
        v[6] = fmaxf(v[6], a.w);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1)
#pragma unroll
        for (int k = 0; k < 7; ++k) v[k] = fmaxf(v[k], __shfl_xor_sync(kFull, v[k], d));
    __shared__ float red[8][8];
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    if (!finite) s_bad = 1;
    if ((threadIdx.x & 31) == 0)
#pragma unroll
        for (int k = 0; k < 7; ++k) red[threadIdx.x >> 5][k] = v[k];
    __syncthreads();
    if (threadIdx.x < 7) {
        float r = red[0][threadIdx.x];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmaxf(r, red[w][threadIdx.x]);
        if (!s_bad && r > -INFINITY) atomicMax(&h->enc[threadIdx.x], enc_f(r));
    } else if (threadIdx.x == 7 && s_bad) {
        atomicExch(&h->enc[7], 1u);
    }
}

// The cell grid from the reduced bounds: cell edge = half the largest pair cutoff, grown until the grid fits `cmax` cells.
__device__ __forceinline__ bool large_make_grid(const LargeHeader *h, float probe, uint32_t cmax, Grid &g, int &ncell) {
    if (h->enc[7]) {
        g = Grid{0.f, 0.f, 0.f, 0.f, 0, 0, 0, 0};
        ncell = 0;
        return false;
    }
    const float mnx = -dec_f(h->enc[0]), mny = -dec_f(h->enc[1]), mnz = -dec_f(h->enc[2]);
    const float mxx = dec_f(h->enc[3]), mxy = dec_f(h->enc[4]), mxz = dec_f(h->enc[5]), rmax = dec_f(h->enc[6]);
    const float cutoff = (2.0f * rmax + 2.0f * probe + kCutSlack) * kCellSafety;
    float c = 0.5f * cutoff;
    const float ex = fmaxf(mxx - mnx, 0.0f), ey = fmaxf(mxy - mny, 0.0f), ez = fmaxf(mxz - mnz, 0.0f);
    float fx = 1.f, fy = 1.f, fz = 1.f;
    for (int it = 0; it < 64; ++it) {
        fx = floorf(ex / c) + 1.0f; fy = floorf(ey / c) + 1.0f; fz = floorf(ez / c) + 1.0f;
        const float nc = fx * fy * fz;
        if (nc <= (float)cmax) break;
        c *= fmaxf(1.05f, cbrtf(nc / (float)cmax));
    }
    g.minx = mnx; g.miny = mny; g.minz = mnz;
    g.inv_c = 1.0f / c;
    g.nx = (int)fx; g.ny = (int)fy; g.nz = (int)fz;
    g.e = (c >= cutoff) ? 1 : 2;
    ncell = g.nx * g.ny * g.nz;
    return true;
}

// Grid (derived redundantly by every block: no one-thread kernel in between) + cell counts.
__global__ void __launch_bounds__(256) large_count_kernel(const float4 *__restrict__ at, int N, LargeHeader *h, float probe,
                                                          uint32_t cmax, int *err_flag, uint32_t *cells, uint32_t *cellid,
                                                          uint32_t *rank) {
    __shared__ Grid s_g;
    __shared__ int s_ncell;
    if (threadIdx.x == 0) {
        Grid g;
        int nc;
        const bool ok = large_make_grid(h, probe, cmax, g, nc);
        s_g = g;
        s_ncell = nc;
        if (blockIdx.x == 0) {
            h->grid = g;
            h->ncell = nc;
            if (!ok) atomicExch(err_flag, 4);
        }
    }
    __syncthreads();
    const Grid g = s_g;
    if (s_ncell == 0) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const float4 a = __ldg(at + i);
        const int c = (cell_coord(a.z, g.minz, g.inv_c, g.nz) * g.ny + cell_coord(a.y, g.miny, g.inv_c, g.ny)) * g.nx +
                      cell_coord(a.x, g.minx, g.inv_c, g.nx);
        cellid[i] = (uint32_t)c;
        rank[i] = atomicAdd(&cells[c], 1u);
    }
}

// Exclusive scan of cells[0, ncell) in ONE kernel (decoupled look-back over 2048-cell tiles; tiles are handed out by an
// atomic counter, so a tile's predecessors are always resident or finished).  cells[ncell] = N.  Tile state (u64, zeroed by
// the workspace memset): bits 62-63 = 1 aggregate known / 2 inclusive prefix known, low bits the value.
// The same pass cuts the cell-sorted order into the work blocks of the atoms kernels: bstart[b] = first cell start at or
// after atom b * blk -- emitted by the cell in front of that start -- and bstart[ceil(N / blk)] = N.  Cell starts
// are the same on every GPU (the order of atoms INSIDE a cell is not: it comes from atomics), so blocks partition the atoms
// identically on every rank of an atom-range split.
__global__ void __launch_bounds__(256) large_scan_kernel(LargeHeader *h, uint32_t *cells, unsigned long long *tiles, uint32_t *bstart,
                                                         uint32_t N, uint32_t blk) {
    const int n = h->ncell;
    __shared__ unsigned s_tile;
    __shared__ uint32_t wsum[8];
    __shared__ uint32_t s_prefix;
    constexpr unsigned long long kAgg = 1ull << 62, kIncl = 2ull << 62, kVal = (1ull << 62) - 1;
    const int ntiles = (n + kScanItems - 1) / kScanItems;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_tile = atomicAdd(&h->tile_counter, 1u);
        __syncthreads();
        const int tile = (int)s_tile;
        if (tile >= ntiles) break;
        const int t0 = tile * kScanItems + threadIdx.x * 8;
        uint32_t v[8], s = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[k] = (t0 + k < n) ? cells[t0 + k] : 0u;
            s += v[k];
        }
        uint32_t incl = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(kFull, incl, d);
            if ((threadIdx.x & 31) >= d) incl += t;
        }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
        __syncthreads();
        uint32_t run = incl - s, total = 0;
        for (int w = 0; w < 8; ++w) {
            if (w < (int)(threadIdx.x >> 5)) run += wsum[w];
            total += wsum[w];
        }
        if (threadIdx.x < 32) {
            uint32_t excl = 0;
            if (tile > 0) {
                if (threadIdx.x == 0) {
                    atomicExch(&tiles[tile], kAgg | total);
                }
                int j = tile - 1;
                for (;;) {
                    const int idx = j - (int)threadIdx.x;
                    unsigned long long st = kIncl;   // tiles in front of tile 0: inclusive prefix 0
                    if (idx >= 0) {
                        do { st = *(volatile unsigned long long *)&tiles[idx]; } while ((st >> 62) == 0ull);
                    }
                    const unsigned has_incl = __ballot_sync(kFull, (st >> 62) == 2ull);
                    const int first = has_incl ? __ffs(has_incl) - 1 : 32;   // nearest tile with a full prefix
                    uint32_t part = ((int)threadIdx.x <= first) ? (uint32_t)(st & kVal) : 0u;
#pragma unroll
                    for (int d = 16; d >= 1; d >>= 1) part += __shfl_xor_sync(kFull, part, d);
                    excl += part;
                    if (has_incl) break;
                    j -= 32;
                }
            }
            if (threadIdx.x == 0) {
                __threadfence();
                atomicExch(&tiles[tile], kIncl | (unsigned long long)(excl + total));
                s_prefix = excl;
            }
        }
        __syncthreads();
        run += s_prefix;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (t0 + k < n) {
                cells[t0 + k] = run;
                if (v[k]) {   // the next cell starts at run + v[k]: it is the first start at or after every block target in (run, run + v[k]]
                    const uint32_t nxt = run + v[k];
                    for (uint32_t b = run / blk + 1; b * blk <= nxt; ++b) bstart[b] = nxt;
                }
            }
            run += v[k];
        }
        if (tile == ntiles - 1 && threadIdx.x == 255) {
            cells[n] = N;
            bstart[0] = 0u;
            bstart[(N + blk - 1) / blk] = N;
        }
    }
}

__global__ void __launch_bounds__(256) large_scatter_kernel(const float4 *__restrict__ at, const uint32_t *__restrict__ cls,
                                                            int N, const LargeHeader *h, const uint32_t *cells,
                                                            const uint32_t *cellid, const uint32_t *rank, float4 *sorted,
                                                            uint32_t *orig, uint32_t *cls_sorted) {
    if (h->ncell == 0) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const uint32_t at_pos = cells[cellid[i]] + rank[i];
        sorted[at_pos] = __ldg(at + i);
        orig[at_pos] = (uint32_t)i;
        if (cls) cls_sorted[at_pos] = cls[i];
    }
}

// Grouped runs: the group labels into the cell-sorted order of large_scatter_kernel.
__global__ void __launch_bounds__(256) large_scatter_groups_kernel(const uint32_t *__restrict__ grp, int N, const LargeHeader *h,
                                                                   const uint32_t *cells, const uint32_t *cellid, const uint32_t *rank,
                                                                   uint32_t *grp_sorted) {
    if (h->ncell == 0) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x)
        grp_sorted[cells[cellid[i]] + rank[i]] = grp[i];
}

// Work block handed out by claim number t: rank r of n owns every n-th GROUP of kLGroup consecutive blocks, so each rank's
// share is spread evenly over the whole structure (surface and interior alike) instead of being one slab of it.
__device__ __forceinline__ unsigned large_owned_block(unsigned t, unsigned rank, unsigned n_ranks) {
    return ((t / kLGroup) * n_ranks + rank) * kLGroup + (t % kLGroup);
}

// Result of one atom (all lanes hold the same values).  Plain run: lane 0 writes the local outputs.  Atom-range split with peer
// writes: lane r writes rank r's vectors -- the local one and, over NVLink, the peers' -- so that when every rank's kernel has
// finished each rank holds the complete vectors and no all-reduce (nor its zero-fill) is needed: the exchange step of the
// split is fused into the kernel that produces the values.
__device__ __forceinline__ void large_store(const KParams &p, int lane, uint32_t gi, uint32_t oi, float *val, float area, uint32_t cnt) {
    if (lane == 0) val[oi] = area;
    if (p.n_peers > 0) {
        if (lane < p.n_peers) {
            if (p.peer_counts[lane]) p.peer_counts[lane][gi] = cnt;
            if (p.peer_atom[lane]) p.peer_atom[lane][gi] = area;
        }
    } else if (lane == 0) {
        if (p.out_counts) p.out_counts[gi] = cnt;
        if (p.out_atom) p.out_atom[gi] = area;
    }
}

// Non-finite input: the reference panics; every output of the structure is blanked instead (quiet NaN, counts 0).
__device__ __forceinline__ void large_blank_outputs(const KParams &p, int N, uint32_t a0) {
    const float qn = __int_as_float(0x7fc00000);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        if (p.out_counts) p.out_counts[a0 + i] = 0u;
        if (p.out_atom) p.out_atom[a0 + i] = qn;
    }
    // (with peer writes every rank detects the bad input itself and blanks its own vectors: out_* are the local ones)
}

// ---------------------------------------------------------------------------------------------------------------------
// Atoms kernel of the large-structure path (no id classes, no statistics flags, n_points <= 1024).
// A warp claims a work block (about kLBlock cell-sorted atoms, whole cells) and, per cell, STAGES the candidate atoms of the
// 5 x 5 x 5 cell block around it -- 25 contiguous runs of the sorted array -- into its own shared-memory strip.  Every atom
// of the cell then tests 32 staged candidates per step with conflict-free LDS.128 (the old kernel went through an index
// list and a scattered global load per candidate: 46 % long-scoreboard stalls at 25 % occupancy,
// profiles/r02a_cfg4_large_atoms.txt), compacts the neighbours into an index list and hands it to the cap-table
// occlusion: cap_atom for n_points <= 128, capm_atom (chunked table) above.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kLCap = 288;    // staged candidates per cell block (largest seen at protein density: 266)
constexpr int kLNb = 128;     // neighbours per atom on the fast path (protein lists peak around 75)

struct StagedAtoms {
    const float4 *a;
    __device__ __forceinline__ float4 operator()(int j) const { return a[j]; }
};

// Candidate rows of cell (cx, cy, cz) -> st[0, total) as atoms, padded to a multiple of 32 with far-away sentinels.
// Returns total (-1: more than kLCap) and the staged index of the first atom of the cell itself.
// The division-free row header, the predicated scan and position stores (as in tight_fill_list) and the neighbour list without
// capacity tests (large_gather) took cfg4 0.187 -> 0.185 ms, cfg5 1.648 -> 1.614 ms (run r04l).
__device__ __forceinline__ int large_stage(const Grid &g, const uint32_t *__restrict__ cells, const float4 *__restrict__ sorted,
                                           int cx, int cy, int cz, float4 *st, int &self0) {
    const int lane = lane_id();
    const int w = 2 * g.e + 1;
    // as in tight_fill_list: lane / w by multiplication (w is 3 or 5), scan with the shuffle's own predicate
    const int q = g.e == 2 ? (lane * 13) >> 6 : (lane * 11) >> 5;
    const int dy = lane - q * w - g.e, dz = q - g.e;
    const int y = cy + dy, z = cz + dz;
    int start = 0, len = 0;
    if (lane < w * w && y >= 0 && y < g.ny && z >= 0 && z < g.nz) {
        const int x0 = max(cx - g.e, 0), x1 = min(cx + g.e, g.nx - 1);
        const int base = (z * g.ny + y) * g.nx;
        start = (int)__ldg(cells + base + x0);
        len = (int)__ldg(cells + base + x1 + 1) - start;
    }
    int incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
        asm volatile("{\n .reg .pred p;\n .reg .b32 t;\n shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n @p add.s32 %0, %0, t;\n}"
                     : "+r"(incl) : "r"(d));
    const int total = __shfl_sync(kFull, incl, 31);
    // the cell's own row is lane e * w + e; its atoms sit (first atom of the cell - row start) into that row
    const int self_lane = g.e * w + g.e;
    const int row_excl = __shfl_sync(kFull, incl - len, self_lane), row_start = __shfl_sync(kFull, start, self_lane);
    self0 = row_excl + ((int)__ldg(cells + (cz * g.ny + cy) * g.nx + cx) - row_start);
    if (total > kLCap) return -1;
    const int maxlen = __reduce_max_sync(kFull, len);
    // positions first (parked in the .x slot of the destination), then one coalesced-by-row copy of the atoms themselves
    {
        uint32_t dsts = (uint32_t)__cvta_generic_to_shared(st + (incl - len));
        int v = start, left = len;
#pragma unroll 1
        for (int t = 0; t < maxlen; t += 4) {
            asm volatile("{\n .reg .pred p0, p1, p2, p3;\n"
                         " setp.gt.s32 p0, %2, 0;\n setp.gt.s32 p1, %2, 1;\n setp.gt.s32 p2, %2, 2;\n setp.gt.s32 p3, %2, 3;\n"
                         " @p0 st.shared.b32 [%0], %1;\n"
                         " @p1 st.shared.b32 [%0+16], %3;\n"
                         " @p2 st.shared.b32 [%0+32], %4;\n"
                         " @p3 st.shared.b32 [%0+48], %5;\n}"
                         :: "r"(dsts), "r"(v), "r"(left), "r"(v + 1), "r"(v + 2), "r"(v + 3) : "memory");
            dsts += 64; v += 4; left -= 4;
        }
    }
    __syncwarp();
    const int padded = (total + 31) & ~31;
#pragma unroll 2
    for (int t = lane; t < padded; t += 32) {
        float4 a = make_float4(1.0e18f, 1.0e18f, 1.0e18f, 0.0f);
        if (t < total) a = __ldg(sorted + __float_as_int(st[t].x));
        st[t] = a;
    }
    __syncwarp();
    return total;
}

// Neighbours of the atom staged at index `self` among st[0, total): indices of all atoms within r_i + r_j + 2 probe (+ slack)
// go to nb[0, k).  Membership is result-neutral (SURVEY.md 8a, A2), so the test may use contracted arithmetic.
__device__ __forceinline__ int large_gather(const float4 *st, int total, int self, const float4 ai, float reach_i, uint16_t *nb) {
    const int lane = lane_id();
    const unsigned lt = lanemask_lt();
    int k = 0;
    int w0 = 0;
#pragma unroll 1
    for (; w0 + 32 < total; w0 += 64) {
        const float4 b0 = st[w0 + lane], b1 = st[w0 + 32 + lane];
        const float dx0 = ai.x - b0.x, dy0 = ai.y - b0.y, dz0 = ai.z - b0.z;
        const float dx1 = ai.x - b1.x, dy1 = ai.y - b1.y, dz1 = ai.z - b1.z;
        const float d0 = fmaf(dx0, dx0, fmaf(dy0, dy0, dz0 * dz0)), d1 = fmaf(dx1, dx1, fmaf(dy1, dy1, dz1 * dz1));
        const float c0 = reach_i + b0.w, c1 = reach_i + b1.w;
        const bool acc0 = (d0 <= c0 * c0) & (w0 + lane != self), acc1 = (d1 <= c1 * c1) & (w0 + 32 + lane != self);
        const unsigned m0 = __ballot_sync(kFull, acc0), m1 = __ballot_sync(kFull, acc1);
        const int at0 = k + __popc(m0 & lt);
        if (acc0) nb[at0] = (uint16_t)(w0 + lane);
        k += __popc(m0);
        const int at1 = k + __popc(m1 & lt);
        if (acc1) nb[at1] = (uint16_t)(w0 + 32 + lane);
        k += __popc(m1);
    }
    if (w0 < total) {
        const float4 b0 = st[w0 + lane];
        const float dx0 = ai.x - b0.x, dy0 = ai.y - b0.y, dz0 = ai.z - b0.z;
        const float d0 = fmaf(dx0, dx0, fmaf(dy0, dy0, dz0 * dz0));
        const float c0 = reach_i + b0.w;
        const bool acc0 = (d0 <= c0 * c0) & (w0 + lane != self);
        const unsigned m0 = __ballot_sync(kFull, acc0);
        const int at0 = k + __popc(m0 & lt);
        if (acc0) nb[at0] = (uint16_t)(w0 + lane);
        k += __popc(m0);
    }
    __syncwarp();
    return k;
}

// Cold path of the cells kernel, out of line: the generic per-atom gather from global memory + the chunked point tests, or
// the list-free streaming routine for neighbourhoods denser than kNbCap.  `scratch` (the warp's staging strip) is reused.
__device__ __noinline__ float large_cold_atom(const KParams &p, const Grid &g, const float4 *__restrict__ sorted,
                                              const uint32_t *__restrict__ cells, int pos, float4 *scratch, int *streamed) {
    const GlobalAtoms atoms{sorted};
    float4 *ent = scratch;
    uint32_t *cand = reinterpret_cast<uint32_t *>(scratch + kNbCap);
    const float4 ai = atoms(pos);
    const int k = gather_candidates(p, g, atoms, cells, (const uint32_t *)nullptr, pos, ai, cand);
    if (k >= 0) {
        const float r = __fadd_rn(ai.w, p.probe);
        const int nfront = build_entries(p, atoms, ai, __fmul_rn(r, r), __fmul_rn(2.0f, r), cand, k, ent);
        return atom_fast(p, ent, k, nfront, reinterpret_cast<uint16_t *>(cand), nullptr);
    }
    *streamed += 1;
    return atom_streaming<GlobalAtoms, uint32_t, false>(p, g, atoms, cells, nullptr, pos, ent, nullptr);
}
// The same for the masked kernels: the atom streams (atom_fast keeps no per-point result) and writes its mask row.
__device__ __noinline__ float large_cold_atom_mask(const KParams &p, const Grid &g, const float4 *__restrict__ sorted,
                                                   const uint32_t *__restrict__ cells, int pos, float4 *scratch, int *streamed,
                                                   uint32_t *mrow) {
    *streamed += 1;
    return atom_streaming<GlobalAtoms, uint32_t, false, true>(p, g, GlobalAtoms{sorted}, cells, nullptr, pos, scratch, nullptr, mrow);
}

// Non-finite input of a masked run: the structure's mask rows are zeros, like its counts.
__device__ __forceinline__ void large_blank_masks(const KParams &p, const MaskParams &mp, int N, uint32_t a0) {
    mask_zero_rows(mp, p.n_points, a0, (size_t)N, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

// HAS_MASK: every atom also writes its exposed-point mask row (mp); cold atoms stream.
template <int NCHP, bool TEX, bool HAS_MASK>
__device__ __forceinline__ void large_cells_body(const KParams &p, int N, uint32_t a0, LargeHeader *h, const float4 *__restrict__ sorted,
                                                 const uint32_t *__restrict__ orig, const uint32_t *__restrict__ cells,
                                                 const uint32_t *__restrict__ bstart, float *val, uint32_t rank, uint32_t n_ranks,
                                                 uint32_t blk, const MaskParams &mp) {
    static_assert(kLCap * 16 >= kNbCap * 16 + kNbCap * 4 + 64, "the cold path's scratch must fit the staging strip");
    __shared__ __align__(16) float4 s_stage[8][kLCap];
    __shared__ __align__(16) uint32_t s_nbp[8][kLNb];
    __shared__ __align__(16) uint16_t s_nb[8][kLCap];   // room for every staged candidate: no capacity test in the gather
    __shared__ __align__(16) float4 s_ptab[NCHP == 1 ? 128 : 1];
    if (h->ncell == 0) {
        large_blank_outputs(p, N, a0);
        if (HAS_MASK) large_blank_masks(p, mp, N, a0);
        return;
    }
    // the grid and the warp index on the uniform datapath (as in tight_kernel_body).  Measured
    // (gpurun_out r04e): cfg4 (NCHP = 1) 0.1875 -> 0.1854 ms, cfg5 (NCHP = 8) 1.65 -> 2.00 ms -- the chunked cap path has no
    // vector registers to spare for the extra moves -- so only the 100-point instance takes it
    Grid g = h->grid;
    const int lane = lane_id();
    int warp = threadIdx.x >> 5;
    if (NCHP == 1) {
        g.minx = uniform_f32(g.minx); g.miny = uniform_f32(g.miny); g.minz = uniform_f32(g.minz); g.inv_c = uniform_f32(g.inv_c);
        g.nx = uniform_i32(g.nx); g.ny = uniform_i32(g.ny); g.nz = uniform_i32(g.nz); g.e = uniform_i32(g.e);
        warp = uniform_i32(warp);
    }
    float4 *const st = s_stage[warp];
    uint16_t *const nb = s_nb[warp];
    const int nbody = (int)min(p.n_points, p.n_body);
    if (NCHP == 1) {
        if (threadIdx.x < 128) {
            const bool v = threadIdx.x < p.n_points;
            s_ptab[threadIdx.x] = make_float4(v ? __ldg(p.px + threadIdx.x) : 0.f, v ? __ldg(p.py + threadIdx.x) : 0.f,
                                              v ? __ldg(p.pz + threadIdx.x) : 0.f, 0.f);
        }
        __syncthreads();
    }
    const unsigned nblocks = ((unsigned)N + blk - 1) / blk;
    const float reach0 = 2.0f * p.probe + kCutSlack;
    unsigned long long pairs = 0;
    int streamed = 0;
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(&h->next_block, 1u);
        t = __shfl_sync(kFull, t, 0);
        const unsigned b = large_owned_block(t, rank, n_ranks);
        if (b >= nblocks) break;
        int pos = (int)__ldg(bstart + b);
        const int pos_end = (int)__ldg(bstart + b + 1);
        while (pos < pos_end) {
            const float4 a_first = __ldg(sorted + pos);
            const int cx = cell_coord(a_first.x, g.minx, g.inv_c, g.nx), cy = cell_coord(a_first.y, g.miny, g.inv_c, g.ny),
                      cz = cell_coord(a_first.z, g.minz, g.inv_c, g.nz);
            const int cid = (cz * g.ny + cy) * g.nx + cx;
            const int cell_begin = (int)__ldg(cells + cid), cell_end = (int)__ldg(cells + cid + 1);
            int self0 = 0;
            int total = large_stage(g, cells, sorted, cx, cy, cz, st, self0);
            for (; pos < cell_end; ++pos) {
                int cnt = -1;
                float radius;
                uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + __ldg(orig + pos)) : nullptr;
                if (total >= 0) {
                    const int self = self0 + (pos - cell_begin);
                    const float4 ai = st[self];
                    radius = ai.w;
                    const int k = large_gather(st, total, self, ai, ai.w + reach0, nb);
                    if (k <= kLNb) {
                        if constexpr (NCHP == 1)
                            cnt = cap_atom<TEX, HAS_MASK>(p.cap, StagedAtoms{st}, ai, p.probe, nb, k, s_ptab, (int)p.n_points, nbody, p.cap_tex,
                                                          mrow);
                        else
                            cnt = capm_atom<NCHP, 9, HAS_MASK>(p.capm_in, p.capm_rg, p.capd, StagedAtoms{st}, ai, p.probe, nb, k, s_nbp[warp],
                                                               p.pts4, (int)p.n_points, nbody, mrow);
                        pairs += (unsigned)k;
                    }
                }
                if (cnt < 0) {   // too many candidates or neighbours for the strips: generic routines, then stage again
                    __syncwarp();
                    radius = __ldg(sorted + pos).w;
                    cnt = HAS_MASK ? (int)large_cold_atom_mask(p, g, sorted, cells, pos, st, &streamed, mrow)
                                   : (int)large_cold_atom(p, g, sorted, cells, pos, st, &streamed);
                    __syncwarp();
                    if (pos + 1 < cell_end) total = large_stage(g, cells, sorted, cx, cy, cz, st, self0);
                }
                large_store(p, lane, a0 + __ldg(orig + pos), __ldg(orig + pos), val, atom_area(radius, p.probe, (float)cnt, p.inv_n), (uint32_t)cnt);
                __syncwarp();
            }
        }
    }
    if (lane == 0 && p.stat) {
        if (pairs) atomicAdd(p.stat + 1, pairs);
        if (streamed) atomicAdd(p.stat + 2, (unsigned long long)streamed);
    }
}

template <int NCHP, bool TEX = false>
__global__ void __launch_bounds__(256, 4) large_cells_kernel(const KParams p, int N, uint32_t a0, LargeHeader *h,
                                                             const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                             const uint32_t *__restrict__ cells, const uint32_t *__restrict__ bstart,
                                                             float *val, uint32_t rank, uint32_t n_ranks, uint32_t blk) {
    large_cells_body<NCHP, TEX, false>(p, N, a0, h, sorted, orig, cells, bstart, val, rank, n_ranks, blk, MaskParams{});
}

template <int NCHP, bool TEX>
__global__ void __launch_bounds__(256, 4) large_cells_masks_kernel(const KParams p, const MaskParams mp, int N, uint32_t a0, LargeHeader *h,
                                                                   const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                                   const uint32_t *__restrict__ cells, const uint32_t *__restrict__ bstart,
                                                                   float *val, uint32_t blk) {
    large_cells_body<NCHP, TEX, true>(p, N, a0, h, sorted, orig, cells, bstart, val, 0, 1, blk, mp);
}

// Generic atoms kernel: id classes, statistics flags, n_points > 1024.  One warp per atom; warps claim work blocks like the
// cells kernel.  Only the atoms of blocks owned by `rank` are evaluated (n_ranks = 1: all).
// HAS_MASK: every atom also writes its exposed-point mask row (mp); atoms that would take atom_fast (id classes above 128
// points, n_points > 1024) stream.
template <bool HAS_MASK>
__device__ __forceinline__ void large_atoms_body(const KParams &p, int N, uint32_t a0, LargeHeader *h, const float4 *__restrict__ sorted,
                                                 const uint32_t *__restrict__ orig, const uint32_t *__restrict__ cls_sorted,
                                                 const uint32_t *__restrict__ cells, const uint32_t *__restrict__ bstart, float *val,
                                                 uint32_t rank, uint32_t n_ranks, uint32_t blk, const MaskParams &mp) {
    __shared__ __align__(16) float4 s_ent[8 * kNbCap];
    __shared__ uint32_t s_cand[8 * kNbCap];       // u32 candidate positions; reused as the u16 survivor queue
    static_assert(kNbCap * 2 >= kQueueCap, "survivor queue must fit the candidate list");
    __shared__ __align__(16) float4 s_ptab[128];
    if (h->ncell == 0) {
        large_blank_outputs(p, N, a0);
        if (HAS_MASK) large_blank_masks(p, mp, N, a0);
        return;
    }
    const Grid g = h->grid;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    float4 *w_ent = s_ent + warp * kNbCap;
    uint32_t *w_cand = s_cand + warp * kNbCap;
    const GlobalAtoms atoms{sorted};
    const bool force_stream = (p.flags & 2u) != 0, stats = (p.flags & 1u) != 0, use_cache = (p.flags & 4u) == 0;
    unsigned long long pairs = 0, streamed = 0;
    const float4 *s_pts = p.n_points <= 128 ? s_ptab : nullptr;
    const bool use_cap = p.cap != nullptr && p.n_points <= 128;
    const int nbody = (int)min(p.n_points, p.n_body);
    if (threadIdx.x < 128) {
        const bool v = threadIdx.x < p.n_points;
        s_ptab[threadIdx.x] = make_float4(v ? __ldg(p.px + threadIdx.x) : 0.f, v ? __ldg(p.py + threadIdx.x) : 0.f,
                                          v ? __ldg(p.pz + threadIdx.x) : 0.f, 0.f);
    }
    __syncthreads();
    const unsigned nblocks = ((unsigned)N + blk - 1) / blk;
    CandCache<uint32_t> cc;
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(&h->next_block, 1u);
        t = __shfl_sync(kFull, t, 0);
        const unsigned b = large_owned_block(t, rank, n_ranks);
        if (b >= nblocks) break;
        cc.cell = -1;
        cc.total = -1;
        const int pend = (int)__ldg(bstart + b + 1);
        for (int pos = (int)__ldg(bstart + b); pos < pend; ++pos) {
            const float4 ai = atoms(pos);
            float cnt;
            int k = -1;
            uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + orig[pos]) : nullptr;
            if (!force_stream && !stats && (!HAS_MASK || use_cap)) {
                const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
                          cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
                const int cid = (cz * g.ny + cy) * g.nx + cx;
                if (use_cache && cid != cc.cell) fill_cache(g, cells, cx, cy, cz, cid, cc);
                k = cc.total >= 0 ? gather_cached(p, atoms, cls_sorted, pos, ai, cc, w_cand)
                                  : gather_candidates(p, g, atoms, cells, cls_sorted, pos, ai, w_cand);
            }
            if (k >= 0 && use_cap) {
                cnt = (float)cap_atom<false, HAS_MASK>(p.cap, atoms, ai, p.probe, w_cand, k, s_ptab, (int)p.n_points, nbody, 0ull, mrow);
                pairs += (unsigned)k;
            } else if (k >= 0) {
                const float r = __fadd_rn(ai.w, p.probe);
                const int nfront = build_entries(p, atoms, ai, __fmul_rn(r, r), __fmul_rn(2.0f, r), w_cand, k, w_ent);
                cnt = atom_fast(p, w_ent, k, nfront, reinterpret_cast<uint16_t *>(w_cand), s_pts);
                pairs += (unsigned)k;
            } else {
                cnt = stats ? atom_streaming<GlobalAtoms, uint32_t, true, HAS_MASK>(p, g, atoms, cells, cls_sorted, pos, w_ent, p.stat, mrow)
                            : atom_streaming<GlobalAtoms, uint32_t, false, HAS_MASK>(p, g, atoms, cells, cls_sorted, pos, w_ent, p.stat, mrow);
                streamed += 1;
            }
            large_store(p, lane, a0 + orig[pos], orig[pos], val, atom_area(ai.w, p.probe, cnt, p.inv_n), (uint32_t)cnt);
            __syncwarp();
        }
    }
    if (lane == 0 && p.stat) {
        if (pairs) atomicAdd(p.stat + 1, pairs);
        if (streamed) atomicAdd(p.stat + 2, streamed);
    }
}

__global__ void __launch_bounds__(256, 2) large_atoms_kernel(const KParams p, int N, uint32_t a0, LargeHeader *h,
                                                             const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                             const uint32_t *__restrict__ cls_sorted, const uint32_t *__restrict__ cells,
                                                             const uint32_t *__restrict__ bstart, float *val, uint32_t rank,
                                                             uint32_t n_ranks, uint32_t blk) {
    large_atoms_body<false>(p, N, a0, h, sorted, orig, cls_sorted, cells, bstart, val, rank, n_ranks, blk, MaskParams{});
}

__global__ void __launch_bounds__(256, 2) large_atoms_masks_kernel(const KParams p, const MaskParams mp, int N, uint32_t a0, LargeHeader *h,
                                                                   const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                                   const uint32_t *__restrict__ cls_sorted, const uint32_t *__restrict__ cells,
                                                                   const uint32_t *__restrict__ bstart, float *val, uint32_t blk) {
    large_atoms_body<true>(p, N, a0, h, sorted, orig, cls_sorted, cells, bstart, val, 0, 1, blk, mp);
}

// One atom of the grouped atoms kernel with the list-based or streaming routines: neighbours cand[0, k) (k < 0: too many,
// streamed).  Atoms: the plain accessor (complex) or GroupAtoms (isolated).
template <class Atoms>
__device__ __forceinline__ float large_eval_atom(const KParams &p, const Grid &g, const Atoms &atoms, const uint32_t *cells,
                                                 const uint32_t *cls_sorted, int pos, const float4 ai, int k, uint32_t *cand,
                                                 float4 *ent, const float4 *s_pts, unsigned long long &streamed) {
    if (k >= 0) {
        const float r = __fadd_rn(ai.w, p.probe);
        const int nfront = build_entries(p, atoms, ai, __fmul_rn(r, r), __fmul_rn(2.0f, r), cand, k, ent);
        return atom_fast(p, ent, k, nfront, reinterpret_cast<uint16_t *>(cand), s_pts);
    }
    streamed += 1;
    return atom_streaming<Atoms, uint32_t, false>(p, g, atoms, cells, cls_sorted, pos, ent, nullptr);
}

// Atoms kernel of grouped runs: every atom in the complex and with its group standing alone.  n_points <= 128: one pass with
// cap_atom_groups over the complex neighbour list; otherwise (and for atoms with more than kNbCap neighbours) two evaluations,
// the second with the atoms of other groups hidden (GroupAtoms).  Writes val (complex areas) and val_iso.
// HAS_MASK: every atom also writes its mask row in the complex (mp) and with its group standing alone (mpi).  The cap path
// writes both from cap_atom_groups; every other atom (n_points > 128, more than kNbCap neighbours) streams both evaluations,
// because atom_fast keeps no per-point result.
// HAS_PAIRS: every atom also writes its partner slots (pp).  The cap path gets them from cap_atom_groups; every other atom with an
// other-group neighbour (or with too many neighbours to tell) enumerates its partners over the cell rows and is evaluated once more
// per partner with only its group and the partner's present (PairAtoms).
template <bool HAS_MASK, bool HAS_PAIRS = false>
__device__ __forceinline__ void large_groups_body(const KParams &p, const GroupParams &gp, int N, uint32_t a0, LargeHeader *h,
                                                  const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                  const uint32_t *__restrict__ cls_sorted, const uint32_t *__restrict__ grp_sorted,
                                                  const uint32_t *__restrict__ cells, const uint32_t *__restrict__ bstart, float *val,
                                                  float *val_iso, uint32_t blk, const MaskParams &mp, const MaskParams &mpi,
                                                  const PairParams &pp = PairParams{}) {
    static_assert(!(HAS_MASK && HAS_PAIRS), "masks and pair slots are separate instantiations");
    __shared__ __align__(16) float4 s_ent[8 * kNbCap];
    __shared__ uint32_t s_cand[8 * kNbCap];
    __shared__ __align__(16) float4 s_ptab[128];
    if (h->ncell == 0) {
        large_blank_outputs(p, N, a0);
        large_blank_outputs(iso_outputs(p, gp), N, a0);
        if (HAS_MASK) {
            large_blank_masks(p, mp, N, a0);
            large_blank_masks(p, mpi, N, a0);
        }
        if (HAS_PAIRS)
            pair_blank_rows(pp, a0, (size_t)N, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
        return;
    }
    const Grid g = h->grid;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    float4 *w_ent = s_ent + warp * kNbCap;
    uint32_t *w_cand = s_cand + warp * kNbCap;
    const GlobalAtoms atoms{sorted};
    unsigned long long pairs = 0, streamed = 0;
    const float4 *s_pts = p.n_points <= 128 ? s_ptab : nullptr;
    const bool use_cap = p.cap != nullptr && p.n_points <= 128;
    const int nbody = (int)min(p.n_points, p.n_body);
    if (threadIdx.x < 128) {
        const bool v = threadIdx.x < p.n_points;
        s_ptab[threadIdx.x] = make_float4(v ? __ldg(p.px + threadIdx.x) : 0.f, v ? __ldg(p.py + threadIdx.x) : 0.f,
                                          v ? __ldg(p.pz + threadIdx.x) : 0.f, 0.f);
    }
    __syncthreads();
    const unsigned nblocks = ((unsigned)N + blk - 1) / blk;
    CandCache<uint32_t> cc;
    for (;;) {
        unsigned b = 0;
        if (lane == 0) b = atomicAdd(&h->next_block, 1u);
        b = __shfl_sync(kFull, b, 0);
        if (b >= nblocks) break;
        cc.cell = -1;
        cc.total = -1;
        const int pend = (int)__ldg(bstart + b + 1);
        for (int pos = (int)__ldg(bstart + b); pos < pend; ++pos) {
            const float4 ai = atoms(pos);
            const uint32_t gi = __ldg(grp_sorted + pos);
            int k = -1;
            if (!HAS_MASK || use_cap) {
                const int cx = cell_coord(ai.x, g.minx, g.inv_c, g.nx), cy = cell_coord(ai.y, g.miny, g.inv_c, g.ny),
                          cz = cell_coord(ai.z, g.minz, g.inv_c, g.nz);
                const int cid = (cz * g.ny + cy) * g.nx + cx;
                if (cid != cc.cell) fill_cache(g, cells, cx, cy, cz, cid, cc);
                k = cc.total >= 0 ? gather_cached(p, atoms, cls_sorted, pos, ai, cc, w_cand)
                                  : gather_candidates(p, g, atoms, cells, cls_sorted, pos, ai, w_cand);
            }
            uint32_t *const mrow = HAS_MASK ? mask_row(mp, p.n_points, a0 + orig[pos]) : nullptr;
            uint32_t *const irow = HAS_MASK ? mask_row(mpi, p.n_points, a0 + orig[pos]) : nullptr;
            float cnt, cnt_iso;
            PairSlot ps;
            if (k >= 0) pairs += (unsigned)k;
            if (k >= 0 && use_cap) {
                int iso;
                cnt = (float)cap_atom_groups<false, HAS_MASK, HAS_PAIRS>(p.cap, atoms, ai, p.probe, w_cand, k, grp_sorted, gi, s_ptab,
                                                                         (int)p.n_points, nbody, 0ull, &iso, mrow, irow, &ps);
                cnt_iso = (float)iso;
            } else if (HAS_PAIRS) {
                bool other = true;   // an atom whose complex neighbours all share its group has no partner
                if (k >= 0) {
                    bool o = false;
                    for (int q = lane; q < k; q += 32) o |= grp_sorted[w_cand[q]] != gi;
                    other = __any_sync(kFull, o);
                }
                cnt = large_eval_atom(p, g, atoms, cells, cls_sorted, pos, ai, k, w_cand, w_ent, s_pts, streamed);
                __syncwarp();
                const GroupAtoms<true> iso_atoms{sorted, grp_sorted, gi};
                const int k2 = cc.total >= 0 ? gather_cached(p, iso_atoms, cls_sorted, pos, ai, cc, w_cand)
                                             : gather_candidates(p, g, iso_atoms, cells, cls_sorted, pos, ai, w_cand);
                cnt_iso = large_eval_atom(p, g, iso_atoms, cells, cls_sorted, pos, ai, k2, w_cand, w_ent, s_pts, streamed);
                ps = pair_empty();
                bool first = true;
                uint32_t gh = 0u;
                const float reach_i = ai.w + 2.0f * p.probe + kCutSlack;
                while (other && cnt_iso > 0.0f &&
                       pair_next_scan(g, cells, atoms, grp_sorted, pos, ai, reach_i, gi, first, gh, gh)) {
                    first = false;
                    __syncwarp();
                    const PairAtoms<true> pair_atoms{sorted, grp_sorted, gi, gh};
                    const int k3 = cc.total >= 0 ? gather_cached(p, pair_atoms, cls_sorted, pos, ai, cc, w_cand)
                                                 : gather_candidates(p, g, pair_atoms, cells, cls_sorted, pos, ai, w_cand);
                    unsigned long long pair_streamed = 0;   // (the statistics count each atom's complex and isolated evaluations only)
                    const float cp = large_eval_atom(p, g, pair_atoms, cells, cls_sorted, pos, ai, k3, w_cand, w_ent, s_pts, pair_streamed);
                    pair_take(ps, gh, (int)cnt_iso - (int)cp);
                }
            } else if (HAS_MASK) {
                cnt = atom_streaming<GlobalAtoms, uint32_t, false, true>(p, g, atoms, cells, cls_sorted, pos, w_ent, nullptr, mrow);
                __syncwarp();
                cnt_iso = atom_streaming<GroupAtoms<true>, uint32_t, false, true>(p, g, GroupAtoms<true>{sorted, grp_sorted, gi}, cells,
                                                                                  cls_sorted, pos, w_ent, nullptr, irow);
                streamed += 2;
            } else {
                cnt = large_eval_atom(p, g, atoms, cells, cls_sorted, pos, ai, k, w_cand, w_ent, s_pts, streamed);
                __syncwarp();
                const GroupAtoms<true> iso_atoms{sorted, grp_sorted, gi};
                const int k2 = cc.total >= 0 ? gather_cached(p, iso_atoms, cls_sorted, pos, ai, cc, w_cand)
                                             : gather_candidates(p, g, iso_atoms, cells, cls_sorted, pos, ai, w_cand);
                cnt_iso = large_eval_atom(p, g, iso_atoms, cells, cls_sorted, pos, ai, k2, w_cand, w_ent, s_pts, streamed);
            }
            const uint32_t oi = orig[pos];
            large_store(p, lane, a0 + oi, oi, val, atom_area(ai.w, p.probe, cnt, p.inv_n), (uint32_t)cnt);
            large_store(iso_outputs(p, gp), lane, a0 + oi, oi, val_iso, atom_area(ai.w, p.probe, cnt_iso, p.inv_n), (uint32_t)cnt_iso);
            if (HAS_PAIRS) pair_store(pp, a0 + oi, ps, ai.w, p.probe, p.inv_n, p.err_flag);
            __syncwarp();
        }
    }
    if (lane == 0 && p.stat) {
        if (pairs) atomicAdd(p.stat + 1, pairs);
        if (streamed) atomicAdd(p.stat + 2, streamed);
    }
}

__global__ void __launch_bounds__(256, 2) large_groups_kernel(const KParams p, const GroupParams gp, int N, uint32_t a0, LargeHeader *h,
                                                              const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                              const uint32_t *__restrict__ cls_sorted, const uint32_t *__restrict__ grp_sorted,
                                                              const uint32_t *__restrict__ cells, const uint32_t *__restrict__ bstart,
                                                              float *val, float *val_iso, uint32_t blk) {
    large_groups_body<false>(p, gp, N, a0, h, sorted, orig, cls_sorted, grp_sorted, cells, bstart, val, val_iso, blk, MaskParams{},
                             MaskParams{});
}

__global__ void __launch_bounds__(256, 2) large_group_pairs_kernel(const KParams p, const GroupParams gp, const PairParams pp, int N,
                                                                   uint32_t a0, LargeHeader *h, const float4 *__restrict__ sorted,
                                                                   const uint32_t *__restrict__ orig, const uint32_t *__restrict__ cls_sorted,
                                                                   const uint32_t *__restrict__ grp_sorted, const uint32_t *__restrict__ cells,
                                                                   const uint32_t *__restrict__ bstart, float *val, float *val_iso, uint32_t blk) {
    large_groups_body<false, true>(p, gp, N, a0, h, sorted, orig, cls_sorted, grp_sorted, cells, bstart, val, val_iso, blk, MaskParams{},
                                   MaskParams{}, pp);
}

__global__ void __launch_bounds__(256, 2) large_groups_masks_kernel(const KParams p, const GroupParams gp, const MaskParams mp,
                                                                    const MaskParams mpi, int N, uint32_t a0, LargeHeader *h,
                                                                    const float4 *__restrict__ sorted, const uint32_t *__restrict__ orig,
                                                                    const uint32_t *__restrict__ cls_sorted,
                                                                    const uint32_t *__restrict__ grp_sorted, const uint32_t *__restrict__ cells,
                                                                    const uint32_t *__restrict__ bstart, float *val, float *val_iso, uint32_t blk) {
    large_groups_body<true>(p, gp, N, a0, h, sorted, orig, cls_sorted, grp_sorted, cells, bstart, val, val_iso, blk, mp, mpi);
}

__device__ __forceinline__ float warp_sum_range(const float *v, uint32_t b, uint32_t e) {
    float t = 0.0f;
    for (uint32_t i = b + lane_id(); i < e; i += 32) t += v[i];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) t += __shfl_xor_sync(kFull, t, d);
    return t;
}

constexpr uint32_t kSeqSumMax = 16384;    // longer atom ranges are summed by a warp (order differs: <= 1e-6 relative)
constexpr uint32_t kSeqChainMax = 65536;  // more segments than this: polar / non-polar totals by a warp tree as well

// Level sums of one large structure, phase 1: one thread per segment, sequential f32 sum in atom order like simd_sum
// (src/utils.rs:14-22); ranges longer than kSeqSumMax atoms by a warp-shuffle tree.  Bit-identity with the reference's
// sequential sums therefore holds for segments (and structures, below) of up to kSeqSumMax atoms; beyond that the sums
// differ in the last bits (north star: 1e-4 relative).  seg_tmp (nullable): the sums again, indexed from the structure's
// first segment, for the protein totals when no segment output was requested.
__global__ void __launch_bounds__(256) large_sums_kernel(const KParams p, uint32_t sid, int N, const float *val,
                                                         const LargeHeader *h, float *seg_tmp) {
    const bool bad = h != nullptr && h->ncell == 0 && N > 0;   // h == nullptr: stand-alone reduction of finished values
    const float qn = __int_as_float(0x7fc00000);
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const int gwarp = gtid >> 5, nwarp = nth >> 5;
    if (!p.seg_be || !(p.out_seg || seg_tmp)) return;
    const uint32_t g0 = p.struct_seg_off[sid], g1 = p.struct_seg_off[sid + 1];
    for (uint32_t k = g0 + gtid; k < g1; k += nth) {
        const uint2 be = p.seg_be[k];
        if (be.y - be.x > kSeqSumMax) continue;
        float t = 0.0f;
        for (uint32_t i = be.x; i < be.y; ++i) t = __fadd_rn(t, val[i]);
        if (bad) t = qn;
        if (p.out_seg) p.out_seg[k] = t;
        if (seg_tmp) seg_tmp[k - g0] = t;
    }
    for (uint32_t k = g0 + gwarp; k < g1; k += nwarp) {
        const uint2 be = p.seg_be[k];
        if (be.y - be.x <= kSeqSumMax) continue;
        float t = warp_sum_range(val, be.x, be.y);
        if (bad) t = qn;
        if (lane_id() == 0) {
            if (p.out_seg) p.out_seg[k] = t;
            if (seg_tmp) seg_tmp[k - g0] = t;
        }
    }
}

// Phase 2 (one block of 64 threads): global_total over all atoms (src/options.rs:404) on warp 0, polar / non-polar running
// sums of the segment sums in segment order (src/options.rs:376-403) on warp 1.  seg_sums: the structure's segment sums
// from phase 1 (indexed from its first segment), or null -> recomputed here.
__global__ void __launch_bounds__(64) large_protein_kernel(const KParams p, uint32_t sid, int N, const float *val,
                                                           const LargeHeader *h, const float *seg_sums) {
    const bool bad = h != nullptr && h->ncell == 0 && N > 0;
    const float qn = __int_as_float(0x7fc00000);
    if (!p.out_protein) return;
    if (threadIdx.x < 32) {
        float t = 0.0f;
        if ((uint32_t)N <= kSeqSumMax) {
            if (threadIdx.x == 0) {
                int i = 0;
                for (; i + 8 <= N; i += 8) {   // loads ahead of the dependent additions
                    float v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[u] = val[i + u];
#pragma unroll
                    for (int u = 0; u < 8; ++u) t = __fadd_rn(t, v[u]);
                }
                for (; i < N; ++i) t = __fadd_rn(t, val[i]);
            }
        } else {
            t = warp_sum_range(val, 0, (uint32_t)N);
        }
        if (threadIdx.x == 0) {
            p.out_protein[3 * (size_t)sid + 0] = bad ? qn : t;
            if (!p.seg_be) { p.out_protein[3 * (size_t)sid + 1] = 0.0f; p.out_protein[3 * (size_t)sid + 2] = bad ? qn : t; }
        }
    } else if (p.seg_be) {
        const uint32_t g0 = p.struct_seg_off[sid], g1 = p.struct_seg_off[sid + 1];
        const uint32_t G = g1 - g0;
        float polar = 0.0f, nonpolar = 0.0f;
        if (seg_sums && G > kSeqChainMax) {
            for (uint32_t k = threadIdx.x - 32; k < G; k += 32) {
                if (p.seg_polar && p.seg_polar[g0 + k]) polar += seg_sums[k];
                else nonpolar += seg_sums[k];
            }
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                polar += __shfl_xor_sync(kFull, polar, d);
                nonpolar += __shfl_xor_sync(kFull, nonpolar, d);
            }
        } else if (threadIdx.x == 32) {
            if (seg_sums) {
                uint32_t k = 0;
                for (; k + 8 <= G; k += 8) {
                    float v[8];
                    bool f[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) { v[u] = seg_sums[k + u]; f[u] = p.seg_polar && p.seg_polar[g0 + k + u]; }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (f[u]) polar = __fadd_rn(polar, v[u]);
                        else nonpolar = __fadd_rn(nonpolar, v[u]);
                    }
                }
                for (; k < G; ++k) {
                    if (p.seg_polar && p.seg_polar[g0 + k]) polar = __fadd_rn(polar, seg_sums[k]);
                    else nonpolar = __fadd_rn(nonpolar, seg_sums[k]);
                }
            } else {
                for (uint32_t k = g0; k < g1; ++k) {
                    const uint2 be = p.seg_be[k];
                    float t = 0.0f;
                    for (uint32_t i = be.x; i < be.y; ++i) t = __fadd_rn(t, val[i]);
                    if (p.seg_polar && p.seg_polar[k]) polar = __fadd_rn(polar, t);
                    else nonpolar = __fadd_rn(nonpolar, t);
                }
            }
        }
        if (threadIdx.x == 32) {
            p.out_protein[3 * (size_t)sid + 1] = bad ? qn : polar;
            p.out_protein[3 * (size_t)sid + 2] = bad ? qn : nonpolar;
        }
    }
}

// Enqueue the level sums of one structure whose per-atom areas sit in val[0, N).  seg_tmp / seg_tmp_cap: scratch for the
// segment sums when the caller wants protein totals but no segment output (null: phase 2 recomputes them, slowly).
inline void large_enqueue_sums(int sm_count, const KParams &kp, uint32_t sid, int N, uint32_t g0, uint32_t nseg, const float *val,
                               const LargeHeader *h, float *seg_tmp, uint32_t seg_tmp_cap, cudaStream_t st, uint32_t *launches) {
    const bool want_seg = kp.seg_be && kp.out_seg, want_prot = kp.out_protein != nullptr;
    if (!want_seg && !want_prot) return;
    float *tmp = (want_prot && !want_seg && kp.seg_be && nseg <= seg_tmp_cap) ? seg_tmp : nullptr;
    if (kp.seg_be && (want_seg || tmp)) {
        const int grid = (int)std::max<uint32_t>(1, std::min<uint32_t>((uint32_t)sm_count * 2, (nseg + 255) / 256));
        large_sums_kernel<<<grid, 256, 0, st>>>(kp, sid, N, val, h, tmp);
        ++*launches;
    }
    if (want_prot) {
        // this structure's segment sums, indexed from its first segment: a slice of the segment output, or the scratch
        const float *sums = want_seg ? kp.out_seg + g0 : tmp;
        large_protein_kernel<<<1, 64, 0, st>>>(kp, sid, N, val, h, sums);
        ++*launches;
    }
}

// xyz[frame][atom][3] + radii[atom] -> float4 {x, y, z, r}; `phase` = index within the frame of element 0.
__global__ void __launch_bounds__(256) pack_frames_kernel(const float *__restrict__ xyz, const float *__restrict__ radii,
                                                          float4 *__restrict__ out, uint32_t n, uint32_t per_frame,
                                                          uint32_t phase) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t a = (phase + i) % per_frame;
    out[i] = make_float4(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], __ldg(radii + a));
}

// labels[atom] shared by every frame -> one label per atom of the chunk (grouped runs of MD frames); `phase` as above.
__global__ void __launch_bounds__(256) expand_frame_labels_kernel(const uint32_t *__restrict__ labels, uint32_t *__restrict__ out,
                                                                  uint32_t n, uint32_t per_frame, uint32_t phase) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = __ldg(labels + (phase + i) % per_frame);
}

// xyz[atom][3] + one palette index per atom -> float4 {x, y, z, palette[index]}.
__global__ void __launch_bounds__(256) pack_indexed_kernel(const float *__restrict__ xyz, const uint8_t *__restrict__ ridx,
                                                           const float *__restrict__ palette, float4 *__restrict__ out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = make_float4(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], __ldg(palette + ridx[i]));
}

inline void large_release(LargeWorkspace &w) {
    cudaFree(w.sorted); cudaFree(w.orig); cudaFree(w.cellid); cudaFree(w.rank); cudaFree(w.cls_sorted);
    cudaFree(w.bstart); cudaFree(w.val); cudaFree(w.zero_block); cudaFree(w.grp_sorted); cudaFree(w.val_iso);
    w = LargeWorkspace{};
}

inline size_t large_tile_cap(uint32_t cells) { return ((size_t)cells + kScanItems - 1) / kScanItems + 1; }

inline int large_reserve(LargeWorkspace &w, uint32_t n_atoms) {
    if (n_atoms <= w.cap_atoms) return 0;
    large_release(w);
    const uint64_t want_cells = std::min<uint64_t>(1ull << 26, std::max<uint64_t>(1ull << 20, 8ull * n_atoms));
    const size_t tiles_bytes = large_tile_cap((uint32_t)want_cells) * 8;
    if (cudaMalloc(&w.sorted, (size_t)n_atoms * 16) != cudaSuccess || cudaMalloc(&w.orig, (size_t)n_atoms * 4) != cudaSuccess ||
        cudaMalloc(&w.cellid, (size_t)n_atoms * 4) != cudaSuccess || cudaMalloc(&w.rank, (size_t)n_atoms * 4) != cudaSuccess ||
        cudaMalloc(&w.cls_sorted, (size_t)n_atoms * 4) != cudaSuccess || cudaMalloc(&w.val, (size_t)n_atoms * 4) != cudaSuccess ||
        cudaMalloc(&w.grp_sorted, (size_t)n_atoms * 4) != cudaSuccess || cudaMalloc(&w.val_iso, (size_t)n_atoms * 4) != cudaSuccess ||
        cudaMalloc(&w.bstart, ((size_t)n_atoms + 2) * 4) != cudaSuccess ||
        cudaMalloc(&w.zero_block, sizeof(LargeHeader) + tiles_bytes + (want_cells + 2) * 4) != cudaSuccess) {
        large_release(w);
        return 3;  // SASA_B200_ERR_OUT_OF_MEMORY
    }
    w.hdr = reinterpret_cast<LargeHeader *>(w.zero_block);
    w.tiles = reinterpret_cast<unsigned long long *>(w.zero_block + sizeof(LargeHeader));
    w.cells = reinterpret_cast<uint32_t *>(w.zero_block + sizeof(LargeHeader) + tiles_bytes);
    w.cap_atoms = n_atoms;
    w.cap_cells = (uint32_t)want_cells;
    return 0;
}

// Enqueue the whole pipeline for each large structure of one launch group: one memset + bounds, count, scan, scatter,
// atoms (+ the level sums when asked for).  `order` / `off` are host arrays.  range_n > 1 selects the atom-range split
// (BASELINE cfg5): the cell list is built for the whole structure, only the work blocks owned by `range_rank` are
// evaluated, and no sums are produced.  Grouped runs (gp set; no atom-range split, no flags) go through
// large_groups_kernel and produce the level sums of both value vectors.  Masked runs (mp set; no atom-range split) take the
// masked instantiations of the cells / atoms kernels; masked grouped runs (gp, mp and mpi set) large_groups_masks_kernel; pairwise
// buried area (gp and pp set) large_group_pairs_kernel.
inline int large_enqueue(int sm_count, LargeWorkspace &w, const KParams &kp, const uint32_t *order, uint32_t n_work,
                         const uint32_t *off, const uint32_t *seg_off, cudaStream_t st, uint32_t *launches,
                         uint32_t range_rank = 0, uint32_t range_n = 1, const GroupParams *gp = nullptr,
                         const MaskParams *mp = nullptr, const MaskParams *mpi = nullptr, const PairParams *pp = nullptr) {
    for (uint32_t q = 0; q < n_work; ++q) {
        const uint32_t sid = order[q];
        const uint32_t a0 = off[sid];
        const int N = (int)(off[sid + 1] - a0);
        const uint32_t nseg = seg_off ? seg_off[sid + 1] - seg_off[sid] : 0;
        if ((uint32_t)N > w.cap_atoms) return 5;
        if (N == 0) {   // nothing to evaluate; the sums of an empty structure are zeros
            if (range_n == 1) large_enqueue_sums(sm_count, kp, sid, 0, seg_off ? seg_off[sid] : 0, nseg, w.val, nullptr, nullptr, 0, st, launches);
            if (gp) large_enqueue_sums(sm_count, iso_outputs(kp, *gp), sid, 0, seg_off ? seg_off[sid] : 0, nseg, w.val_iso, nullptr, nullptr, 0, st, launches);
            continue;
        }
        const float4 *at = kp.xyzr + a0;
        const uint32_t *cls = kp.cls ? kp.cls + a0 : nullptr;
        // cell budget of this structure: at most 8 cells per atom (sparser boxes get larger cells), so that the memset
        // below and the scan stay proportional to the structure rather than to the largest one the context has seen
        const uint32_t cmax = (uint32_t)std::min<uint64_t>(w.cap_cells, std::max<uint64_t>(1u << 16, 8ull * (uint64_t)N));
        const size_t zero_bytes = sizeof(LargeHeader) + large_tile_cap(w.cap_cells) * 8 + ((size_t)cmax + 2) * 4;
        if (cudaMemsetAsync(w.zero_block, 0, zero_bytes, st) != cudaSuccess) return 2;
        const int gb = std::max(1, std::min((N + 1023) / 1024, sm_count * 2));
        const int gc = std::max(1, std::min((N + 255) / 256, sm_count * 8));
        const int gs = (int)std::max<size_t>(1, std::min<size_t>(large_tile_cap(cmax), (size_t)sm_count * 4));
        large_bounds_kernel<<<gb, 256, 0, st>>>(at, N, w.hdr);
        large_count_kernel<<<gc, 256, 0, st>>>(at, N, w.hdr, kp.probe, cmax, kp.err_flag, w.cells, w.cellid, w.rank);
        // atoms per work block: kLBlock for structures that fill the machine, fewer for small ones so that every resident warp
        // slot sees eight blocks or more (a 2,600-atom structure in blocks of 8 would occupy 7 % of the warp slots; an eighth
        // of the 1M-atom capsid in blocks of 8 is 3.3 blocks per slot: a fifth of the kernel was the wait for the 4-block warps)
        const int owned = (int)(((uint64_t)N + range_n - 1) / range_n);
        const uint32_t blk = (uint32_t)std::max(1, std::min(kLBlock, owned / (sm_count * 32 * 8)));
        large_scan_kernel<<<gs, 256, 0, st>>>(w.hdr, w.cells, w.tiles, w.bstart, (uint32_t)N, blk);
        large_scatter_kernel<<<gc, 256, 0, st>>>(at, cls, N, w.hdr, w.cells, w.cellid, w.rank, w.sorted, w.orig, w.cls_sorted);
        const bool table = (kp.n_points <= 128 && kp.cap) || (kp.n_points > 128 && kp.n_points <= 1024 && kp.capm_in);
        if (gp) {
            large_scatter_groups_kernel<<<gc, 256, 0, st>>>(gp->grp + a0, N, w.hdr, w.cells, w.cellid, w.rank, w.grp_sorted);
            const int ga = std::max(1, std::min((N + 8 * (int)blk - 1) / (8 * (int)blk), sm_count * 2));
            if (pp)
                large_group_pairs_kernel<<<ga, 256, 0, st>>>(kp, *gp, *pp, N, a0, w.hdr, w.sorted, w.orig, cls ? w.cls_sorted : nullptr,
                                                             w.grp_sorted, w.cells, w.bstart, w.val, w.val_iso, blk);
            else if (mp)
                large_groups_masks_kernel<<<ga, 256, 0, st>>>(kp, *gp, *mp, *mpi, N, a0, w.hdr, w.sorted, w.orig, cls ? w.cls_sorted : nullptr,
                                                              w.grp_sorted, w.cells, w.bstart, w.val, w.val_iso, blk);
            else
                large_groups_kernel<<<ga, 256, 0, st>>>(kp, *gp, N, a0, w.hdr, w.sorted, w.orig, cls ? w.cls_sorted : nullptr, w.grp_sorted,
                                                        w.cells, w.bstart, w.val, w.val_iso, blk);
            *launches += 1;
        } else if (!cls && (kp.flags & 3u) == 0 && table) {
            const int ga = std::max(1, std::min((owned + 8 * (int)blk - 1) / (8 * (int)blk), sm_count * 4));
            // chunked tables are always laid out for eight chunks (the fused kernel shares them): one instantiation
#define SASA_LARGE_CELLS(NCHP, TEX)                                                                                                   \
    if (mp) large_cells_masks_kernel<NCHP, TEX><<<ga, 256, 0, st>>>(kp, *mp, N, a0, w.hdr, w.sorted, w.orig, w.cells, w.bstart, w.val, blk); \
    else large_cells_kernel<NCHP, TEX><<<ga, 256, 0, st>>>(kp, N, a0, w.hdr, w.sorted, w.orig, w.cells, w.bstart, w.val, range_rank, range_n, blk)
            if (kp.n_points <= 128) {
                // Structures of at least kLargeTexAtoms atoms read the cap table through the texture path, as the fused kernel does.
                // Measured (run r05d): cfg4, 150 k atoms, 0.1846 -> 0.1776 ms; one call on one small structure gets SLOWER
                // (1,283 atoms 79 -> 92 us, 2,622 atoms 77 -> 84 us: a texture fetch has the longer latency and these runs are
                // latency-bound), 19 k / 32 k atoms 120 -> 119 / 160 -> 153 us.
                constexpr int kLargeTexAtoms = 16384;
                if (kp.cap_tex && N >= kLargeTexAtoms) {
                    SASA_LARGE_CELLS(1, true);
                } else {
                    SASA_LARGE_CELLS(1, false);
                }
            } else {
                SASA_LARGE_CELLS(8, false);
            }
#undef SASA_LARGE_CELLS
        } else {
            const int ga = std::max(1, std::min((owned + 8 * (int)blk - 1) / (8 * (int)blk), sm_count * 2));
            if (mp)
                large_atoms_masks_kernel<<<ga, 256, 0, st>>>(kp, *mp, N, a0, w.hdr, w.sorted, w.orig, cls ? w.cls_sorted : nullptr, w.cells,
                                                             w.bstart, w.val, blk);
            else
                large_atoms_kernel<<<ga, 256, 0, st>>>(kp, N, a0, w.hdr, w.sorted, w.orig, cls ? w.cls_sorted : nullptr, w.cells, w.bstart,
                                                       w.val, range_rank, range_n, blk);
        }
        *launches += 5;
        // level sums (not in the atom-range split, where the per-atom values of the other ranks are missing); the `rank`
        // array is free after the scatter and serves as scratch for the segment sums
        if (range_n == 1)
            large_enqueue_sums(sm_count, kp, sid, N, seg_off ? seg_off[sid] : 0, nseg, w.val, w.hdr, reinterpret_cast<float *>(w.rank),
                               w.cap_atoms, st, launches);
        if (gp)
            large_enqueue_sums(sm_count, iso_outputs(kp, *gp), sid, N, seg_off ? seg_off[sid] : 0, nseg, w.val_iso, w.hdr,
                               reinterpret_cast<float *>(w.rank), w.cap_atoms, st, launches);
        if (cudaGetLastError() != cudaSuccess) return 2;
    }
    return 0;
}

}  // namespace sasa
