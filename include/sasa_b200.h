/*
 * sasa_b200.h -- C ABI of the B200 (sm_100a) Shrake-Rupley engine.
 *
 * This is the drop-in boundary for ONE path of maxall41/RustSASA (crate rust-sasa 0.9.2):
 *
 *     pub fn calculate_sasa_internal(atoms: &[Atom], probe_radius: f32,
 *                                    n_points: usize, threads: isize) -> Vec<f32>
 *                                                        (reference src/lib.rs:249-298)
 *
 * together with the neighbour build in front of it (src/lib.rs:69-84,
 * src/structures/spatial_grid.rs:28-465) and the numeric part of the level sums behind
 * it (SASAProcessor::process_atoms, src/options.rs:142-149, :195-232, :292-315,
 * :370-410; simd_sum, src/utils.rs:14-22).  Everything else in the crate (pdbtbx
 * parsing, radius lookup, result structs, CLI) stays host-side and unchanged; see
 * INTEGRATION.md for the Rust `extern "C"` block and the replacement body of
 * calculate_sasa_internal that binds these symbols.
 *
 * Conventions
 *   - plain pointers and sizes only; no CUDA or torch types appear in any signature
 *     (streams are passed as void* holding a cudaStream_t -- including the special handles cudaStreamLegacy (0x1)
 *     and cudaStreamPerThread (0x2) -- and NULL = the context's own non-blocking stream, which is NOT ordered with
 *     the caller's default stream: synchronise with sasa_b200_batch_sync);
 *   - every call returns a sasa_b200_status; sasa_b200_last_error() gives the text;
 *     nothing in the library aborts the process and there is NO CPU fallback: if no
 *     CUDA device is present sasa_b200_create() fails with SASA_B200_ERR_CUDA;
 *   - atoms travel as packed float4 {x, y, z, radius} (16 B/atom) instead of the 40-byte
 *     rust `Atom` (src/structures/atomic.rs:13-24) -- `Option<isize>` has no stable C
 *     layout and parent_id is never read by the path;
 *   - `Atom.id` only matters through equality (atoms with equal ids never occlude each
 *     other, src/lib.rs:124-126, spatial_grid.rs:313-316), so it travels as an optional
 *     u32 class array `id_class`; NULL means "all ids distinct";
 *   - a batch is CSR: struct_off[S+1] atom offsets; output segments (residues or chains)
 *     are [begin, end) atom ranges RELATIVE to their structure's first atom, grouped per
 *     structure by struct_seg_off[S+1].  Ranges may be empty or repeated (the reference's
 *     HashMap::insert last-writer-wins behaviour is expressed by repeating a range);
 *   - `simd_lanes` in {4, 8, 16} selects which pulp build of the reference is mirrored
 *     for the scalar-tail rule (src/lib.rs:104-106, :162-218): points
 *     [0, lanes*floor(n/lanes)) use the fma-nested dot and `<`, the rest the unfused dot
 *     and `<=`.  8 = AVX2 (x86-64-v3), 16 = AVX-512, 4 = NEON.  For n_points = 100 and
 *     960 the 8- and 16-lane splits coincide.
 */
#ifndef SASA_B200_H
#define SASA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SASA_B200_ABI_VERSION 1

#if defined(__GNUC__)
#define SASA_B200_API __attribute__((visibility("default")))
#else
#define SASA_B200_API
#endif

typedef enum sasa_b200_status {
    SASA_B200_OK = 0,
    SASA_B200_ERR_INVALID_ARGUMENT = 1,
    SASA_B200_ERR_CUDA = 2,        /* CUDA runtime / driver failure, or no device */
    SASA_B200_ERR_OUT_OF_MEMORY = 3,
    SASA_B200_ERR_NON_FINITE = 4,  /* NaN/inf coordinate or radius (the reference panics here) */
    SASA_B200_ERR_UNSUPPORTED = 5
} sasa_b200_status;

typedef struct sasa_b200_ctx sasa_b200_ctx;     /* one per (process, device); shareable between threads */
typedef struct sasa_b200_batch sasa_b200_batch; /* topology of a batch: reusable across runs   */
typedef struct sasa_b200_job sasa_b200_job;     /* one host-buffer run in flight (submit .. wait) */

/* Numeric parameters of one run: the arguments of calculate_sasa_internal
 * (src/lib.rs:249-254) plus the lane count of the mirrored reference build. */
typedef struct sasa_b200_params {
    float probe_radius;  /* default 1.4   (src/options.rs:500) */
    uint32_t n_points;   /* default 100   (src/options.rs:501) */
    uint32_t simd_lanes; /* 4, 8 or 16; 0 = 8 */
    int32_t threads;     /* accepted for signature compatibility, ignored on the GPU path */
    uint32_t flags;      /* SASA_B200_FLAG_* */
} sasa_b200_params;

#define SASA_B200_FLAG_NONE 0u
/* Count "boundary" sphere points: points whose test against some neighbour j lies within
 * boundary_tol = 1e-5 A^2 of that sphere, |d^2 - R_j^2| = |2 R_i (dot - limit)| <= tol
 * (SURVEY.md 8b numerics contract).  Uses the slower streaming kernel. */
#define SASA_B200_FLAG_BOUNDARY_STATS 1u
/* Force the streaming (list-free) kernel everywhere; a cross-check for the fast path. */
#define SASA_B200_FLAG_FORCE_STREAMING 2u

/* Output pointers; every one may be NULL (= not wanted).  Sizes refer to the batch. */
typedef struct sasa_b200_outputs {
    uint32_t *counts;   /* [n_atoms]   exposed sphere points per atom (exact integers)         */
    float *atom_sasa;   /* [n_atoms]   AtomLevel: ((4*pi*R^2) * count) * (1/n), src/lib.rs:220-222 */
    float *seg_sasa;    /* [n_segments] ResidueLevel / ChainLevel sums                          */
    float *protein;     /* [3*S] ProteinLevel {global_total, polar_total, non_polar_total}       */
} sasa_b200_outputs;

typedef struct sasa_b200_stats {
    uint64_t n_atoms;
    uint64_t n_structures;
    uint64_t boundary_points; /* only with SASA_B200_FLAG_BOUNDARY_STATS */
    uint64_t neighbor_pairs;  /* sum over atoms of the tight neighbour-list length (fast path) */
    uint64_t streamed_atoms;  /* atoms that took the streaming kernel path                     */
    float h2d_ms, kernel_ms, d2h_ms, total_ms; /* CUDA-event times of the last run_host call   */
    uint32_t gpu_launches;    /* kernels launched by the last run call                          */
} sasa_b200_stats;

/* ---- context ---------------------------------------------------------------------- */
SASA_B200_API int sasa_b200_abi_version(void);
/* Number of CUDA devices this process can use (0 and SASA_B200_ERR_CUDA without a driver / device). */
SASA_B200_API int sasa_b200_device_count(int *out_count);
/* device < 0 selects the current CUDA device. */
SASA_B200_API int sasa_b200_create(int device, sasa_b200_ctx **out_ctx);
SASA_B200_API void sasa_b200_destroy(sasa_b200_ctx *ctx);
/* Message of the last failing call on this context (or of the last failing create when ctx
 * is NULL).  The pointer stays valid until the next call on the same context. */
SASA_B200_API const char *sasa_b200_last_error(const sasa_b200_ctx *ctx);
/* Page-locked host memory for the pipelined host entry points (optional but ~2x faster). */
SASA_B200_API int sasa_b200_alloc_pinned(size_t bytes, void **out_ptr);
SASA_B200_API int sasa_b200_free_pinned(void *ptr);
/* The golden-spiral sphere points the kernels use (src/lib.rs:43-66), computed on the host
 * with libm exactly like the reference; xyz receives n_points * 3 floats (x0,y0,z0,x1,...). */
SASA_B200_API int sasa_b200_sphere_points(uint32_t n_points, float *xyz);

/* ---- replaces calculate_sasa_internal (src/lib.rs:249-298) -------------------------
 * One structure, host buffers, synchronous.  Safe to call from many threads at once on one context (the reference's
 * directory mode does, src/main.rs:375, :439): each call runs on a stream and workspace of its own.  xyzr = n_atoms * 4 floats.  ids may be NULL
 * (all distinct) or n_atoms 64-bit Atom.id values.  out_sasa receives n_atoms floats;
 * out_counts (nullable) the integer exposed-point counts.  n_atoms == 0 is a no-op
 * (tests/sanity.rs:148-157). */
SASA_B200_API int sasa_b200_calculate_sasa_internal(sasa_b200_ctx *ctx, const float *xyzr, const uint64_t *ids, size_t n_atoms,
                                      float probe_radius, size_t n_points, ptrdiff_t threads, float *out_sasa,
                                      uint32_t *out_counts);

/* ---- batched path (what CLI directory mode, src/main.rs:342-480, becomes) ----------
 * Topology of a batch.  struct_off: S+1 atom offsets (struct_off[0] == 0).  Segments are
 * optional (seg_be == NULL -> n_segments = 0): seg_be holds n_segments pairs
 * {begin, end}, struct_seg_off S+1 offsets into the pair table, seg_polar (nullable)
 * n_segments flags used only for the ProteinLevel polar / non-polar split
 * (POLAR_AMINO_ACIDS, src/utils/consts.rs:7-16). */
SASA_B200_API int sasa_b200_batch_create(sasa_b200_ctx *ctx, const uint64_t *struct_off, size_t n_structures,
                           const uint32_t *seg_be, const uint64_t *struct_seg_off, const uint8_t *seg_polar,
                           sasa_b200_batch **out_batch);
SASA_B200_API void sasa_b200_batch_destroy(sasa_b200_batch *batch);

/* Host buffers in, host buffers out; H2D copies, kernels and D2H copies are pipelined over
 * several CUDA streams inside the call, which returns when every requested output is in
 * host memory.  xyzr: n_atoms*4 floats.  id_class: NULL or n_atoms u32. */
SASA_B200_API int sasa_b200_batch_run_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                             const sasa_b200_params *params, const sasa_b200_outputs *out,
                             sasa_b200_stats *stats /* nullable */);

/* The same run as an asynchronous pair (SURVEY.md 8b: "async submit/wait pair for stream overlap").  submit enqueues the
 * copies and kernels and returns; the input and output buffers belong to the run until sasa_b200_job_wait returns (use
 * page-locked buffers: copies from pageable memory make submit block).  wait blocks until every requested output is in host
 * memory, reports deferred errors and releases the job handle.  Several jobs of DIFFERENT batches may be in flight on one
 * context, from any threads; a batch itself carries one run at a time.  This is what lets a caller parse and pack tile
 * k + 1 while tile k is on the GPU (directory mode, src/main.rs:342-480). */
SASA_B200_API int sasa_b200_batch_submit_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_job **out_job);
SASA_B200_API int sasa_b200_batch_submit_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                       const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_job **out_job);
SASA_B200_API int sasa_b200_job_wait(sasa_b200_job *job, sasa_b200_stats *stats /* nullable */);

/* Same computation with every data pointer (xyzr, id_class, outputs) already in DEVICE
 * memory; enqueues on `stream` (a cudaStream_t, NULL = the context's stream) and returns
 * without synchronising. */
SASA_B200_API int sasa_b200_batch_run_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                               const sasa_b200_params *params, const sasa_b200_outputs *d_out, void *stream);
/* Blocks until work enqueued by run_device on the context's own stream has finished and
 * reports deferred errors (e.g. SASA_B200_ERR_NON_FINITE). */
SASA_B200_API int sasa_b200_batch_sync(sasa_b200_batch *batch, sasa_b200_stats *stats /* nullable */);

/* Grouped runs: buried surface area in one pass.  group holds one label per atom; only equality within a structure matters.
 *   out           the complex: exactly what sasa_b200_batch_run_host / _device give for the same input, bit for bit.
 *   out_isolated  every atom as the engine computes it when its group runs alone (the group's atoms as their own structure,
 *                 in original order, same id_class rule): neighbour j occludes atom i only if group[j] == group[i].  Level sums
 *                 use the batch's segments with the same summation order, so they equal the sums over the isolated per-atom
 *                 areas bit for bit wherever the plain run's sums are sequential (<= 16,384 atoms per sum).
 * Buried area = isolated - complex; the caller derives it.  count_isolated[i] >= count[i]; one group for all atoms gives
 * isolated == complex; one group per atom gives count_isolated[i] == n_points.  Every output field of both structs is
 * nullable.  group == NULL: SASA_B200_ERR_INVALID_ARGUMENT; params->flags != 0: SASA_B200_ERR_UNSUPPORTED.  Non-finite
 * input: SASA_B200_ERR_NON_FINITE with both output sets NaN-filled for that structure.  The host form uses the per-chunk
 * pipeline; the device form behaves like sasa_b200_batch_run_device (stream-ordered, errors via sasa_b200_batch_sync). */
SASA_B200_API int sasa_b200_batch_run_groups_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                    const uint32_t *group, const sasa_b200_params *params, const sasa_b200_outputs *out,
                                    const sasa_b200_outputs *out_isolated, sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_run_groups_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                      const uint32_t *d_group, const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                      const sasa_b200_outputs *d_out_isolated, void *stream);

/* Exposed-point masks: which sphere points of every atom are solvent-accessible (the dot surface), from the same pass as the
 * counts.  exposed holds W = (n_points + 31) / 32 u32 words per atom, atoms in batch order (the indexing of counts): bit b of
 * word w of atom i is set exactly when point 32 w + b -- in the order of sasa_b200_sphere_points -- is exposed; bits at or
 * above n_points are zero, and the popcount of atom i's row equals counts[i].  out / d_out are bit for bit what
 * sasa_b200_batch_run_host / _device give for the same input (every field nullable); every n_points, simd_lanes, id_class and
 * flag the plain run accepts is accepted.  exposed == NULL with atoms in the batch, or a buffer size (n_atoms * W * 4 bytes)
 * that overflows size_t: SASA_B200_ERR_INVALID_ARGUMENT.  Non-finite input: SASA_B200_ERR_NON_FINITE with zero mask rows for
 * that structure.  The host form uses the per-chunk pipeline; the device form behaves like sasa_b200_batch_run_device
 * (stream-ordered, errors via sasa_b200_batch_sync). */
SASA_B200_API int sasa_b200_batch_run_masks_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                   const sasa_b200_params *params, const sasa_b200_outputs *out,
                                   uint32_t *exposed, sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_run_masks_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                     const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                     uint32_t *d_exposed, void *stream);

/* Grouped runs with exposed-point masks: interface patches in one pass.
 *   out / out_isolated  bit for bit what sasa_b200_batch_run_groups_* gives for the same input; every field nullable.
 *   exposed             the layout of sasa_b200_batch_run_masks_*, and bit for bit that entry point's masks (the complex).
 *   exposed_isolated    the same layout; atom i's row is its mask with its group standing alone (the engine's mask when the
 *                       group's atoms run as their own structure).
 * So popcount(exposed row i) == counts[i], popcount(exposed_isolated row i) == count_isolated[i], exposed[i] & ~exposed_isolated[i]
 * == 0, and the points of atom i that other groups bury -- the interface patch -- are exposed_isolated[i] & ~exposed[i], with
 * popcount count_isolated[i] - counts[i].  group == NULL, either mask pointer NULL with atoms in the batch, or a mask buffer
 * size that overflows size_t: SASA_B200_ERR_INVALID_ARGUMENT; params->flags != 0: SASA_B200_ERR_UNSUPPORTED.  Non-finite input:
 * SASA_B200_ERR_NON_FINITE with both output sets NaN-filled and both mask row sets zeroed for that structure.  The host form
 * uses the per-chunk pipeline; the device form behaves like sasa_b200_batch_run_groups_device (stream-ordered, errors via
 * sasa_b200_batch_sync). */
SASA_B200_API int sasa_b200_batch_run_groups_masks_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                          const uint32_t *group, const sasa_b200_params *params, const sasa_b200_outputs *out,
                                          const sasa_b200_outputs *out_isolated, uint32_t *exposed, uint32_t *exposed_isolated,
                                          sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_run_groups_masks_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                            const uint32_t *d_group, const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                            const sasa_b200_outputs *d_out_isolated, uint32_t *d_exposed,
                                            uint32_t *d_exposed_isolated, void *stream);

/* Pairwise buried area: which partner group buries how much of every atom, from one grouped pass.  For atom i of group g and
 * another group h of the same structure, buried_h(i) = count_isolated(i) - count_{g+h}(i), where count_{g+h}(i) is i's count
 * when only the atoms of g and h exist (in original order, same id_class rule): the points of i open with g alone that at least
 * one atom of h hides.  The slot area is the reference's area expression on that count, ((4*pi*R^2) * buried_h(i)) * (1/n),
 * bit for bit what atom_sasa would hold for that radius and count.  K = max_partners slots per atom, atoms in batch order (the
 * indexing of counts): slot s of atom i is element i * K + s.  The slots in use hold the partners with buried_h(i) > 0 in
 * ascending label order; the rest hold partner = UINT32_MAX, count 0 and area 0.0f.  A slot is in use exactly when its count
 * is non-zero, so the label UINT32_MAX is not reserved.  Partners are enumerated among the atom's neighbours in the complex.
 * So buried_h(i) <= count_isolated(i) - count(i), max_h buried_h(i) <= count_isolated(i) - count(i) <= sum_h buried_h(i)
 * (a point hidden by two partners counts for both), and with exactly two groups in a structure the one slot in use holds
 * count_isolated(i) - count(i). */
typedef struct sasa_b200_pair_outputs {
    uint32_t max_partners;     /* K: slots per atom, 1..16                                                           */
    uint32_t *partner;         /* [n_atoms*K] partner group label per slot, UINT32_MAX = unused                      */
    uint32_t *buried_counts;   /* [n_atoms*K] nullable: buried_h(i)                                                  */
    float *buried_area;        /* [n_atoms*K] nullable: the area expression above on buried_counts                   */
    uint32_t *partners_needed; /* nullable, ONE u32: the largest number of partners of an atom in this run           */
} sasa_b200_pair_outputs;      /* (host pointers for _host, device pointers for _device)                             */

/* out / out_isolated: bit for bit what sasa_b200_batch_run_groups_* gives for the same input; every field nullable.  An atom
 * with more than K partners gets its K lowest-label partners, and the call returns SASA_B200_ERR_INVALID_ARGUMENT with a
 * message naming the K the batch needs; *partners_needed receives that maximum on every run, successful or not, and out /
 * out_isolated are still complete.  group == NULL, pairs or pairs->partner NULL with atoms in the batch, K outside 1..16 or a
 * slot-buffer size that overflows size_t: SASA_B200_ERR_INVALID_ARGUMENT; params->flags != 0: SASA_B200_ERR_UNSUPPORTED.
 * Non-finite input: SASA_B200_ERR_NON_FINITE with both output sets NaN-filled for that structure and its slots set to
 * partner UINT32_MAX, count 0, area NaN.  An empty batch does nothing.  The host form uses the per-chunk pipeline; the device
 * form behaves like sasa_b200_batch_run_groups_device: stream-ordered, with the too-few-slots error deferred to
 * sasa_b200_batch_sync like SASA_B200_ERR_NON_FINITE (which takes precedence when both occur). */
SASA_B200_API int sasa_b200_batch_run_group_pairs_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                         const uint32_t *group, const sasa_b200_params *params, const sasa_b200_outputs *out,
                                         const sasa_b200_outputs *out_isolated, const sasa_b200_pair_outputs *pairs,
                                         sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_run_group_pairs_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                           const uint32_t *d_group, const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                           const sasa_b200_outputs *d_out_isolated, const sasa_b200_pair_outputs *d_pairs,
                                           void *stream);

/* MD-trajectory form (what mdsasa-bolt feeds calculate_sasa_internal per frame): a batch
 * created with S = n_frames equal-sized structures; xyz holds n_frames * n_atoms_per_frame
 * * 3 floats, radii n_atoms_per_frame floats shared by every frame (12 B/atom/frame on the
 * wire instead of 16). */
SASA_B200_API int sasa_b200_batch_run_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                    const sasa_b200_params *params, const sasa_b200_outputs *out,
                                    sasa_b200_stats *stats /* nullable */);

/* Grouped runs of MD frames: buried surface area per frame along a trajectory, in the 12-byte frames form.  The batch, xyz
 * and radii are exactly as in sasa_b200_batch_run_frames_host; group holds n_atoms_per_frame labels shared by every frame
 * (only equality within a frame matters).  They cross the wire once per run and are expanded on the device, so a frame costs
 * 12 B/atom on the wire as in the plain frames form.
 *   out           bit for bit what sasa_b200_batch_run_frames_host gives for the same input; every field nullable.
 *   out_isolated  bit for bit what sasa_b200_batch_run_groups_host gives for the same coordinates packed as float4 with the
 *                 labels tiled over the frames; every field nullable.
 * xyz, radii or group NULL with atoms in the batch, out_isolated NULL, or frames of unequal size: SASA_B200_ERR_INVALID_ARGUMENT;
 * params->flags != 0: SASA_B200_ERR_UNSUPPORTED.  Non-finite input: SASA_B200_ERR_NON_FINITE with both output sets NaN-filled
 * for that frame only.  Uses the per-chunk pipeline of the host entry points.  submit / sasa_b200_job_wait split the run like
 * sasa_b200_batch_submit_host: the buffers belong to the run until the wait returns, and a batch carries one run at a time. */
SASA_B200_API int sasa_b200_batch_run_groups_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                           const uint32_t *group, const sasa_b200_params *params,
                                           const sasa_b200_outputs *out, const sasa_b200_outputs *out_isolated,
                                           sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_submit_groups_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                              const uint32_t *group, const sasa_b200_params *params,
                                              const sasa_b200_outputs *out, const sasa_b200_outputs *out_isolated,
                                              sasa_b200_job **out_job);

/* Pairwise buried area of MD frames: per frame, how much of every group each partner group buries, summed on the device.  The
 * batch, xyz, radii and group are exactly as in sasa_b200_batch_run_groups_frames_host; the labels must be 0 .. n_labels - 1.
 * The run is the pairwise buried-area run of sasa_b200_batch_run_group_pairs_host on the frames (K = max(1, n_labels - 1) slots
 * per atom, so no atom can have more partners than slots); its slot rows stay in device memory and only their sums come back.
 *   pair_area      [S * L * L]: element (s * L + g) * L + h is the sum of the slot areas with partner h over the atoms of group
 *                  g in frame s -- started at 0.0, added in float64, in the frame's atom order.  This is what
 *                  rustsasa_b200.group_pair_table computes from the slots on the host, bit for bit.  The diagonal is 0, and a
 *                  label with no atoms has zero rows and columns.
 *   seg_pair_area  [n_segments * L], nullable: element q * L + h is the same float64 atom-order sum over segment q's atom range
 *                  (relative to its frame's first atom, as everywhere in this ABI). */
typedef struct sasa_b200_pair_sums {
    uint32_t n_labels;       /* L, 1..17: group labels are 0 .. L - 1                                                 */
    double *pair_area;       /* [S * L * L]                                                                           */
    double *seg_pair_area;   /* [n_segments * L], nullable                                                            */
} sasa_b200_pair_sums;       /* (host pointers)                                                                       */

/* out: bit for bit sasa_b200_batch_run_frames_host; out_isolated: bit for bit sasa_b200_batch_run_groups_frames_host; every
 * field of both nullable.  xyz, radii or group NULL with atoms in the batch, out_isolated NULL, sums or sums->pair_area NULL
 * with atoms in the batch, n_labels outside 1..17, a label >= n_labels, frames of unequal size or an output size that overflows
 * size_t: SASA_B200_ERR_INVALID_ARGUMENT; params->flags != 0: SASA_B200_ERR_UNSUPPORTED.  Non-finite input:
 * SASA_B200_ERR_NON_FINITE with both output sets NaN-filled, and the frame's L x L block and all its segment rows NaN, for that
 * frame only.  An empty batch does nothing.  Uses the per-chunk pipeline; submit / sasa_b200_job_wait split the run as for
 * sasa_b200_batch_submit_groups_frames_host. */
SASA_B200_API int sasa_b200_batch_run_group_pairs_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                                const uint32_t *group, const sasa_b200_params *params,
                                                const sasa_b200_outputs *out, const sasa_b200_outputs *out_isolated,
                                                const sasa_b200_pair_sums *sums, sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_submit_group_pairs_frames_host(sasa_b200_batch *batch, const float *xyz, const float *radii,
                                                   const uint32_t *group, const sasa_b200_params *params,
                                                   const sasa_b200_outputs *out, const sasa_b200_outputs *out_isolated,
                                                   const sasa_b200_pair_sums *sums, sasa_b200_job **out_job);

/* Indexed-radius form: 13 bytes per atom on the wire instead of 16.  Proteins use a handful of distinct radii (ProtOr,
 * radii/protor.config, has ten), so the extraction step (build_atoms_and_mapping, src/options.rs:81-116) can emit
 * coordinates as 3 floats per atom plus ONE BYTE per atom indexing a palette of at most 256 radii.  With eight GPUs pulling
 * their batches over PCIe at once the host copy is the limiter, and it scales with the bytes.  Same results as the float4
 * form bit for bit; the fused kernels read this form directly.  xyz: n_atoms * 3 floats; radius_index: n_atoms bytes. */
SASA_B200_API int sasa_b200_batch_run_indexed_host(sasa_b200_batch *batch, const float *xyz, const uint8_t *radius_index,
                                     const float *palette, size_t n_palette, const uint32_t *id_class,
                                     const sasa_b200_params *params, const sasa_b200_outputs *out,
                                     sasa_b200_stats *stats /* nullable */);
SASA_B200_API int sasa_b200_batch_submit_indexed_host(sasa_b200_batch *batch, const float *xyz, const uint8_t *radius_index,
                                        const float *palette, size_t n_palette, const uint32_t *id_class,
                                        const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_job **out_job);

/* Atom-range split of large structures over several GPUs (BASELINE.json config 5: a 1M-atom capsid at 960 points
 * split across 8 GPUs).  The reference has no counterpart -- its neighbour build is serial and its atom loop is a
 * rayon par_iter inside one process (src/lib.rs:278-290); this is that par_iter cut across devices.  Every rank
 * holds ALL atoms of the batch, rebuilds the cell list redundantly (cheaper than exchanging it) and evaluates
 * only slice `rank` of `n_ranks` of each structure's CELL-SORTED atom order, i.e. a spatially compact slab (cut at
 * cell boundaries, which are identical on every rank, so the slices partition the atoms exactly).
 * counts / atom_sasa are written for the slice's atoms and ZERO elsewhere, so the element-wise sum over ranks
 * (ncclAllReduce on the device variant) equals the single-GPU result bit for bit.  Level sums are not produced
 * here: reduce the summed per-atom vector with sasa_b200_batch_reduce_device or on the host. */
SASA_B200_API int sasa_b200_batch_run_atom_range_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                          const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                          uint32_t *d_counts /* nullable */, float *d_atom_sasa /* nullable */, void *stream);
/* The same with the exchange step fused into the kernel: peer_counts[r] / peer_atom_sasa[r] (host arrays of n_ranks device
 * pointers, each valid on THIS device -- the local vector for r == rank, the peers' vectors mapped over NVLink / NVSwitch,
 * e.g. the buffer_ptrs of a torch symmetric-memory allocation or cudaIpc handles) receive the values of the atoms this rank
 * owns as they are produced.  Nothing is zero-filled and nothing is reduced afterwards: once every rank's kernel has finished
 * (a barrier across ranks, not provided here) every rank holds the complete vectors.  Either array may be NULL; n_ranks <= 8.
 * The caller also keeps ranks from overwriting vectors a peer is still reading (a barrier before the call). */
SASA_B200_API int sasa_b200_batch_run_atom_range_peers_device(sasa_b200_batch *batch, const float *d_xyzr, const uint32_t *d_id_class,
                                                const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                                uint32_t *const *peer_counts, float *const *peer_atom_sasa, void *stream);
SASA_B200_API int sasa_b200_batch_run_atom_range_host(sasa_b200_batch *batch, const float *xyzr, const uint32_t *id_class,
                                        const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                        uint32_t *out_counts /* nullable */, float *out_atom_sasa /* nullable */,
                                        sasa_b200_stats *stats /* nullable */);

/* The level sums alone (the numeric part of process_atoms, src/options.rs:195-232, :292-315, :370-410) over a
 * finished per-atom SASA vector in device memory: d_seg_sasa [n_segments] and d_protein [3*S], both nullable.
 * One small launch per structure -- meant for the few large structures of the atom-range split. */
SASA_B200_API int sasa_b200_batch_reduce_device(sasa_b200_batch *batch, const float *d_atom_sasa, float *d_seg_sasa,
                                  float *d_protein, void *stream);

/* Convenience: create + run_host + destroy. */
SASA_B200_API int sasa_b200_run_batch(sasa_b200_ctx *ctx, const float *xyzr, const uint32_t *id_class, const uint64_t *struct_off,
                        size_t n_structures, const uint32_t *seg_be, const uint64_t *struct_seg_off,
                        const uint8_t *seg_polar, const sasa_b200_params *params, const sasa_b200_outputs *out,
                        sasa_b200_stats *stats /* nullable */);

#ifdef __cplusplus
}
#endif
#endif /* SASA_B200_H */
