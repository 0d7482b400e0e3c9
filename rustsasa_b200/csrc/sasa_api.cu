// sasa_api.cu -- host side of libsasa_b200.so: the C ABI declared in include/sasa_b200.h.
//
// One context per (process, device).  A batch object holds the topology of a set of structures (CSR
// offsets, output segments) and the launch plan derived from it: structures are bucketed by size into
// shared-memory configurations of the fused per-structure kernel, ordered largest-first inside each
// bucket, and cut into chunks so that the host entry point can overlap the H2D copy of chunk c+1 with
// the kernels of chunk c and the D2H copy of chunk c-1 on separate CUDA streams.
//
// There is deliberately no CPU implementation in this library: without a CUDA device every entry point
// fails with SASA_B200_ERR_CUDA.
#include "../../include/sasa_b200.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#include "sasa_large.cuh"
#include "sasa_pair_sums.cuh"
#include "sasa_small.cuh"
#include "sasa_tight.cuh"

using namespace sasa;

namespace {

thread_local std::string g_create_error;

struct Points {
    float *d = nullptr;    // 3*n floats: x[n] y[n] z[n]
    uint4 *cap = nullptr;  // cap table (sasa_cap.cuh), n <= 128 only
    cudaTextureObject_t cap_tex = 0;   // the same table as a linear uint4 texture (the fused kernel reads it through the texture pipe)
    // 128 < n <= 1024: the points as float4 and the chunked cap table (inner / ring masks in separate arrays)
    float4 *d4 = nullptr;
    uint4 *capm_in = nullptr, *capm_rg = nullptr;
    CapDims capd = {};
};

// The fused kernels of one shared-memory configuration, by attribute slot (kernel_slot).
constexpr int kKernelSlots = 14;
struct Proto {
    int nt, minb;
    uint32_t cmax;
    uint32_t cap[4];                 // max_atoms(...), index = has_cls + 2 * grouped
    const void *fn[kKernelSlots];
};
// Slots: plain runs has_cls + 2 * tight, masked runs 4 + the same (tight: n_points <= 128, no statistics / forced streaming),
// grouped runs 8 + has_cls, masked grouped runs 10 + has_cls and pairwise buried area 12 + has_cls (always tight: they take no
// flags, and with n_points > 128 they take the large-structure path).
int kernel_slot(bool grouped, bool masked, bool has_cls, bool tight, bool pairs = false) {
    if (pairs) return 12 + (has_cls ? 1 : 0);
    return grouped ? (masked ? 10 : 8) + (has_cls ? 1 : 0) : (masked ? 4 : 0) + (has_cls ? 1 : 0) + (tight ? 2 : 0);
}
#define SASA_PROTO(NT, MINB, CMAX)                                                                                     \
    Proto { NT, MINB, CMAX, { max_atoms(NT, MINB, CMAX, false), max_atoms(NT, MINB, CMAX, true),                       \
                              max_atoms(NT, MINB, CMAX, false, true), max_atoms(NT, MINB, CMAX, true, true) },         \
            { (const void *)sasa_small_kernel<NT, MINB, false, CMAX>, (const void *)sasa_small_kernel<NT, MINB, true, CMAX>, \
              (const void *)sasa_tight_kernel<NT, MINB, false, CMAX>, (const void *)sasa_tight_kernel<NT, MINB, true, CMAX>, \
              (const void *)sasa_small_masks_kernel<NT, MINB, false, CMAX>,                                            \
              (const void *)sasa_small_masks_kernel<NT, MINB, true, CMAX>,                                             \
              (const void *)sasa_tight_masks_kernel<NT, MINB, false, CMAX>,                                            \
              (const void *)sasa_tight_masks_kernel<NT, MINB, true, CMAX>,                                             \
              (const void *)sasa_tight_groups_kernel<NT, MINB, false, CMAX>,                                           \
              (const void *)sasa_tight_groups_kernel<NT, MINB, true, CMAX>,                                            \
              (const void *)sasa_tight_groups_masks_kernel<NT, MINB, false, CMAX>,                                     \
              (const void *)sasa_tight_groups_masks_kernel<NT, MINB, true, CMAX>,                                      \
              (const void *)sasa_tight_group_pairs_kernel<NT, MINB, false, CMAX>,                                      \
              (const void *)sasa_tight_group_pairs_kernel<NT, MINB, true, CMAX> } }
// Shared-memory configurations of the fused kernel.  nmax is derived from the per-CTA budget that lets `minb` CTAs share one SM
// (228 KB per SM, 1 KB reserved per CTA, 227 KB per CTA max); both keep 32 warps resident per SM (64 registers/thread).
const Proto kProtos[] = {SASA_PROTO(512, 2, 8192), SASA_PROTO(1024, 1, 16384)};
#undef SASA_PROTO
constexpr int kNumProtos = sizeof(kProtos) / sizeof(kProtos[0]);

struct SmallCfg {
    int nt, minb;
    uint32_t cap[4];   // atom capacity, index = has_cls + 2 * grouped (compile-time constants of the configuration)
    uint32_t cmax;
    size_t smem[4];    // dynamic shared memory of a launch, same index
    int proto;
};

// Streams of the pipelined host entry points.  cfg2 end to end, device-side span (tools/exp_e2e.py, one B200): 2 streams 5.92 ms,
// 3: 5.26 ms, 4: 5.29 ms, 6: 5.37 ms (5.00 ms as one device-resident launch).
constexpr int kStreams = 3;
constexpr size_t kChunkAtoms = 1000000;
constexpr size_t kMaxGatedChunks = 1024;              // chunks of one gated single-launch run (more: the per-chunk launches)
constexpr size_t kGatedMaxOutBytes = 32u << 20;        // outputs above this go through device memory and D2H copies
constexpr uint32_t kSingleLargeMin = 1024;   // atoms from which a lone structure takes the large-structure path
constexpr size_t kMaxSlots = 16;

// Everything one one-structure call needs, owned for the duration of the call.
struct SingleSlot {
    cudaStream_t st = nullptr;
    LargeWorkspace large;
    char *d_buf = nullptr;
    size_t d_bytes = 0;
    char *h_pin = nullptr;
    size_t h_bytes = 0;
    bool busy = false;
};

}  // namespace

// One host-buffer run in flight (sasa_b200_batch_submit_host .. sasa_b200_job_wait).
struct sasa_b200_job {
    sasa_b200_batch *batch = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // timing: first enqueue .. everything done
    void *d_arena = nullptr;                    // stream-ordered allocation holding inputs, outputs and the status words
    unsigned long long *h_status = nullptr;     // pinned: [0] error flag, [1..3] statistics
    uint32_t *h_ready = nullptr;                // pinned: cumulative structure counts of the chunks (gated single-launch pipeline)
    std::chrono::steady_clock::time_point t_begin;
    uint32_t launches = 0;
    bool active = false;
    const sasa_b200_pair_outputs *pairs = nullptr;   // pairwise buried-area runs: the caller's slot outputs (partners_needed is
                                                     // written when the job is waited for)
};

struct sasa_b200_job;
struct sasa_b200_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t streams[kStreams] = {};
    // fork/join helpers: the launches of one chunk (one per shared-memory bucket) run on sibling streams so that the
    // tail of one kernel is back-filled by the CTAs of the next instead of idling the SMs
    static constexpr int kSide = 3;
    cudaStream_t side[kSide] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[kSide] = {};
    std::map<uint32_t, Points> points;
    int *d_err = nullptr;
    unsigned long long *d_stat = nullptr;
    uint32_t *d_needed = nullptr;   // pairwise buried area, device form: partners needed by the last run [0] and since the last sync [1]
    std::vector<SmallCfg> cfgs;
    std::string err;
    std::mutex mu;
    // grow-only device arena for the host entry points
    void *arena = nullptr;
    size_t arena_bytes = 0;
    // grow-only workspace of the large-structure path, shared by every batch of the context (a per-batch workspace cost
    // nine cudaMalloc / cudaFree pairs per call: 6 ms for one 6,000-atom structure through calculate_sasa_internal).
    // Uses on different streams are chained through ev_large.
    LargeWorkspace large;
    cudaEvent_t ev_large = nullptr;
    bool large_used = false;
    bool attr_done[kNumProtos][kKernelSlots] = {};  // shared-memory attribute set (at a kernel's first launch)
    // jobs: one per host-buffer run in flight (submit / wait); recycled, so events and the pinned status word are made once
    std::vector<sasa_b200_job *> free_jobs;
    cudaEvent_t ev_tail[kStreams] = {};   // end of the previous job on each copy stream (the next job's first stream waits on them)
    bool tail_valid = false;
    // slots of the one-structure calls: own stream, own workspace, own staging -- callers on different threads do not
    // serialise on the context (the reference's directory mode calls the engine from every rayon worker, src/main.rs:375)
    std::vector<std::unique_ptr<SingleSlot>> slots;
    std::mutex slot_mu;
    std::condition_variable slot_cv;
};

namespace {

int fail(sasa_b200_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    else g_create_error = buf;
    return code;
}

#define CU_TRY(ctx, expr)                                                                                      \
    do {                                                                                                       \
        cudaError_t e__ = (expr);                                                                              \
        if (e__ != cudaSuccess)                                                                                \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? SASA_B200_ERR_OUT_OF_MEMORY : SASA_B200_ERR_CUDA, \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__);          \
    } while (0)

// generate_sphere_points, reference src/lib.rs:43-66: golden-section spiral evaluated with the host libm
// (CUDA's sinf/cosf/acosf are not bit-identical to glibc's, so the points are never computed on the device).
void sphere_points_host(uint32_t n, float *x, float *y, float *z) {
    const float golden = 1.618034f;
    const float inc = (2.0f * 3.14159265358979323846f) * golden;
    const float inv = 1.0f / (float)n;
    for (uint32_t i = 0; i < n; ++i) {
        const float fi = (float)i;
        const float incl = std::acos(1.0f - 2.0f * (fi * inv));
        const float az = inc * fi;
        const float si = std::sin(incl);
        x[i] = si * std::cos(az);
        y[i] = si * std::sin(az);
        z[i] = std::cos(incl);
    }
}

int get_points(sasa_b200_ctx *ctx, uint32_t n, const Points **out) {
    auto it = ctx->points.find(n);
    if (it == ctx->points.end()) {
        std::vector<float> h(3 * (size_t)n);
        sphere_points_host(n, h.data(), h.data() + n, h.data() + 2 * (size_t)n);
        Points P;
        CU_TRY(ctx, cudaMalloc(&P.d, h.size() * sizeof(float)));
        CU_TRY(ctx, cudaMemcpy(P.d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
        if (n <= 128) {   // the point sets of the tight kernel get their cap table (built once per context and n_points)
            std::vector<uint32_t> t(kCapTableBins * 8);
            cap_build_table(n, h.data(), h.data() + n, h.data() + 2 * (size_t)n, t.data());
            CU_TRY(ctx, cudaMalloc(&P.cap, t.size() * sizeof(uint32_t)));
            CU_TRY(ctx, cudaMemcpy(P.cap, t.data(), t.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
            cudaResourceDesc rd = {};
            rd.resType = cudaResourceTypeLinear;
            rd.res.linear.devPtr = P.cap;
            rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
            rd.res.linear.sizeInBytes = t.size() * sizeof(uint32_t);
            cudaTextureDesc td = {};
            td.readMode = cudaReadModeElementType;
            CU_TRY(ctx, cudaCreateTextureObject(&P.cap_tex, &rd, &td, nullptr));
        } else if (n <= 1024) {   // chunked table for the large-structure path (sasa_cap.cuh, capm_atom)
            // 64 direction bins per axis: a 96^2 / 128^2 grid measured 1.55 / 1.54 ms against 1.60 ms on cfg5 (run r02l) for
            // 2.3x / 4x the table.  Always eight chunk slots: capm_atom<8> serves every 128 < n <= 1024.
            P.capd = cap_dims(64, kCapmL, 8);
            const size_t words = cap_multi_words(P.capd);
            std::vector<uint32_t> tin(words), trg(words);
            cap_build_table_multi(n, h.data(), h.data() + n, h.data() + 2 * (size_t)n, P.capd, tin.data(), trg.data());
            std::vector<float> h4(4 * (size_t)n, 0.0f);
            for (uint32_t i = 0; i < n; ++i) {
                h4[4 * (size_t)i + 0] = h[i];
                h4[4 * (size_t)i + 1] = h[n + i];
                h4[4 * (size_t)i + 2] = h[2 * (size_t)n + i];
            }
            CU_TRY(ctx, cudaMalloc(&P.d4, h4.size() * sizeof(float)));
            CU_TRY(ctx, cudaMemcpy(P.d4, h4.data(), h4.size() * sizeof(float), cudaMemcpyHostToDevice));
            CU_TRY(ctx, cudaMalloc(&P.capm_in, words * sizeof(uint32_t)));
            CU_TRY(ctx, cudaMalloc(&P.capm_rg, words * sizeof(uint32_t)));
            CU_TRY(ctx, cudaMemcpy(P.capm_in, tin.data(), words * sizeof(uint32_t), cudaMemcpyHostToDevice));
            CU_TRY(ctx, cudaMemcpy(P.capm_rg, trg.data(), words * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        it = ctx->points.emplace(n, P).first;
    }
    *out = &it->second;
    return SASA_B200_OK;
}

// The configurations of the context, smallest atom capacity first.
int build_cfgs(sasa_b200_ctx *ctx) {
    for (int i = 0; i < kNumProtos; ++i) {
        const Proto &pr = kProtos[i];
        SmallCfg c{pr.nt, pr.minb, {pr.cap[0], pr.cap[1], pr.cap[2], pr.cap[3]}, pr.cmax, {0, 0, 0, 0}, i};
        for (int v = 0; v < 4; ++v) c.smem[v] = small_layout(c.cap[v], c.cmax, c.nt / 32, (v & 1) == 1, v >= 2).total;
        if (*std::min_element(c.cap, c.cap + 4) == 0 || *std::max_element(c.smem, c.smem + 4) > ctx->smem_optin)
            return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "the fused kernels are laid out for 228 KB of shared memory per SM (B200); this device offers %zu per block",
                        ctx->smem_optin);
        // (the MaxDynamicSharedMemorySize attribute is set at a kernel's first launch, enqueue_chunk: touching every
        // instantiation here made the driver load every one of them at context creation)
        ctx->cfgs.push_back(c);
    }
    std::sort(ctx->cfgs.begin(), ctx->cfgs.end(), [](const SmallCfg &a, const SmallCfg &b) { return a.cap[0] < b.cap[0]; });
    return SASA_B200_OK;
}

uint32_t cfg_capacity(const sasa_b200_ctx *, const SmallCfg &c, bool has_cls, bool grouped = false) {
    return c.cap[(has_cls ? 1 : 0) + (grouped ? 2 : 0)];
}

struct Launch {
    int cfg;          // index into ctx->cfgs, or -1 for the large-structure path
    uint32_t order_off, n_work;
    uint32_t counter; // index into the work-counter array
};

struct Chunk {
    uint32_t s0, s1;      // structure range
    uint64_t a0, a1;      // atom range
    uint64_t g0, g1;      // segment range
    std::vector<Launch> launches;
};

}  // namespace

struct sasa_b200_batch {
    sasa_b200_ctx *ctx = nullptr;
    size_t S = 0, n_atoms = 0, n_seg = 0;
    bool has_polar = false;
    bool single_latency = false;   // one-structure convenience calls: prefer the multi-CTA large-structure path (see build_plan)
    std::vector<uint32_t> h_off;      // S+1
    std::vector<uint32_t> h_seg_off;  // S+1
    // launch plans, index = variant + 2*mode + 4*grouped; variant: 0 without / 1 with id classes (capacities differ);
    // mode: 0 = chunked for the pipelined host entry points, 1 = one chunk for device-resident runs; grouped: the plans of
    // sasa_b200_batch_run_groups_* (8 B more shared memory per atom)
    std::vector<Chunk> plan[8];
    std::vector<uint32_t> h_order[8];
    // gated single-launch pipeline (host plans 0 / 1 only): the whole batch as ONE queue in an order that follows the arrival of
    // the chunks, and per queue position the number of chunks that must have arrived (empty: the plan does not qualify)
    std::vector<uint32_t> h_gorder[2], h_gneed[2];
    uint32_t *d_gorder[2] = {nullptr, nullptr}, *d_gneed[2] = {nullptr, nullptr};
    uint32_t n_counters[8] = {};
    uint32_t max_large = 0;             // largest structure that takes the large-structure path in any ungrouped plan (workspace size)
    uint32_t max_large_v[8] = {};       // ... per plan: a structure may fit the fused kernels without id classes only
    uint32_t max_struct = 0;            // largest structure (grouped runs with n_points > 128 take the large-structure path throughout)
    // device topology
    uint32_t *d_off = nullptr, *d_seg_off = nullptr, *d_order[8] = {}, *d_counters = nullptr;
    uint2 *d_seg_be = nullptr;
    uint8_t *d_polar = nullptr;
    sasa_b200_stats last = {};
    uint32_t launches_last = 0;
    sasa_b200_job *in_flight = nullptr;   // the work counters belong to one run at a time
};

namespace {

// Queue of the gated single-launch pipeline: CHUNK-MAJOR -- the structures of chunk 0 largest-first (ties: lower index first),
// then those of chunk 1, ... -- so that a CTA only ever waits for the chunk the copy stream is working on and a slow copy (eight
// ranks sharing one host, pageable input) degrades the run gracefully: everything that has arrived is worked on, the end is the
// last chunk's copy plus its work.
void build_gated_order(sasa_b200_batch *b, int variant) {
    std::vector<uint32_t> &order = b->h_gorder[variant], &need = b->h_gneed[variant];
    order.clear();
    need.clear();
    const std::vector<Chunk> &plan = b->plan[variant];
    if (b->max_large_v[variant] != 0 || plan.size() < 2 || plan.size() > kMaxGatedChunks) return;
    const int cfg0 = plan[0].launches.empty() ? -1 : plan[0].launches[0].cfg;
    for (const Chunk &ch : plan)
        if (ch.launches.size() != 1 || ch.launches[0].cfg < 0 || ch.launches[0].cfg != cfg0) return;
    auto atoms_of = [&](uint32_t sidx) { return b->h_off[sidx + 1] - b->h_off[sidx]; };
    for (size_t c = 0; c < plan.size(); ++c) {
        const size_t first = order.size();
        for (uint32_t i = plan[c].s0; i < plan[c].s1; ++i) order.push_back(i);
        std::stable_sort(order.begin() + first, order.end(), [&](uint32_t x, uint32_t y) { return atoms_of(x) > atoms_of(y); });
        need.resize(order.size(), (uint32_t)(c + 1));
    }
}

int arena_reserve(sasa_b200_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->arena_bytes) return SASA_B200_OK;
    if (ctx->arena) cudaFree(ctx->arena);
    ctx->arena = nullptr;
    ctx->arena_bytes = 0;
    const size_t want = bytes + bytes / 8 + (1 << 20);
    CU_TRY(ctx, cudaMalloc(&ctx->arena, want));
    ctx->arena_bytes = want;
    return SASA_B200_OK;
}

void build_plan(sasa_b200_batch *b, int variant) {
    sasa_b200_ctx *ctx = b->ctx;
    const bool has_cls = (variant & 1) == 1, grouped = (variant & 4) != 0;
    static const size_t chunk_env = [] {
        const char *e = getenv("SASA_B200_CHUNK_ATOMS");   // tuning aid: atoms per pipelined chunk of the host entry points
        return e ? (size_t)atoll(e) : kChunkAtoms;
    }();
    const size_t chunk_atoms = (variant & 2) ? ~(size_t)0 : chunk_env;
    std::vector<uint32_t> cap;
    for (const SmallCfg &c : ctx->cfgs) cap.push_back(cfg_capacity(ctx, c, has_cls, grouped));
    std::vector<Chunk> &plan = b->plan[variant];
    std::vector<uint32_t> &order = b->h_order[variant];
    plan.clear();
    order.clear();
    uint32_t counters = 0;
    uint32_t s = 0;
    while (s < b->S) {
        Chunk ch;
        ch.s0 = s;
        ch.a0 = b->h_off[s];
        // the first chunks are smaller so that the first kernel starts after a short copy (ramp 1/8, 1/4, 1/2, 1, 1, ...)
        constexpr size_t ramp_levels = 3;
        const size_t ramp = plan.size() < ramp_levels && chunk_atoms != ~(size_t)0 ? chunk_atoms >> (ramp_levels - plan.size()) : chunk_atoms;
        while (s < b->S && (b->h_off[s] - ch.a0 < ramp || s == ch.s0)) ++s;
        // equal-sized structures (MD frames) finish in lock step: cut the chunk at a whole number of waves of the
        // widest configuration so that no launch ends with a mostly idle last round
        if (s < b->S && chunk_atoms != ~(size_t)0) {
            const uint32_t n0 = b->h_off[ch.s0 + 1] - b->h_off[ch.s0];
            bool uniform = true;
            for (uint32_t i = ch.s0; i < s && uniform; ++i) uniform = (b->h_off[i + 1] - b->h_off[i]) == n0;
            if (uniform) {
                size_t k = 0;
                while (k < cap.size() && n0 > cap[k]) ++k;
                if (k < cap.size()) {
                    const uint32_t slots = (uint32_t)(ctx->sm_count * ctx->cfgs[k].minb);
                    uint32_t want = ((s - ch.s0 + slots - 1) / slots) * slots;
                    while (s < b->S && s - ch.s0 < want && b->h_off[s + 1] - b->h_off[s] == n0) ++s;
                }
            }
        }
        ch.s1 = s;
        ch.a1 = b->h_off[s];
        ch.g0 = b->h_seg_off.empty() ? 0 : b->h_seg_off[ch.s0];
        ch.g1 = b->h_seg_off.empty() ? 0 : b->h_seg_off[ch.s1];
        // bucket the chunk's structures
        std::vector<std::vector<uint32_t>> bucket(ctx->cfgs.size() + 1);
        for (uint32_t i = ch.s0; i < ch.s1; ++i) {
            const uint32_t n = b->h_off[i + 1] - b->h_off[i];
            size_t k = 0;
            while (k < cap.size() && n > cap[k]) ++k;
            // A lone structure in a fused kernel occupies ONE SM (297 us per call at 1,283 atoms, 373 us at 2,622); the
            // large-structure path spreads it over the GPU (171 us at 6,065 atoms, 264 us at 32,500).  Only the
            // one-structure convenience entry points ask for this; explicit batches keep the fused kernels.
            if (b->single_latency && b->S == 1 && n >= kSingleLargeMin) k = cap.size();
            bucket[k].push_back(i);
            if (k == cap.size()) {
                if (!grouped) b->max_large = std::max(b->max_large, n);   // (grouped runs reserve the workspace at run time)
                b->max_large_v[variant] = std::max(b->max_large_v[variant], n);
            }
        }
        // One launch per chunk wherever that costs little: every extra bucket is an extra kernel with its own ramp-up
        // and tail (measured on the proteome batch: 953 vs 875 M atoms/s end to end).  If the widest fused
        // configuration in use holds a fifth or more of the chunk's fused atoms, the smaller buckets join it.
        for (size_t k = cap.size(); k-- > 1;) {
            if (bucket[k].empty()) continue;
            uint64_t atoms_k = 0, atoms_below = 0;
            for (uint32_t i : bucket[k]) atoms_k += b->h_off[i + 1] - b->h_off[i];
            for (size_t j = 0; j < k; ++j)
                for (uint32_t i : bucket[j]) atoms_below += b->h_off[i + 1] - b->h_off[i];
            if (atoms_below && atoms_k * 5 >= atoms_k + atoms_below) {
                for (size_t j = 0; j < k; ++j) {
                    bucket[k].insert(bucket[k].end(), bucket[j].begin(), bucket[j].end());
                    bucket[j].clear();
                }
            }
            break;   // only the widest bucket in use absorbs
        }
        for (size_t k = 0; k < bucket.size(); ++k) {
            if (bucket[k].empty()) continue;
            std::stable_sort(bucket[k].begin(), bucket[k].end(), [&](uint32_t x, uint32_t y) {
                return b->h_off[x + 1] - b->h_off[x] > b->h_off[y + 1] - b->h_off[y];
            });
            Launch L;
            L.cfg = k < cap.size() ? (int)k : -1;
            L.order_off = (uint32_t)order.size();
            L.n_work = (uint32_t)bucket[k].size();
            L.counter = counters++;
            order.insert(order.end(), bucket[k].begin(), bucket[k].end());
            ch.launches.push_back(L);
        }
        plan.push_back(std::move(ch));
    }
    b->n_counters[variant] = counters;
}

struct RunArgs {
    const float4 *d_xyzr;
    const uint32_t *d_cls;
    sasa_b200_outputs d_out;
    sasa_b200_params prm;
    const Points *pts;
};

// Sphere points, cap tables and numeric parameters of a run.
void fill_run_params(KParams *kp, const Points *pts, const sasa_b200_params &prm) {
    const uint32_t n = prm.n_points;
    kp->cap = pts->cap;
    kp->cap_tex = (unsigned long long)pts->cap_tex;
    kp->capm_in = pts->capm_in;
    kp->capm_rg = pts->capm_rg;
    kp->pts4 = pts->d4;
    kp->capd = pts->capd;
    kp->px = pts->d;
    kp->py = pts->d + n;
    kp->pz = pts->d + 2 * (size_t)n;
    kp->n_points = n;
    const uint32_t lanes = prm.simd_lanes ? prm.simd_lanes : 8;
    kp->n_body = (n / lanes) * lanes;
    kp->inv_n = 1.0f / (float)n;
    kp->probe = prm.probe_radius;
    // the two-phase point tests of the generic kernel (atom_fast): neighbours nearer than 4 A first, phase 1 against 4..16 of
    // them, the broadcast form of phase 2 above 16 survivors
    kp->near2 = 4.0f * 4.0f;
    kp->bcast_min = 16;
    kp->m_min = 4;
    kp->m_max = 16;
    kp->flags = prm.flags;
}

int make_kparams(sasa_b200_batch *b, const RunArgs &ra, KParams *kp) {
    sasa_b200_ctx *ctx = b->ctx;
    memset(kp, 0, sizeof *kp);
    kp->xyzr = ra.d_xyzr;
    kp->cls = ra.d_cls;
    kp->struct_off = b->d_off;
    kp->seg_be = b->d_seg_be;
    kp->struct_seg_off = b->d_seg_off;
    kp->seg_polar = b->d_polar;
    kp->out_counts = ra.d_out.counts;
    kp->out_atom = ra.d_out.atom_sasa;
    kp->out_seg = b->n_seg ? ra.d_out.seg_sasa : nullptr;
    kp->out_protein = ra.d_out.protein;
    fill_run_params(kp, ra.pts, ra.prm);
    kp->err_flag = ctx->d_err;
    kp->stat = ctx->d_stat;
    return SASA_B200_OK;
}

int check_params(sasa_b200_ctx *ctx, const sasa_b200_params *p) {
    if (!p) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "params is NULL");
    if (p->n_points == 0 || p->n_points > (1u << 24))
        return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "n_points must be in [1, 2^24], got %u", p->n_points);
    if (p->simd_lanes != 0 && p->simd_lanes != 4 && p->simd_lanes != 8 && p->simd_lanes != 16)
        return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "simd_lanes must be 0, 4, 8 or 16, got %u", p->simd_lanes);
    if (!std::isfinite(p->probe_radius) || p->probe_radius < 0.0f)
        return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "probe_radius must be finite and >= 0");
    return SASA_B200_OK;
}

// Enqueue every kernel of one chunk: the first fused launch on `st`, the others on sibling streams forked from and
// joined back into `st` (so the caller still sees one stream-ordered unit of work).  Large-structure pipelines stay
// on `st`.
// gp: grouped runs (group labels and isolated outputs), else null.  mp: exposed-point masks, else null.  mpi: the isolated
// masks of a masked grouped run (gp and mp set), else null.  pp: the partner slots of a pairwise buried-area run (gp set), else null.
int enqueue_chunk(sasa_b200_batch *b, int variant, const Chunk &ch, const KParams &base, cudaStream_t st,
                  uint32_t *launches, const uint32_t *order_override = nullptr, const GroupParams *gp = nullptr,
                  const MaskParams *mp = nullptr, const MaskParams *mpi = nullptr, const PairParams *pp = nullptr) {
    sasa_b200_ctx *ctx = b->ctx;
    int n_small = 0;
    for (const Launch &L : ch.launches) n_small += L.cfg >= 0;
    // device-resident runs only: in the pipelined host path the sibling streams would be shared by chunks in flight on
    // different copy streams and delay their D2H (measured: -5 % end to end), while the next chunk back-fills anyway
    const bool fork = (variant & 2) && n_small > 1 && n_small <= sasa_b200_ctx::kSide + 1;
    if (fork) CU_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
    int small_idx = 0, forked = 0;
    // grouped runs with more than 128 points: no fused kernel, every structure takes the large-structure path
    const bool all_large = gp && base.n_points > 128;
    for (const Launch &L : ch.launches) {
        KParams kp = base;
        kp.order = order_override ? order_override : b->d_order[variant] + L.order_off;
        kp.n_work = L.n_work;
        kp.work_counter = b->d_counters + L.counter;
        if (L.cfg < 0 || all_large) {
            if (ctx->large_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_large, 0));
            int rc = large_enqueue(ctx->sm_count, ctx->large, kp, &b->h_order[variant][L.order_off], L.n_work,
                                   b->h_off.data(), b->h_seg_off.empty() ? nullptr : b->h_seg_off.data(), st, launches, 0, 1, gp, mp, mpi, pp);
            if (rc != 0) return fail(ctx, rc, "large-structure path failed: %s", cudaGetErrorString(cudaGetLastError()));
            CU_TRY(ctx, cudaEventRecord(ctx->ev_large, st));
            ctx->large_used = true;
            continue;
        }
        const SmallCfg &c = ctx->cfgs[L.cfg];
        const bool has_cls = (variant & 1) == 1, grouped = gp != nullptr;
        kp.nmax = cfg_capacity(ctx, c, has_cls, grouped);
        kp.cmax = c.cmax;
        const size_t smem = c.smem[(has_cls ? 1 : 0) + (grouped ? 2 : 0)];
        const int grid = (int)std::min<uint32_t>(L.n_work, (uint32_t)(ctx->sm_count * c.minb));
        cudaStream_t ls = st;
        if (fork && small_idx > 0) {
            ls = ctx->side[small_idx - 1];
            CU_TRY(ctx, cudaStreamWaitEvent(ls, ctx->ev_fork, 0));
        }
        // (kernel arguments past the kernel's own are not read)
        void *args[] = {(void *)&kp, gp ? (void *)gp : (void *)mp, pp ? (void *)pp : (void *)mp, (void *)mpi};
        const bool tight = kp.n_points <= 128 && (kp.flags & 3u) == 0;
        const int slot = kernel_slot(grouped, mp != nullptr, has_cls, tight, pp != nullptr);
        const void *fn = kProtos[c.proto].fn[slot];
        if (!ctx->attr_done[c.proto][slot]) {
            cudaError_t ea = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (ea != cudaSuccess)
                return fail(ctx, SASA_B200_ERR_CUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize=%zu) failed: %s", smem, cudaGetErrorString(ea));
            ctx->attr_done[c.proto][slot] = true;
        }
        cudaError_t e = cudaLaunchKernel(fn, dim3(grid), dim3(c.nt), args, smem, ls);
        if (e != cudaSuccess) return fail(ctx, SASA_B200_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
        if (ls != st) {
            CU_TRY(ctx, cudaEventRecord(ctx->ev_join[small_idx - 1], ls));
            forked = small_idx;
        }
        ++small_idx;
        ++*launches;
    }
    for (int i = 0; i < forked; ++i) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_join[i], 0));
    return SASA_B200_OK;
}

int finish_run(sasa_b200_batch *b, sasa_b200_stats *stats) {
    sasa_b200_ctx *ctx = b->ctx;
    int h_err = 0;
    unsigned long long h_stat[3] = {0, 0, 0};
    CU_TRY(ctx, cudaMemcpy(&h_err, ctx->d_err, sizeof h_err, cudaMemcpyDeviceToHost));
    CU_TRY(ctx, cudaMemcpy(h_stat, ctx->d_stat, sizeof h_stat, cudaMemcpyDeviceToHost));
    b->last.n_atoms = b->n_atoms;
    b->last.n_structures = b->S;
    b->last.boundary_points = h_stat[0];
    b->last.neighbor_pairs = h_stat[1];
    b->last.streamed_atoms = h_stat[2];
    b->last.gpu_launches = b->launches_last;
    if (stats) *stats = b->last;
    if (h_err == SASA_B200_ERR_NON_FINITE)
        return fail(ctx, SASA_B200_ERR_NON_FINITE, "non-finite coordinate or radius in the input (the reference panics here)");
    if (h_err == SASA_B200_ERR_INVALID_ARGUMENT) {   // only raised by the pairs kernels: an atom with more partners than slots
        uint32_t need = 0;
        CU_TRY(ctx, cudaMemcpy(&need, ctx->d_needed + 1, sizeof need, cudaMemcpyDeviceToHost));
        return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "too few partner slots: the batch needs max_partners = %u", need);
    }
    if (h_err) return fail(ctx, h_err, "device-side error %d", h_err);
    return SASA_B200_OK;
}

}  // namespace

// =====================================================================================================
extern "C" {

int sasa_b200_abi_version(void) { return SASA_B200_ABI_VERSION; }

const char *sasa_b200_last_error(const sasa_b200_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int sasa_b200_device_count(int *out_count) {
    if (!out_count) return SASA_B200_ERR_INVALID_ARGUMENT;
    *out_count = 0;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return fail(nullptr, SASA_B200_ERR_CUDA, "no CUDA device available (%s)", cudaGetErrorString(e));
    *out_count = count;
    return SASA_B200_OK;
}

int sasa_b200_create(int device, sasa_b200_ctx **out_ctx) {
    if (!out_ctx) return fail(nullptr, SASA_B200_ERR_INVALID_ARGUMENT, "out_ctx is NULL");
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, SASA_B200_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0) {
        if ((e = cudaGetDevice(&device)) != cudaSuccess) return fail(nullptr, SASA_B200_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
    }
    if (device >= count) return fail(nullptr, SASA_B200_ERR_INVALID_ARGUMENT, "device %d out of range (%d devices)", device, count);
    sasa_b200_ctx *ctx = new sasa_b200_ctx();
    ctx->device = device;
    auto bail = [&](int code, const char *what, cudaError_t ce) {
        int rc = fail(nullptr, code, "%s: %s", what, cudaGetErrorString(ce));
        delete ctx;
        return rc;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaGetDeviceProperties", e);
    if (prop.major < 10) {
        int rc = fail(nullptr, SASA_B200_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                      device, prop.major, prop.minor);
        delete ctx;
        return rc;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    for (int i = 0; i < kStreams; ++i)
        if ((e = cudaStreamCreateWithFlags(&ctx->streams[i], cudaStreamNonBlocking)) != cudaSuccess)
            return bail(SASA_B200_ERR_CUDA, "cudaStreamCreate", e);
    for (int i = 0; i < sasa_b200_ctx::kSide; ++i) {
        if ((e = cudaStreamCreateWithFlags(&ctx->side[i], cudaStreamNonBlocking)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaStreamCreate", e);
        if ((e = cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaEventCreate", e);
    }
    if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_large, cudaEventDisableTiming)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaEventCreate", e);
    for (int i = 0; i < kStreams; ++i)
        if ((e = cudaEventCreateWithFlags(&ctx->ev_tail[i], cudaEventDisableTiming)) != cudaSuccess) return bail(SASA_B200_ERR_CUDA, "cudaEventCreate", e);
    {   // per-batch topology arrays come from the stream-ordered pool: keep freed blocks cached instead of returning them
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    if ((e = cudaMalloc(&ctx->d_err, sizeof(int))) != cudaSuccess) return bail(SASA_B200_ERR_OUT_OF_MEMORY, "cudaMalloc", e);
    if ((e = cudaMalloc(&ctx->d_stat, 3 * sizeof(unsigned long long))) != cudaSuccess) return bail(SASA_B200_ERR_OUT_OF_MEMORY, "cudaMalloc", e);
    if ((e = cudaMalloc(&ctx->d_needed, 2 * sizeof(uint32_t))) != cudaSuccess) return bail(SASA_B200_ERR_OUT_OF_MEMORY, "cudaMalloc", e);
    cudaMemset(ctx->d_needed, 0, 2 * sizeof(uint32_t));
    cudaMemset(ctx->d_err, 0, sizeof(int));
    cudaMemset(ctx->d_stat, 0, 3 * sizeof(unsigned long long));
    int rc = build_cfgs(ctx);
    if (rc != SASA_B200_OK) {
        g_create_error = ctx->err;
        sasa_b200_destroy(ctx);
        return rc;
    }
    *out_ctx = ctx;
    return SASA_B200_OK;
}

void sasa_b200_destroy(sasa_b200_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto &kv : ctx->points) {
        if (kv.second.cap_tex) cudaDestroyTextureObject(kv.second.cap_tex);
        cudaFree(kv.second.d); cudaFree(kv.second.cap); cudaFree(kv.second.d4); cudaFree(kv.second.capm_in); cudaFree(kv.second.capm_rg);
    }
    for (int i = 0; i < kStreams; ++i)
        if (ctx->streams[i]) cudaStreamDestroy(ctx->streams[i]);
    for (int i = 0; i < sasa_b200_ctx::kSide; ++i) {
        if (ctx->side[i]) cudaStreamDestroy(ctx->side[i]);
        if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_large) cudaEventDestroy(ctx->ev_large);
    for (int i = 0; i < kStreams; ++i)
        if (ctx->ev_tail[i]) cudaEventDestroy(ctx->ev_tail[i]);
    for (sasa_b200_job *j : ctx->free_jobs) {
        cudaEventDestroy(j->ev0);
        cudaEventDestroy(j->ev1);
        cudaFreeHost(j->h_status);
        cudaFreeHost(j->h_ready);
        delete j;
    }
    for (auto &sp : ctx->slots) {
        if (sp->st) cudaStreamDestroy(sp->st);
        large_release(sp->large);
        cudaFree(sp->d_buf);
        cudaFreeHost(sp->h_pin);
    }
    large_release(ctx->large);
    cudaFree(ctx->d_err);
    cudaFree(ctx->d_stat);
    cudaFree(ctx->d_needed);
    cudaFree(ctx->arena);
    delete ctx;
}

int sasa_b200_alloc_pinned(size_t bytes, void **out_ptr) {
    if (!out_ptr) return SASA_B200_ERR_INVALID_ARGUMENT;
    cudaError_t e = cudaHostAlloc(out_ptr, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(nullptr, SASA_B200_ERR_OUT_OF_MEMORY, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
    return SASA_B200_OK;
}

int sasa_b200_free_pinned(void *ptr) {
    if (!ptr) return SASA_B200_OK;
    return cudaFreeHost(ptr) == cudaSuccess ? SASA_B200_OK : SASA_B200_ERR_CUDA;
}

int sasa_b200_sphere_points(uint32_t n_points, float *xyz) {
    if (!xyz || n_points == 0) return SASA_B200_ERR_INVALID_ARGUMENT;
    std::vector<float> h(3 * (size_t)n_points);
    sphere_points_host(n_points, h.data(), h.data() + n_points, h.data() + 2 * (size_t)n_points);
    for (uint32_t i = 0; i < n_points; ++i) {
        xyz[3 * i + 0] = h[i];
        xyz[3 * i + 1] = h[n_points + i];
        xyz[3 * i + 2] = h[2 * (size_t)n_points + i];
    }
    return SASA_B200_OK;
}

static int batch_create_impl(sasa_b200_ctx *ctx, const uint64_t *struct_off, size_t S, const uint32_t *seg_be,
                             const uint64_t *struct_seg_off, const uint8_t *seg_polar, sasa_b200_batch **out_batch,
                             bool single_latency) {
    if (!ctx) return SASA_B200_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!out_batch || (!struct_off && S)) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "struct_off / out_batch is NULL");
    *out_batch = nullptr;
    if (S && struct_off[0] != 0) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "struct_off[0] must be 0");
    for (size_t i = 0; i < S; ++i)
        if (struct_off[i + 1] < struct_off[i]) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "struct_off must be non-decreasing");
    if (S && struct_off[S] >= (1ull << 32)) return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "more than 2^32 atoms in one batch");
    if (S >= (1ull << 31)) return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "too many structures");
    if (seg_be && !struct_seg_off) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "seg_be without struct_seg_off");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    sasa_b200_batch *b = new sasa_b200_batch();
    b->ctx = ctx;
    b->S = S;
    b->single_latency = single_latency;
    b->h_off.resize(S + 1, 0);
    for (size_t i = 0; i <= S && S; ++i) b->h_off[i] = (uint32_t)struct_off[i];
    b->n_atoms = S ? b->h_off[S] : 0;
    auto cleanup = [&](int rc) {
        sasa_b200_batch_destroy(b);
        return rc;
    };
    if (seg_be && S) {
        if (struct_seg_off[0] != 0) return cleanup(fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "struct_seg_off[0] must be 0"));
        for (size_t i = 0; i < S; ++i)
            if (struct_seg_off[i + 1] < struct_seg_off[i]) return cleanup(fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "struct_seg_off must be non-decreasing"));
        if (struct_seg_off[S] >= (1ull << 32)) return cleanup(fail(ctx, SASA_B200_ERR_UNSUPPORTED, "too many segments"));
        b->n_seg = struct_seg_off[S];
        b->h_seg_off.resize(S + 1);
        for (size_t i = 0; i <= S; ++i) b->h_seg_off[i] = (uint32_t)struct_seg_off[i];
        for (size_t s = 0; s < S; ++s) {
            const uint32_t n = b->h_off[s + 1] - b->h_off[s];
            for (uint64_t k = struct_seg_off[s]; k < struct_seg_off[s + 1]; ++k)
                if (seg_be[2 * k] > seg_be[2 * k + 1] || seg_be[2 * k + 1] > n)
                    return cleanup(fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "segment %llu of structure %zu is not a range inside its structure",
                                        (unsigned long long)k, s));
        }
    }
    for (int v = 0; v < 8; ++v) build_plan(b, v);
    for (int v = 0; v < 2; ++v) build_gated_order(b, v);
    for (size_t i = 0; i < S; ++i) b->max_struct = std::max(b->max_struct, b->h_off[i + 1] - b->h_off[i]);
#define B_TRY(expr)                                                                                            \
    do {                                                                                                       \
        cudaError_t e__ = (expr);                                                                              \
        if (e__ != cudaSuccess)                                                                                \
            return cleanup(fail(ctx, e__ == cudaErrorMemoryAllocation ? SASA_B200_ERR_OUT_OF_MEMORY : SASA_B200_ERR_CUDA, \
                                "%s failed: %s", #expr, cudaGetErrorString(e__)));                             \
    } while (0)
    cudaStream_t ps = ctx->streams[0];
    B_TRY(cudaSetDevice(ctx->device));
    B_TRY(cudaMallocAsync(&b->d_off, (S + 1) * sizeof(uint32_t), ps));
    B_TRY(cudaMemcpyAsync(b->d_off, b->h_off.data(), (S + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ps));
    for (int v = 0; v < 8; ++v) {
        B_TRY(cudaMallocAsync(&b->d_order[v], std::max<size_t>(1, b->h_order[v].size()) * sizeof(uint32_t), ps));
        if (!b->h_order[v].empty())
            B_TRY(cudaMemcpyAsync(b->d_order[v], b->h_order[v].data(), b->h_order[v].size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ps));
    }
    for (int v = 0; v < 2; ++v) {
        if (b->h_gorder[v].empty()) continue;
        B_TRY(cudaMallocAsync(&b->d_gorder[v], b->h_gorder[v].size() * sizeof(uint32_t), ps));
        B_TRY(cudaMallocAsync(&b->d_gneed[v], b->h_gneed[v].size() * sizeof(uint32_t), ps));
        B_TRY(cudaMemcpyAsync(b->d_gorder[v], b->h_gorder[v].data(), b->h_gorder[v].size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ps));
        B_TRY(cudaMemcpyAsync(b->d_gneed[v], b->h_gneed[v].data(), b->h_gneed[v].size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ps));
    }
    B_TRY(cudaMallocAsync(&b->d_counters, std::max<uint32_t>(1, *std::max_element(b->n_counters, b->n_counters + 8)) * sizeof(uint32_t), ps));
    if (b->n_seg) {
        B_TRY(cudaMallocAsync(&b->d_seg_be, b->n_seg * sizeof(uint2), ps));
        B_TRY(cudaMemcpyAsync(b->d_seg_be, seg_be, b->n_seg * sizeof(uint2), cudaMemcpyHostToDevice, ps));
        B_TRY(cudaMallocAsync(&b->d_seg_off, (S + 1) * sizeof(uint32_t), ps));
        B_TRY(cudaMemcpyAsync(b->d_seg_off, b->h_seg_off.data(), (S + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ps));
        if (seg_polar) {
            B_TRY(cudaMallocAsync(&b->d_polar, b->n_seg, ps));
            B_TRY(cudaMemcpyAsync(b->d_polar, seg_polar, b->n_seg, cudaMemcpyHostToDevice, ps));
            b->has_polar = true;
        }
    }
    B_TRY(cudaStreamSynchronize(ps));   // the caller's arrays may go away; the topology is complete for any stream from here on
    if (b->max_large) {   // (ctx->mu is held since the top of this function)
        if (b->max_large > ctx->large.cap_atoms) cudaDeviceSynchronize();   // growing frees buffers a run in flight may still use
        int rc = large_reserve(ctx->large, b->max_large);
        if (rc) return cleanup(fail(ctx, rc, "allocating the large-structure workspace (%u atoms) failed", b->max_large));
    }
#undef B_TRY
    *out_batch = b;
    return SASA_B200_OK;
}

int sasa_b200_batch_create(sasa_b200_ctx *ctx, const uint64_t *struct_off, size_t S, const uint32_t *seg_be,
                           const uint64_t *struct_seg_off, const uint8_t *seg_polar, sasa_b200_batch **out_batch) {
    return batch_create_impl(ctx, struct_off, S, seg_be, struct_seg_off, seg_polar, out_batch, false);
}

void sasa_b200_batch_destroy(sasa_b200_batch *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaDeviceSynchronize();
    cudaStream_t ps = b->ctx->streams[0];
    if (b->d_off) cudaFreeAsync(b->d_off, ps);
    if (b->d_seg_off) cudaFreeAsync(b->d_seg_off, ps);
    for (int v = 0; v < 8; ++v)
        if (b->d_order[v]) cudaFreeAsync(b->d_order[v], ps);
    for (int v = 0; v < 2; ++v) {
        if (b->d_gorder[v]) cudaFreeAsync(b->d_gorder[v], ps);
        if (b->d_gneed[v]) cudaFreeAsync(b->d_gneed[v], ps);
    }
    if (b->d_counters) cudaFreeAsync(b->d_counters, ps);
    if (b->d_seg_be) cudaFreeAsync(b->d_seg_be, ps);
    if (b->d_polar) cudaFreeAsync(b->d_polar, ps);
    delete b;
}

// Checks of the grouped entry points (after check_params), and the large-structure workspace their plan needs: structures that
// no longer fit the fused kernels with the group arrays, or -- n_points > 128 -- every structure.  (ctx->mu is held.)
static int prepare_groups(sasa_b200_batch *b, const uint32_t *group, const sasa_b200_params *params, const sasa_b200_outputs *out_iso,
                          int variant) {
    sasa_b200_ctx *ctx = b->ctx;
    if (!group && b->n_atoms) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "group is NULL");
    if (!out_iso) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    if (params->flags != 0)
        return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "grouped runs support no flags (boundary statistics, forced streaming), got %u", params->flags);
    const uint32_t need = params->n_points > 128 ? b->max_struct : b->max_large_v[variant];
    if (need > ctx->large.cap_atoms) {
        cudaDeviceSynchronize();   // growing frees buffers a run in flight may still use
        int rc = large_reserve(ctx->large, need);
        if (rc) return fail(ctx, rc, "allocating the large-structure workspace (%u atoms) failed", need);
    }
    return SASA_B200_OK;
}

// Checks of the masked entry points (after check_params): a mask buffer for every atom whose size fits a size_t.  name: the
// buffer's argument name, for the error message.
static int check_masks(sasa_b200_batch *b, const uint32_t *exposed, const sasa_b200_params *params, const char *name = "exposed") {
    if (!exposed && b->n_atoms) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "%s is NULL", name);
    if (b->n_atoms && mask_words(params->n_points) > SIZE_MAX / 4 / b->n_atoms)
        return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "the mask buffer (%zu atoms x %u words) overflows size_t", b->n_atoms,
                    mask_words(params->n_points));
    return SASA_B200_OK;
}

// Checks of the pairwise buried-area entry points: slot outputs for every atom, 1..16 slots per atom, a slot buffer whose size
// fits a size_t.
static int check_pairs(sasa_b200_batch *b, const sasa_b200_pair_outputs *pairs) {
    if (!pairs) return b->n_atoms ? fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "pairs is NULL") : SASA_B200_OK;
    if (pairs->max_partners < 1 || pairs->max_partners > 16)
        return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "max_partners must be 1..16, got %u", pairs->max_partners);
    if (!pairs->partner && b->n_atoms) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "pairs->partner is NULL");
    if (b->n_atoms && pairs->max_partners > SIZE_MAX / 4 / b->n_atoms)
        return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "the slot buffers (%zu atoms x %u slots) overflow size_t", b->n_atoms,
                    pairs->max_partners);
    return SASA_B200_OK;
}

// d_iso: grouped runs; masked: d_exposed receives the exposed-point masks, and with d_iso d_exposed_iso the isolated ones.
// pairs (with d_iso): pairwise buried area, d_pairs receives the partner slots.
static int run_device_impl(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class, const uint32_t *d_group,
                           const sasa_b200_params *params, const sasa_b200_outputs *d_out, const sasa_b200_outputs *d_iso, void *stream,
                           bool masked = false, uint32_t *d_exposed = nullptr, uint32_t *d_exposed_iso = nullptr, bool pairs = false,
                           const sasa_b200_pair_outputs *d_pairs = nullptr) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!d_out || (!d_xyzr && b->n_atoms)) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_xyzr / d_out is NULL");
    int rc = check_params(ctx, params);
    if (rc) return rc;
    const bool grouped = d_iso != nullptr;
    if (masked && (rc = check_masks(b, d_exposed, params)) != 0) return rc;
    if (masked && grouped && (rc = check_masks(b, d_exposed_iso, params, "exposed_isolated")) != 0) return rc;
    const MaskParams mp{d_exposed}, mpi{d_exposed_iso};
    const int variant = (d_id_class ? 1 : 0) + 2 + (grouped ? 4 : 0);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (grouped && (rc = prepare_groups(b, d_group, params, d_iso, variant)) != 0) return rc;
    if (pairs && (rc = check_pairs(b, d_pairs)) != 0) return rc;
    if (pairs && !d_pairs) pairs = false;   // (an empty batch: no slots to write)
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->streams[0];
    PairParams pp{};
    if (pairs) {
        pp = PairParams{d_pairs->partner, d_pairs->buried_counts, d_pairs->buried_area, ctx->d_needed, d_pairs->max_partners};
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_needed, 0, sizeof(uint32_t), st));
    }
    RunArgs ra;
    ra.d_xyzr = reinterpret_cast<const float4 *>(d_xyzr);
    ra.d_cls = d_id_class;
    ra.d_out = *d_out;
    GroupParams gp{};
    if (grouped) gp = GroupParams{d_group, d_iso->counts, d_iso->atom_sasa, b->n_seg ? d_iso->seg_sasa : nullptr, d_iso->protein};
    ra.prm = *params;
    if ((rc = get_points(ctx, params->n_points, &ra.pts)) != 0) return rc;
    KParams base;
    make_kparams(b, ra, &base);
    b->launches_last = 0;
    if (b->n_counters[variant])
        CU_TRY(ctx, cudaMemsetAsync(b->d_counters, 0, b->n_counters[variant] * sizeof(uint32_t), st));
    for (const Chunk &ch : b->plan[variant])
        if ((rc = enqueue_chunk(b, variant, ch, base, st, &b->launches_last, nullptr, grouped ? &gp : nullptr, masked ? &mp : nullptr,
                                masked && grouped ? &mpi : nullptr, pairs ? &pp : nullptr)) != 0)
            return rc;
    if (pairs && d_pairs->partners_needed)
        CU_TRY(ctx, cudaMemcpyAsync(d_pairs->partners_needed, ctx->d_needed, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    return SASA_B200_OK;
}

int sasa_b200_batch_run_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class,
                               const sasa_b200_params *params, const sasa_b200_outputs *d_out, void *stream) {
    return run_device_impl(b, d_xyzr, d_id_class, nullptr, params, d_out, nullptr, stream);
}

int sasa_b200_batch_run_groups_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class, const uint32_t *d_group,
                                      const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                      const sasa_b200_outputs *d_out_isolated, void *stream) {
    if (b && !d_out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_out_isolated is NULL");
    return run_device_impl(b, d_xyzr, d_id_class, d_group, params, d_out, d_out_isolated, stream);
}

int sasa_b200_batch_run_masks_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class, const sasa_b200_params *params,
                                     const sasa_b200_outputs *d_out, uint32_t *d_exposed, void *stream) {
    return run_device_impl(b, d_xyzr, d_id_class, nullptr, params, d_out, nullptr, stream, true, d_exposed);
}

int sasa_b200_batch_run_groups_masks_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class, const uint32_t *d_group,
                                            const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                            const sasa_b200_outputs *d_out_isolated, uint32_t *d_exposed, uint32_t *d_exposed_isolated,
                                            void *stream) {
    if (b && !d_out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_out_isolated is NULL");
    return run_device_impl(b, d_xyzr, d_id_class, d_group, params, d_out, d_out_isolated, stream, true, d_exposed, d_exposed_isolated);
}

int sasa_b200_batch_run_group_pairs_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class, const uint32_t *d_group,
                                           const sasa_b200_params *params, const sasa_b200_outputs *d_out,
                                           const sasa_b200_outputs *d_out_isolated, const sasa_b200_pair_outputs *d_pairs, void *stream) {
    if (b && !d_out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_out_isolated is NULL");
    return run_device_impl(b, d_xyzr, d_id_class, d_group, params, d_out, d_out_isolated, stream, false, nullptr, nullptr, true, d_pairs);
}

int sasa_b200_batch_sync(sasa_b200_batch *b, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaDeviceSynchronize());
    int rc = finish_run(b, stats);
    cudaMemset(ctx->d_err, 0, sizeof(int));
    cudaMemset(ctx->d_stat, 0, 3 * sizeof(unsigned long long));
    cudaMemset(ctx->d_needed, 0, 2 * sizeof(uint32_t));
    return rc;
}

// ---- host-buffer runs as jobs ---------------------------------------------------------------------------------------
// submit: everything of one run is enqueued -- H2D copies, kernels, D2H copies into the caller's buffers, chunk by chunk on
// three streams -- and the call returns; wait: blocks on the job's last event and reports.  The context mutex is held only
// while enqueueing, so callers on several threads interleave their jobs instead of queueing for whole runs.  A job owns a
// stream-ordered arena (cudaMallocAsync; the pool keeps freed blocks) and its own error / statistics words.
static sasa_b200_job *job_acquire(sasa_b200_ctx *ctx) {
    sasa_b200_job *j = nullptr;
    if (!ctx->free_jobs.empty()) {
        j = ctx->free_jobs.back();
        ctx->free_jobs.pop_back();
    } else {
        j = new sasa_b200_job();
        if (cudaEventCreate(&j->ev0) != cudaSuccess || cudaEventCreate(&j->ev1) != cudaSuccess ||
            cudaHostAlloc((void **)&j->h_status, 5 * sizeof(unsigned long long), cudaHostAllocDefault) != cudaSuccess ||
            cudaHostAlloc((void **)&j->h_ready, kMaxGatedChunks * sizeof(uint32_t), cudaHostAllocDefault) != cudaSuccess) {
            if (j->ev0) cudaEventDestroy(j->ev0);
            if (j->ev1) cudaEventDestroy(j->ev1);
            if (j->h_status) cudaFreeHost(j->h_status);
            if (j->h_ready) cudaFreeHost(j->h_ready);
            delete j;
            return nullptr;
        }
    }
    return j;
}

// Failure after work was queued: nothing may still write into the caller's buffers or read the arena once the call returns.
static int job_abort(sasa_b200_ctx *ctx, sasa_b200_job *j, int rc) {
    for (int i = 0; i < kStreams; ++i) cudaStreamSynchronize(ctx->streams[i]);
    if (j->d_arena) cudaFreeAsync(j->d_arena, ctx->streams[0]);
    j->d_arena = nullptr;
    if (j->batch) j->batch->in_flight = nullptr;
    j->active = false;
    ctx->tail_valid = false;
    ctx->free_jobs.push_back(j);
    cudaGetLastError();
    return rc;
}

static int submit_host_impl(sasa_b200_batch *b, const float *xyzr, const float *xyz3, const float *radii,
                            const uint32_t *id_class, const sasa_b200_params *params, const sasa_b200_outputs *out,
                            sasa_b200_job **out_job, const uint8_t *ridx = nullptr, size_t n_palette = 0,
                            const uint32_t *group = nullptr, const sasa_b200_outputs *out_iso = nullptr, bool masked = false,
                            uint32_t *exposed = nullptr, uint32_t *exposed_iso = nullptr, bool pairs = false,
                            const sasa_b200_pair_outputs *pair_out = nullptr, const sasa_b200_pair_sums *sums = nullptr) {
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!out || !out_job) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out / out_job is NULL");
    *out_job = nullptr;
    if (b->n_atoms && !xyzr && !(xyz3 && radii)) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "atom data is NULL");
    if (b->in_flight) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "this batch already has a run in flight: wait for it first");
    int rc = check_params(ctx, params);
    if (rc) return rc;
    const bool grouped = out_iso != nullptr;   // sasa_b200_batch_run_groups_host: per-chunk pipeline only
    if (masked && (rc = check_masks(b, exposed, params)) != 0) return rc;
    if (masked && grouped && (rc = check_masks(b, exposed_iso, params, "exposed_isolated")) != 0) return rc;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t N = b->n_atoms, S = b->S, G = b->n_seg;
    const size_t W = mask_words(params->n_points);
    const int variant = (id_class ? 1 : 0) + (grouped ? 4 : 0);
    if (grouped && (rc = prepare_groups(b, group, params, out_iso, variant)) != 0) return rc;
    // sums (pairwise buried area of MD frames): the slot rows stay in the arena, only their sums per frame and segment come back
    if (pairs && !sums && (rc = check_pairs(b, pair_out)) != 0) return rc;
    if (pairs && !sums && !pair_out) pairs = false;   // (an empty batch: no slots to write)
    const bool indexed = xyz3 != nullptr && ridx != nullptr;   // 13 B/atom: coordinates + a palette index per atom
    const bool frames = xyz3 != nullptr;                       // any 12-byte coordinate form
    size_t fN = 0;  // atoms per frame (MD form) / palette entries (indexed form)
    if (indexed) {
        fN = n_palette;
    } else if (frames) {
        fN = S ? b->h_off[1] - b->h_off[0] : 0;
        for (size_t s = 0; s < S; ++s)
            if (b->h_off[s + 1] - b->h_off[s] != fN)
                return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "run_frames needs equal-sized structures");
    }
    if (indexed && (n_palette == 0 || n_palette > 256)) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "the radius palette holds 1..256 entries");
    // K = L - 1 slots hold every partner an atom can have, so the too-few-slots failure of the pairs kernels cannot occur
    const uint32_t L = sums ? sums->n_labels : 0;
    if (sums) {
        if (L < 1 || L > kPairSumsMaxLabels) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "n_labels must be 1..%u, got %u", kPairSumsMaxLabels, L);
        if (!sums->pair_area && N) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "sums->pair_area is NULL");
        for (size_t i = 0; i < fN; ++i)
            if (group[i] >= L)
                return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "group[%zu] = %u is not below n_labels = %u", i, group[i], L);
        if ((N && std::max<size_t>(1, L - 1) > SIZE_MAX / 4 / N) || (S && (size_t)L * L > SIZE_MAX / 8 / S) || (G && L > SIZE_MAX / 8 / G))
            return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "the pair outputs (%zu frames, %zu segments, %u labels) overflow size_t", S, G, L);
        if (!N) pairs = false;
    }
    const bool want_sums = sums && sums->pair_area;
    const bool want_seg_sums = want_sums && sums->seg_pair_area && G;
    const size_t K = sums ? std::max<size_t>(1, L - 1) : pairs ? pair_out->max_partners : 0;
    // grouped MD form: `group` holds the fN labels of one frame, shared by every frame; they cross the wire once and are
    // expanded on the device chunk by chunk (expand_frame_labels_kernel)
    const bool frame_labels = frames && grouped;
    const Points *pts = nullptr;
    if ((rc = get_points(ctx, params->n_points, &pts)) != 0) return rc;
    sasa_b200_job *job = job_acquire(ctx);
    if (!job) return fail(ctx, SASA_B200_ERR_CUDA, "creating the job's events / status word failed");
    job->batch = b;
    job->t_begin = std::chrono::steady_clock::now();
    job->launches = 0;
    job->pairs = pairs ? pair_out : nullptr;
    // carve the arena
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o = 0;
    const size_t o_status = o; o += 256;
    const size_t o_xyzr = o;   o += al(N * 16);
    const size_t o_xyz3 = o;   o += frames ? al(N * 12) : 0;
    const size_t o_rad = o;    o += frames ? al(fN * 4) : 0;
    const size_t o_ridx = o;   o += indexed ? al(N) : 0;
    const size_t o_cls = o;    o += id_class ? al(N * 4) : 0;
    const size_t o_cnt = o;    o += out->counts ? al(N * 4) : 0;
    const size_t o_atom = o;   o += out->atom_sasa ? al(N * 4) : 0;
    const size_t o_seg = o;    o += (out->seg_sasa && G) ? al(G * 4) : 0;
    const size_t o_prot = o;   o += out->protein ? al(S * 12) : 0;
    const size_t o_grp = o;    o += grouped ? al(N * 4) : 0;
    const size_t o_lab = o;    o += frame_labels ? al(fN * 4) : 0;
    const size_t o_icnt = o;   o += (grouped && out_iso->counts) ? al(N * 4) : 0;
    const size_t o_iatom = o;  o += (grouped && out_iso->atom_sasa) ? al(N * 4) : 0;
    const size_t o_iseg = o;   o += (grouped && out_iso->seg_sasa && G) ? al(G * 4) : 0;
    const size_t o_iprot = o;  o += (grouped && out_iso->protein) ? al(S * 12) : 0;
    const size_t o_mask = o;   o += masked ? al(N * W * 4) : 0;
    const size_t o_imask = o;  o += (masked && grouped) ? al(N * W * 4) : 0;
    const size_t o_ppart = o;  o += pairs ? al(N * K * 4) : 0;
    const size_t o_pcnt = o;   o += (pairs && pair_out && pair_out->buried_counts) ? al(N * K * 4) : 0;
    const size_t o_parea = o;  o += (pairs && (sums || pair_out->buried_area)) ? al(N * K * 4) : 0;
    const size_t o_psum = o;   o += want_sums ? al(S * L * L * 8) : 0;
    const size_t o_pseg = o;   o += want_seg_sums ? al(G * L * 8) : 0;
    cudaStream_t s0 = ctx->streams[0];
    // the previous job may still be running on the sibling streams: this job's first stream starts behind all of them
    if (ctx->tail_valid)
        for (int i = 1; i < kStreams; ++i) cudaStreamWaitEvent(s0, ctx->ev_tail[i], 0);
    {
        cudaError_t e = cudaMallocAsync(&job->d_arena, o + 256, s0);
        if (e != cudaSuccess) {
            job->d_arena = nullptr;
            job_abort(ctx, job, 0);
            return fail(ctx, e == cudaErrorMemoryAllocation ? SASA_B200_ERR_OUT_OF_MEMORY : SASA_B200_ERR_CUDA,
                        "cudaMallocAsync(%zu) failed: %s", o + 256, cudaGetErrorString(e));
        }
    }
    b->in_flight = job;
    job->active = true;
#define J_TRY(expr)                                                                                                       \
    do {                                                                                                                  \
        cudaError_t e__ = (expr);                                                                                         \
        if (e__ != cudaSuccess)                                                                                           \
            return job_abort(ctx, job, fail(ctx, e__ == cudaErrorMemoryAllocation ? SASA_B200_ERR_OUT_OF_MEMORY : SASA_B200_ERR_CUDA, \
                                            "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__)); \
    } while (0)
    char *base_p = static_cast<char *>(job->d_arena);
    RunArgs ra;
    ra.d_xyzr = reinterpret_cast<const float4 *>(base_p + o_xyzr);
    ra.d_cls = id_class ? reinterpret_cast<const uint32_t *>(base_p + o_cls) : nullptr;
    ra.d_out.counts = out->counts ? reinterpret_cast<uint32_t *>(base_p + o_cnt) : nullptr;
    ra.d_out.atom_sasa = out->atom_sasa ? reinterpret_cast<float *>(base_p + o_atom) : nullptr;
    ra.d_out.seg_sasa = (out->seg_sasa && G) ? reinterpret_cast<float *>(base_p + o_seg) : nullptr;
    ra.d_out.protein = out->protein ? reinterpret_cast<float *>(base_p + o_prot) : nullptr;
    GroupParams gp{};
    if (grouped) {
        gp.grp = reinterpret_cast<const uint32_t *>(base_p + o_grp);
        gp.counts = out_iso->counts ? reinterpret_cast<uint32_t *>(base_p + o_icnt) : nullptr;
        gp.atom = out_iso->atom_sasa ? reinterpret_cast<float *>(base_p + o_iatom) : nullptr;
        gp.seg = (out_iso->seg_sasa && G) ? reinterpret_cast<float *>(base_p + o_iseg) : nullptr;
        gp.protein = out_iso->protein ? reinterpret_cast<float *>(base_p + o_iprot) : nullptr;
    }
    const MaskParams mp{masked ? reinterpret_cast<uint32_t *>(base_p + o_mask) : nullptr};
    const MaskParams mpi{(masked && grouped) ? reinterpret_cast<uint32_t *>(base_p + o_imask) : nullptr};
    // ---- gated single-launch pipeline ----------------------------------------------------------------------------------
    // Thirteen launches of 148 persistent CTAs cost the pipelined run 0.25 ms over the same work as ONE launch (CTA start-ups
    // with a cold first structure, per-chunk instead of batch-wide queue; DESIGN.md section 6).  When every chunk of the plan is one
    // launch of the same fused configuration, the whole batch is therefore ONE launch over the chunk-major queue: the copy
    // stream raises a counter in device memory after every chunk's copy, a CTA that claims a queue position beyond it waits
    // (wait_ready, sasa_small.cuh), and the kernel writes its results straight into the caller's page-locked buffers --
    // there is no D2H stage to order behind individual chunks.  Needs outputs the device can address (pinned / registered
    // host memory) of moderate size; anything else takes the per-chunk launches below.
    bool gated = variant < 2 && !masked && !b->h_gorder[variant].empty();
    if (gated) {
        const size_t out_bytes = (out->counts ? N * 4 : 0) + (out->atom_sasa ? N * 4 : 0) + ((out->seg_sasa && G) ? G * 4 : 0) +
                                 (out->protein ? S * 12 : 0);
        if (out_bytes > kGatedMaxOutBytes) gated = false;
        auto mapped = [&](const void *host, void **dev) {
            if (!host) { *dev = nullptr; return true; }
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return false; }
            if (at.type != cudaMemoryTypeHost || !at.devicePointer) return false;
            *dev = at.devicePointer;
            return true;
        };
        void *dc = nullptr, *da = nullptr, *ds = nullptr, *dp = nullptr;
        if (gated && mapped(out->counts, &dc) && mapped(out->atom_sasa, &da) && mapped((out->seg_sasa && G) ? out->seg_sasa : nullptr, &ds) &&
            mapped(out->protein, &dp)) {
            ra.d_out.counts = static_cast<uint32_t *>(dc);
            ra.d_out.atom_sasa = static_cast<float *>(da);
            ra.d_out.seg_sasa = static_cast<float *>(ds);
            ra.d_out.protein = static_cast<float *>(dp);
        } else {
            gated = false;
        }
    }
    ra.prm = *params;
    ra.pts = pts;
    KParams kbase;
    make_kparams(b, ra, &kbase);
    unsigned long long *d_status = reinterpret_cast<unsigned long long *>(base_p + o_status);
    kbase.err_flag = reinterpret_cast<int *>(d_status);
    kbase.stat = d_status + 1;
    // pairwise buried area: the partners-needed words sit behind the statistics (status word 4) and come back with them
    PairParams pp{};
    if (pairs)
        pp = PairParams{reinterpret_cast<uint32_t *>(base_p + o_ppart),
                        (pair_out && pair_out->buried_counts) ? reinterpret_cast<uint32_t *>(base_p + o_pcnt) : nullptr,
                        (sums || pair_out->buried_area) ? reinterpret_cast<float *>(base_p + o_parea) : nullptr,
                        reinterpret_cast<uint32_t *>(d_status + 4), (uint32_t)K};
    double *d_psum = reinterpret_cast<double *>(base_p + o_psum), *d_pseg = reinterpret_cast<double *>(base_p + o_pseg);
    // MD form: the fused kernels read the 12-byte coordinates and the shared radius table directly; only batches with
    // structures on the large-structure path still expand to float4 first
    // (per plan: round 1 asked "any plan", so a 5,001-atom frame -- fused without id classes, large path with them -- lost both
    // the fused unpack and the three-stream overlap: cfg3 ran 18.4 ms end to end where the kernels take 12.9 ms)
    // (grouped runs with n_points > 128 take the large-structure path for every structure, whatever the plan says)
    const bool fused_frames = frames && b->max_large_v[variant] == 0 && !(grouped && params->n_points > 128);
    if (fused_frames) {
        kbase.xyz3 = reinterpret_cast<const float *>(base_p + o_xyz3);
        kbase.radii = reinterpret_cast<const float *>(base_p + o_rad);
        if (indexed) kbase.ridx = reinterpret_cast<const uint8_t *>(base_p + o_ridx);
    }
    J_TRY(cudaMemsetAsync(d_status, 0, 128, s0));   // status words + the ready counter of the gated pipeline (at +64 bytes)
    if (b->n_counters[variant]) J_TRY(cudaMemsetAsync(b->d_counters, 0, b->n_counters[variant] * sizeof(uint32_t), s0));
    if (frames && fN) J_TRY(cudaMemcpyAsync(base_p + o_rad, radii, fN * 4, cudaMemcpyHostToDevice, s0));
    if (frame_labels && fN) J_TRY(cudaMemcpyAsync(base_p + o_lab, group, fN * 4, cudaMemcpyHostToDevice, s0));
    J_TRY(cudaEventRecord(job->ev0, s0));
    for (int i = 1; i < kStreams; ++i) J_TRY(cudaStreamWaitEvent(ctx->streams[i], job->ev0, 0));
    size_t ci = 0;
    // the large-structure workspace is shared by all chunks: keep such batches on a single stream
    const int nstreams = b->max_large_v[variant] || (grouped && params->n_points > 128) ? 1 : kStreams;
    if (gated) {
        // the one kernel first (it starts at once and waits for chunk 0 at the gate), then the copies on the first stream
        uint32_t *d_ready = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(d_status) + 64);
        KParams kg = kbase;
        kg.ready = d_ready;
        kg.need = b->d_gneed[variant];
        Chunk all;
        all.s0 = 0; all.s1 = (uint32_t)S; all.a0 = 0; all.a1 = N; all.g0 = 0; all.g1 = G;
        Launch L = b->plan[variant][0].launches[0];
        L.n_work = 0;
        for (const Chunk &ch : b->plan[variant]) L.n_work += ch.launches[0].n_work;
        all.launches.push_back(L);
        cudaStream_t sk = ctx->streams[1];
        if ((rc = enqueue_chunk(b, variant, all, kg, sk, &job->launches, b->d_gorder[variant])) != 0) return job_abort(ctx, job, rc);
        size_t c = 0;
        for (const Chunk &ch : b->plan[variant]) {
            const size_t na = ch.a1 - ch.a0;
            if (na) {
                if (frames) {
                    J_TRY(cudaMemcpyAsync(base_p + o_xyz3 + ch.a0 * 12, xyz3 + ch.a0 * 3, na * 12, cudaMemcpyHostToDevice, s0));
                    if (indexed) J_TRY(cudaMemcpyAsync(base_p + o_ridx + ch.a0, ridx + ch.a0, na, cudaMemcpyHostToDevice, s0));
                } else {
                    J_TRY(cudaMemcpyAsync(base_p + o_xyzr + ch.a0 * 16, xyzr + ch.a0 * 4, na * 16, cudaMemcpyHostToDevice, s0));
                }
                if (id_class) J_TRY(cudaMemcpyAsync(base_p + o_cls + ch.a0 * 4, id_class + ch.a0, na * 4, cudaMemcpyHostToDevice, s0));
            }
            job->h_ready[c] = (uint32_t)(c + 1);
            J_TRY(cudaMemcpyAsync(d_ready, &job->h_ready[c], sizeof(uint32_t), cudaMemcpyHostToDevice, s0));
            ++c;
        }
    } else
    for (const Chunk &ch : b->plan[variant]) {
        cudaStream_t st = ctx->streams[ci++ % nstreams];
        const size_t na = ch.a1 - ch.a0;
        if (na) {
            if (frames) {
                J_TRY(cudaMemcpyAsync(base_p + o_xyz3 + ch.a0 * 12, xyz3 + ch.a0 * 3, na * 12, cudaMemcpyHostToDevice, st));
                if (indexed) J_TRY(cudaMemcpyAsync(base_p + o_ridx + ch.a0, ridx + ch.a0, na, cudaMemcpyHostToDevice, st));
                if (!fused_frames) {
                    if (indexed)
                        pack_indexed_kernel<<<(unsigned)((na + 255) / 256), 256, 0, st>>>(
                            reinterpret_cast<const float *>(base_p + o_xyz3) + ch.a0 * 3, reinterpret_cast<const uint8_t *>(base_p + o_ridx) + ch.a0,
                            reinterpret_cast<const float *>(base_p + o_rad), reinterpret_cast<float4 *>(base_p + o_xyzr) + ch.a0, (uint32_t)na);
                    else
                        pack_frames_kernel<<<(unsigned)((na + 255) / 256), 256, 0, st>>>(
                            reinterpret_cast<const float *>(base_p + o_xyz3) + ch.a0 * 3, reinterpret_cast<const float *>(base_p + o_rad),
                            reinterpret_cast<float4 *>(base_p + o_xyzr) + ch.a0, (uint32_t)na, (uint32_t)fN, (uint32_t)(ch.a0 % (fN ? fN : 1)));
                    ++job->launches;
                }
            } else {
                J_TRY(cudaMemcpyAsync(base_p + o_xyzr + ch.a0 * 16, xyzr + ch.a0 * 4, na * 16, cudaMemcpyHostToDevice, st));
            }
            if (id_class) J_TRY(cudaMemcpyAsync(base_p + o_cls + ch.a0 * 4, id_class + ch.a0, na * 4, cudaMemcpyHostToDevice, st));
            if (frame_labels) {
                expand_frame_labels_kernel<<<(unsigned)((na + 255) / 256), 256, 0, st>>>(
                    reinterpret_cast<const uint32_t *>(base_p + o_lab), reinterpret_cast<uint32_t *>(base_p + o_grp) + ch.a0, (uint32_t)na,
                    (uint32_t)fN, (uint32_t)(ch.a0 % fN));
                ++job->launches;
            } else if (grouped) {
                J_TRY(cudaMemcpyAsync(base_p + o_grp + ch.a0 * 4, group + ch.a0, na * 4, cudaMemcpyHostToDevice, st));
            }
        }
        if ((rc = enqueue_chunk(b, variant, ch, kbase, st, &job->launches, nullptr, grouped ? &gp : nullptr, masked ? &mp : nullptr,
                                (masked && grouped) ? &mpi : nullptr, pairs ? &pp : nullptr)) != 0)
            return job_abort(ctx, job, rc);
        if (na && out->counts)
            J_TRY(cudaMemcpyAsync(out->counts + ch.a0, base_p + o_cnt + ch.a0 * 4, na * 4, cudaMemcpyDeviceToHost, st));
        if (na && out->atom_sasa)
            J_TRY(cudaMemcpyAsync(out->atom_sasa + ch.a0, base_p + o_atom + ch.a0 * 4, na * 4, cudaMemcpyDeviceToHost, st));
        if (na && masked)
            J_TRY(cudaMemcpyAsync(exposed + ch.a0 * W, base_p + o_mask + ch.a0 * W * 4, na * W * 4, cudaMemcpyDeviceToHost, st));
        if (out->seg_sasa && ch.g1 > ch.g0)
            J_TRY(cudaMemcpyAsync(out->seg_sasa + ch.g0, base_p + o_seg + ch.g0 * 4, (ch.g1 - ch.g0) * 4, cudaMemcpyDeviceToHost, st));
        if (out->protein && ch.s1 > ch.s0)
            J_TRY(cudaMemcpyAsync(out->protein + 3 * (size_t)ch.s0, base_p + o_prot + 12 * (size_t)ch.s0,
                                  12 * (size_t)(ch.s1 - ch.s0), cudaMemcpyDeviceToHost, st));
        if (grouped) {
            if (na && out_iso->counts)
                J_TRY(cudaMemcpyAsync(out_iso->counts + ch.a0, base_p + o_icnt + ch.a0 * 4, na * 4, cudaMemcpyDeviceToHost, st));
            if (na && out_iso->atom_sasa)
                J_TRY(cudaMemcpyAsync(out_iso->atom_sasa + ch.a0, base_p + o_iatom + ch.a0 * 4, na * 4, cudaMemcpyDeviceToHost, st));
            if (out_iso->seg_sasa && ch.g1 > ch.g0)
                J_TRY(cudaMemcpyAsync(out_iso->seg_sasa + ch.g0, base_p + o_iseg + ch.g0 * 4, (ch.g1 - ch.g0) * 4, cudaMemcpyDeviceToHost, st));
            if (out_iso->protein && ch.s1 > ch.s0)
                J_TRY(cudaMemcpyAsync(out_iso->protein + 3 * (size_t)ch.s0, base_p + o_iprot + 12 * (size_t)ch.s0,
                                      12 * (size_t)(ch.s1 - ch.s0), cudaMemcpyDeviceToHost, st));
            if (na && masked)
                J_TRY(cudaMemcpyAsync(exposed_iso + ch.a0 * W, base_p + o_imask + ch.a0 * W * 4, na * W * 4, cudaMemcpyDeviceToHost, st));
        }
        if (want_sums && ch.s1 > ch.s0) {
            // the chunk's slot rows -> per-frame L x L blocks and per-segment rows, behind the chunk's kernels on its stream
            const uint32_t ns = ch.s1 - ch.s0;
            pair_sums_kernel<<<(ns + 3) / 4, 128, 0, st>>>(b->d_off, gp.grp, pp.partner, pp.area, (uint32_t)K, L, ch.s0, ch.s1, d_psum);
            ++job->launches;
            if (want_seg_sums && ch.g1 > ch.g0) {
                const size_t nt = (ch.g1 - ch.g0) * L;
                seg_pair_sums_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(b->d_off, b->d_seg_off, b->d_seg_be, pp.partner, pp.area,
                                                                                   (uint32_t)K, L, ch.s0, ch.s1, (uint32_t)ch.g0,
                                                                                   (uint32_t)ch.g1, d_psum, d_pseg);
                ++job->launches;
            }
            J_TRY(cudaGetLastError());
            const size_t blk = (size_t)L * L;
            J_TRY(cudaMemcpyAsync(sums->pair_area + ch.s0 * blk, d_psum + ch.s0 * blk, ns * blk * 8, cudaMemcpyDeviceToHost, st));
            if (want_seg_sums && ch.g1 > ch.g0)
                J_TRY(cudaMemcpyAsync(sums->seg_pair_area + ch.g0 * L, d_pseg + ch.g0 * L, (ch.g1 - ch.g0) * L * 8, cudaMemcpyDeviceToHost, st));
        }
        if (na && pairs && pair_out) {
            J_TRY(cudaMemcpyAsync(pair_out->partner + ch.a0 * K, base_p + o_ppart + ch.a0 * K * 4, na * K * 4, cudaMemcpyDeviceToHost, st));
            if (pair_out->buried_counts)
                J_TRY(cudaMemcpyAsync(pair_out->buried_counts + ch.a0 * K, base_p + o_pcnt + ch.a0 * K * 4, na * K * 4, cudaMemcpyDeviceToHost,
                                      st));
            if (pair_out->buried_area)
                J_TRY(cudaMemcpyAsync(pair_out->buried_area + ch.a0 * K, base_p + o_parea + ch.a0 * K * 4, na * K * 4, cudaMemcpyDeviceToHost,
                                      st));
        }
    }
    // join the sibling streams into the first one, read the status words back, free the arena in stream order
    for (int i = 1; i < kStreams; ++i) {
        J_TRY(cudaEventRecord(ctx->ev_tail[i], ctx->streams[i]));
        J_TRY(cudaStreamWaitEvent(s0, ctx->ev_tail[i], 0));
    }
    ctx->tail_valid = true;
    J_TRY(cudaMemcpyAsync(job->h_status, d_status, pairs ? 40 : 32, cudaMemcpyDeviceToHost, s0));
    J_TRY(cudaEventRecord(job->ev1, s0));
    J_TRY(cudaFreeAsync(job->d_arena, s0));
    job->d_arena = nullptr;
#undef J_TRY
    *out_job = job;
    return SASA_B200_OK;
}

static int wait_job_impl(sasa_b200_job *job, sasa_b200_stats *stats) {
    sasa_b200_batch *b = job->batch;
    sasa_b200_ctx *ctx = b->ctx;
    cudaError_t e = cudaEventSynchronize(job->ev1);   // no lock: other threads keep submitting meanwhile
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = SASA_B200_OK;
    if (e != cudaSuccess) {
        rc = fail(ctx, SASA_B200_ERR_CUDA, "waiting for the run failed: %s", cudaGetErrorString(e));
    } else {
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, job->ev0, job->ev1);
        b->last = sasa_b200_stats{};
        b->last.kernel_ms = ms;   // device-side span of the whole pipelined run (copies overlapped with kernels)
        b->last.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - job->t_begin).count();
        b->last.n_atoms = b->n_atoms;
        b->last.n_structures = b->S;
        b->last.boundary_points = job->h_status[1];
        b->last.neighbor_pairs = job->h_status[2];
        b->last.streamed_atoms = job->h_status[3];
        b->last.gpu_launches = job->launches;
        b->launches_last = job->launches;
        if (stats) *stats = b->last;
        const int h_err = (int)(job->h_status[0] & 0xffffffffull);
        const uint32_t need = (uint32_t)(job->h_status[4] & 0xffffffffull);   // pairwise buried area: partners needed
        if (job->pairs && job->pairs->partners_needed) *job->pairs->partners_needed = need;
        if (h_err == SASA_B200_ERR_NON_FINITE)
            rc = fail(ctx, SASA_B200_ERR_NON_FINITE, "non-finite coordinate or radius in the input (the reference panics here)");
        else if (job->pairs && h_err == SASA_B200_ERR_INVALID_ARGUMENT)
            rc = fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "too few partner slots: max_partners = %u, the batch needs max_partners = %u",
                      job->pairs->max_partners, need);
        else if (h_err)
            rc = fail(ctx, h_err, "device-side error %d", h_err);
    }
    b->in_flight = nullptr;
    job->active = false;
    ctx->free_jobs.push_back(job);
    return rc;
}

static int run_host_impl(sasa_b200_batch *b, const float *xyzr, const float *xyz3, const float *radii,
                         const uint32_t *id_class, const sasa_b200_params *params, const sasa_b200_outputs *out,
                         sasa_b200_stats *stats) {
    sasa_b200_job *job = nullptr;
    int rc = submit_host_impl(b, xyzr, xyz3, radii, id_class, params, out, &job);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_submit_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class, const sasa_b200_params *params,
                                const sasa_b200_outputs *out, sasa_b200_job **out_job) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    return submit_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, out_job);
}

int sasa_b200_batch_submit_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii, const sasa_b200_params *params,
                                       const sasa_b200_outputs *out, sasa_b200_job **out_job) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!xyz || !radii) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyz / radii is NULL");
    return submit_host_impl(b, nullptr, xyz, radii, nullptr, params, out, out_job);
}

int sasa_b200_batch_submit_indexed_host(sasa_b200_batch *b, const float *xyz, const uint8_t *radius_index, const float *palette,
                                        size_t n_palette, const uint32_t *id_class, const sasa_b200_params *params,
                                        const sasa_b200_outputs *out, sasa_b200_job **out_job) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (b->n_atoms && (!xyz || !radius_index || !palette)) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyz / radius_index / palette is NULL");
    return submit_host_impl(b, nullptr, xyz, palette, id_class, params, out, out_job, radius_index, n_palette);
}

int sasa_b200_batch_run_indexed_host(sasa_b200_batch *b, const float *xyz, const uint8_t *radius_index, const float *palette,
                                     size_t n_palette, const uint32_t *id_class, const sasa_b200_params *params,
                                     const sasa_b200_outputs *out, sasa_b200_stats *stats) {
    sasa_b200_job *job = nullptr;
    int rc = sasa_b200_batch_submit_indexed_host(b, xyz, radius_index, palette, n_palette, id_class, params, out, &job);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_job_wait(sasa_b200_job *job, sasa_b200_stats *stats) {
    if (!job || !job->active) return SASA_B200_ERR_INVALID_ARGUMENT;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_run_groups_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class, const uint32_t *group,
                                    const sasa_b200_params *params, const sasa_b200_outputs *out,
                                    const sasa_b200_outputs *out_isolated, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    sasa_b200_job *job = nullptr;
    int rc = submit_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, &job, nullptr, 0, group, out_isolated);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_submit_groups_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii, const uint32_t *group,
                                              const sasa_b200_params *params, const sasa_b200_outputs *out,
                                              const sasa_b200_outputs *out_isolated, sasa_b200_job **out_job) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    if (b->n_atoms && (!xyz || !radii)) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyz / radii is NULL");
    return submit_host_impl(b, nullptr, xyz, radii, nullptr, params, out, out_job, nullptr, 0, group, out_isolated);
}

int sasa_b200_batch_run_groups_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii, const uint32_t *group,
                                           const sasa_b200_params *params, const sasa_b200_outputs *out,
                                           const sasa_b200_outputs *out_isolated, sasa_b200_stats *stats) {
    sasa_b200_job *job = nullptr;
    int rc = sasa_b200_batch_submit_groups_frames_host(b, xyz, radii, group, params, out, out_isolated, &job);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_submit_group_pairs_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii, const uint32_t *group,
                                                   const sasa_b200_params *params, const sasa_b200_outputs *out,
                                                   const sasa_b200_outputs *out_isolated, const sasa_b200_pair_sums *sums,
                                                   sasa_b200_job **out_job) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    if (b->n_atoms && (!xyz || !radii)) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyz / radii is NULL");
    if (!sums && b->n_atoms) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "sums is NULL");
    return submit_host_impl(b, nullptr, xyz, radii, nullptr, params, out, out_job, nullptr, 0, group, out_isolated, false, nullptr,
                            nullptr, sums != nullptr, nullptr, sums);
}

int sasa_b200_batch_run_group_pairs_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii, const uint32_t *group,
                                                const sasa_b200_params *params, const sasa_b200_outputs *out,
                                                const sasa_b200_outputs *out_isolated, const sasa_b200_pair_sums *sums,
                                                sasa_b200_stats *stats) {
    sasa_b200_job *job = nullptr;
    int rc = sasa_b200_batch_submit_group_pairs_frames_host(b, xyz, radii, group, params, out, out_isolated, sums, &job);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_run_masks_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class, const sasa_b200_params *params,
                                   const sasa_b200_outputs *out, uint32_t *exposed, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_job *job = nullptr;
    int rc = submit_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, &job, nullptr, 0, nullptr, nullptr, true, exposed);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_run_groups_masks_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class, const uint32_t *group,
                                          const sasa_b200_params *params, const sasa_b200_outputs *out,
                                          const sasa_b200_outputs *out_isolated, uint32_t *exposed, uint32_t *exposed_isolated,
                                          sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    sasa_b200_job *job = nullptr;
    int rc = submit_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, &job, nullptr, 0, group, out_isolated, true, exposed,
                              exposed_isolated);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_run_group_pairs_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class, const uint32_t *group,
                                         const sasa_b200_params *params, const sasa_b200_outputs *out,
                                         const sasa_b200_outputs *out_isolated, const sasa_b200_pair_outputs *pairs, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!out_isolated) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "out_isolated is NULL");
    sasa_b200_job *job = nullptr;
    int rc = submit_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, &job, nullptr, 0, group, out_isolated, false, nullptr,
                              nullptr, true, pairs);
    if (rc) return rc;
    return wait_job_impl(job, stats);
}

int sasa_b200_batch_run_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class,
                             const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    return run_host_impl(b, xyzr, nullptr, nullptr, id_class, params, out, stats);
}

int sasa_b200_batch_run_frames_host(sasa_b200_batch *b, const float *xyz, const float *radii,
                                    const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (!xyz || !radii) return fail(b->ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyz / radii is NULL");
    return run_host_impl(b, nullptr, xyz, radii, nullptr, params, out, stats);
}

// Atom-range split (BASELINE cfg5): every structure of the batch goes through the global-cell-list path and only
// slice `rank` of `n_ranks` of its cell-sorted atom order is evaluated.  Outputs are zero-filled first, so summing
// the per-rank vectors (ncclAllReduce over NVLink, or on the host) reproduces the single-GPU result bit for bit.
static int run_atom_range_locked(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_cls, const sasa_b200_params *params,
                                 uint32_t rank, uint32_t n_ranks, uint32_t *d_counts, float *d_atom, cudaStream_t st,
                                 uint32_t *const *peer_counts = nullptr, float *const *peer_atom = nullptr) {
    sasa_b200_ctx *ctx = b->ctx;
    int rc = check_params(ctx, params);
    if (rc) return rc;
    if (n_ranks == 0 || rank >= n_ranks) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "rank %u out of range (%u ranks)", rank, n_ranks);
    if (params->flags & (SASA_B200_FLAG_BOUNDARY_STATS | SASA_B200_FLAG_FORCE_STREAMING))
        return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "statistics flags are not available in the atom-range split");
    uint32_t max_atoms = 0;
    for (size_t s = 0; s < b->S; ++s) max_atoms = std::max(max_atoms, b->h_off[s + 1] - b->h_off[s]);
    if (max_atoms > ctx->large.cap_atoms) cudaDeviceSynchronize();
    if (max_atoms && (rc = large_reserve(ctx->large, max_atoms)) != 0)
        return fail(ctx, rc, "allocating the large-structure workspace (%u atoms) failed", max_atoms);
    RunArgs ra;
    ra.d_xyzr = reinterpret_cast<const float4 *>(d_xyzr);
    ra.d_cls = d_cls;
    ra.d_out = sasa_b200_outputs{d_counts, d_atom, nullptr, nullptr};
    ra.prm = *params;
    if ((rc = get_points(ctx, params->n_points, &ra.pts)) != 0) return rc;
    KParams kp;
    make_kparams(b, ra, &kp);
    kp.seg_be = nullptr;
    kp.out_seg = nullptr;
    b->launches_last = 0;
    const bool peers = peer_counts != nullptr || peer_atom != nullptr;
    if (peers) {
        // every atom's owner writes it into every rank's vectors: nothing to zero, nothing to reduce afterwards
        if (n_ranks > 8) return fail(ctx, SASA_B200_ERR_UNSUPPORTED, "peer writes support at most 8 ranks, got %u", n_ranks);
        kp.n_peers = (int)n_ranks;
        for (uint32_t r = 0; r < n_ranks; ++r) {
            kp.peer_counts[r] = peer_counts ? peer_counts[r] : nullptr;
            kp.peer_atom[r] = peer_atom ? peer_atom[r] : nullptr;
        }
        kp.out_counts = peer_counts ? peer_counts[rank] : nullptr;   // the local vectors (non-finite input blanks them)
        kp.out_atom = peer_atom ? peer_atom[rank] : nullptr;
    } else {
        if (d_counts && b->n_atoms) CU_TRY(ctx, cudaMemsetAsync(d_counts, 0, b->n_atoms * sizeof(uint32_t), st));
        if (d_atom && b->n_atoms) CU_TRY(ctx, cudaMemsetAsync(d_atom, 0, b->n_atoms * sizeof(float), st));
    }
    std::vector<uint32_t> order(b->S);
    std::iota(order.begin(), order.end(), 0u);
    if (ctx->large_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_large, 0));
    rc = large_enqueue(ctx->sm_count, ctx->large, kp, order.data(), (uint32_t)b->S, b->h_off.data(), nullptr, st, &b->launches_last, rank,
                       n_ranks);
    if (rc == 0) {
        CU_TRY(ctx, cudaEventRecord(ctx->ev_large, st));
        ctx->large_used = true;
    }
    if (rc != 0) return fail(ctx, rc, "large-structure path failed: %s", cudaGetErrorString(cudaGetLastError()));
    return SASA_B200_OK;
}

int sasa_b200_batch_run_atom_range_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class,
                                          const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                          uint32_t *d_counts, float *d_atom_sasa, void *stream) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!d_xyzr && b->n_atoms) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_xyzr is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    return run_atom_range_locked(b, d_xyzr, d_id_class, params, rank, n_ranks, d_counts, d_atom_sasa,
                                 stream ? (cudaStream_t)stream : ctx->streams[0]);
}

int sasa_b200_batch_run_atom_range_peers_device(sasa_b200_batch *b, const float *d_xyzr, const uint32_t *d_id_class,
                                                const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                                uint32_t *const *peer_counts, float *const *peer_atom_sasa, void *stream) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!d_xyzr && b->n_atoms) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_xyzr is NULL");
    if (!peer_counts && !peer_atom_sasa) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "peer_counts and peer_atom_sasa are both NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    return run_atom_range_locked(b, d_xyzr, d_id_class, params, rank, n_ranks, nullptr, nullptr,
                                 stream ? (cudaStream_t)stream : ctx->streams[0], peer_counts, peer_atom_sasa);
}

int sasa_b200_batch_run_atom_range_host(sasa_b200_batch *b, const float *xyzr, const uint32_t *id_class,
                                        const sasa_b200_params *params, uint32_t rank, uint32_t n_ranks,
                                        uint32_t *out_counts, float *out_atom_sasa, sasa_b200_stats *stats) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!xyzr && b->n_atoms) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyzr is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t N = b->n_atoms;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_xyzr = 0, o_cls = al(N * 16), o_cnt = o_cls + (id_class ? al(N * 4) : 0), o_atom = o_cnt + al(N * 4);
    int rc = arena_reserve(ctx, o_atom + al(N * 4) + 256);
    if (rc) return rc;
    char *base_p = static_cast<char *>(ctx->arena);
    cudaStream_t st = ctx->streams[0];
    if (N) {
        CU_TRY(ctx, cudaMemcpyAsync(base_p + o_xyzr, xyzr, N * 16, cudaMemcpyHostToDevice, st));
        if (id_class) CU_TRY(ctx, cudaMemcpyAsync(base_p + o_cls, id_class, N * 4, cudaMemcpyHostToDevice, st));
    }
    rc = run_atom_range_locked(b, reinterpret_cast<const float *>(base_p + o_xyzr),
                               id_class ? reinterpret_cast<const uint32_t *>(base_p + o_cls) : nullptr, params, rank, n_ranks,
                               reinterpret_cast<uint32_t *>(base_p + o_cnt), reinterpret_cast<float *>(base_p + o_atom), st);
    if (rc) return rc;
    if (N && out_counts) CU_TRY(ctx, cudaMemcpyAsync(out_counts, base_p + o_cnt, N * 4, cudaMemcpyDeviceToHost, st));
    if (N && out_atom_sasa) CU_TRY(ctx, cudaMemcpyAsync(out_atom_sasa, base_p + o_atom, N * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    b->last = sasa_b200_stats{};
    rc = finish_run(b, stats);
    cudaMemset(ctx->d_err, 0, sizeof(int));
    cudaMemset(ctx->d_stat, 0, 3 * sizeof(unsigned long long));
    return rc;
}

int sasa_b200_batch_reduce_device(sasa_b200_batch *b, const float *d_atom_sasa, float *d_seg_sasa, float *d_protein, void *stream) {
    if (!b) return SASA_B200_ERR_INVALID_ARGUMENT;
    sasa_b200_ctx *ctx = b->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!d_atom_sasa && b->n_atoms) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "d_atom_sasa is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->streams[0];
    KParams kp;
    memset(&kp, 0, sizeof kp);
    kp.struct_off = b->d_off;
    kp.seg_be = b->d_seg_be;
    kp.struct_seg_off = b->d_seg_off;
    kp.seg_polar = b->d_polar;
    kp.out_seg = b->n_seg ? d_seg_sasa : nullptr;
    kp.out_protein = d_protein;
    b->launches_last = 0;
    for (size_t s = 0; s < b->S; ++s) {
        const uint32_t a0 = b->h_off[s];
        const int N = (int)(b->h_off[s + 1] - a0);
        const uint32_t g0 = b->h_seg_off.empty() ? 0 : b->h_seg_off[s];
        const uint32_t nseg = b->h_seg_off.empty() ? 0 : b->h_seg_off[s + 1] - g0;
        large_enqueue_sums(ctx->sm_count, kp, (uint32_t)s, N, g0, nseg, d_atom_sasa + a0, nullptr, nullptr, 0, st, &b->launches_last);
    }
    CU_TRY(ctx, cudaGetLastError());
    return SASA_B200_OK;
}

// ---- one structure per call ---------------------------------------------------------------------------------------------
// What SASAOptions::process does in the reference: one structure, host buffers, synchronous (BASELINE config 1).  The call
// takes a slot -- stream, large-structure workspace, device buffer and pinned staging of its own -- so that concurrent
// callers (the reference's directory mode, src/main.rs:375, :439) overlap instead of queueing on the context; the
// structure goes down the multi-CTA large-structure path (a lone structure in a fused kernel would occupy one SM), and
// inputs / outputs / status each travel in ONE copy.  About a dozen runtime calls in all.
static SingleSlot *slot_acquire(sasa_b200_ctx *ctx) {
    std::unique_lock<std::mutex> lk(ctx->slot_mu);
    for (;;) {
        for (auto &sp : ctx->slots)
            if (!sp->busy) {
                sp->busy = true;
                return sp.get();
            }
        if (ctx->slots.size() < kMaxSlots) {
            auto sp = std::make_unique<SingleSlot>();
            if (cudaStreamCreateWithFlags(&sp->st, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
            sp->busy = true;
            ctx->slots.push_back(std::move(sp));
            return ctx->slots.back().get();
        }
        ctx->slot_cv.wait(lk);
    }
}

static void slot_release(sasa_b200_ctx *ctx, SingleSlot *sl) {
    {
        std::lock_guard<std::mutex> lk(ctx->slot_mu);
        sl->busy = false;
    }
    ctx->slot_cv.notify_one();
}

static int single_run(sasa_b200_ctx *ctx, const float *xyzr, const uint32_t *cls, size_t N, const uint32_t *seg_be, size_t G,
                      const uint8_t *seg_polar, const sasa_b200_params *params, const sasa_b200_outputs *out,
                      sasa_b200_stats *stats, std::string *err_text) {
    const auto t_begin = std::chrono::steady_clock::now();
    const Points *pts = nullptr;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        int rc = check_params(ctx, params);
        if (rc == 0) rc = get_points(ctx, params->n_points, &pts);
        if (rc) {
            *err_text = ctx->err;
            return rc;
        }
    }
    auto failed = [&](int code, const char *what, cudaError_t e) {
        *err_text = std::string(what) + ": " + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? (int)SASA_B200_ERR_OUT_OF_MEMORY : code;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(ctx->device)) != cudaSuccess) return failed(SASA_B200_ERR_CUDA, "cudaSetDevice", e);
    SingleSlot *sl = slot_acquire(ctx);
    if (!sl) return failed(SASA_B200_ERR_CUDA, "creating a slot stream", cudaGetLastError());
    struct Release {
        sasa_b200_ctx *c;
        SingleSlot *s;
        ~Release() { slot_release(c, s); }
    } release{ctx, sl};
    // layout (offsets shared by the device buffer and the pinned staging): inputs | outputs | status
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const bool segs = seg_be != nullptr && G > 0;
    size_t o = 0;
    const size_t o_xyzr = o;  o += al(N * 16);
    const size_t o_cls = o;   o += cls ? al(N * 4) : 0;
    const size_t o_seg = o;   o += segs ? al(G * 8) : 0;
    const size_t o_pol = o;   o += (segs && seg_polar) ? al(G) : 0;
    const size_t o_off = o;   o += 256;   // struct_off {0, N}, struct_seg_off {0, G}
    const size_t in_bytes = o;
    const size_t o_atom = o;  o += out->atom_sasa ? al(N * 4) : 0;
    const size_t o_cnt = o;   o += out->counts ? al(N * 4) : 0;
    const size_t o_sseg = o;  o += (segs && out->seg_sasa) ? al(G * 4) : 0;
    const size_t o_prot = o;  o += out->protein ? 256 : 0;
    const size_t out_bytes = o - in_bytes;
    const size_t o_hdr = o;   o += al(sizeof(LargeHeader));
    if (o > sl->d_bytes) {
        cudaStreamSynchronize(sl->st);
        cudaFree(sl->d_buf);
        cudaFreeHost(sl->h_pin);
        sl->d_buf = nullptr; sl->h_pin = nullptr; sl->d_bytes = sl->h_bytes = 0;
        const size_t want = o + o / 4 + (64 << 10);
        if ((e = cudaMalloc((void **)&sl->d_buf, want)) != cudaSuccess) return failed(SASA_B200_ERR_CUDA, "cudaMalloc", e);
        if ((e = cudaHostAlloc((void **)&sl->h_pin, want, cudaHostAllocDefault)) != cudaSuccess) return failed(SASA_B200_ERR_CUDA, "cudaHostAlloc", e);
        // the sections of the layout are 256-byte aligned and travel in one copy each way: define the gaps once
        memset(sl->h_pin, 0, want);
        cudaMemset(sl->d_buf, 0, want);
        sl->d_bytes = sl->h_bytes = want;
    }
    if (N > sl->large.cap_atoms) {
        cudaStreamSynchronize(sl->st);
        if (large_reserve(sl->large, (uint32_t)std::max<size_t>(N + N / 4, 4096)) != 0) {
            *err_text = "allocating the large-structure workspace failed";
            return SASA_B200_ERR_OUT_OF_MEMORY;
        }
    }
    char *h = sl->h_pin, *d = sl->d_buf;
    memcpy(h + o_xyzr, xyzr, N * 16);
    if (cls) memcpy(h + o_cls, cls, N * 4);
    if (segs) memcpy(h + o_seg, seg_be, G * 8);
    if (segs && seg_polar) memcpy(h + o_pol, seg_polar, G);
    {
        uint32_t *off = reinterpret_cast<uint32_t *>(h + o_off);
        off[0] = 0; off[1] = (uint32_t)N; off[2] = 0; off[3] = (uint32_t)G;
    }
    if ((e = cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, sl->st)) != cudaSuccess) return failed(SASA_B200_ERR_CUDA, "H2D copy", e);
    KParams kp;
    memset(&kp, 0, sizeof kp);
    kp.xyzr = reinterpret_cast<const float4 *>(d + o_xyzr);
    kp.cls = cls ? reinterpret_cast<const uint32_t *>(d + o_cls) : nullptr;
    kp.struct_off = reinterpret_cast<const uint32_t *>(d + o_off);
    if (segs) {
        kp.seg_be = reinterpret_cast<const uint2 *>(d + o_seg);
        kp.struct_seg_off = reinterpret_cast<const uint32_t *>(d + o_off) + 2;
        kp.seg_polar = seg_polar ? reinterpret_cast<const uint8_t *>(d + o_pol) : nullptr;
    }
    kp.out_atom = out->atom_sasa ? reinterpret_cast<float *>(d + o_atom) : nullptr;
    kp.out_counts = out->counts ? reinterpret_cast<uint32_t *>(d + o_cnt) : nullptr;
    kp.out_seg = (segs && out->seg_sasa) ? reinterpret_cast<float *>(d + o_sseg) : nullptr;
    kp.out_protein = out->protein ? reinterpret_cast<float *>(d + o_prot) : nullptr;
    fill_run_params(&kp, pts, *params);
    kp.err_flag = &sl->large.hdr->err;
    kp.stat = sl->large.hdr->stat;
    const uint32_t order[1] = {0}, offs[2] = {0, (uint32_t)N}, soff[2] = {0, (uint32_t)G};
    uint32_t launches = 0;
    int rc = large_enqueue(ctx->sm_count, sl->large, kp, order, 1, offs, segs ? soff : nullptr, sl->st, &launches);
    if (rc) {
        cudaStreamSynchronize(sl->st);
        *err_text = std::string("large-structure path failed: ") + cudaGetErrorString(cudaGetLastError());
        return rc;
    }
    if (out_bytes && (e = cudaMemcpyAsync(h + in_bytes, d + in_bytes, out_bytes, cudaMemcpyDeviceToHost, sl->st)) != cudaSuccess)
        return failed(SASA_B200_ERR_CUDA, "D2H copy", e);
    if ((e = cudaMemcpyAsync(h + o_hdr, sl->large.hdr, sizeof(LargeHeader), cudaMemcpyDeviceToHost, sl->st)) != cudaSuccess)
        return failed(SASA_B200_ERR_CUDA, "D2H copy", e);
    if ((e = cudaStreamSynchronize(sl->st)) != cudaSuccess) return failed(SASA_B200_ERR_CUDA, "cudaStreamSynchronize", e);
    if (out->atom_sasa) memcpy(out->atom_sasa, h + o_atom, N * 4);
    if (out->counts) memcpy(out->counts, h + o_cnt, N * 4);
    if (segs && out->seg_sasa) memcpy(out->seg_sasa, h + o_sseg, G * 4);
    if (out->protein) memcpy(out->protein, h + o_prot, 12);
    const LargeHeader *hh = reinterpret_cast<const LargeHeader *>(h + o_hdr);
    if (stats) {
        *stats = sasa_b200_stats{};
        stats->n_atoms = N;
        stats->n_structures = 1;
        stats->boundary_points = hh->stat[0];
        stats->neighbor_pairs = hh->stat[1];
        stats->streamed_atoms = hh->stat[2];
        stats->gpu_launches = launches;
        stats->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
    if (hh->err == SASA_B200_ERR_NON_FINITE) {
        *err_text = "non-finite coordinate or radius in the input (the reference panics here)";
        return SASA_B200_ERR_NON_FINITE;
    }
    if (hh->err) {
        *err_text = "device-side error " + std::to_string(hh->err);
        return hh->err;
    }
    return SASA_B200_OK;
}

int sasa_b200_run_batch(sasa_b200_ctx *ctx, const float *xyzr, const uint32_t *id_class, const uint64_t *struct_off,
                        size_t S, const uint32_t *seg_be, const uint64_t *struct_seg_off, const uint8_t *seg_polar,
                        const sasa_b200_params *params, const sasa_b200_outputs *out, sasa_b200_stats *stats) {
    if (!ctx) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (S == 1 && struct_off && struct_off[0] == 0 && struct_off[1] > 0 && struct_off[1] < (1ull << 31) && xyzr && out && params &&
        (!seg_be || struct_seg_off)) {
        const size_t N = (size_t)struct_off[1];
        const size_t G = seg_be ? (size_t)(struct_seg_off[1] - struct_seg_off[0]) : 0;
        bool ok = !seg_be || struct_seg_off[0] == 0;
        for (size_t k = 0; ok && k < G; ++k) ok = seg_be[2 * k] <= seg_be[2 * k + 1] && seg_be[2 * k + 1] <= N;
        if (ok) {
            std::string text;
            const int rc = single_run(ctx, xyzr, id_class, N, seg_be, G, seg_polar, params, out, stats, &text);
            if (rc) {
                std::lock_guard<std::mutex> lk(ctx->mu);
                ctx->err = text;
            }
            return rc;
        }
    }
    sasa_b200_batch *b = nullptr;
    int rc = batch_create_impl(ctx, struct_off, S, seg_be, struct_seg_off, seg_polar, &b, S == 1);
    if (rc) return rc;
    rc = sasa_b200_batch_run_host(b, xyzr, id_class, params, out, stats);
    sasa_b200_batch_destroy(b);
    return rc;
}

int sasa_b200_calculate_sasa_internal(sasa_b200_ctx *ctx, const float *xyzr, const uint64_t *ids, size_t n_atoms,
                                      float probe_radius, size_t n_points, ptrdiff_t threads, float *out_sasa,
                                      uint32_t *out_counts) {
    if (!ctx) return SASA_B200_ERR_INVALID_ARGUMENT;
    if (n_atoms == 0) return SASA_B200_OK;  // empty in, empty out (tests/sanity.rs:148-157)
    if (!xyzr || !out_sasa) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "xyzr / out_sasa is NULL");
    if (n_points > (1u << 24)) return fail(ctx, SASA_B200_ERR_INVALID_ARGUMENT, "n_points too large");
    // Atom.id only matters through equality: rank the ids densely, and drop them when all are distinct.
    std::vector<uint32_t> cls;
    if (ids) {
        std::unordered_map<uint64_t, uint32_t> rank;
        rank.reserve(n_atoms * 2);
        cls.resize(n_atoms);
        for (size_t i = 0; i < n_atoms; ++i) cls[i] = rank.emplace(ids[i], (uint32_t)rank.size()).first->second;
        if (rank.size() == n_atoms) cls.clear();
    }
    const uint64_t off[2] = {0, n_atoms};
    sasa_b200_params prm{probe_radius, (uint32_t)n_points, 8, (int32_t)threads, 0};
    sasa_b200_outputs out{out_counts, out_sasa, nullptr, nullptr};
    return sasa_b200_run_batch(ctx, xyzr, cls.empty() ? nullptr : cls.data(), off, 1, nullptr, nullptr, nullptr, &prm, &out, nullptr);
}

}  // extern "C"
