// locohd_capi.cu — implementation of the C ABI declared in include/locohd_b200.h.
// Host-side orchestration only: validation (LoCoHD::build, locohd.rs:289-389), device memory, stream
// ordering and the launch sequence K0 -> K1 -> scan -> K1' -> K2.  No CPU fallback exists: every entry point
// needs a CUDA device.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "locohd_kernels.cuh"

using namespace locohd;

namespace {
std::mutex g_err_mutex;
std::string g_global_err;

// A job list grouped into tiles (plan_job_tiles) and whether score_tile_kernel pays for that grouping (tiles_pay);
// the same list in wide tiles and whether they are filled well enough for score_wide_kernel (wide_tiles_pay)
struct TilePlan {
    std::vector<ScoreTile> tiles;
    bool pays = false;
    std::vector<WideTile> wide;
    bool wide_pays = false;
};
}

struct locohd_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    uint64_t tile_launches = 0;
    uint64_t wide_launches = 0;   // the part of tile_launches that ran score_wide_kernel
    // tile plan of the last job list (a benchmark step, the next block of frames: the same list again)
    std::vector<locohd_job> tile_cache_jobs;
    TilePlan tile_cache_plan;
    bool has_params = false;
    KParams kp{};
    int n_categories = 0;
    // device-side parameter storage
    double* d_cat_w = nullptr;
    double* d_cat_sw = nullptr;
    WfDev* d_wfs = nullptr;
    WfDev h_wf0{};                 // host copy of weight function 0 (selects kernel specialisations)
    uint64_t* d_tag_pairs = nullptr;
    double* d_sqrt_tbl = nullptr;
    double* d_rsqrt_tbl = nullptr;
    int* d_err = nullptr;
    ScanStats* d_scan = nullptr;   // three slots: [0] anchor order, [1] environment sizes, [2] a chunk of a graph
    FusedStats* d_fstats = nullptr;  // fused gather: store cursor, sample sum, largest environment, overflow word
    unsigned long long* d_score_cursor = nullptr;   // scoring kernel: next unclaimed pair
    // pinned host mirrors: the error word and the gather statistics come back with asynchronous copies queued before
    // the stream synchronisation (no separate blocking cudaMemcpy per synchronisation point)
    int* h_err = nullptr;
    FusedStats* h_fstats = nullptr;   // two slots: [0] sizing sample, [1] result of the fused gather
    ScanStats* h_scan = nullptr;      // d_scan[2]: the entries of a chunk of a graph (locohd_score_within[_condensed])
    // pinned staging area of the one-call entry point (small calls: all inputs travel in one copy)
    unsigned char* h_stage = nullptr;
    size_t h_stage_bytes = 0;
    struct {   // sizing state of the fused gather, carried from call to call (fused_gather alone reads and writes it)
        int cap_hint = kFusedCap;               // members per environment the fused gather starts with (512 or 1024)
        uint64_t n_anchors = 0, capacity = 0;   // store size that worked for the last call of this shape (0: none)
        double threshold = 0.0;
        int cap = 0;
    } store_hist;
    // Large device buffers (environment stores, scratch) are recycled per context: the stream-ordered pool of the
    // driver splits and re-merges multi-GB blocks unpredictably, which shows up as 30-60 ms stalls per call.
    std::mutex cache_mu;
    std::unordered_map<void*, size_t> big_live;           // big blocks handed out
    std::vector<std::pair<size_t, void*>> big_free;       // big blocks ready for reuse (same stream: ordered)
    // per-kernel-group event timing
    bool prof_on = false;
    struct ProfRec { int group; cudaEvent_t a, b; };
    std::vector<ProfRec> prof;
};

namespace {
// Brackets the launches issued in its scope with a pair of events when profiling is enabled.
struct ProfScope {
    locohd_ctx* ctx;
    cudaEvent_t a = nullptr, b = nullptr;
    int group;
    ProfScope(locohd_ctx* c, int g) : ctx(c), group(g) {
        if (!ctx->prof_on) return;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, ctx->stream);
    }
    ~ProfScope() {
        if (!a) return;
        cudaEventRecord(b, ctx->stream);
        ctx->prof.push_back({group, a, b});
    }
};
}

struct locohd_structs {
    locohd_ctx* ctx = nullptr;
    uint64_t n_structs = 0, n_prims = 0;
    uint64_t max_prims = 0;          // largest structure
    uint64_t* d_prim_off = nullptr;
    double* d_xyz = nullptr;
    uint8_t* d_cat = nullptr;
    uint32_t* d_tag = nullptr;
    StructMeta* d_meta = nullptr;
    float4* d_pf = nullptr;
    PrimRec* d_pd = nullptr;
    uint32_t* d_porig = nullptr;
    uint32_t* d_sorted_pos = nullptr;
    uint32_t* d_cell_start = nullptr;
    uint32_t* d_cell_fill = nullptr;
    bool cells_valid = false;
    double cell_threshold = 0.0;
    unsigned char* block = nullptr;  // the one device block the arrays above are views into (structs_layout)
    StructsView view() const {
        StructsView v;
        v.n_structs = n_structs; v.prim_off = d_prim_off; v.xyz = d_xyz; v.cat = d_cat; v.tag = d_tag;
        v.meta = d_meta; v.pf = d_pf; v.pd = d_pd; v.porig = d_porig; v.sorted_pos = d_sorted_pos; v.cell_start = d_cell_start;
        v.cell_fill = d_cell_fill;
        return v;
    }
};

struct locohd_envset {
    locohd_ctx* ctx = nullptr;
    uint64_t n_env = 0, total = 0;   // total = members actually stored (sum of the sizes)
    uint64_t capacity = 0;           // entries of the store (even-rounded upper bounds)
    unsigned max_count = 0;
    bool key_is_w = false;
    uint64_t* d_off = nullptr;       // [n_env + 1]
    uint32_t* d_count = nullptr;
    uint64_t* d_key = nullptr;       // packed keys (see EnvView)
    double* d_dist = nullptr;        // plain distances, kept only for locohd_envset_dump
    uint32_t* d_idx = nullptr;       // primitive indices, kept only for locohd_envset_dump
    EnvView view() const {
        EnvView v;
        v.n_env = n_env; v.off = d_off; v.count = d_count; v.key = d_key; v.key_is_w = key_is_w ? 1 : 0;
        return v;
    }
};

// A threshold graph in CSR form (locohd_score_within[_condensed]): row r holds the columns indices[indptr[r] ..
// indptr[r + 1]) with their scores.
struct locohd_graph {
    locohd_ctx* ctx = nullptr;
    uint64_t rows = 0, cols = 0, nnz = 0;
    uint64_t* d_indptr = nullptr;    // [rows + 1]
    uint32_t* d_indices = nullptr;   // [nnz]
    double* d_scores = nullptr;      // [nnz]
};

namespace {

int fail(locohd_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    else {
        std::lock_guard<std::mutex> g(g_err_mutex);
        g_global_err = buf;
    }
    return code;
}

#define CU(ctx, expr)                                                                                         \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return fail(ctx, LOCOHD_ERR_CUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e__), __FILE__, \
                        __LINE__, cudaGetErrorString(e__));                                                   \
    } while (0)

#define TRY_ST(expr)             \
    do {                         \
        int st__ = (expr);       \
        if (st__) return st__;   \
    } while (0)

const char* status_text(int code) {
    switch (code) {
        case LOCOHD_ERR_LEN_MISMATCH: return "Lists seq and dists must have equal lengths!";
        case LOCOHD_ERR_FIRST_NOT_ZERO: return "The dists list must start with a distance of 0!";
        case LOCOHD_ERR_UNKNOWN_CATEGORY: return "Category not found!";
        case LOCOHD_ERR_ZERO_NORM: return "Zero norm error for a PMF";
        case LOCOHD_ERR_NEGATIVE_POINT: return "Invalid input value: all weight function inputs must be non-negative!";
        case LOCOHD_ERR_NAN: return "NaN or non-finite value in the input";
        case LOCOHD_ERR_EMPTY_ENV: return "Empty environment (non-positive or NaN threshold distance?)";
        case LOCOHD_ERR_INDEX: return "Anchor or environment index out of range";
        case LOCOHD_ERR_DMX_SHAPE: return "Expected matrices with the same length";
        case LOCOHD_ERR_BAD_PARAM: return "weight function index out of range";
        case LOCOHD_ERR_CUDA: return "internal device error";
        default: return "error";
    }
}

// Device allocations are stream-ordered on the context stream; blocks of kBigBlock bytes and more are recycled
// through the context's cache (best fit with at most 25 % slack).
constexpr size_t kBigBlock = 16u << 20;
constexpr size_t kBigCacheEntries = 32;

int dev_alloc_bytes(locohd_ctx* ctx, void** out, size_t bytes) {
    *out = nullptr;
    if (bytes == 0) bytes = 1;
    if (bytes >= kBigBlock) {
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        int best = -1;
        for (int i = 0; i < (int)ctx->big_free.size(); ++i) {
            const size_t sz = ctx->big_free[i].first;
            if (sz >= bytes && sz - bytes <= bytes / 4 && (best < 0 || sz < ctx->big_free[best].first)) best = i;
        }
        if (best >= 0) {
            *out = ctx->big_free[best].second;
            ctx->big_live[*out] = ctx->big_free[best].first;
            ctx->big_free.erase(ctx->big_free.begin() + best);
            return 0;
        }
    }
    void* p = nullptr;
    CU(ctx, cudaMallocAsync(&p, bytes, ctx->stream));
    if (bytes >= kBigBlock) {
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        ctx->big_live[p] = bytes;
    }
    *out = p;
    return 0;
}

void dev_free_bytes(locohd_ctx* ctx, void* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        auto it = ctx->big_live.find(p);
        if (it != ctx->big_live.end()) {
            const size_t sz = it->second;
            ctx->big_live.erase(it);
            if (ctx->big_free.size() >= kBigCacheEntries) {   // drop the smallest cached block
                size_t k = 0;
                for (size_t i = 1; i < ctx->big_free.size(); ++i) if (ctx->big_free[i].first < ctx->big_free[k].first) k = i;
                cudaFreeAsync(ctx->big_free[k].second, ctx->stream);
                ctx->big_free.erase(ctx->big_free.begin() + k);
            }
            ctx->big_free.emplace_back(sz, p);
            return;
        }
    }
    cudaFreeAsync(p, ctx->stream);
}

template <class T>
int dev_alloc(locohd_ctx* ctx, T** out, uint64_t n) {
    void* p = nullptr;
    const int st = dev_alloc_bytes(ctx, &p, (size_t)n * sizeof(T));
    *out = static_cast<T*>(p);
    return st;
}
template <class T>
void dev_free(locohd_ctx* ctx, T*& p) {
    dev_free_bytes(ctx, (void*)p);
    p = nullptr;
}

bool is_device_ptr(const locohd_ctx* ctx, const void* p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return (at.type == cudaMemoryTypeDevice && at.device == ctx->device) || at.type == cudaMemoryTypeManaged;
}

// Input array that may be host or device memory: `ptr` is always device-accessible afterwards.
template <class T>
struct InBuf {
    locohd_ctx* ctx = nullptr;
    const T* ptr = nullptr;
    T* owned = nullptr;
    ~InBuf() { if (owned) dev_free_bytes(ctx, owned); }
    int load(locohd_ctx* c, const T* src, uint64_t n) {
        ctx = c;
        if (!src || n == 0) { ptr = nullptr; return 0; }
        if (is_device_ptr(c, src)) { ptr = src; return 0; }
        TRY_ST(dev_alloc(c, &owned, n));
        CU(c, cudaMemcpyAsync(owned, src, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
        ptr = owned;
        return 0;
    }
};

// Output array that may be host or device memory.
template <class T>
struct OutBuf {
    locohd_ctx* ctx = nullptr;
    T* ptr = nullptr;
    T* owned = nullptr;
    T* user = nullptr;
    uint64_t n = 0;
    ~OutBuf() { if (owned) dev_free_bytes(ctx, owned); }
    int prepare(locohd_ctx* c, T* dst, uint64_t count) {
        ctx = c; user = dst; n = count;
        if (!dst) { ptr = nullptr; return 0; }
        if (is_device_ptr(c, dst)) { ptr = dst; return 0; }
        TRY_ST(dev_alloc(c, &owned, count));
        ptr = owned;
        return 0;
    }
    int commit() {  // enqueue the device -> host copy when the destination is host memory
        if (owned && n) CU(ctx, cudaMemcpyAsync(user, owned, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
        return 0;
    }
};

int sync_and_check(locohd_ctx* ctx) {
    CU(ctx, cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    const int code = *ctx->h_err;
    if (code) {
        CU(ctx, cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
        return fail(ctx, code, "%s", status_text(code));
    }
    return 0;
}

int need_params(locohd_ctx* ctx) {
    if (!ctx) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null context");
    if (!ctx->has_params) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "locohd_ctx_set_params has not been called");
    return 0;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int small_int_exponent(double v) {
    if (v >= 0.0 && v <= 64.0 && std::floor(v) == v) return (int)v;
    return -1;
}

// WeightFunction::build validation (weight_function.rs:22-93)
int make_wf(locohd_ctx* ctx, const locohd_weight_function& in, WfDev* out) {
    WfDev w{};
    w.kind = in.kind;
    w.n = in.n_params;
    w.int_a = w.int_b = -1;
    w.monotone = 0;
    w.pad = 0;
    w.inv_range = w.inv_norm = 0.0;
    if (in.n_params < 0 || in.n_params > LOCOHD_MAX_WF_PARAMS)
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "weight function with %d parameters (max %d)", in.n_params,
                    LOCOHD_MAX_WF_PARAMS);
    for (int i = 0; i < in.n_params; ++i) w.p[i] = in.params[i];
    const double* p = in.params;
    switch (in.kind) {
        case LOCOHD_WF_HYPER_EXP: {
            if (in.n_params % 2 != 0)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"hyper_exp\" there must be an even number of parameters!");
            double norm = 0.0;
            for (int i = 0; i < in.n_params; ++i)
                if (!(p[i] > 0.0))
                    return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"hyper_exp\" all parameters must be positive!");
            for (int i = 0; i < in.n_params / 2; ++i) norm += p[i];
            w.inv_norm = 1.0 / norm;
            break;
        }
        case LOCOHD_WF_DAGUM:
            if (in.n_params != 3)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"dagum\" there must be exactly 3 parameters!");
            if (p[0] < 0.0 || p[1] < 0.0 || p[2] < 0.0)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"dagum\" all parameters must be positive!");
            break;
        case LOCOHD_WF_UNIFORM:
            if (in.n_params != 2)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"uniform\" there must be exactly 2 parameters!");
            if (p[0] < 0.0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"uniform\" the first parameter must be non-negative!");
            if (p[1] <= 0.0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"uniform\" the second parameter must be positive!");
            if (!(p[0] < p[1])) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"uniform\" the first parameter must be smaller than the second!");
            w.inv_range = 1.0 / (p[1] - p[0]);
            w.monotone = 1;
            break;
        case LOCOHD_WF_KUMARASWAMY:
            if (in.n_params != 4)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"kumaraswamy\" there must be exactly 4 parameters!");
            if (p[0] < 0.0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"kumaraswamy\" the first parameter must be non-negative!");
            if (p[1] <= 0.0 || p[2] <= 0.0 || p[3] <= 0.0)
                return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"kumaraswamy\" after the first parameter all parameters must be positive!");
            if (!(p[0] < p[1])) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "For function \"kumaraswamy\" the first parameter must be smaller than the second!");
            w.inv_range = 1.0 / (p[1] - p[0]);
            w.int_a = small_int_exponent(p[2]);
            w.int_b = small_int_exponent(p[3]);
            w.monotone = (w.int_a >= 0 && w.int_b >= 0) ? 1 : 0;
            break;
        default:
            return fail(ctx, LOCOHD_ERR_BAD_PARAM, "No function implemented with kind %d!", in.kind);
    }
    {   // CDF(+inf) with the reference's formulas (cdfs.rs:5-63)
        const double inf = std::numeric_limits<double>::infinity();
        switch (in.kind) {
            case LOCOHD_WF_DAGUM: w.w_inf = std::pow(1.0 + std::pow(inf / p[1], -p[0]), -p[2]); break;
            case LOCOHD_WF_HYPER_EXP: {
                double sum = 0.0, norm = 0.0;
                for (int i = 0; i < in.n_params / 2; ++i) { sum += p[i] * std::exp(-p[in.n_params / 2 + i] * inf); norm += p[i]; }
                w.w_inf = 1.0 - sum / norm;
                break;
            }
            default: w.w_inf = 1.0;
        }
    }
    *out = w;
    return 0;
}

int ensure_cells(locohd_structs* s, double threshold) {
    locohd_ctx* ctx = s->ctx;
    if (s->cells_valid && s->cell_threshold == threshold) return 0;
    { ProfScope ps(ctx, LOCOHD_PROF_CELLS); ctx->launches += launch_build_cells(s->view(), threshold, s->max_prims, ctx->stream); }
    CU(ctx, cudaGetLastError());
    s->cells_valid = true;
    s->cell_threshold = threshold;
    return 0;
}

int read_scan_stats(locohd_ctx* ctx, int slot, ScanStats* host) {
    CU(ctx, cudaMemcpyAsync(host, ctx->d_scan + slot, sizeof(ScanStats), cudaMemcpyDeviceToHost, ctx->stream));
    return sync_and_check(ctx);
}

int read_fused_stats(locohd_ctx* ctx, int slot, FusedStats* host) {
    if (cudaMemcpyAsync(&ctx->h_fstats[slot], ctx->d_fstats, sizeof(FusedStats), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess)
        return fail(ctx, LOCOHD_ERR_CUDA, "copy of the gather statistics failed");
    TRY_ST(sync_and_check(ctx));
    *host = ctx->h_fstats[slot];
    return 0;
}

void destroy_envset(locohd_envset* e) {
    if (!e) return;
    locohd_ctx* ctx = e->ctx;
    DeviceGuard g(ctx->device);
    dev_free(ctx, e->d_off); dev_free(ctx, e->d_count); dev_free(ctx, e->d_key); dev_free(ctx, e->d_dist);
    dev_free(ctx, e->d_idx);
    delete e;
}

constexpr uint64_t kBoundAnchors = 32768;
constexpr uint32_t kSampleStride = 16;

// Store entries of the fused gather for n_anchors environments of at most `cap` members gathered by `grid` blocks:
// the `history` size when not 0 (the store size that worked for the last call of this shape), else for calls of up to
// kBoundAnchors anchors (one structure pair is the typical call of the reference API) the bound `cap` per environment,
// else the sum `sample` of the FP32 upper-bound sizes of every kSampleStride-th anchor.
uint64_t fused_store_capacity(uint64_t n_anchors, int cap, unsigned grid, uint64_t sample, uint64_t history) {
    if (history) return history;
    // sampled sizes are FP32 upper bounds; even-rounding adds at most one entry per environment, every warp can leave
    // most of a chunk unused at every refill and at the end
    const double est = n_anchors <= kBoundAnchors ? (double)n_anchors * (double)cap
                                                  : (double)sample * (double)kSampleStride * 1.03 + 65536.0;
    const double waste = 1.0 + (double)cap / (double)kFusedChunk;
    const uint64_t capacity = (uint64_t)((est + (double)n_anchors) * waste) + (uint64_t)grid * kFusedWarps * kFusedChunk + 2 * kFusedChunk;
    // The sample differs a little from call to call (cell order depends on atomics): round the size up to 4
    // significant bits so that repeated calls ask the block cache for the same size (a fresh multi-GB
    // cudaMallocAsync costs 0.5-2 s).
    for (uint64_t step = 1ull << 62; step >= 32; step >>= 1)
        if (capacity & step) { step >>= 4; return (capacity + step - 1) & ~(step - 1); }
    return capacity;
}

// The fused gather: env_fused_kernel gathers, sorts and packs every environment in one launch.  It runs the 512-member
// instantiation, or the 1024-member one once a call has reported larger environments (the hint stays with the context
// until a 1024 run sees none above 384 members).  *built stays false, with no store allocated, when an environment has
// more than 1024 members or the store overflows for another reason than the cap.
int fused_gather(locohd_ctx* ctx, const StructsView& sv, locohd_envset* e, const uint32_t* d_anchor_struct,
                 const uint32_t* d_anchor_prim, double threshold, int keep_indices, const uint32_t* d_order,
                 const uint2* d_order_rec, bool* built) {
    const uint64_t n_anchors = e->n_env;
    const bool by_bound = n_anchors <= kBoundAnchors;
    auto& h = ctx->store_hist;
    // A call of the same shape as the last one (a benchmark step, the next block of trajectory frames) takes the store
    // size that worked then and skips the sizing pass and its synchronisation.  If that store turns out too small, the
    // history is dropped and the call is redone once, sized by a sample like a first call.
    for (int attempt = 0; attempt < 2; ++attempt) {
        const uint64_t history = !by_bound && h.n_anchors == n_anchors && h.threshold == threshold && h.cap == h.cap_hint ? h.capacity : 0;
        cudaMemsetAsync(ctx->d_fstats, 0, sizeof(FusedStats), ctx->stream);
        FusedStats fs{};
        if (!by_bound && !history) {
            { ProfScope ps(ctx, LOCOHD_PROF_COUNT);
              ctx->launches += launch_env_sample(sv, ctx->kp, n_anchors, d_order, d_anchor_struct, d_anchor_prim, threshold,
                                                 kSampleStride, &ctx->d_fstats->sample, ctx->stream); }
            TRY_ST(read_fused_stats(ctx, 0, &fs));
        }
        for (int cap = h.cap_hint; cap <= kFusedCapBig; cap *= 2) {
            const unsigned grid = fused_grid(ctx->kp, &ctx->h_wf0, e->key_is_w ? 1 : 0, keep_indices != 0, cap, n_anchors);
            const uint64_t capacity = fused_store_capacity(n_anchors, cap, grid, fs.sample, history);
            TRY_ST(dev_alloc(ctx, &e->d_key, capacity));
            if (keep_indices) { TRY_ST(dev_alloc(ctx, &e->d_idx, capacity)); TRY_ST(dev_alloc(ctx, &e->d_dist, capacity)); }
            EnvBuild b{};   // ub, off and cat stay null: the fused kernel needs neither sizes nor scratch
            b.n_env = n_anchors; b.order = d_order; b.order_rec = d_order_rec; b.off_out = e->d_off; b.count = e->d_count;
            b.key = e->d_key; b.idx = e->d_idx; b.dist = e->d_dist; b.key_is_w = e->key_is_w ? 1 : 0; b.key_is_sq = 1;
            cudaMemsetAsync(&ctx->d_fstats->cursor, 0, sizeof(unsigned long long), ctx->stream);
            cudaMemsetAsync(&ctx->d_fstats->max_count, 0, 2 * sizeof(unsigned int), ctx->stream);
            { ProfScope ps(ctx, LOCOHD_PROF_FILL);
              ctx->launches += launch_env_fused(sv, ctx->kp, &ctx->h_wf0, d_anchor_struct, d_anchor_prim, threshold, b, cap,
                                                ctx->d_fstats, capacity, grid, ctx->stream); }
            CU(ctx, cudaGetLastError());
            FusedStats fr{}; TRY_ST(read_fused_stats(ctx, 1, &fr));
            if (!fr.overflow) {
                // remember the size for the next call of this shape unless it was a tight fit
                h.n_anchors = n_anchors; h.threshold = threshold; h.cap = cap;
                h.capacity = (!by_bound && (double)fr.cursor <= 0.94 * (double)capacity) ? capacity : 0;
                if (cap == kFusedCapBig && fr.max_count <= (unsigned)(kFusedCap * 3 / 4)) h.cap_hint = kFusedCap;
                e->capacity = capacity; e->total = fr.cursor < capacity ? fr.cursor : capacity; e->max_count = fr.max_count;
                *built = true;
                return 0;
            }
            dev_free(ctx, e->d_key); dev_free(ctx, e->d_idx); dev_free(ctx, e->d_dist);
            if (fr.overflow == 8u) h.cap_hint = kFusedCapBig;   // only "more members than cap": on with 1024 members
            if (history) { h.capacity = 0; break; }           // the history-sized store was too small: sample
            if (fr.overflow != 8u) return 0;                  // the larger instantiation will not help
        }
        if (!history) return 0;                               // an environment has more than 1024 members
    }
    return 0;
}

// The multi-kernel gather, for every environment size and threshold: K1a upper-bound sizes -> scan -> store
// allocation -> K1b exact gather into the store -> K1c per-environment sort + CDF + key packing.  One host
// synchronisation (the store size).  *d_cat is allocated here; the caller releases it with its own scratch.
int multi_kernel_gather(locohd_ctx* ctx, const StructsView& sv, locohd_envset* e, const uint32_t* d_anchor_struct,
                        const uint32_t* d_anchor_prim, double threshold, int keep_indices, const uint32_t* d_order,
                        uint32_t* d_ub, uint64_t* d_scratch, uint8_t** d_cat) {
    { ProfScope ps(ctx, LOCOHD_PROF_COUNT);
      ctx->launches += launch_env_count(sv, ctx->kp, e->n_env, d_order, d_anchor_struct, d_anchor_prim, threshold, d_ub, ctx->stream); }
    { ProfScope ps(ctx, LOCOHD_PROF_SCAN); ctx->launches += launch_scan(d_ub, e->n_env, 1, e->d_off, d_scratch, ctx->d_scan + 1, ctx->stream); }
    ScanStats ss{};
    TRY_ST(read_scan_stats(ctx, 1, &ss));
    e->capacity = ss.total + 2;
    e->max_count = ss.max_value;   // upper bound of every environment size
    TRY_ST(dev_alloc(ctx, &e->d_key, e->capacity)); TRY_ST(dev_alloc(ctx, d_cat, e->capacity));
    if (keep_indices) { TRY_ST(dev_alloc(ctx, &e->d_idx, e->capacity)); TRY_ST(dev_alloc(ctx, &e->d_dist, e->capacity)); }
    EnvBuild b{};
    b.n_env = e->n_env; b.order = d_order; b.ub = d_ub; b.off = e->d_off; b.count = e->d_count; b.key = e->d_key;
    b.cat = *d_cat; b.idx = e->d_idx; b.dist = e->d_dist; b.key_is_w = e->key_is_w ? 1 : 0; b.key_is_sq = 1;
    { ProfScope ps(ctx, LOCOHD_PROF_FILL); ctx->launches += launch_env_fill(sv, ctx->kp, d_anchor_struct, d_anchor_prim, threshold, b, ctx->stream); }
    { ProfScope ps(ctx, LOCOHD_PROF_SORT); ctx->launches += launch_env_sort(ctx->kp, b, e->max_count, threshold, ctx->stream); }
    CU(ctx, cudaGetLastError());
    e->total = ss.total;  // stored entries (upper bound of the member count; exact sizes are in d_count)
    return 0;
}

// Environments of a list of anchors (kd-tree build + env_from_idx, locohd.rs:504-542): K0 cells (cached per
// threshold), the anchors in cell order, then the fused gather, or the multi-kernel gather when the fused one does not
// apply or falls back.  The fused kernel works with r^2 in the f32 exponent range (fixed-point sort keys, f32-seeded
// square roots); LOCOHD_LEGACY_GATHER takes the multi-kernel gather for every call.
int build_envset(locohd_ctx* ctx, locohd_structs* s, uint64_t n_anchors, const uint32_t* d_anchor_struct,
                 const uint32_t* d_anchor_prim, double threshold, int keep_indices, const LaunchOverrides& ov,
                 locohd_envset** out) {
    if (!(threshold > 0.0))  // NaN included: nothing passes `d2 < r*r`, the reference then panics on dists[0]
        return fail(ctx, LOCOHD_ERR_EMPTY_ENV, "threshold_distance must be positive (got %g): every environment would be empty", threshold);
    if (n_anchors > 0xFFFFFFF0ull) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "more than 2^32 anchors in one call");
    TRY_ST(ensure_cells(s, threshold));
    locohd_envset* e = new locohd_envset();
    e->ctx = ctx;
    e->n_env = n_anchors;
    e->key_is_w = ctx->kp.n_wf == 1;  // a single weight function: the store holds W(distance) directly
    uint32_t *d_order = nullptr, *d_slot_cnt = nullptr, *d_ub = nullptr;
    uint2* d_order_rec = nullptr;
    uint64_t *d_slot_off = nullptr, *d_scratch = nullptr;
    uint8_t* d_cat = nullptr;
    auto release = [&]() {  // stream-ordered: freed after the kernels of this call have run
        dev_free(ctx, d_order); dev_free(ctx, d_order_rec); dev_free(ctx, d_slot_cnt); dev_free(ctx, d_ub); dev_free(ctx, d_slot_off);
        dev_free(ctx, d_scratch); dev_free(ctx, d_cat);
    };
    auto bail = [&](int st) { release(); destroy_envset(e); return st; };
    int st;
    if ((st = dev_alloc(ctx, &e->d_count, n_anchors)) || (st = dev_alloc(ctx, &e->d_off, n_anchors + 1))) return bail(st);
    const StructsView sv = s->view();
    if (n_anchors == 0) { cudaMemsetAsync(e->d_off, 0, sizeof(uint64_t), ctx->stream); *out = e; return 0; }
    const uint64_t n_prims = s->n_prims;
    const uint64_t scratch_n = std::max(scan_scratch_entries(n_prims + 1), scan_scratch_entries(n_anchors));
    if ((st = dev_alloc(ctx, &d_order, n_anchors)) || (st = dev_alloc(ctx, &d_order_rec, n_anchors)) || (st = dev_alloc(ctx, &d_slot_cnt, n_prims + 1)) ||
        (st = dev_alloc(ctx, &d_slot_off, n_prims + 2)) || (st = dev_alloc(ctx, &d_scratch, scratch_n)) ||
        (st = dev_alloc(ctx, &d_ub, n_anchors)))
        return bail(st);
    { ProfScope ps(ctx, LOCOHD_PROF_OTHER);
      ctx->launches += launch_anchor_order(sv, ctx->kp, n_anchors, d_anchor_struct, d_anchor_prim, n_prims, d_slot_cnt,
                                           d_slot_off, d_scratch, ctx->d_scan, d_order, d_order_rec, ctx->stream); }
    bool built = false;
    if (!ov.legacy_gather && threshold * threshold < 1.0e30)
        st = fused_gather(ctx, sv, e, d_anchor_struct, d_anchor_prim, threshold, keep_indices, d_order, d_order_rec, &built);
    if (!st && !built)
        st = multi_kernel_gather(ctx, sv, e, d_anchor_struct, d_anchor_prim, threshold, keep_indices, d_order, d_ub, d_scratch, &d_cat);
    if (st) return bail(st);
    release();
    *out = e;
    return 0;
}

// Groups a list of equally sized jobs into tiles of <= kTileDim x kTileDim jobs that share runs of environments
// (greedy, in list order: a job joins the open tile while its A run and its B run fit the tile's rows and columns and
// its cell is free).  batch.py::blocked_pairs lists an all-vs-all ensemble so that this recovers its 4 x 4 blocks.
std::vector<ScoreTile> group_job_tiles(const std::vector<locohd_job>& jobs, const std::vector<uint64_t>& joff) {
    std::vector<ScoreTile> tiles;
    ScoreTile t;
    int rows = 0, cols = 0;
    auto open = [&]() {
        for (int k = 0; k < kTileDim; ++k) { t.a_first[k] = kTileNone; t.b_first[k] = kTileNone; }
        for (int k = 0; k < kTileDim * kTileDim; ++k) t.out_first[k] = kTileNone;
        rows = cols = 0;
    };
    open();
    for (size_t j = 0; j < jobs.size(); ++j) {
        for (;;) {
            int r = 0, c = 0;
            while (r < rows && t.a_first[r] != jobs[j].a_first) ++r;
            while (c < cols && t.b_first[c] != jobs[j].b_first) ++c;
            if (r < kTileDim && c < kTileDim && t.out_first[r * kTileDim + c] == kTileNone) {
                if (r == rows) t.a_first[rows++] = jobs[j].a_first;
                if (c == cols) t.b_first[cols++] = jobs[j].b_first;
                t.out_first[r * kTileDim + c] = joff[j];
                break;
            }
            tiles.push_back(t);   // does not fit: close the tile, the job opens the next one
            open();
        }
    }
    if (rows) tiles.push_back(t);
    return tiles;
}

// The same for job lists in any order (plain row-major (i, j) order of an ensemble, shuffled lists) and for tiles of
// any size DIM: the distinct A runs and B runs are ranked, a job belongs to block (rank_a / DIM, rank_b / DIM) and
// sits in cell (rank_a % DIM, rank_b % DIM) of it; blocks are scored in (block row, block column) order, which keeps
// the structures of a block row in L2.  A job named twice opens a second tile of its block.  O(n log n) on the host,
// so at DIM = 4 it is only tried when the list order itself does not tile.  More than max_tiles tiles: stops and
// returns no tiles (a list that cannot fill its tiles).
template <int DIM>
std::vector<TileDesc<DIM>> group_job_tiles_sorted(const std::vector<locohd_job>& jobs, const std::vector<uint64_t>& joff,
                                                  size_t max_tiles = SIZE_MAX) {
    std::vector<uint64_t> av(jobs.size()), bv(jobs.size());
    for (size_t j = 0; j < jobs.size(); ++j) { av[j] = jobs[j].a_first; bv[j] = jobs[j].b_first; }
    std::sort(av.begin(), av.end()); av.erase(std::unique(av.begin(), av.end()), av.end());
    std::sort(bv.begin(), bv.end()); bv.erase(std::unique(bv.begin(), bv.end()), bv.end());
    struct Item { uint64_t block; uint32_t cell; uint32_t job; };
    std::vector<Item> items(jobs.size());
    for (size_t j = 0; j < jobs.size(); ++j) {
        const uint64_t ra = (uint64_t)(std::lower_bound(av.begin(), av.end(), jobs[j].a_first) - av.begin());
        const uint64_t rb = (uint64_t)(std::lower_bound(bv.begin(), bv.end(), jobs[j].b_first) - bv.begin());
        items[j] = {((ra / DIM) << 32) | (rb / DIM), (uint32_t)((ra % DIM) * DIM + rb % DIM), (uint32_t)j};
    }
    std::stable_sort(items.begin(), items.end(), [](const Item& x, const Item& y) { return x.block < y.block; });
    std::vector<TileDesc<DIM>> tiles;
    size_t lo = 0;
    while (lo < items.size()) {
        size_t hi = lo;
        while (hi < items.size() && items[hi].block == items[lo].block) ++hi;
        size_t first_tile = tiles.size();
        for (size_t k = lo; k < hi; ++k) {
            const Item& it = items[k];
            const int r = (int)(it.cell / DIM), c = (int)(it.cell % DIM);
            size_t t = first_tile;   // first tile of this block whose cell is still free
            while (t < tiles.size() && tiles[t].out_first[it.cell] != kTileNone) ++t;
            if (t == tiles.size()) {
                if (tiles.size() == max_tiles) return {};
                tiles.emplace_back();
                TileDesc<DIM>& nt = tiles.back();
                for (int q = 0; q < DIM; ++q) { nt.a_first[q] = kTileNone; nt.b_first[q] = kTileNone; }
                for (int q = 0; q < DIM * DIM; ++q) nt.out_first[q] = kTileNone;
            }
            tiles[t].a_first[r] = jobs[it.job].a_first;
            tiles[t].b_first[c] = jobs[it.job].b_first;
            tiles[t].out_first[it.cell] = joff[it.job];
        }
        lo = hi;
    }
    return tiles;
}

// A row of a tile is one warp, four pairs wide; full tiles run 1.5 x the pair kernel's rate (profiles/r6a).  The tile
// kernel pays when the rows are mostly filled and a team mostly has work for its four warps (one-against-many lists -
// trajectory frames against frame 0 - give tiles of a single row: three of four warps would idle).
uint64_t tile_rows(const std::vector<ScoreTile>& tiles) {
    uint64_t rows = 0;
    for (const ScoreTile& t : tiles)
        for (int r = 0; r < kTileDim; ++r) rows += t.a_first[r] != kTileNone ? 1 : 0;
    return rows;
}

bool tiles_pay(const std::vector<ScoreTile>& tiles, uint64_t n_jobs) {
    const uint64_t rows = tile_rows(tiles);
    return !tiles.empty() && n_jobs * 10 >= rows * kTileDim * 6 && rows >= 3 * tiles.size();
}

// A wide tile is one CTA of 1024 lanes, one per cell: it pays when at least 80 % of the cells hold a job.  Measured
// against the 4 x 4 tiles (B200, profiles/r16a_wide_tiles.md): 1.20 x on the 1000-member ensemble in blocked order
// (92 % filled), 0.98 x on 96 members (74 %); the 4 x 4 tiles, whose rows are one warp each, waste fewer lanes.
constexpr uint64_t kWideFillPct = 80;
size_t wide_tiles_max(uint64_t n_jobs) { return (size_t)(n_jobs * 100 / (kWideFillPct * kWideDim * kWideDim)); }

// The list order itself (batch.py::blocked_pairs) when its tiles pay, else the sorted grouping (any other order).
// Lists of fewer than 4 jobs, of unequal jobs or of empty jobs get no tiles.
TilePlan plan_job_tiles(const std::vector<locohd_job>& jobs, const std::vector<uint64_t>& joff) {
    TilePlan plan;
    if (jobs.size() < 4 || jobs[0].n == 0) return plan;
    for (const locohd_job& j : jobs)
        if (j.n != jobs[0].n) return plan;
    plan.tiles = group_job_tiles(jobs, joff);
    plan.pays = tiles_pay(plan.tiles, jobs.size());
    if (!plan.pays) {
        plan.tiles = group_job_tiles_sorted<kTileDim>(jobs, joff);
        plan.pays = tiles_pay(plan.tiles, jobs.size());
    }
    const size_t wide_max = wide_tiles_max(jobs.size());
    if (wide_max > 0) {
        plan.wide = group_job_tiles_sorted<kWideDim>(jobs, joff, wide_max);
        plan.wide_pays = !plan.wide.empty();
    }
    return plan;
}

int run_score(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_pairs,
              const uint32_t* d_pairs, const locohd_job* d_jobs, const uint64_t* d_job_off, uint64_t n_jobs,
              uint64_t uniform_n, const uint32_t* d_wf_idx, double* d_out, const LaunchOverrides& ov,
              const ScoreTile* d_tiles = nullptr, uint64_t n_tiles = 0, const WideTile* d_wide = nullptr) {
    ScoreArgs sa{};
    sa.tiles = d_tiles; sa.n_tiles = n_tiles;
    if (d_wide) { sa.wide_tiles = d_wide; sa.wide = 1; }
    sa.a = a->view(); sa.b = b->view();
    sa.n_pairs = n_pairs; sa.pairs = d_pairs; sa.jobs = d_jobs; sa.job_pair_off = d_job_off; sa.n_jobs = n_jobs;
    sa.uniform_n = uniform_n; sa.wf_idx = d_wf_idx; sa.out = d_out; sa.stage_cap = 0; sa.only_unstaged = 0; sa.table_n = 0;
    sa.cursor = ctx->d_score_cursor; sa.run = 1;
    int n;
    if (a->key_is_w != b->key_is_w) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "environment sets were built with different weight-function modes");
    const double mean_a = a->n_env ? (double)a->total / (double)a->n_env : 0.0;
    const double mean_b = b->n_env ? (double)b->total / (double)b->n_env : 0.0;
    { ProfScope ps(ctx, LOCOHD_PROF_SCORE);
      n = launch_score(sa, ctx->kp, a->max_count, b->max_count, mean_a, mean_b, ov, ctx->stream); }
    if (n < 0) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "shared memory budget exceeded for %d categories", ctx->kp.C);
    ctx->launches += n;
    if (d_tiles || d_wide) ctx->tile_launches += n;
    if (d_wide) ctx->wide_launches += n;
    CU(ctx, cudaGetLastError());
    return 0;
}

int check_wf_indices(locohd_ctx* ctx, const uint32_t* wf_idx, uint64_t n) {
    if (!wf_idx) return 0;
    if (is_device_ptr(ctx, wf_idx)) {
        // device-resident indices: checked by a kernel (LOCOHD_ERR_BAD_PARAM in the device error word, reported at
        // the call's synchronisation); the scoring kernels clamp the index, so nothing is read out of bounds
        ctx->launches += launch_validate_wf_idx(wf_idx, n, (uint32_t)ctx->kp.n_wf, ctx->d_err, ctx->stream);
        return 0;
    }
    for (uint64_t i = 0; i < n; ++i)
        if (wf_idx[i] >= (uint32_t)ctx->kp.n_wf)
            return fail(ctx, LOCOHD_ERR_BAD_PARAM, "weight function index %u out of range (%d functions)", wf_idx[i], ctx->kp.n_wf);
    return 0;
}

}  // namespace

#define API_BEGIN(ctx_expr)                                                                       \
    locohd_ctx* ctx__ = (ctx_expr);                                                               \
    if (!ctx__) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null context");                      \
    DeviceGuard guard__(ctx__->device);                                                           \
    try {
#define API_END()                                                                                 \
    } catch (const std::bad_alloc&) {                                                             \
        return fail(ctx__, LOCOHD_ERR_CUDA, "host out of memory");                               \
    } catch (const std::exception& ex) {                                                          \
        return fail(ctx__, LOCOHD_ERR_CUDA, "exception: %s", ex.what());                         \
    }

extern "C" {

int locohd_abi_version(void) { return LOCOHD_ABI_VERSION; }

int locohd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* locohd_last_error(const locohd_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    std::lock_guard<std::mutex> g(g_err_mutex);
    static thread_local std::string copy;
    copy = g_global_err;
    return copy.c_str();
}

int locohd_ctx_create(int device, locohd_ctx** out) {
    if (!out) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null output pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(nullptr, LOCOHD_ERR_NO_DEVICE,
                    "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return fail(nullptr, LOCOHD_ERR_NO_DEVICE, "device %d out of range (%d devices)", device, n);
    DeviceGuard g(device);
    locohd_ctx* ctx = new locohd_ctx();
    ctx->device = device;
    auto bail = [&](cudaError_t ce) {
        fail(nullptr, LOCOHD_ERR_CUDA, "context creation failed: %s", cudaGetErrorString(ce));
        delete ctx;
        return (int)LOCOHD_ERR_CUDA;
    };
    cudaError_t ce;
    if ((ce = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(ce);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    if ((ce = cudaMalloc(&ctx->d_err, sizeof(int))) != cudaSuccess) return bail(ce);
    if ((ce = cudaMemset(ctx->d_err, 0, sizeof(int))) != cudaSuccess) return bail(ce);
    if ((ce = cudaMalloc(&ctx->d_scan, 3 * sizeof(ScanStats))) != cudaSuccess) return bail(ce);
    if ((ce = cudaMalloc(&ctx->d_fstats, sizeof(FusedStats))) != cudaSuccess) return bail(ce);
    if ((ce = cudaMalloc(&ctx->d_score_cursor, sizeof(unsigned long long))) != cudaSuccess) return bail(ce);
    if ((ce = cudaHostAlloc((void**)&ctx->h_err, sizeof(int), cudaHostAllocDefault)) != cudaSuccess) return bail(ce);
    if ((ce = cudaHostAlloc((void**)&ctx->h_fstats, 2 * sizeof(FusedStats), cudaHostAllocDefault)) != cudaSuccess) return bail(ce);
    if ((ce = cudaHostAlloc((void**)&ctx->h_scan, sizeof(ScanStats), cudaHostAllocDefault)) != cudaSuccess) return bail(ce);
    *ctx->h_err = 0;
    if ((ce = cudaMalloc(&ctx->d_sqrt_tbl, kSqrtTableSize * sizeof(double))) != cudaSuccess) return bail(ce);
    if ((ce = cudaMalloc(&ctx->d_rsqrt_tbl, kSqrtTableSize * sizeof(double))) != cudaSuccess) return bail(ce);
    std::vector<double> t(kSqrtTableSize), r(kSqrtTableSize);
    for (int k = 0; k < kSqrtTableSize; ++k) {
        t[k] = std::sqrt((double)k);
        r[k] = k ? 1.0 / std::sqrt((double)k) : 0.0;
    }
    if ((ce = cudaMemcpy(ctx->d_sqrt_tbl, t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(ce);
    if ((ce = cudaMemcpy(ctx->d_rsqrt_tbl, r.data(), r.size() * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(ce);
    *out = ctx;
    return 0;
}

void locohd_ctx_destroy(locohd_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& blk : ctx->big_free) cudaFreeAsync(blk.second, ctx->stream);
    ctx->big_free.clear();
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_cat_w); cudaFree(ctx->d_cat_sw); cudaFree(ctx->d_wfs); cudaFree(ctx->d_tag_pairs);
    cudaFree(ctx->d_sqrt_tbl); cudaFree(ctx->d_rsqrt_tbl); cudaFree(ctx->d_err); cudaFree(ctx->d_scan);
    cudaFree(ctx->d_fstats); cudaFree(ctx->d_score_cursor);
    cudaFreeHost(ctx->h_err); cudaFreeHost(ctx->h_fstats); cudaFreeHost(ctx->h_scan); cudaFreeHost(ctx->h_stage);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

void* locohd_ctx_stream(locohd_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

uint64_t locohd_ctx_launch_count(const locohd_ctx* ctx) { return ctx ? ctx->launches : 0; }
uint64_t locohd_ctx_tile_launches(const locohd_ctx* ctx) { return ctx ? ctx->tile_launches : 0; }
uint64_t locohd_ctx_wide_launches(const locohd_ctx* ctx) { return ctx ? ctx->wide_launches : 0; }

int locohd_ctx_synchronize(locohd_ctx* ctx) {
    API_BEGIN(ctx)
    return sync_and_check(ctx);
    API_END()
}

int locohd_ctx_profile_enable(locohd_ctx* ctx, int on) {
    API_BEGIN(ctx)
    ctx->prof_on = on != 0;
    return 0;
    API_END()
}

int locohd_ctx_profile_read(locohd_ctx* ctx, double* ms, uint64_t* launches) {
    API_BEGIN(ctx)
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (auto& r : ctx->prof) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess && r.group >= 0 && r.group < LOCOHD_PROF_GROUPS) {
            if (ms) ms[r.group] += t;
            if (launches) launches[r.group] += 1;
        }
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    ctx->prof.clear();
    return 0;
    API_END()
}

int locohd_measure_fp64_tflops(locohd_ctx* ctx, double* out_tflops) {
    API_BEGIN(ctx)
    if (!out_tflops) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null output");
    cudaDeviceProp prop;
    CU(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    double* scratch = nullptr;
    TRY_ST(dev_alloc(ctx, &scratch, 1));
    const int blocks = prop.multiProcessorCount * 8, iters = 1 << 16;
    cudaEvent_t a, b;
    CU(ctx, cudaEventCreate(&a)); CU(ctx, cudaEventCreate(&b));
    launch_fp64_peak(scratch, blocks, 1 << 12, ctx->stream);  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        CU(ctx, cudaEventRecord(a, ctx->stream));
        launch_fp64_peak(scratch, blocks, iters, ctx->stream);
        CU(ctx, cudaEventRecord(b, ctx->stream));
        CU(ctx, cudaEventSynchronize(b));
        float msf = 0.f;
        CU(ctx, cudaEventElapsedTime(&msf, a, b));
        const double flops = 2.0 * 8.0 * (double)iters * 256.0 * (double)blocks;
        if (msf > 0.f) best = std::max(best, flops / (msf * 1e-3) / 1e12);
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    dev_free(ctx, scratch);
    *out_tflops = best;
    return 0;
    API_END()
}

int locohd_host_alloc(uint64_t bytes, void** out) {
    if (!out) return LOCOHD_ERR_BAD_PARAM;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); *out = nullptr; return fail(nullptr, LOCOHD_ERR_CUDA, "cudaHostAlloc: %s", cudaGetErrorString(e)); }
    return 0;
}

void locohd_host_free(void* p) { if (p) cudaFreeHost(p); }

int locohd_ctx_set_params(locohd_ctx* ctx, const locohd_params* params) {
    API_BEGIN(ctx)
    if (!params) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null params");
    const int C = params->n_categories;
    // LoCoHD::build (locohd.rs:305-346)
    if (C <= 0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "The number of possible categories (primitive types) cannot be zero!");
    if (C > LOCOHD_MAX_CATEGORIES)
        return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "at most %d categories are supported (got %d)", LOCOHD_MAX_CATEGORIES, C);
    std::vector<double> w(C, 1.0), sw(C, 1.0);
    bool unit = true;
    if (params->category_weights) {
        int bad = 0;
        for (int i = 0; i < C; ++i) {
            w[i] = params->category_weights[i];
            if (!(w[i] > 0.0)) ++bad;
            if (w[i] != 1.0) unit = false;
            sw[i] = std::sqrt(w[i]);
        }
        if (bad)
            return fail(ctx, LOCOHD_ERR_BAD_PARAM, "LoCoHD parameter 'category_weights' must only contain positive values! Instead, it contains %d non-positive values!", bad);
    }
    // StatisticalDistance::build (statistical_distances.rs:97-121)
    if (params->sd_kind < LOCOHD_SD_HELLINGER || params->sd_kind > LOCOHD_SD_RENYI)
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "Invalid statistical distance kind %d!", params->sd_kind);
    if (params->n_weight_functions < 1) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "at least one weight function is required");
    std::vector<WfDev> wfs(params->n_weight_functions);
    for (int i = 0; i < params->n_weight_functions; ++i) TRY_ST(make_wf(ctx, params->weight_functions[i], &wfs[i]));
    if (params->tpr_kind != LOCOHD_TPR_WITHOUT_LIST && params->tpr_kind != LOCOHD_TPR_WITH_LIST)
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "Invalid tag pairing rule kind %d!", params->tpr_kind);
    std::vector<uint64_t> pairs;
    if (params->tpr_kind == LOCOHD_TPR_WITH_LIST && params->n_tag_pairs) {
        pairs.assign(params->tag_pairs, params->tag_pairs + params->n_tag_pairs);
        std::sort(pairs.begin(), pairs.end());
        pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());
    }

    CU(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->d_cat_w); cudaFree(ctx->d_cat_sw); cudaFree(ctx->d_wfs); cudaFree(ctx->d_tag_pairs);
    ctx->d_cat_w = ctx->d_cat_sw = nullptr; ctx->d_wfs = nullptr; ctx->d_tag_pairs = nullptr;
    ctx->has_params = false;
    CU(ctx, cudaMalloc(&ctx->d_cat_w, C * sizeof(double)));
    CU(ctx, cudaMalloc(&ctx->d_cat_sw, C * sizeof(double)));
    CU(ctx, cudaMalloc(&ctx->d_wfs, wfs.size() * sizeof(WfDev)));
    CU(ctx, cudaMemcpy(ctx->d_cat_w, w.data(), C * sizeof(double), cudaMemcpyHostToDevice));
    CU(ctx, cudaMemcpy(ctx->d_cat_sw, sw.data(), C * sizeof(double), cudaMemcpyHostToDevice));
    CU(ctx, cudaMemcpy(ctx->d_wfs, wfs.data(), wfs.size() * sizeof(WfDev), cudaMemcpyHostToDevice));
    ctx->h_wf0 = wfs[0];
    if (!pairs.empty()) {
        CU(ctx, cudaMalloc(&ctx->d_tag_pairs, pairs.size() * sizeof(uint64_t)));
        CU(ctx, cudaMemcpy(ctx->d_tag_pairs, pairs.data(), pairs.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
    }
    KParams k{};
    k.C = C;
    k.sd_kind = params->sd_kind;
    k.sd_p0 = params->sd_params[0];
    k.sd_p1 = params->sd_params[1];
    k.hell2 = (params->sd_kind == LOCOHD_SD_HELLINGER && params->sd_params[0] == 2.0) ? 1 : 0;
    k.unit_w = unit ? 1 : 0;
    k.tpr_kind = params->tpr_kind;
    k.tpr_accept_same = params->tpr_accept_same ? 1 : 0;
    k.tpr_accepted_pairs = params->tpr_accepted_pairs ? 1 : 0;
    k.tpr_ordered = params->tpr_ordered ? 1 : 0;
    k.n_tag_pairs = pairs.size();
    k.tag_pairs = ctx->d_tag_pairs;
    k.cat_w = ctx->d_cat_w;
    k.cat_sw = ctx->d_cat_sw;
    k.wfs = ctx->d_wfs;
    k.n_wf = (int)wfs.size();
    k.sqrt_tbl = ctx->d_sqrt_tbl;
    k.rsqrt_tbl = ctx->d_rsqrt_tbl;
    k.err = ctx->d_err;
    ctx->kp = k;
    ctx->n_categories = C;
    ctx->has_params = true;
    return 0;
    API_END()
}

// ---------------------------------------------------------------------------------------------- structures
// Places arrays one after another in one device block, each at a multiple of 256 bytes: the alignment the kernels
// would get from a cudaMallocAsync block of its own.
struct BlockCursor {
    size_t end = 0;
    size_t take(size_t bytes) {
        const size_t at = (end + 255) & ~(size_t)255;
        end = at + bytes;
        return at;
    }
};

// Byte offsets of the arrays of a structure set in its device block.  The block starts with `head` bytes that the
// caller uses for arrays of its own (locohd_from_primitives: those of the call).  The arrays that come from the host
// follow, so that the head and they form one range [0, upload_end) that one copy can fill.
struct StructsLayout {
    size_t prim_off, xyz, tag, upload_end, cat, meta, pf, pd, porig, sorted_pos, cell_start, cell_fill, bytes;
};

static StructsLayout structs_layout(uint64_t n_structs, uint64_t n_prims, size_t head) {
    BlockCursor c{head};
    StructsLayout l;
    l.prim_off = c.take((n_structs + 1) * sizeof(uint64_t));
    l.xyz = c.take(3 * n_prims * sizeof(double));
    l.tag = c.take(n_prims * sizeof(uint32_t));
    l.upload_end = c.end;
    l.cat = c.take(n_prims);
    l.meta = c.take(n_structs * sizeof(StructMeta));
    l.pf = c.take(n_prims * sizeof(float4));
    l.pd = c.take(n_prims * sizeof(PrimRec));
    l.porig = c.take(n_prims * sizeof(uint32_t));
    l.sorted_pos = c.take(n_prims * sizeof(uint32_t));
    l.cell_start = c.take(cell_entries(n_prims, n_structs) * sizeof(uint32_t));
    l.cell_fill = c.take(cell_entries(n_prims, n_structs) * sizeof(uint32_t));
    l.bytes = c.end;
    return l;
}

// A structure set whose arrays are views into one new device block laid out by `l`; offs: host copy of the
// n_structs + 1 primitive offsets.  The contents of the arrays are the caller's to upload.
static int structs_alloc(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* offs, const StructsLayout& l,
                         locohd_structs** out) {
    locohd_structs* s = new locohd_structs();
    unsigned char* d = nullptr;
    if (int st = dev_alloc(ctx, &d, l.bytes)) { delete s; return st; }
    s->ctx = ctx; s->n_structs = n_structs; s->n_prims = offs[n_structs]; s->block = d;
    for (uint64_t k = 0; k < n_structs; ++k) s->max_prims = std::max<uint64_t>(s->max_prims, offs[k + 1] - offs[k]);
    s->d_prim_off = reinterpret_cast<uint64_t*>(d + l.prim_off);
    s->d_xyz = reinterpret_cast<double*>(d + l.xyz);
    s->d_tag = reinterpret_cast<uint32_t*>(d + l.tag);
    s->d_cat = d + l.cat;
    s->d_meta = reinterpret_cast<StructMeta*>(d + l.meta);
    s->d_pf = reinterpret_cast<float4*>(d + l.pf);
    s->d_pd = reinterpret_cast<PrimRec*>(d + l.pd);
    s->d_porig = reinterpret_cast<uint32_t*>(d + l.porig);
    s->d_sorted_pos = reinterpret_cast<uint32_t*>(d + l.sorted_pos);
    s->d_cell_start = reinterpret_cast<uint32_t*>(d + l.cell_start);
    s->d_cell_fill = reinterpret_cast<uint32_t*>(d + l.cell_fill);
    *out = s;
    return 0;
}

// Coordinates arrive as f64 (24 B per primitive) or as f32 (12 B, widened on the device: exact).
static int upload_xyz(locohd_ctx* ctx, double* d_xyz, const void* xyz, bool f32, uint64_t n3) {
    if (!n3) return 0;
    if (!f32) {
        CU(ctx, cudaMemcpyAsync(d_xyz, xyz, n3 * sizeof(double), cudaMemcpyDefault, ctx->stream));
        return 0;
    }
    InBuf<float> in;
    TRY_ST(in.load(ctx, static_cast<const float*>(xyz), n3));
    ctx->launches += launch_widen_xyz(in.ptr, d_xyz, n3, ctx->stream);
    return 0;   // a temporary of `in` is released stream-ordered, after the kernel
}

static int structs_create_impl(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* prim_offsets, const void* xyz,
                               bool f32, const uint16_t* category, const uint32_t* tag, locohd_structs** out) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!out || !prim_offsets) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    *out = nullptr;
    if (n_structs == 0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "at least one structure is required");
    // prim_offsets must be readable on the host to size the allocations
    std::vector<uint64_t> offs(n_structs + 1);
    if (is_device_ptr(ctx, prim_offsets)) {
        CU(ctx, cudaMemcpy(offs.data(), prim_offsets, offs.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    } else {
        std::memcpy(offs.data(), prim_offsets, offs.size() * sizeof(uint64_t));
    }
    if (offs[0] != 0) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "prim_offsets[0] must be 0");
    for (uint64_t s = 0; s < n_structs; ++s) {
        if (offs[s + 1] < offs[s]) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "prim_offsets must be non-decreasing");
        if (offs[s + 1] - offs[s] > 0xFFFFFFFFull) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "structure %llu has more than 2^32 primitives", (unsigned long long)s);
    }
    const uint64_t n = offs[n_structs];
    if (n && (!xyz || !category || !tag)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null primitive arrays");
    locohd_structs* s = nullptr;
    TRY_ST(structs_alloc(ctx, n_structs, offs.data(), structs_layout(n_structs, n, 0), &s));
    auto bail = [&](int st) { locohd_structs_destroy(s); return st; };
    int st;
    cudaError_t ce = cudaMemcpyAsync(s->d_prim_off, offs.data(), offs.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (ce == cudaSuccess && n) ce = cudaMemcpyAsync(s->d_tag, tag, n * sizeof(uint32_t), cudaMemcpyDefault, ctx->stream);
    if (ce != cudaSuccess) return bail(fail(ctx, LOCOHD_ERR_CUDA, "upload failed: %s", cudaGetErrorString(ce)));
    if ((st = upload_xyz(ctx, s->d_xyz, xyz, f32, 3 * n))) return bail(st);
    {
        InBuf<uint16_t> cat16;
        if ((st = cat16.load(ctx, category, n))) return bail(st);
        ctx->launches += launch_convert_categories(cat16.ptr, s->d_cat, n, ctx->kp.C, ctx->stream);
    }
    ctx->launches += launch_validate_xyz(s->d_xyz, 3 * n, ctx->d_err, ctx->stream);
    // offs (host vector) is consumed by an async copy: wait before it goes out of scope
    if ((st = sync_and_check(ctx))) return bail(st);
    *out = s;
    return 0;
    API_END()
}

int locohd_structs_create(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* prim_offsets, const double* xyz,
                          const uint16_t* category, const uint32_t* tag, locohd_structs** out) {
    return structs_create_impl(ctx, n_structs, prim_offsets, xyz, false, category, tag, out);
}

int locohd_structs_create_f32(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* prim_offsets, const float* xyz,
                              const uint16_t* category, const uint32_t* tag, locohd_structs** out) {
    return structs_create_impl(ctx, n_structs, prim_offsets, xyz, true, category, tag, out);
}

void locohd_structs_destroy(locohd_structs* s) {
    if (!s) return;
    locohd_ctx* ctx = s->ctx;
    DeviceGuard g(ctx->device);
    dev_free_bytes(ctx, s->block);
    delete s;
}

void locohd_structs_drop_cells(locohd_structs* s) { if (s) s->cells_valid = false; }

static int update_xyz_impl(locohd_structs* s, const void* xyz, bool f32) {
    if (!s) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null structures");
    API_BEGIN(s->ctx)
    locohd_ctx* ctx = s->ctx;
    if (s->n_prims && !xyz) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null xyz");
    s->cells_valid = false;
    if (s->n_prims) {
        TRY_ST(upload_xyz(ctx, s->d_xyz, xyz, f32, 3 * s->n_prims));
        ctx->launches += launch_validate_xyz(s->d_xyz, 3 * s->n_prims, ctx->d_err, ctx->stream);
    }
    return sync_and_check(ctx);
    API_END()
}

int locohd_structs_update_xyz(locohd_structs* s, const double* xyz) { return update_xyz_impl(s, xyz, false); }
int locohd_structs_update_xyz_f32(locohd_structs* s, const float* xyz) { return update_xyz_impl(s, xyz, true); }

int locohd_structs_update_from_atoms(locohd_structs* s, uint64_t first_struct, uint64_t n_frames, uint64_t n_atoms,
                                     const float* atom_xyz, uint64_t n_prims, const uint32_t* segment_start,
                                     const uint32_t* atom_index, uint64_t n_atom_refs) {
    if (!s) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null structures");
    API_BEGIN(s->ctx)
    locohd_ctx* ctx = s->ctx;
    if (n_frames == 0) return 0;
    if (first_struct + n_frames > s->n_structs) return fail(ctx, LOCOHD_ERR_INDEX, "frames address structures beyond the set");
    if (!segment_start || (n_atom_refs && !atom_index) || (n_atoms && !atom_xyz)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (n_atom_refs > 0xFFFFFFFFull) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "more than 2^32 atom references in a topology");
    // every updated structure must have the topology's primitive count (same topology for all frames)
    std::vector<uint64_t> offs(n_frames + 1);
    CU(ctx, cudaMemcpy(offs.data(), s->d_prim_off + first_struct, offs.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    for (uint64_t f = 0; f < n_frames; ++f)
        if (offs[f + 1] - offs[f] != n_prims)
            return fail(ctx, LOCOHD_ERR_LEN_MISMATCH, "structure %llu has %llu primitives, the topology yields %llu",
                        (unsigned long long)(first_struct + f), (unsigned long long)(offs[f + 1] - offs[f]),
                        (unsigned long long)n_prims);
    InBuf<float> atoms;
    InBuf<uint32_t> seg, idx;
    TRY_ST(atoms.load(ctx, atom_xyz, 3 * n_atoms * n_frames));
    TRY_ST(seg.load(ctx, segment_start, n_prims + 1));
    TRY_ST(idx.load(ctx, atom_index, n_atom_refs));
    s->cells_valid = false;
    double* dst = s->d_xyz + 3 * offs[0];
    ctx->launches += launch_centroids(atoms.ptr, n_atoms, n_frames, seg.ptr, idx.ptr, n_prims, dst, ctx->d_err, ctx->stream);
    ctx->launches += launch_validate_xyz(dst, 3 * n_prims * n_frames, ctx->d_err, ctx->stream);
    return sync_and_check(ctx);
    API_END()
}

// -------------------------------------------------------------------------------------------- environments
int locohd_envset_build(locohd_ctx* ctx, locohd_structs* s, uint64_t n_anchors, const uint32_t* anchor_struct,
                        const uint32_t* anchor_prim, double threshold, int keep_indices, locohd_envset** out) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!s || !out || (n_anchors && !anchor_prim)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (s->ctx != ctx) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "structures belong to another context");
    *out = nullptr;
    InBuf<uint32_t> as, ap;
    TRY_ST(as.load(ctx, anchor_struct, n_anchors));
    TRY_ST(ap.load(ctx, anchor_prim, n_anchors));
    TRY_ST(build_envset(ctx, s, n_anchors, as.ptr, ap.ptr, threshold, keep_indices, read_launch_overrides(), out));
    // the anchor arrays may be temporaries that are released (stream-ordered) when this scope ends
    return 0;
    API_END()
}

// Rows as environments (from_dmxs / from_coords, locohd.rs:410-476): row r becomes environment r, copied unsorted into
// the store and sorted there.  With host offsets `row_off` (ragged input, checked by the caller) row r is
// values[row_off[r], row_off[r + 1]) and row_len is the longest row; without them every row has row_len entries: row r
// is values[r * row_len, (r + 1) * row_len) or the distances of point r to the row_len points `xyz`.  Row r is
// co-sorted with the first categories (utils.rs:25-39).
static int rows_envset(locohd_ctx* ctx, uint64_t n_rows, const uint64_t* row_off, uint64_t row_len,
                       const double* values, const double* xyz, const uint16_t* category, locohd_envset** out) {
    if (!out || (row_len && !category)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    *out = nullptr;
    if (row_len > 0xFFFFFFFFull) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "rows longer than 2^32");
    // every row starts at an even entry of the store
    uint64_t n_in = xyz ? 3 * row_len : n_rows * row_len, total = n_rows * ((row_len + 1) & ~1ull);
    std::vector<uint64_t> store_off;
    if (row_off) {
        store_off.assign(n_rows + 1, 0);
        for (uint64_t r = 0; r < n_rows; ++r) store_off[r + 1] = store_off[r] + ((row_off[r + 1] - row_off[r] + 1) & ~1ull);
        n_in = row_off[n_rows];
        total = store_off[n_rows];
    }
    InBuf<double> in;
    InBuf<uint16_t> cat16;
    InBuf<uint64_t> d_row_off, d_store_off;
    TRY_ST(in.load(ctx, xyz ? xyz : values, n_in));
    TRY_ST(cat16.load(ctx, category, row_len));
    if (row_off) {
        TRY_ST(d_row_off.load(ctx, row_off, n_rows + 1));
        TRY_ST(d_store_off.load(ctx, store_off.data(), n_rows + 1));
    }
    locohd_envset* e = new locohd_envset();
    e->ctx = ctx; e->n_env = n_rows; e->total = total; e->capacity = total + 2;
    e->max_count = (unsigned)row_len;
    e->key_is_w = ctx->kp.n_wf == 1;
    uint8_t *d_cat8 = nullptr, *d_cat = nullptr;
    auto bail = [&](int st) { dev_free(ctx, d_cat8); dev_free(ctx, d_cat); destroy_envset(e); return st; };
    int st;
    if ((st = dev_alloc(ctx, &d_cat8, row_len)) || (st = dev_alloc(ctx, &e->d_count, n_rows)) ||
        (st = dev_alloc(ctx, &e->d_off, n_rows + 1)) || (st = dev_alloc(ctx, &e->d_key, e->capacity)) ||
        (st = dev_alloc(ctx, &d_cat, e->capacity)) || (st = dev_alloc(ctx, &e->d_idx, e->capacity)) ||
        (st = dev_alloc(ctx, &e->d_dist, e->capacity)))
        return bail(st);
    ctx->launches += launch_convert_categories(cat16.ptr, d_cat8, row_len, ctx->kp.C, ctx->stream);
    if (xyz) ctx->launches += launch_validate_xyz(in.ptr, 3 * row_len, ctx->d_err, ctx->stream);
    EnvBuild b{};
    b.n_env = n_rows; b.off = e->d_off; b.count = e->d_count; b.key = e->d_key; b.cat = d_cat; b.idx = e->d_idx;
    b.dist = e->d_dist; b.key_is_w = e->key_is_w ? 1 : 0; b.key_is_sq = 0; b.check_first_zero = 1;
    {
        ProfScope ps(ctx, LOCOHD_PROF_OTHER);
        ctx->launches += launch_rows_copy(xyz ? nullptr : in.ptr, xyz ? in.ptr : nullptr, d_cat8, n_rows, row_len,
                                          d_row_off.ptr, d_store_off.ptr, e->d_off, e->d_count, b, ctx->stream);
    }
    {
        ProfScope ps(ctx, LOCOHD_PROF_SORT);
        ctx->launches += launch_env_sort(ctx->kp, b, e->max_count, 0.0, ctx->stream);
    }
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return bail(fail(ctx, LOCOHD_ERR_CUDA, "launch failed: %s", cudaGetErrorString(ce)));
    if ((st = sync_and_check(ctx))) return bail(st);   // also keeps store_off alive until its copy is done
    dev_free(ctx, d_cat8); dev_free(ctx, d_cat);
    *out = e;
    return 0;
}

int locohd_envset_from_rows(locohd_ctx* ctx, uint64_t n_rows, uint64_t row_len, const double* dmx,
                            const uint16_t* category, locohd_envset** out) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!dmx) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null distance matrix");
    return rows_envset(ctx, n_rows, nullptr, row_len, dmx, nullptr, category, out);
    API_END()
}

int locohd_envset_from_coords(locohd_ctx* ctx, uint64_t n_points, const double* xyz, const uint16_t* category,
                              locohd_envset** out) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!xyz) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null coordinates");
    return rows_envset(ctx, n_points, nullptr, n_points, nullptr, xyz, category, out);
    API_END()
}

// Host checks of ragged rows (locohd_envset_from_ragged_rows, locohd_from_rows_grad): copies the offsets (host or
// device memory) to in_off and sets *max_len to the longest row.
static int ragged_rows_check(locohd_ctx* ctx, uint64_t n_rows, const uint64_t* row_offsets, const double* values,
                             const uint16_t* category, uint64_t n_categories_given, std::vector<uint64_t>& in_off,
                             uint64_t* max_len) {
    if (!row_offsets) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    in_off.assign(n_rows + 1, 0);
    if (is_device_ptr(ctx, row_offsets)) CU(ctx, cudaMemcpy(in_off.data(), row_offsets, in_off.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    else std::memcpy(in_off.data(), row_offsets, in_off.size() * sizeof(uint64_t));
    *max_len = 0;
    for (uint64_t r = 0; r < n_rows; ++r) {
        if (in_off[r + 1] < in_off[r]) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "row_offsets must be non-decreasing");
        const uint64_t len = in_off[r + 1] - in_off[r];
        if (len == 0) return fail(ctx, LOCOHD_ERR_EMPTY_ENV, "row %llu is empty (the reference panics on dists[0])", (unsigned long long)r);
        if (len > 0xFFFFFFFFull) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "rows longer than 2^32");
        if (len > n_categories_given)   // sort_together indexes the categories by the row's indices (utils.rs:33-36)
            return fail(ctx, LOCOHD_ERR_LEN_MISMATCH, "row %llu has %llu distances but only %llu categories were given",
                        (unsigned long long)r, (unsigned long long)len, (unsigned long long)n_categories_given);
        *max_len = std::max(*max_len, len);
    }
    if (in_off[n_rows] && (!values || !category)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    return 0;
}

int locohd_envset_from_ragged_rows(locohd_ctx* ctx, uint64_t n_rows, const uint64_t* row_offsets, const double* values,
                                   const uint16_t* category, uint64_t n_categories_given, locohd_envset** out) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!out) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    *out = nullptr;
    std::vector<uint64_t> in_off;
    uint64_t max_len = 0;
    TRY_ST(ragged_rows_check(ctx, n_rows, row_offsets, values, category, n_categories_given, in_off, &max_len));
    return rows_envset(ctx, n_rows, in_off.data(), max_len, values, nullptr, category, out);
    API_END()
}

void locohd_envset_destroy(locohd_envset* e) { destroy_envset(e); }
uint64_t locohd_envset_size(const locohd_envset* e) { return e ? e->n_env : 0; }
uint64_t locohd_envset_total_members(const locohd_envset* e) {
    if (!e || !e->n_env) return 0;
    // exact member count = sum of the sizes (the store itself is sized by upper bounds)
    DeviceGuard g(e->ctx->device);
    cudaStreamSynchronize(e->ctx->stream);
    std::vector<uint32_t> cnt(e->n_env);
    if (cudaMemcpy(cnt.data(), e->d_count, e->n_env * sizeof(uint32_t), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    uint64_t t = 0;
    for (uint32_t c : cnt) t += c;
    return t;
}

int locohd_envset_dump(locohd_ctx* ctx, const locohd_envset* e, uint64_t* offsets, double* distances,
                       uint16_t* categories, uint32_t* prim_indices) {
    API_BEGIN(ctx)
    if (!e) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null envset");
    TRY_ST(sync_and_check(ctx));
    // The store leaves slack after every environment (its offsets come from upper bounds): the dump is compact,
    // offsets = running sum of the exact sizes.
    const uint64_t n = e->n_env;
    std::vector<uint64_t> off(n + 1, 0), canon(n + 1, 0);
    std::vector<uint32_t> cnt(n);
    if (n) {
        CU(ctx, cudaMemcpy(off.data(), e->d_off, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
        CU(ctx, cudaMemcpy(cnt.data(), e->d_count, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    }
    for (uint64_t i = 0; i < n; ++i) canon[i + 1] = canon[i] + cnt[i];
    const uint64_t total = canon[n];
    if (offsets) CU(ctx, cudaMemcpy(offsets, canon.data(), (n + 1) * sizeof(uint64_t), cudaMemcpyDefault));
    std::vector<uint64_t> keys;
    if ((categories || (distances && !e->d_dist)) && total) {
        keys.resize(e->capacity);
        CU(ctx, cudaMemcpy(keys.data(), e->d_key, e->capacity * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    }
    if (distances && total) {
        std::vector<double> outv(total);
        if (e->d_dist) {
            std::vector<double> raw(e->capacity);
            CU(ctx, cudaMemcpy(raw.data(), e->d_dist, e->capacity * sizeof(double), cudaMemcpyDeviceToHost));
            for (uint64_t i = 0; i < n; ++i) std::copy(raw.begin() + off[i], raw.begin() + off[i] + cnt[i], outv.begin() + canon[i]);
        } else if (!e->key_is_w) {
            // without the parity arrays the distances are only known up to the 8 mantissa bits that hold the category
            for (uint64_t i = 0; i < n; ++i)
                for (uint32_t k = 0; k < cnt[i]; ++k) {
                    const uint64_t bits = keys[off[i] + k] & ~kCatMask;
                    std::memcpy(&outv[canon[i] + k], &bits, sizeof(double));
                }
        } else {
            return fail(ctx, LOCOHD_ERR_BAD_PARAM, "envset was built without keep_indices: distances are not kept");
        }
        CU(ctx, cudaMemcpy(distances, outv.data(), total * sizeof(double), cudaMemcpyDefault));
    }
    if (categories && total) {
        std::vector<uint16_t> c16(total);
        for (uint64_t i = 0; i < n; ++i)
            for (uint32_t k = 0; k < cnt[i]; ++k) {
                const uint8_t c = (uint8_t)(keys[off[i] + k] & kCatMask);
                c16[canon[i] + k] = c == kUnknownCat8 ? (uint16_t)LOCOHD_UNKNOWN_CATEGORY : c;
            }
        CU(ctx, cudaMemcpy(categories, c16.data(), total * sizeof(uint16_t), cudaMemcpyDefault));
    }
    if (prim_indices && total) {
        if (!e->d_idx) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "envset was built without keep_indices");
        std::vector<uint32_t> raw(e->capacity), outv(total);
        CU(ctx, cudaMemcpy(raw.data(), e->d_idx, e->capacity * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < n; ++i) std::copy(raw.begin() + off[i], raw.begin() + off[i] + cnt[i], outv.begin() + canon[i]);
        CU(ctx, cudaMemcpy(prim_indices, outv.data(), total * sizeof(uint32_t), cudaMemcpyDefault));
    }
    return 0;
    API_END()
}

// ------------------------------------------------------------------------------------------------ scoring
int locohd_score_pairs(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_pairs,
                       const uint32_t* pairs, const uint32_t* wf_idx, double* out_scores) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!a || !b || (n_pairs && (!pairs || !out_scores))) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    TRY_ST(check_wf_indices(ctx, wf_idx, n_pairs));
    InBuf<uint32_t> pr, wf;
    TRY_ST(pr.load(ctx, pairs, 2 * n_pairs));
    TRY_ST(wf.load(ctx, wf_idx, n_pairs));
    OutBuf<double> out;
    TRY_ST(out.prepare(ctx, out_scores, n_pairs));
    TRY_ST(run_score(ctx, a, b, n_pairs, pr.ptr, nullptr, nullptr, 0, 0, wf.ptr, out.ptr, read_launch_overrides()));
    TRY_ST(out.commit());
    return sync_and_check(ctx);
    API_END()
}

int locohd_plan_job_tiles(uint64_t n_jobs, const locohd_job* jobs, uint64_t* out_tiles, uint64_t* out_rows, int* out_pays) {
    if (n_jobs && !jobs) return LOCOHD_ERR_BAD_PARAM;
    try {
        std::vector<locohd_job> hj(jobs, jobs + n_jobs);   // host memory only: this is a host-side query
        std::vector<uint64_t> joff(n_jobs + 1, 0);
        for (uint64_t j = 0; j < n_jobs; ++j) joff[j + 1] = joff[j] + hj[j].n;
        const TilePlan plan = plan_job_tiles(hj, joff);
        if (out_tiles) *out_tiles = plan.tiles.size();
        if (out_rows) *out_rows = tile_rows(plan.tiles);
        if (out_pays) *out_pays = plan.pays ? 1 : 0;
        return LOCOHD_OK;
    } catch (const std::exception&) {
        return LOCOHD_ERR_CUDA;
    }
}

int locohd_tile_unit(uint64_t n_tiles, uint64_t n_anchors, uint64_t slice, uint64_t unit, uint64_t* out_tile,
                     uint64_t* out_anchor) {
    if (!out_tile || !out_anchor || n_anchors == 0 || n_tiles > (~0ull) / n_anchors || unit >= n_tiles * n_anchors)
        return LOCOHD_ERR_BAD_PARAM;
    const TileOrder o = make_tile_order(n_tiles, n_anchors, slice);
    tile_unit<uint64_t>(o, unit, out_tile, out_anchor);
    if (((n_tiles * n_anchors) >> 32) == 0) {   // the kernel's 32-bit path must agree
        uint32_t t32 = 0, p32 = 0;
        tile_unit<uint32_t>(o, (uint32_t)unit, &t32, &p32);
        if (t32 != *out_tile || p32 != *out_anchor) return LOCOHD_ERR_CUDA;
    }
    return LOCOHD_OK;
}

int locohd_tile_geometry(int n_categories, uint32_t max_a, uint32_t max_b, int* teams, int* cp, int* rep_n,
                         int* table_n) {
    if (!teams) return LOCOHD_ERR_BAD_PARAM;
    KParams p{};
    p.C = n_categories;
    p.hell2 = 1;
    p.unit_w = 1;
    const TileGeometry g = tile_geometry(p, max_a, max_b, 1, read_launch_overrides());
    *teams = g.teams;
    if (cp) *cp = g.cp;
    if (rep_n) *rep_n = g.rep_n;
    if (table_n) *table_n = g.table_n;
    return LOCOHD_OK;
}

// Pairs of environments of a and b take the tile kernels: W-keyed sets, the configuration the kernels have
// (tile_geometry) and at least kTileMinTeams teams per SM.
static bool tile_route(const locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, const LaunchOverrides& ov) {
    return a->key_is_w && b->key_is_w && !ov.no_tiles &&
           tile_geometry(ctx->kp, a->max_count, b->max_count, 1, ov).teams >= kTileMinTeams;
}

int locohd_score_jobs(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_jobs,
                      const locohd_job* jobs, const uint32_t* wf_idx, double* out_scores, double* out_job_means) {
    return locohd_score_jobs_stats(ctx, a, b, n_jobs, jobs, wf_idx, out_scores, out_job_means, nullptr, nullptr);
}

int locohd_score_jobs_stats(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_jobs,
                            const locohd_job* jobs, const uint32_t* wf_idx, double* out_scores, double* out_job_means,
                            double* out_anchor_means, double* out_anchor_stds) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!a || !b || (n_jobs && !jobs)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    // the job table is read on the host to lay out the output
    std::vector<locohd_job> hj(n_jobs);
    if (n_jobs) {
        if (is_device_ptr(ctx, jobs)) CU(ctx, cudaMemcpy(hj.data(), jobs, n_jobs * sizeof(locohd_job), cudaMemcpyDeviceToHost));
        else std::memcpy(hj.data(), jobs, n_jobs * sizeof(locohd_job));
    }
    std::vector<uint64_t> joff(n_jobs + 1, 0);
    bool uniform = n_jobs > 0;
    for (uint64_t j = 0; j < n_jobs; ++j) {
        if (hj[j].a_first + hj[j].n > a->n_env || hj[j].b_first + hj[j].n > b->n_env)
            return fail(ctx, LOCOHD_ERR_INDEX, "job %llu addresses environments beyond the env-set", (unsigned long long)j);
        joff[j + 1] = joff[j] + hj[j].n;
        if (hj[j].n != hj[0].n) uniform = false;
    }
    const uint64_t n_pairs = joff[n_jobs];
    const bool anchor_stats = out_anchor_means || out_anchor_stds;
    if (n_pairs && !out_scores && !out_job_means && !anchor_stats) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "no output requested");
    if (anchor_stats && !(uniform && hj[0].n))
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "per-anchor statistics need jobs of one common, non-zero size");
    const uint64_t n_per_job = n_jobs ? hj[0].n : 0;
    TRY_ST(check_wf_indices(ctx, wf_idx, n_pairs));
    InBuf<locohd_job> dj;
    InBuf<uint64_t> djoff;
    InBuf<uint32_t> wf;
    TRY_ST(dj.load(ctx, hj.data(), n_jobs));
    TRY_ST(djoff.load(ctx, joff.data(), n_jobs + 1));
    TRY_ST(wf.load(ctx, wf_idx, n_pairs));
    OutBuf<double> out, means, amean, astd;
    double *d_scores_tmp = nullptr, *d_stat = nullptr;
    auto cleanup = [&](int st) { dev_free(ctx, d_scores_tmp); dev_free(ctx, d_stat); return st; };
    int st;
    if ((st = out.prepare(ctx, out_scores, n_pairs))) return cleanup(st);
    double* d_scores = out.ptr;
    if (!d_scores) { if ((st = dev_alloc(ctx, &d_scores_tmp, n_pairs))) return cleanup(st); d_scores = d_scores_tmp; }
    if ((st = means.prepare(ctx, out_job_means, n_jobs)) || (st = amean.prepare(ctx, out_anchor_means, n_per_job)) ||
        (st = astd.prepare(ctx, out_anchor_stds, n_per_job)))
        return cleanup(st);
    if (anchor_stats && (st = dev_alloc(ctx, &d_stat, 2 * n_per_job))) return cleanup(st);
    // Jobs that share runs of environments (an all-vs-all ensemble in 4 x 4 blocks) go to the tile kernel, which
    // stages every environment once per tile instead of once per pair.  It pays when the tiles are mostly full and
    // at least 6 teams fit an SM: below that, one pair per warp with a stage of its own is the better kernel.  Lists
    // that fill 32 x 32 tiles well go to the wide tile kernel when its stage fits (one lane per pair, no per-pair
    // split: 1.2 x the rate of the 4 x 4 tiles on the 1000-member ensemble, profiles/r16a_wide_tiles.md).
    const LaunchOverrides ov = read_launch_overrides();
    InBuf<ScoreTile> dtiles;
    InBuf<WideTile> dwide;
    TilePlan plan;   // alive until the call's final synchronisation
    if (!wf_idx && tile_route(ctx, a, b, ov)) {
        if (!ctx->tile_cache_plan.tiles.empty() && ctx->tile_cache_jobs.size() == hj.size() &&
            std::memcmp(ctx->tile_cache_jobs.data(), hj.data(), hj.size() * sizeof(locohd_job)) == 0) {
            plan = ctx->tile_cache_plan;   // the list of the previous call: 2 ms instead of 25 for 500 000 jobs
        } else {
            plan = plan_job_tiles(hj, joff);
            if (!plan.tiles.empty()) {   // a list without tiles is planned at once and does not evict the cached one
                ctx->tile_cache_jobs = hj;
                ctx->tile_cache_plan = plan;
            }
        }
        if (!(plan.wide_pays && ov.wide_tiles && wide_geometry(ctx->kp, a->max_count, b->max_count, 1, ov).fits))
            plan.wide_pays = false;
        if (plan.wide_pays) {
            if ((st = dwide.load(ctx, plan.wide.data(), plan.wide.size()))) return cleanup(st);
        } else if (plan.pays && (st = dtiles.load(ctx, plan.tiles.data(), plan.tiles.size()))) {
            return cleanup(st);
        }
    }
    const uint64_t n_tiles = plan.wide_pays ? plan.wide.size() : plan.pays ? plan.tiles.size() : 0;
    st = run_score(ctx, a, b, n_pairs, nullptr, dj.ptr, djoff.ptr, n_jobs, (uniform && hj[0].n) ? hj[0].n : 0,
                   wf.ptr, d_scores, ov, (n_tiles && !plan.wide_pays) ? dtiles.ptr : nullptr, n_tiles,
                   (n_tiles && plan.wide_pays) ? dwide.ptr : nullptr);
    if (!st && (means.ptr || anchor_stats)) {
        ProfScope ps(ctx, LOCOHD_PROF_OTHER);
        if (means.ptr) ctx->launches += launch_job_means(d_scores, djoff.ptr, n_jobs, means.ptr, ctx->stream);
        if (anchor_stats)
            ctx->launches += launch_anchor_stats(d_scores, n_per_job, n_jobs, d_stat, d_stat + n_per_job, amean.ptr,
                                                 astd.ptr, ctx->stream);
    }
    if (!st) st = out.commit();
    if (!st) st = means.commit();
    if (!st) st = amean.commit();
    if (!st) st = astd.commit();
    const int st2 = sync_and_check(ctx);  // also keeps hj/joff alive until the copies are done
    return cleanup(st ? st : st2);
    API_END()
}

// Scratch of one cross-matrix chunk: its scores (unless they go straight to a device output) and, on the pair-kernel
// route, its explicit pairs.  256 MB: a chunk of a 10^5-column matrix still has ~300 rows (3 x 10^7 pairs, far more
// than one launch needs to fill the GPU), and the rows of a chunk stay in L2 while the column blocks pass.
constexpr uint64_t kCrossScratchBytes = 256ull << 20;

// Route and weight function of the pairs of two ranges (locohd_score_cross, locohd_score_condensed and their graph
// forms): the tile kernel under the condition of locohd_score_jobs_stats (W-keyed sets - one weight function, so
// wf_idx is 0 -, Hellinger-2 with unit weights, C <= 16, >= 6 teams); else explicit pairs on the pair kernel, with the
// chosen weight function as the kernels' function 0.
struct PairRoute {
    LaunchOverrides ov;
    bool tiles;
    KParams kp;
};

static PairRoute pair_route(const locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint32_t wf_idx) {
    PairRoute r;
    r.ov = read_launch_overrides();
    r.tiles = tile_route(ctx, a, b, r.ov);
    r.kp = ctx->kp;
    r.kp.wfs = ctx->d_wfs + wf_idx;
    r.kp.n_wf = 1;
    return r;
}

// Rows per chunk of an n_a x n_b cross matrix whose entries take per_entry bytes of scratch (0: none, one chunk).
// Chunks of R whole rows (R a multiple of 4): a chunk of the dense output is one contiguous block, and the k nearest
// of a row are found in one pass over it.
static uint64_t cross_chunk_rows(uint64_t n_a, uint64_t n_b, uint64_t per_entry, const LaunchOverrides& ov) {
    uint64_t R = per_entry ? kCrossScratchBytes / (per_entry * n_b) : n_a;
    if (ov.cross_rows && ov.cross_rows < R) R = ov.cross_rows;
    R = std::max<uint64_t>(R / 4 * 4, 4);
    return std::min<uint64_t>(R, (n_a + 3) / 4 * 4);
}

// Scores environments a_first + i (i < rows) of a against b_first + j (j < cols) of b into scores[i * cols + j] on
// the route's kernel; d_pairs: room for the 2 rows cols pair entries of the pair route.
static int score_cross_chunk(locohd_ctx* ctx, const PairRoute& r, const locohd_envset* a, uint64_t a_first,
                             const locohd_envset* b, uint64_t b_first, uint64_t rows, uint64_t cols, double* scores,
                             uint32_t* d_pairs) {
    int n = 0;
    {
        ProfScope ps(ctx, LOCOHD_PROF_SCORE);
        ScoreArgs sa{};
        sa.a = a->view(); sa.b = b->view();
        sa.out = scores;
        sa.cursor = ctx->d_score_cursor; sa.run = 1;
        sa.n_pairs = rows * cols;
        if (r.tiles) {
            sa.cross = CrossGrid{a_first, b_first, rows, cols};
            n = launch_score_cross(sa, r.kp, a->max_count, b->max_count, r.ov, ctx->stream);
        } else {
            ctx->launches += launch_cross_pairs(a_first, b_first, rows, cols, d_pairs, ctx->stream);
            sa.pairs = d_pairs;
            const double mean_a = a->n_env ? (double)a->total / (double)a->n_env : 0.0;
            const double mean_b = b->n_env ? (double)b->total / (double)b->n_env : 0.0;
            n = launch_score(sa, r.kp, a->max_count, b->max_count, mean_a, mean_b, r.ov, ctx->stream);
        }
    }
    if (n < 0) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "shared memory budget exceeded for %d categories", ctx->kp.C);
    ctx->launches += n;
    if (r.tiles) ctx->tile_launches += n;
    return 0;
}

// Chunks of whole row blocks (4 rows from `first`) of the condensed vector of n environments: the scores of a chunk
// are one contiguous slice of the vector.  A chunk takes row blocks while its scores fit the scratch budget (entries
// of per_score bytes; 0: no scratch, one chunk), so the chunks further down, whose rows are shorter, take more of
// them; one row block may exceed the budget (rows of more than 8 M columns).
struct CondensedChunks {
    uint64_t n, nb, max_blocks, budget;
    CondensedChunks(uint64_t n_, uint64_t per_score, const LaunchOverrides& ov)
        : n(n_), nb((n_ + 3) / 4), max_blocks(ov.cross_rows ? std::max<uint64_t>(ov.cross_rows / 4, 1) : (n_ + 3) / 4),
          budget(per_score ? kCrossScratchBytes / per_score : ~0ull) {}
    uint64_t row_base(uint64_t i) const { return n * i - triangle<uint64_t>(i); }   // condensed index of (i, i + 1)
    uint64_t scores_of(uint64_t rb0, uint64_t rb1) const { return row_base(std::min(4 * rb1, n)) - row_base(4 * rb0); }
    uint64_t end(uint64_t rb0) const {   // the row block after the chunk that starts at rb0
        uint64_t rb1 = rb0 + 1;
        while (rb1 < nb && rb1 - rb0 < max_blocks && scores_of(rb0, rb1 + 1) <= budget) ++rb1;
        return rb1;
    }
    uint64_t scratch() const { return std::min(scores_of(0, nb), std::max(budget, scores_of(0, 1))); }   // largest chunk
};

// Scores the chunk of row blocks [rb0, rb1) of the condensed vector into `scores` (its slice) on the route's kernel;
// d_pairs: room for the chunk's pair entries on the pair route.
static int score_condensed_chunk(locohd_ctx* ctx, const PairRoute& r, const locohd_envset* s, uint64_t first,
                                 const CondensedChunks& c, uint64_t rb0, uint64_t rb1, double* scores, uint32_t* d_pairs) {
    const uint64_t i0 = 4 * rb0;
    int launched = 0;
    {
        ProfScope ps(ctx, LOCOHD_PROF_SCORE);
        ScoreArgs sa{};
        sa.a = s->view(); sa.b = sa.a;
        sa.out = scores;
        sa.n_pairs = c.scores_of(rb0, rb1);
        sa.cursor = ctx->d_score_cursor; sa.run = 1;
        if (r.tiles) {
            sa.condensed = CondensedGrid{first, c.n, rb0, rb1 - rb0, c.row_base(i0)};
            launched = launch_score_condensed(sa, r.kp, s->max_count, r.ov, ctx->stream);
        } else {
            ctx->launches += launch_condensed_pairs(first, c.n, i0, std::min(4 * rb1, c.n) - i0, d_pairs, ctx->stream);
            sa.pairs = d_pairs;
            const double mean = s->n_env ? (double)s->total / (double)s->n_env : 0.0;
            launched = launch_score(sa, r.kp, s->max_count, s->max_count, mean, mean, r.ov, ctx->stream);
        }
    }
    if (launched < 0) return fail(ctx, LOCOHD_ERR_UNSUPPORTED, "shared memory budget exceeded for %d categories", ctx->kp.C);
    ctx->launches += launched;
    if (r.tiles) ctx->tile_launches += launched;
    return 0;
}

int locohd_score_cross(locohd_ctx* ctx, const locohd_envset* a, uint64_t a_first, uint64_t n_a, const locohd_envset* b,
                       uint64_t b_first, uint64_t n_b, uint32_t wf_idx, int skip_self, double* out_scores, uint32_t k,
                       double* out_knn_scores, uint32_t* out_knn_index) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!a || !b) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (a_first > a->n_env || n_a > a->n_env - a_first || b_first > b->n_env || n_b > b->n_env - b_first)
        return fail(ctx, LOCOHD_ERR_INDEX, "cross range beyond the env-set: A [%llu, +%llu) of %llu, B [%llu, +%llu) of %llu",
                    (unsigned long long)a_first, (unsigned long long)n_a, (unsigned long long)a->n_env,
                    (unsigned long long)b_first, (unsigned long long)n_b, (unsigned long long)b->n_env);
    const bool knn = out_knn_scores || out_knn_index;
    if (!out_scores && !knn) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "no output requested");
    if (knn != (k != 0) || k > 32) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "k = %u: k-nearest outputs need 1 <= k <= 32", k);
    if (skip_self && a != b) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "skip_self needs the same env-set on both sides");
    if (n_b > 0xFFFFFFFEull) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "more than 2^32 - 2 columns");
    // rows whose own environment lies inside the column range have one column fewer
    const bool self_in_range = skip_self && a_first < b_first + n_b && b_first < a_first + n_a;
    if (knn && (uint64_t)k > n_b - (self_in_range ? 1 : 0))
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "k = %u exceeds the %llu eligible columns", k,
                    (unsigned long long)(n_b - (self_in_range ? 1 : 0)));
    TRY_ST(check_wf_indices(ctx, &wf_idx, 1));
    if (a->key_is_w != b->key_is_w) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "environment sets were built with different weight-function modes");
    if (!n_a || !n_b) return 0;

    const PairRoute route = pair_route(ctx, a, b, wf_idx);
    const bool direct = out_scores && is_device_ptr(ctx, out_scores);   // scores go straight to the caller's matrix
    const uint64_t R = cross_chunk_rows(n_a, n_b, (direct ? 0 : 8) + (route.tiles ? 0 : 8), route.ov);
    OutBuf<double> kscores;
    OutBuf<uint32_t> kindex;
    TRY_ST(kscores.prepare(ctx, out_knn_scores, knn ? n_a * k : 0));
    TRY_ST(kindex.prepare(ctx, out_knn_index, knn ? n_a * k : 0));
    double* d_chunk = nullptr;
    uint32_t* d_pairs = nullptr;
    auto cleanup = [&](int st) { dev_free(ctx, d_chunk); dev_free(ctx, d_pairs); return st; };
    int st = 0;
    if (!direct && (st = dev_alloc(ctx, &d_chunk, R * n_b))) return cleanup(st);
    if (!route.tiles && (st = dev_alloc(ctx, &d_pairs, 2 * R * n_b))) return cleanup(st);
    const int64_t self_off = skip_self ? (int64_t)a_first - (int64_t)b_first : INT64_MIN;
    for (uint64_t row0 = 0; row0 < n_a && !st; row0 += R) {
        const uint64_t rows = std::min(R, n_a - row0);
        double* scores = direct ? out_scores + row0 * n_b : d_chunk;
        if ((st = score_cross_chunk(ctx, route, a, a_first + row0, b, b_first, rows, n_b, scores, d_pairs))) break;
        if (knn) {
            ProfScope ps(ctx, LOCOHD_PROF_OTHER);
            ctx->launches += launch_row_topk(scores, rows, n_b, (int)k, skip_self ? self_off + (int64_t)row0 : INT64_MIN,
                                             kscores.ptr ? kscores.ptr + row0 * k : nullptr,
                                             kindex.ptr ? kindex.ptr + row0 * k : nullptr, ctx->stream);
        }
        if (cudaGetLastError() != cudaSuccess) { st = fail(ctx, LOCOHD_ERR_CUDA, "cross-matrix launch failed"); break; }
        if (out_scores && !direct &&
            cudaMemcpyAsync(out_scores + row0 * n_b, d_chunk, rows * n_b * sizeof(double), cudaMemcpyDeviceToHost,
                            ctx->stream) != cudaSuccess)
            st = fail(ctx, LOCOHD_ERR_CUDA, "copy of a cross-matrix chunk failed");
    }
    if (!st) st = kscores.commit();
    if (!st) st = kindex.commit();
    const int st2 = sync_and_check(ctx);
    return cleanup(st ? st : st2);
    API_END()
}

int locohd_score_condensed(locohd_ctx* ctx, const locohd_envset* s, uint64_t first, uint64_t n, uint32_t wf_idx,
                           double* out_scores) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!s) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (first > s->n_env || n > s->n_env - first)
        return fail(ctx, LOCOHD_ERR_INDEX, "condensed range beyond the env-set: [%llu, +%llu) of %llu",
                    (unsigned long long)first, (unsigned long long)n, (unsigned long long)s->n_env);
    // One triangle stands for the matrix only where the score is symmetric in its two environments.
    if (ctx->kp.sd_kind != LOCOHD_SD_HELLINGER && ctx->kp.sd_kind != LOCOHD_SD_KOLMOGOROV_SMIRNOV)
        return fail(ctx, LOCOHD_ERR_BAD_PARAM,
                    "condensed scores need a symmetric statistical distance (Hellinger or Kolmogorov-Smirnov); "
                    "locohd_score_cross gives both triangles of an asymmetric one");
    if (n > 0xFFFFFFFEull) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "more than 2^32 - 2 environments");
    TRY_ST(check_wf_indices(ctx, &wf_idx, 1));
    if (n < 2) return 0;
    if (!out_scores) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "no output");

    // Route and weight function as in locohd_score_cross with the range on both sides.
    const PairRoute route = pair_route(ctx, s, s, wf_idx);
    const bool direct = is_device_ptr(ctx, out_scores);   // scores go straight to the caller's vector
    const uint64_t per_score = (direct ? 0 : 8) + (route.tiles ? 0 : 8);
    const CondensedChunks chunks(n, per_score, route.ov);
    const uint64_t scratch = per_score ? chunks.scratch() : 0;
    double* d_chunk = nullptr;
    uint32_t* d_pairs = nullptr;
    auto cleanup = [&](int st) { dev_free(ctx, d_chunk); dev_free(ctx, d_pairs); return st; };
    int st = 0;
    if (!direct && (st = dev_alloc(ctx, &d_chunk, scratch))) return cleanup(st);
    if (!route.tiles && (st = dev_alloc(ctx, &d_pairs, 2 * scratch))) return cleanup(st);
    for (uint64_t rb0 = 0, rb1; rb0 < chunks.nb && !st; rb0 = rb1) {
        rb1 = chunks.end(rb0);
        const uint64_t base = chunks.row_base(4 * rb0), count = chunks.scores_of(rb0, rb1);
        if (!count) continue;   // the last row alone: it has no pair
        double* scores = direct ? out_scores + base : d_chunk;
        if ((st = score_condensed_chunk(ctx, route, s, first, chunks, rb0, rb1, scores, d_pairs))) break;
        if (cudaGetLastError() != cudaSuccess) { st = fail(ctx, LOCOHD_ERR_CUDA, "condensed launch failed"); break; }
        if (!direct && cudaMemcpyAsync(out_scores + base, d_chunk, count * sizeof(double), cudaMemcpyDeviceToHost,
                                       ctx->stream) != cudaSuccess)
            st = fail(ctx, LOCOHD_ERR_CUDA, "copy of a condensed chunk failed");
    }
    const int st2 = sync_and_check(ctx);
    return cleanup(st ? st : st2);
    API_END()
}

// One call of locohd_score_within[_condensed]: the graph grows chunk by chunk.  Per chunk the rows' entries are
// counted, scanned and the total read back (one synchronisation), the storage grows to hold them, and the fill kernel
// writes them behind the entries of the earlier chunks.  Everything is freed unless finish() hands the graph out.
struct GraphBuild {
    locohd_ctx* ctx;
    locohd_graph* g = nullptr;
    uint64_t cap = 0;                    // entries the storage of g holds room for
    double* d_chunk = nullptr;           // scores of a chunk
    uint32_t* d_pairs = nullptr;         // pair list of a chunk (pair route)
    uint32_t* d_counts = nullptr;        // entries per row of a chunk
    uint64_t* d_off = nullptr;           // their exclusive scan [rows + 1]
    uint64_t* d_scan_scratch = nullptr;

    explicit GraphBuild(locohd_ctx* c) : ctx(c) {}
    ~GraphBuild() {
        dev_free(ctx, d_chunk); dev_free(ctx, d_pairs); dev_free(ctx, d_counts); dev_free(ctx, d_off);
        dev_free(ctx, d_scan_scratch);
        destroy_graph(g);
    }
    // An empty graph of rows x cols, and scratch for chunks of at most chunk_rows rows and chunk_scores scores.
    int start(uint64_t rows, uint64_t cols, uint64_t chunk_rows, uint64_t chunk_scores, bool pair_route) {
        g = new locohd_graph();
        g->ctx = ctx; g->rows = rows; g->cols = cols;
        TRY_ST(dev_alloc(ctx, &g->d_indptr, rows + 1));
        CU(ctx, cudaMemsetAsync(g->d_indptr, 0, (rows + 1) * sizeof(uint64_t), ctx->stream));
        if (!chunk_rows) return 0;
        TRY_ST(dev_alloc(ctx, &d_chunk, chunk_scores));
        if (pair_route) TRY_ST(dev_alloc(ctx, &d_pairs, 2 * chunk_scores));
        TRY_ST(dev_alloc(ctx, &d_counts, chunk_rows));
        TRY_ST(dev_alloc(ctx, &d_off, chunk_rows + 1));
        return dev_alloc(ctx, &d_scan_scratch, scan_scratch_entries(chunk_rows));
    }
    // Moves the entries to storage for exactly nc >= nnz entries.
    int resize(uint64_t nc) {
        uint32_t* ni = nullptr;
        double* ns = nullptr;
        if (nc && (dev_alloc(ctx, &ni, nc) || dev_alloc(ctx, &ns, nc))) {
            cudaGetLastError();
            dev_free(ctx, ni); dev_free(ctx, ns);
            return fail(ctx, LOCOHD_ERR_CUDA, "no device memory for a graph of %llu entries (%llu entries reached)",
                        (unsigned long long)nc, (unsigned long long)g->nnz);
        }
        if (g->nnz) {
            CU(ctx, cudaMemcpyAsync(ni, g->d_indices, g->nnz * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            CU(ctx, cudaMemcpyAsync(ns, g->d_scores, g->nnz * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        dev_free(ctx, g->d_indices); dev_free(ctx, g->d_scores);
        g->d_indices = ni; g->d_scores = ns;
        cap = nc;
        return 0;
    }
    // Geometric growth: the storage never holds room for more than twice the entries reached.
    int reserve(uint64_t need) { return need <= cap ? 0 : resize(std::max(need, 2 * cap)); }
    // The entries of one chunk, scored into d_chunk.
    int add(const GraphChunk& c, bool within) {
        {
            ProfScope ps(ctx, LOCOHD_PROF_OTHER);
            ctx->launches += launch_graph_count(c, within, d_counts, ctx->stream);
            ctx->launches += launch_scan(d_counts, c.rows, 0, d_off, d_scan_scratch, ctx->d_scan + 2, ctx->stream);
        }
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaMemcpyAsync(ctx->h_scan, ctx->d_scan + 2, sizeof(ScanStats), cudaMemcpyDeviceToHost, ctx->stream));
        TRY_ST(sync_and_check(ctx));   // also surfaces the scoring kernel's errors of this chunk
        const uint64_t entries = ctx->h_scan->total;
        TRY_ST(reserve(g->nnz + entries));
        {
            ProfScope ps(ctx, LOCOHD_PROF_OTHER);
            ctx->launches += launch_graph_fill(c, within, d_off, g->nnz, g->d_indptr, g->d_indices, g->d_scores,
                                               ctx->stream);
        }
        CU(ctx, cudaGetLastError());
        g->nnz += entries;
        return 0;
    }
    // Closes the last row (the chunk of the condensed vector's last row alone is never launched), trims the storage to
    // the entries and hands the graph out.
    int finish(locohd_graph** out) {
        CU(ctx, cudaMemcpyAsync(g->d_indptr + g->rows, &g->nnz, sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        if (cap > g->nnz) TRY_ST(resize(g->nnz));
        TRY_ST(sync_and_check(ctx));
        *out = g;
        g = nullptr;
        return 0;
    }
    static void destroy_graph(locohd_graph* gr) {
        if (!gr) return;
        locohd_ctx* c = gr->ctx;
        DeviceGuard dg(c->device);
        dev_free(c, gr->d_indptr); dev_free(c, gr->d_indices); dev_free(c, gr->d_scores);
        delete gr;
    }
};

int locohd_score_within(locohd_ctx* ctx, const locohd_envset* a, uint64_t a_first, uint64_t n_a, const locohd_envset* b,
                        uint64_t b_first, uint64_t n_b, uint32_t wf_idx, int skip_self, double max_score,
                        locohd_graph** out) {
    API_BEGIN(ctx)
    if (out) *out = nullptr;
    TRY_ST(need_params(ctx));
    if (!a || !b || !out) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (a_first > a->n_env || n_a > a->n_env - a_first || b_first > b->n_env || n_b > b->n_env - b_first)
        return fail(ctx, LOCOHD_ERR_INDEX, "graph range beyond the env-set: A [%llu, +%llu) of %llu, B [%llu, +%llu) of %llu",
                    (unsigned long long)a_first, (unsigned long long)n_a, (unsigned long long)a->n_env,
                    (unsigned long long)b_first, (unsigned long long)n_b, (unsigned long long)b->n_env);
    if (skip_self && a != b) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "skip_self needs the same env-set on both sides");
    if (n_b > 0xFFFFFFFEull) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "more than 2^32 - 2 columns");
    if (std::isnan(max_score)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "max_score is NaN");
    TRY_ST(check_wf_indices(ctx, &wf_idx, 1));
    if (a->key_is_w != b->key_is_w) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "environment sets were built with different weight-function modes");

    // Route and chunks as in locohd_score_cross; the scores of a chunk always go to the scratch.
    const PairRoute route = pair_route(ctx, a, b, wf_idx);
    const uint64_t R = n_a && n_b ? cross_chunk_rows(n_a, n_b, route.tiles ? 8 : 16, route.ov) : 0;
    GraphBuild gb(ctx);
    int st = gb.start(n_a, n_b, R, R * n_b, !route.tiles);
    const int64_t self_off = skip_self ? (int64_t)a_first - (int64_t)b_first : INT64_MIN;
    for (uint64_t row0 = 0; R && row0 < n_a && !st; row0 += R) {
        const uint64_t rows = std::min(R, n_a - row0);
        if ((st = score_cross_chunk(ctx, route, a, a_first + row0, b, b_first, rows, n_b, gb.d_chunk, gb.d_pairs))) break;
        if (cudaGetLastError() != cudaSuccess) { st = fail(ctx, LOCOHD_ERR_CUDA, "graph launch failed"); break; }
        st = gb.add(GraphChunk{gb.d_chunk, rows, n_b, row0, skip_self ? self_off + (int64_t)row0 : INT64_MIN, max_score},
                    false);
    }
    if (!st) st = gb.finish(out);
    const int st2 = sync_and_check(ctx);
    return st ? st : st2;
    API_END()
}

int locohd_score_within_condensed(locohd_ctx* ctx, const locohd_envset* s, uint64_t first, uint64_t n, uint32_t wf_idx,
                                  double max_score, locohd_graph** out) {
    API_BEGIN(ctx)
    if (out) *out = nullptr;
    TRY_ST(need_params(ctx));
    if (!s || !out) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if (first > s->n_env || n > s->n_env - first)
        return fail(ctx, LOCOHD_ERR_INDEX, "graph range beyond the env-set: [%llu, +%llu) of %llu",
                    (unsigned long long)first, (unsigned long long)n, (unsigned long long)s->n_env);
    if (ctx->kp.sd_kind != LOCOHD_SD_HELLINGER && ctx->kp.sd_kind != LOCOHD_SD_KOLMOGOROV_SMIRNOV)
        return fail(ctx, LOCOHD_ERR_BAD_PARAM,
                    "an upper-triangle graph needs a symmetric statistical distance (Hellinger or Kolmogorov-Smirnov); "
                    "locohd_score_within gives both triangles of an asymmetric one");
    if (n > 0xFFFFFFFEull) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "more than 2^32 - 2 environments");
    if (std::isnan(max_score)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "max_score is NaN");
    TRY_ST(check_wf_indices(ctx, &wf_idx, 1));

    // Route and chunks as in locohd_score_condensed; the scores of a chunk always go to the scratch.
    const PairRoute route = pair_route(ctx, s, s, wf_idx);
    const CondensedChunks chunks(n, route.tiles ? 8 : 16, route.ov);
    GraphBuild gb(ctx);
    int st = gb.start(n, n, n < 2 ? 0 : n, n < 2 ? 0 : chunks.scratch(), !route.tiles);
    for (uint64_t rb0 = 0, rb1; n >= 2 && rb0 < chunks.nb && !st; rb0 = rb1) {
        rb1 = chunks.end(rb0);
        if (!chunks.scores_of(rb0, rb1)) continue;   // the last row alone: finish() closes it
        if ((st = score_condensed_chunk(ctx, route, s, first, chunks, rb0, rb1, gb.d_chunk, gb.d_pairs))) break;
        if (cudaGetLastError() != cudaSuccess) { st = fail(ctx, LOCOHD_ERR_CUDA, "graph launch failed"); break; }
        const uint64_t i0 = 4 * rb0;
        st = gb.add(GraphChunk{gb.d_chunk, std::min(4 * rb1, n) - i0, n, i0, INT64_MIN, max_score}, true);
    }
    if (!st) st = gb.finish(out);
    const int st2 = sync_and_check(ctx);
    return st ? st : st2;
    API_END()
}

int locohd_graph_shape(const locohd_graph* g, uint64_t* rows, uint64_t* cols, uint64_t* nnz) {
    if (!g) return fail(nullptr, LOCOHD_ERR_BAD_PARAM, "null graph");
    if (rows) *rows = g->rows;
    if (cols) *cols = g->cols;
    if (nnz) *nnz = g->nnz;
    return 0;
}

int locohd_graph_copy(locohd_ctx* ctx, const locohd_graph* g, uint64_t* indptr, uint32_t* indices, double* scores) {
    API_BEGIN(ctx)
    if (!g) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null graph");
    if (indptr) CU(ctx, cudaMemcpyAsync(indptr, g->d_indptr, (g->rows + 1) * sizeof(uint64_t), cudaMemcpyDefault, ctx->stream));
    if (indices && g->nnz)
        CU(ctx, cudaMemcpyAsync(indices, g->d_indices, g->nnz * sizeof(uint32_t), cudaMemcpyDefault, ctx->stream));
    if (scores && g->nnz) CU(ctx, cudaMemcpyAsync(scores, g->d_scores, g->nnz * sizeof(double), cudaMemcpyDefault, ctx->stream));
    return sync_and_check(ctx);
    API_END()
}

void locohd_graph_destroy(locohd_graph* g) { GraphBuild::destroy_graph(g); }

int locohd_condensed_unit(uint64_t n, uint64_t row_block0, uint64_t row_blocks, uint64_t unit, uint64_t* out_row_block,
                          uint64_t* out_col_block) {
    const uint64_t nb = n / 4 + (n % 4 != 0);
    if (!out_row_block || !out_col_block || row_blocks == 0 || row_block0 > nb || row_blocks > nb - row_block0)
        return LOCOHD_ERR_BAD_PARAM;
    const unsigned __int128 R = row_blocks,
                            units = R * (R + 1) / 2 + R * (unsigned __int128)(nb - row_block0 - row_blocks);
    if ((units >> 64) != 0 || unit >= (uint64_t)units) return LOCOHD_ERR_BAD_PARAM;
    uint64_t dr = 0, dc = 0;
    condensed_unit<uint64_t>(row_blocks, unit, &dr, &dc);
    if ((units >> 32) == 0) {   // the kernel's 32-bit path must agree
        uint32_t r32 = 0, c32 = 0;
        condensed_unit<uint32_t>((uint32_t)row_blocks, (uint32_t)unit, &r32, &c32);
        if (r32 != dr || c32 != dc) return LOCOHD_ERR_CUDA;
    }
    *out_row_block = row_block0 + dr;
    *out_col_block = row_block0 + dc;
    return LOCOHD_OK;
}

int locohd_score_anchor_lists(locohd_ctx* ctx, const uint16_t* seq_a, uint64_t len_a, const double* dists_a,
                              uint64_t dlen_a, const uint16_t* seq_b, uint64_t len_b, const double* dists_b,
                              uint64_t dlen_b, uint32_t wf_idx, double* out_score) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (!out_score) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null output");
    if (len_a != dlen_a || len_b != dlen_b) return fail(ctx, LOCOHD_ERR_LEN_MISMATCH, "%s", status_text(LOCOHD_ERR_LEN_MISMATCH));
    if (len_a == 0 || len_b == 0) return fail(ctx, LOCOHD_ERR_EMPTY_ENV, "from_anchors needs non-empty lists (the reference panics on dists[0])");
    if (wf_idx >= (uint32_t)ctx->kp.n_wf) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "weight function index out of range");
    InBuf<uint16_t> sa16, sb16;
    InBuf<double> da, db;
    TRY_ST(sa16.load(ctx, seq_a, len_a)); TRY_ST(sb16.load(ctx, seq_b, len_b));
    TRY_ST(da.load(ctx, dists_a, len_a)); TRY_ST(db.load(ctx, dists_b, len_b));
    uint8_t *sa8 = nullptr, *sb8 = nullptr;
    TRY_ST(dev_alloc(ctx, &sa8, len_a));
    if (int ast = dev_alloc(ctx, &sb8, len_b)) { dev_free(ctx, sa8); return ast; }
    ctx->launches += launch_convert_categories(sa16.ptr, sa8, len_a, ctx->kp.C, ctx->stream);
    ctx->launches += launch_convert_categories(sb16.ptr, sb8, len_b, ctx->kp.C, ctx->stream);
    OutBuf<double> out;
    int st = out.prepare(ctx, out_score, 1);
    if (!st) {
        ctx->launches += launch_anchor_lists(ctx->kp, sa8, len_a, da.ptr, sb8, len_b, db.ptr, wf_idx, out.ptr, ctx->stream);
        st = out.commit();
    }
    const int st2 = sync_and_check(ctx);
    dev_free(ctx, sa8); dev_free(ctx, sb8);
    return st ? st : st2;
    API_END()
}

// The shared head of locohd_from_primitives and locohd_from_primitives_grad: one structure set holding A then B, its
// inputs uploaded, categories converted, coordinates validated and the 2 P environments built.  The members release
// the set and the environments, and keep the host arrays of the upload alive until the caller has synchronised.
struct PrimCall {
    locohd_structs* s = nullptr;
    locohd_envset* env = nullptr;
    size_t o_job = 0, o_as = 0, o_ap = 0, o_wf = 0;   // the call's arrays at the start of the block of `s`
    uint64_t offs[3] = {0, 0, 0};
    std::vector<uint32_t> h_anchor, h_split;
    ~PrimCall() { if (env) destroy_envset(env); if (s) locohd_structs_destroy(s); }
    const unsigned char* at(size_t o) const { return s->block + o; }
};

// Validates the arguments; with n_pairs = 0 it returns 0 and builds nothing (pc.s stays null).
static int prim_call_build(locohd_ctx* ctx, uint64_t n_a, const double* xyz_a, const uint16_t* cat_a,
                           const uint32_t* tag_a, uint64_t n_b, const double* xyz_b, const uint16_t* cat_b,
                           const uint32_t* tag_b, uint64_t n_pairs, const uint32_t* anchors, const uint32_t* wf_idx,
                           double threshold, bool has_out, int keep_indices, const LaunchOverrides& ov, PrimCall& pc) {
    TRY_ST(need_params(ctx));
    if (n_pairs && (!anchors || !has_out)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    if ((n_a && (!xyz_a || !cat_a || !tag_a)) || (n_b && (!xyz_b || !cat_b || !tag_b)))
        return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null primitive arrays");
    if (n_pairs == 0) return 0;
    if (!(threshold > 0.0))
        return fail(ctx, LOCOHD_ERR_EMPTY_ENV, "threshold_distance must be positive (got %g): every environment would be empty", threshold);
    TRY_ST(check_wf_indices(ctx, wf_idx, n_pairs));
    const uint64_t n = n_a + n_b;
    // Its device block starts with the arrays of the call: the job, the anchors of the 2 P environments ([0, P) belong
    // to A, [P, 2 P) to B), the categories as given and the per-pair weight function indices.  Everything the host
    // sends lands in the range [0, upload_end) of the block.
    BlockCursor head;
    pc.o_job = head.take(sizeof(locohd_job));
    pc.o_as = head.take(2 * n_pairs * sizeof(uint32_t));
    pc.o_ap = head.take(2 * n_pairs * sizeof(uint32_t));
    const size_t o_cat16 = head.take(n * sizeof(uint16_t));
    pc.o_wf = head.take(wf_idx ? n_pairs * sizeof(uint32_t) : 0);
    const StructsLayout l = structs_layout(2, n, head.end);
    // Small calls with host inputs (the typical call of the reference API: one structure pair) are packed into one
    // pinned staging buffer and sent with one copy: a dozen pageable copies of ~10 us each otherwise dominate such a
    // call.  Any other call copies every input into its place in the block.
    const bool host_in = !is_device_ptr(ctx, xyz_a) && !is_device_ptr(ctx, xyz_b) && !is_device_ptr(ctx, cat_a) &&
                         !is_device_ptr(ctx, cat_b) && !is_device_ptr(ctx, tag_a) && !is_device_ptr(ctx, tag_b) &&
                         !is_device_ptr(ctx, anchors) && !(wf_idx && is_device_ptr(ctx, wf_idx));
    unsigned char* h = nullptr;
    if (host_in && l.upload_end <= (8u << 20)) {
        if (ctx->h_stage_bytes < l.upload_end) {
            if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
            ctx->h_stage = nullptr; ctx->h_stage_bytes = 0;
            const size_t want = std::max<size_t>(l.upload_end * 2, 1u << 20);
            if (cudaHostAlloc((void**)&ctx->h_stage, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); ctx->h_stage = nullptr; }
            else ctx->h_stage_bytes = want;
        }
        h = ctx->h_stage;
    }
    // the A/B split of the anchors is built on the host (device anchors are copied back first)
    const uint32_t* an = anchors;
    if (is_device_ptr(ctx, anchors)) {
        pc.h_anchor.resize(2 * n_pairs);
        CU(ctx, cudaMemcpy(pc.h_anchor.data(), anchors, 2 * n_pairs * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        an = pc.h_anchor.data();
    }
    if (!h) pc.h_split.resize(4 * n_pairs);
    uint32_t* has = h ? reinterpret_cast<uint32_t*>(h + pc.o_as) : pc.h_split.data();
    uint32_t* hap = h ? reinterpret_cast<uint32_t*>(h + pc.o_ap) : pc.h_split.data() + 2 * n_pairs;
    for (uint64_t i = 0; i < n_pairs; ++i) {
        has[i] = 0; hap[i] = an[2 * i];
        has[n_pairs + i] = 1; hap[n_pairs + i] = an[2 * i + 1];
    }
    pc.offs[1] = n_a; pc.offs[2] = n;
    TRY_ST(structs_alloc(ctx, 2, pc.offs, l, &pc.s));
    unsigned char* d = pc.s->block;
    cudaError_t ce = cudaSuccess;
    auto put = [&](size_t at, const void* src, size_t bytes) {
        if (!bytes || ce != cudaSuccess) return;
        if (h) std::memcpy(h + at, src, bytes);
        else ce = cudaMemcpyAsync(d + at, src, bytes, cudaMemcpyDefault, ctx->stream);
    };
    const locohd_job job{0, n_pairs, n_pairs};
    put(pc.o_job, &job, sizeof job);
    put(l.prim_off, pc.offs, sizeof pc.offs);
    put(l.xyz, xyz_a, 3 * n_a * sizeof(double));
    put(l.xyz + 3 * n_a * sizeof(double), xyz_b, 3 * n_b * sizeof(double));
    put(l.tag, tag_a, n_a * sizeof(uint32_t));
    put(l.tag + n_a * sizeof(uint32_t), tag_b, n_b * sizeof(uint32_t));
    put(o_cat16, cat_a, n_a * sizeof(uint16_t));
    put(o_cat16 + n_a * sizeof(uint16_t), cat_b, n_b * sizeof(uint16_t));
    if (wf_idx) put(pc.o_wf, wf_idx, n_pairs * sizeof(uint32_t));
    if (h) {
        ce = cudaMemcpyAsync(d, h, l.upload_end, cudaMemcpyHostToDevice, ctx->stream);
    } else {
        put(pc.o_as, has, 2 * n_pairs * sizeof(uint32_t));
        put(pc.o_ap, hap, 2 * n_pairs * sizeof(uint32_t));
    }
    if (ce != cudaSuccess) return fail(ctx, LOCOHD_ERR_CUDA, "upload failed: %s", cudaGetErrorString(ce));
    ctx->launches += launch_convert_categories(reinterpret_cast<const uint16_t*>(d + o_cat16), pc.s->d_cat, n, ctx->kp.C, ctx->stream);
    ctx->launches += launch_validate_xyz(pc.s->d_xyz, 3 * n, ctx->d_err, ctx->stream);
    return build_envset(ctx, pc.s, 2 * n_pairs, reinterpret_cast<const uint32_t*>(d + pc.o_as),
                        reinterpret_cast<const uint32_t*>(d + pc.o_ap), threshold, keep_indices, ov, &pc.env);
}

int locohd_from_primitives(locohd_ctx* ctx, uint64_t n_a, const double* xyz_a, const uint16_t* cat_a,
                           const uint32_t* tag_a, uint64_t n_b, const double* xyz_b, const uint16_t* cat_b,
                           const uint32_t* tag_b, uint64_t n_pairs, const uint32_t* anchors,
                           const uint32_t* wf_idx, double threshold, double* out_scores) {
    API_BEGIN(ctx)
    const LaunchOverrides ov = read_launch_overrides();
    PrimCall pc;
    TRY_ST(prim_call_build(ctx, n_a, xyz_a, cat_a, tag_a, n_b, xyz_b, cat_b, tag_b, n_pairs, anchors, wf_idx,
                           threshold, out_scores != nullptr, 0, ov, pc));
    if (!pc.s) return 0;
    OutBuf<double> out;
    int st = out.prepare(ctx, out_scores, n_pairs);
    if (!st) st = run_score(ctx, pc.env, pc.env, n_pairs, nullptr, reinterpret_cast<const locohd_job*>(pc.at(pc.o_job)),
                            nullptr, 1, n_pairs, wf_idx ? reinterpret_cast<const uint32_t*>(pc.at(pc.o_wf)) : nullptr,
                            out.ptr, ov);
    if (!st) st = out.commit();
    const int st2 = sync_and_check(ctx);   // also keeps the host arrays of the upload alive until it is done
    return st ? st : st2;
    API_END()
}

int locohd_from_primitives_grad(locohd_ctx* ctx, uint64_t n_a, const double* xyz_a, const uint16_t* cat_a,
                                const uint32_t* tag_a, uint64_t n_b, const double* xyz_b, const uint16_t* cat_b,
                                const uint32_t* tag_b, uint64_t n_pairs, const uint32_t* anchors,
                                const uint32_t* wf_idx, double threshold, const double* pair_weights,
                                double* out_scores, double* out_grad_a, double* out_grad_b) {
    API_BEGIN(ctx)
    if ((n_a && !out_grad_a) || (n_b && !out_grad_b)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null gradient array");
    const LaunchOverrides ov = read_launch_overrides();
    PrimCall pc;
    TRY_ST(prim_call_build(ctx, n_a, xyz_a, cat_a, tag_a, n_b, xyz_b, cat_b, tag_b, n_pairs, anchors, wf_idx,
                           threshold, true, 1, ov, pc));
    OutBuf<double> ga, gb, out;
    TRY_ST(ga.prepare(ctx, out_grad_a, 3 * n_a));
    TRY_ST(gb.prepare(ctx, out_grad_b, 3 * n_b));
    if (n_a) CU(ctx, cudaMemsetAsync(ga.ptr, 0, 3 * n_a * sizeof(double), ctx->stream));
    if (n_b) CU(ctx, cudaMemsetAsync(gb.ptr, 0, 3 * n_b * sizeof(double), ctx->stream));
    int st = 0;
    if (pc.s) {
        InBuf<double> pw;
        double* d_scores = nullptr;   // scores are always computed; a caller without `out_scores` gets them dropped
        if (!(st = pw.load(ctx, pair_weights, n_pairs)))
            st = out_scores ? out.prepare(ctx, out_scores, n_pairs) : dev_alloc(ctx, &d_scores, n_pairs);
        if (!st) {
            GradArgs g{};
            for (int side = 0; side < 2; ++side)
                g.side[side] = {pc.env->view(), pc.env->d_dist, pc.env->d_idx, side ? n_pairs : 0};
            g.xyz = pc.s->d_xyz; g.prim_off = pc.s->d_prim_off; g.n_structs = 2;
            g.anchor_struct = reinterpret_cast<const uint32_t*>(pc.at(pc.o_as));
            g.anchor_prim = reinterpret_cast<const uint32_t*>(pc.at(pc.o_ap));
            g.n_pairs = n_pairs;
            g.wf_idx = wf_idx ? reinterpret_cast<const uint32_t*>(pc.at(pc.o_wf)) : nullptr;
            g.pair_weights = pw.ptr;
            g.out = out_scores ? out.ptr : d_scores;
            g.grad[0] = ga.ptr; g.grad[1] = gb.ptr;
            int nl;
            { ProfScope ps(ctx, LOCOHD_PROF_SCORE); nl = launch_score_grad(g, ctx->kp, GradTarget::kCoords, ctx->stream); }
            if (nl < 0) st = fail(ctx, LOCOHD_ERR_UNSUPPORTED, "shared memory budget exceeded for %d categories", ctx->kp.C);
            else ctx->launches += nl;
            if (!st && cudaPeekAtLastError() != cudaSuccess)
                st = fail(ctx, LOCOHD_ERR_CUDA, "launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        if (!st) st = out.commit();
        dev_free(ctx, d_scores);
    }
    if (!st) st = ga.commit();
    if (!st) st = gb.commit();
    const int st2 = sync_and_check(ctx);
    return st ? st : st2;
    API_END()
}

// --------------------------------------------------------------------- gradients of from_dmxs / from_coords
// The two row sets of one gradient call, released with it (stream-ordered).
struct RowSets {
    locohd_envset* e[2] = {nullptr, nullptr};
    ~RowSets() { destroy_envset(e[0]); destroy_envset(e[1]); }
};

// Scores of the row pairs p of two row sets and g_p dS_p/dt of every entry (score_grad_kernel<kEntries>): entry c of row
// p of side s goes to d_grad[s][d_entry_off[s][p] + c].  wf_idx, pair_weights and out_scores may be host or device
// memory; the caller synchronises.
static int rows_grad(locohd_ctx* ctx, const RowSets& rs, uint64_t n_rows, const uint32_t* wf_idx,
                     const double* pair_weights, double* out_scores, const uint64_t* const d_entry_off[2],
                     double* const d_grad[2]) {
    InBuf<uint32_t> wf;
    InBuf<double> pw;
    OutBuf<double> out;
    double* d_scores = nullptr;   // scores are always computed; a caller without `out_scores` gets them dropped
    int st = wf.load(ctx, wf_idx, n_rows);
    if (!st) st = pw.load(ctx, pair_weights, n_rows);
    if (!st) st = out_scores ? out.prepare(ctx, out_scores, n_rows) : dev_alloc(ctx, &d_scores, n_rows);
    if (!st) {
        GradArgs g{};
        for (int side = 0; side < 2; ++side) {
            g.side[side] = {rs.e[side]->view(), rs.e[side]->d_dist, rs.e[side]->d_idx, 0};
            g.entry_off[side] = d_entry_off[side];
            g.entry_grad[side] = d_grad[side];
        }
        g.n_pairs = n_rows;
        g.wf_idx = wf.ptr;
        g.pair_weights = pw.ptr;
        g.out = out_scores ? out.ptr : d_scores;
        int nl;
        { ProfScope ps(ctx, LOCOHD_PROF_SCORE); nl = launch_score_grad(g, ctx->kp, GradTarget::kEntries, ctx->stream); }
        if (nl < 0) st = fail(ctx, LOCOHD_ERR_UNSUPPORTED, "shared memory budget exceeded for %d categories", ctx->kp.C);
        else ctx->launches += nl;
        if (!st && cudaPeekAtLastError() != cudaSuccess)
            st = fail(ctx, LOCOHD_ERR_CUDA, "launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!st) st = out.commit();
    dev_free(ctx, d_scores);
    return st;
}

int locohd_from_rows_grad(locohd_ctx* ctx, uint64_t n_rows,
                          const uint64_t* row_offsets_a, const double* values_a, const uint16_t* category_a,
                          uint64_t n_categories_a,
                          const uint64_t* row_offsets_b, const double* values_b, const uint16_t* category_b,
                          uint64_t n_categories_b,
                          const uint32_t* wf_idx, const double* pair_weights,
                          double* out_scores, double* out_grad_a, double* out_grad_b) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    const uint64_t* offsets[2] = {row_offsets_a, row_offsets_b};
    const double* values[2] = {values_a, values_b};
    const uint16_t* cats[2] = {category_a, category_b};
    const uint64_t n_cats[2] = {n_categories_a, n_categories_b};
    double* grads[2] = {out_grad_a, out_grad_b};
    std::vector<uint64_t> in_off[2];
    uint64_t max_len[2];
    for (int s = 0; s < 2; ++s) {
        TRY_ST(ragged_rows_check(ctx, n_rows, offsets[s], values[s], cats[s], n_cats[s], in_off[s], &max_len[s]));
        if (in_off[s][n_rows] && !grads[s]) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null gradient array");
    }
    TRY_ST(check_wf_indices(ctx, wf_idx, n_rows));
    if (n_rows == 0) return 0;
    RowSets rs;
    InBuf<uint64_t> d_off[2];
    OutBuf<double> g[2];
    for (int s = 0; s < 2; ++s) {
        TRY_ST(rows_envset(ctx, n_rows, in_off[s].data(), max_len[s], values[s], nullptr, cats[s], &rs.e[s]));
        TRY_ST(d_off[s].load(ctx, in_off[s].data(), n_rows));
        TRY_ST(g[s].prepare(ctx, grads[s], in_off[s][n_rows]));
    }
    const uint64_t* entry_off[2] = {d_off[0].ptr, d_off[1].ptr};
    double* entry_grad[2] = {g[0].ptr, g[1].ptr};
    int st = rows_grad(ctx, rs, n_rows, wf_idx, pair_weights, out_scores, entry_off, entry_grad);
    if (!st) st = g[0].commit();
    if (!st) st = g[1].commit();
    const int st2 = sync_and_check(ctx);   // also keeps in_off alive until its copies are done
    return st ? st : st2;
    API_END()
}

int locohd_from_coords_grad(locohd_ctx* ctx, uint64_t n_points, const double* xyz_a, const uint16_t* cat_a,
                            const double* xyz_b, const uint16_t* cat_b, const uint32_t* wf_idx,
                            const double* pair_weights, double* out_scores, double* out_grad_a, double* out_grad_b) {
    API_BEGIN(ctx)
    TRY_ST(need_params(ctx));
    if (n_points && (!xyz_a || !xyz_b)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null coordinates");
    if (n_points && (!out_grad_a || !out_grad_b)) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null gradient array");
    TRY_ST(check_wf_indices(ctx, wf_idx, n_points));
    if (n_points == 0) return 0;
    const double* xyz[2] = {xyz_a, xyz_b};
    const uint16_t* cats[2] = {cat_a, cat_b};
    double* grads[2] = {out_grad_a, out_grad_b};
    RowSets rs;
    InBuf<double> x[2];
    OutBuf<double> g[2];
    double* G[2] = {nullptr, nullptr};   // dense [n][n] per side: entry (i, j) of row i at i n + j
    auto release = [&](int st) { dev_free(ctx, G[0]); dev_free(ctx, G[1]); return st; };
    int st = 0;
    for (int s = 0; s < 2 && !st; ++s) {
        st = rows_envset(ctx, n_points, nullptr, n_points, nullptr, xyz[s], cats[s], &rs.e[s]);
        if (!st) st = x[s].load(ctx, xyz[s], 3 * n_points);
        if (!st) st = g[s].prepare(ctx, grads[s], 3 * n_points);
        if (!st) st = dev_alloc(ctx, &G[s], n_points * n_points);
    }
    std::vector<uint64_t> row_off(n_points);
    for (uint64_t r = 0; r < n_points; ++r) row_off[r] = r * n_points;
    InBuf<uint64_t> d_off;
    if (!st) st = d_off.load(ctx, row_off.data(), n_points);
    if (!st) {
        const uint64_t* entry_off[2] = {d_off.ptr, d_off.ptr};
        st = rows_grad(ctx, rs, n_points, wf_idx, pair_weights, out_scores, entry_off, G);
    }
    if (!st) {
        ProfScope ps(ctx, LOCOHD_PROF_OTHER);
        for (int s = 0; s < 2; ++s) ctx->launches += launch_coords_chain(x[s].ptr, G[s], n_points, g[s].ptr, ctx->stream);
        if (cudaPeekAtLastError() != cudaSuccess)
            st = fail(ctx, LOCOHD_ERR_CUDA, "launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!st) st = g[0].commit();
    if (!st) st = g[1].commit();
    const int st2 = sync_and_check(ctx);   // also keeps row_off alive until its copy is done
    return release(st ? st : st2);
    API_END()
}

// ----------------------------------------------------------------------------------------------- leaf math
// W(x) (density = false) or w(x) = W'(x) at n points
static int wf_points(locohd_ctx* ctx, const locohd_weight_function* wf, uint64_t n, const double* x, double* out,
                     bool density) {
    if (!wf || (n && (!x || !out))) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "null argument");
    WfDev w;
    TRY_ST(make_wf(ctx, *wf, &w));
    WfDev* d_w = nullptr;
    TRY_ST(dev_alloc(ctx, &d_w, 1));
    if (cudaMemcpyAsync(d_w, &w, sizeof w, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
        dev_free(ctx, d_w);
        return fail(ctx, LOCOHD_ERR_CUDA, "upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    InBuf<double> in;
    OutBuf<double> o;
    int st = in.load(ctx, x, n);
    if (!st) st = o.prepare(ctx, out, n);
    if (!st) {
        ctx->launches += density ? launch_wf_density(d_w, n, in.ptr, o.ptr, ctx->d_err, ctx->stream)
                                 : launch_wf_points(d_w, n, in.ptr, o.ptr, ctx->d_err, ctx->stream);
        st = o.commit();
    }
    const int st2 = sync_and_check(ctx);
    dev_free(ctx, d_w);
    return st ? st : st2;
}

int locohd_wf_integral_points(locohd_ctx* ctx, const locohd_weight_function* wf, uint64_t n, const double* x,
                              double* out) {
    API_BEGIN(ctx)
    return wf_points(ctx, wf, n, x, out, false);
    API_END()
}

int locohd_wf_density_points(locohd_ctx* ctx, const locohd_weight_function* wf, uint64_t n, const double* x,
                             double* out) {
    API_BEGIN(ctx)
    return wf_points(ctx, wf, n, x, out, true);
    API_END()
}

int locohd_sd_run(locohd_ctx* ctx, int32_t sd_kind, const double* sd_params, int32_t n_categories, uint64_t n,
                  const double* p1, const double* p2, double* out) {
    API_BEGIN(ctx)
    if (sd_kind < LOCOHD_SD_HELLINGER || sd_kind > LOCOHD_SD_RENYI) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "Invalid statistical distance kind %d!", sd_kind);
    if (n_categories <= 0 || (n && (!p1 || !p2 || !out))) return fail(ctx, LOCOHD_ERR_BAD_PARAM, "bad argument");
    const double q0 = sd_params ? sd_params[0] : 0.0, q1 = sd_params ? sd_params[1] : 0.0;
    InBuf<double> a, b;
    OutBuf<double> o;
    TRY_ST(a.load(ctx, p1, n * n_categories));
    TRY_ST(b.load(ctx, p2, n * n_categories));
    TRY_ST(o.prepare(ctx, out, n));
    ctx->launches += launch_sd_run(sd_kind, q0, q1, n_categories, n, a.ptr, b.ptr, o.ptr, ctx->stream);
    TRY_ST(o.commit());
    return sync_and_check(ctx);
    API_END()
}

}  // extern "C"
