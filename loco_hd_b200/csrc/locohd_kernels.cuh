// locohd_kernels.cuh — internal interface between the C ABI (locohd_capi.cu) and the sm_100a kernels
// (locohd_kernels.cu).  Not installed; the public boundary is include/locohd_b200.h.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "locohd_math.cuh"

namespace locohd {

constexpr uint8_t kUnknownCat8 = 0xFF;
constexpr int kSqrtTableSize = 4096;
constexpr uint64_t kCatMask = 0xFFull;  // low byte of a packed key = category

// One primitive in cell-sorted order: exact coordinates for the FP64 membership test and distance.
struct __align__(32) PrimRec {
    double x, y, z;
    uint32_t tag;   // interned tag id
    uint32_t cat;   // category id (0..254) or kUnknownCat8
};

// Per-structure cell grid (built for one threshold).
struct __align__(16) StructMeta {
    double ox, oy, oz;   // grid origin = bounding-box minimum
    double inv_cell;     // 1 / cell edge along y and z (cell edge >= threshold / 2 * (1 + 1e-6))
    int nx, ny, nz;
    int reach;           // neighbour cells to visit on each side along y and z (at most 2)
    float thr2f;         // conservative squared radius for the FP32 prefilter
    float cellf;         // cell edge as f32 (0: a single cell, no row pruning)
    float prune_r;       // row pruning (fused gather): conservative radius in the f32 relative coordinates
    float inv_cellxf;    // 1 / x cell edge as f32
    double inv_cell_x;   // 1 / x cell edge: cells are up to 4 times finer along x (the fastest axis), which costs no
                         // extra rows and lets the gather cut every row close to the sphere
    int reach_x;         // neighbour cells along x
    int pad0;
    double r2_safe;      // fused gather: squared radius below which the kd-tree crate's per-axis box test cannot reject
                         // ((r - 8.9e-16 (max |coordinate| of the structure + r))^2 (1 - 1e-15); 0: always test)
};
static_assert(sizeof(StructMeta) == 96, "env_fused_kernel loads the record as six 16-byte words");

// Kernel-visible parameter block of one LoCoHD instance (LoCoHD struct, locohd.rs:42-55).
struct KParams {
    int C;
    int sd_kind;
    double sd_p0, sd_p1;
    int hell2;    // Hellinger with exponent exactly 2 -> sqrt-table fast path
    int unit_w;   // all category weights == 1
    int tpr_kind, tpr_accept_same, tpr_accepted_pairs, tpr_ordered;
    uint64_t n_tag_pairs;
    const uint64_t* tag_pairs;  // sorted
    const double* cat_w;        // [C]
    const double* cat_sw;       // [C] sqrt(w)
    const WfDev* wfs;
    int n_wf;
    const double* sqrt_tbl;     // sqrt(k), k < kSqrtTableSize
    const double* rsqrt_tbl;    // 1/sqrt(k)
    int* err;                   // device error word (first locohd_status raised by a kernel)
};

// cells of structure s live at cell_start[cell_base(s) ...]: at most max(2 N_s, 8) cells + 1 end marker
__host__ __device__ inline uint64_t cell_base(uint64_t prim_off_s, uint64_t s) { return 2 * prim_off_s + 9 * s; }
__host__ __device__ inline uint64_t cell_entries(uint64_t n_prims, uint64_t n_structs) { return 2 * n_prims + 9 * n_structs; }

struct StructsView {
    uint64_t n_structs;
    const uint64_t* prim_off;     // [n_structs + 1]
    const double* xyz;            // raw [n_prims][3]
    const uint8_t* cat;           // raw [n_prims]
    const uint32_t* tag;          // raw [n_prims]
    StructMeta* meta;             // [n_structs]
    float4* pf;                   // cell-sorted: (x - ox, y - oy, z - oz) as f32, w = tag bits
    PrimRec* pd;                  // cell-sorted exact records
    uint32_t* porig;              // cell-sorted position -> index inside the structure, original order (parity dumps)
    uint32_t* sorted_pos;         // original index -> cell-sorted position (inside the structure)
    uint32_t* cell_start;         // [cell_entries]: first cell-sorted position of every cell
    uint32_t* cell_fill;          // [cell_entries]: scratch cursor of the counting sort
};

// Sorted environments.  Member k of environment e is key[off[e] + k], k < count[e]; a key is the f64 bit pattern of
// W(distance) (key_is_w) or of the distance with the low mantissa byte replaced by the member's category.
struct EnvView {
    uint64_t n_env;
    const uint64_t* off;
    const uint32_t* count;
    const uint64_t* key;
    int key_is_w;
};

struct ScanStats {  // written by the scan kernels, read back by the host
    unsigned long long total;
    unsigned int max_value;
    unsigned int pad;
};

// fused gather (env_fused_kernel)
// warps per CTA (one anchor per warp at a time): one CTA per SM for the 512-member instantiation - the warps of a CTA
// work on consecutive anchors of the cell order and share their candidate rows in L1; measured 24.6 / 23.6 / 22.6 ms
// at 4 / 8 / 16 warps per CTA with the same 32 warps per SM
constexpr int kFusedWarps = 32;     // the 512-member instantiation, and the largest warps-per-CTA (store sizing)
__host__ __device__ constexpr int fused_warps(int cap, bool debug) { return cap == 512 ? (debug ? 16 : kFusedWarps) : 8; }  // debug: the parity arrays need more shared memory per warp
constexpr int kFusedCap = 512;      // members per environment (default instantiation)
constexpr int kFusedCapBig = 1024;  // second instantiation, used when the first reports larger environments
constexpr int kFusedChunk = 2048;   // store entries a warp reserves with one atomicAdd
constexpr int kScoreRun = 16;       // consecutive pairs a scoring warp claims with one atomicAdd
constexpr uint64_t kIdentityOrderMax = 2048;   // calls of up to this many anchors keep the caller's anchor order

struct FusedStats {  // written by env_fused_kernel, read back by the host
    unsigned long long cursor;     // store entries handed out (multiple of kFusedChunk)
    unsigned long long sample;     // sum of the sampled upper-bound sizes (env_tile_kernel<false> with a stride)
    unsigned int max_count;        // largest environment
    unsigned int overflow;         // != 0: bit 3 = an environment exceeded CAP, bit 0 = store exhausted, bit 1 = reach
};

struct EnvBuild {
    uint64_t n_env;
    const uint32_t* order;    // environments in cell order of their anchors
    const uint2* order_rec;   // (structure, cell-sorted position) of the anchor at every place of `order`
    const uint32_t* ub;       // FP32-prefilter upper bound of every environment size
    const uint64_t* off;      // exclusive scan of the (even-rounded) upper bounds
    uint64_t* off_out;        // fused gather: store offset of every environment (written by the kernel)
    uint32_t* count;          // exact sizes (written by the fill kernel)
    uint64_t* key;            // store: plain distances (f64 bits) until the sort kernel packs them
    uint8_t* cat;             // categories of the unsorted members (scratch)
    uint32_t* idx;            // primitive indices (debug/parity) or nullptr
    double* dist;             // sorted plain distances (debug/parity) or nullptr
    int key_is_w;
    int key_is_sq;            // unsorted keys are squared distances (gather) rather than distances (rows)
    int check_first_zero;     // rows mode: the smallest distance of a row must be 0 (locohd.rs:74-77)
};

// A tile of jobs that share environment runs: up to kTileDim runs of env-set A (rows) against up to kTileDim runs of
// env-set B (columns), every job of the tile with the same number of anchors.  An all-vs-all ensemble listed in
// 4 x 4 blocks (batch.py::blocked_pairs) is exactly a list of such tiles.  score_tile_kernel stages the <= 8
// environments of (tile, anchor) once and scores the <= 16 anchor pairs they form.
constexpr int kTileDim = 4;
constexpr uint64_t kTileNone = ~0ull;
struct __align__(16) ScoreTile {
    uint64_t a_first[kTileDim];                 // first environment of row r in env-set A (kTileNone: no such row)
    uint64_t b_first[kTileDim];                 // first environment of column c in env-set B
    uint64_t out_first[kTileDim * kTileDim];    // index of the first score of job (r, c) in `out` (kTileNone: no job)
};

// Order of the units (tile, anchor) of a tile launch.  Tile-major order (all anchors of a tile, then the next tile)
// re-reads an environment from DRAM for almost every tile it takes part in: the 8 structures of a tile hold 60 MB of
// environments on the 1000-structure ensemble, so only the row structures survive in L2 from one tile to the next
// (ncu: 459 B of DRAM reads per anchor pair, 29 x the algorithmic bytes of the step).  Sliced order: the anchors are
// cut into slices of `slice` consecutive anchors and ALL tiles are visited for one slice before the next slice
// starts; the environments of one slice of every structure (slice x 1.5 MB there) stay in L2 while the ~31 000
// tiles pass over them, and every environment comes from DRAM once per launch.
struct TileOrder {
    uint64_t slice;       // anchors per slice (= n: one slice, tile-major order)
    uint64_t per_slice;   // units of a full slice = n_tiles * slice
    uint64_t full;        // units in full slices
    uint64_t base_last;   // first anchor of the short last slice
    uint64_t last;        // its anchors (0: n is a multiple of slice)
};
__host__ __device__ inline TileOrder make_tile_order(uint64_t n_tiles, uint64_t n, uint64_t slice) {
    TileOrder o;
    if (slice == 0 || slice > n) slice = n;
    o.slice = slice;
    o.per_slice = n_tiles * slice;
    o.full = slice ? (n / slice) * o.per_slice : 0;
    o.base_last = slice ? (n / slice) * slice : 0;
    o.last = n - o.base_last;
    return o;
}
template <class T>
__host__ __device__ inline void tile_unit(const TileOrder& o, T u, T* tile, T* p) {
    if (u < (T)o.full) {
        const T s = u / (T)o.per_slice, r = u - s * (T)o.per_slice;
        const T t = r / (T)o.slice;
        *tile = t;
        *p = s * (T)o.slice + (r - t * (T)o.slice);
    } else {
        const T r = u - (T)o.full;
        const T t = r / (T)o.last;
        *tile = t;
        *p = (T)o.base_last + (r - t * (T)o.last);
    }
}

struct ScoreArgs {
    const ScoreTile* tiles;        // tile mode (score_tile_kernel): jobs grouped by the host, uniform_n anchors each
    uint64_t n_tiles;
    EnvView a, b;
    uint64_t n_pairs;
    const uint32_t* pairs;         // explicit mode: [n_pairs][2]; nullptr -> job mode
    const locohd_job* jobs;        // job mode
    const uint64_t* job_pair_off;  // [n_jobs + 1]
    uint64_t n_jobs;
    uint64_t uniform_n;            // > 0: every job has this many pairs
    const uint32_t* wf_idx;        // per pair or nullptr
    double* out;
    int stage_cap;                 // members (A + B) a warp can stage in shared memory
    int only_unstaged;             // second pass: score only the pairs the fast kernel skipped
    int table_n;                   // sqrt / rsqrt table entries staged by the fast kernel
    int rep_n;                     // tile kernel: head entries of the count-indexed tables replicated per bank pair
    TileOrder order;               // tile kernel: unit -> (tile, anchor), slice by slice (read from the parameter bank)
    unsigned long long* cursor;    // fast kernel: next unclaimed pair (zeroed before the launch); warps claim runs of
                                   // `run` consecutive pairs, so all resident warps work at one moving frontier
    unsigned run;                  // pairs per claim: kScoreRun for large launches, fewer when the launch has fewer
                                   // pairs than 4 runs per resident warp (single structure pairs: latency)
};

// ---- launchers (all asynchronous on `st`; each returns the number of kernel launches it made) ----
int launch_convert_categories(const uint16_t* in, uint8_t* out, uint64_t n, int C, cudaStream_t st);
int launch_validate_xyz(const double* xyz, uint64_t n3, int* err, cudaStream_t st);
// max_prims: size of the largest structure (selects the shared-memory variant of the counting sort)
int launch_build_cells(const StructsView& s, double threshold, uint64_t max_prims, cudaStream_t st);
// anchors -> cell order: slot_cnt / slot_off are scratch of n_prims (+1) entries
int launch_anchor_order(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* anchor_struct,
                        const uint32_t* anchor_prim, uint64_t n_prims, uint32_t* slot_cnt, uint64_t* slot_off,
                        uint64_t* scan_scratch, ScanStats* stats, uint32_t* order, uint2* order_rec, cudaStream_t st);
uint64_t scan_scratch_entries(uint64_t n);
// exclusive scan of u32 values (optionally rounded up to even) into u64 offsets [n + 1]; stats->total / max_value
int launch_scan(const uint32_t* values, uint64_t n, int round_even, uint64_t* off, uint64_t* scratch, ScanStats* stats,
                cudaStream_t st);
int launch_env_count(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* order,
                     const uint32_t* anchor_struct, const uint32_t* anchor_prim, double threshold, uint32_t* ub,
                     cudaStream_t st);
// sum of the upper-bound sizes of every stride-th anchor (in cell order) -> *sum
int launch_env_sample(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* order,
                      const uint32_t* anchor_struct, const uint32_t* anchor_prim, double threshold, uint32_t stride,
                      unsigned long long* sum, cudaStream_t st);
// fused gather + sort + pack: grid from fused_grid(); the store needs room for the members plus one kFusedChunk per
// warp of the grid
// host_wf: host copy of weight function 0 (selects the CDF specialisation)
unsigned fused_grid(const KParams& p, const WfDev* host_wf, int key_is_w, bool debug, int cap, uint64_t n_env);
int launch_env_fused(const StructsView& s, const KParams& p, const WfDev* host_wf, const uint32_t* anchor_struct,
                     const uint32_t* anchor_prim, double threshold, const EnvBuild& b, int cap, FusedStats* stats,
                     uint64_t capacity, unsigned grid, cudaStream_t st);
int launch_env_fill(const StructsView& s, const KParams& p, const uint32_t* anchor_struct, const uint32_t* anchor_prim,
                    double threshold, const EnvBuild& b, cudaStream_t st);
// sorts every environment of the store in place and packs the keys; max_count bounds the environment sizes
int launch_env_sort(const KParams& p, const EnvBuild& b, unsigned max_count, double threshold, cudaStream_t st);
// rows into the store, unsorted: values (or the distances among the row_len points xyz) of rows of row_len entries,
// or, with in_off / out_off, of ragged rows (row_len: the longest row) at those offsets of the input and the store
int launch_rows_copy(const double* values, const double* xyz, const uint8_t* cat, uint64_t n_rows, uint64_t row_len,
                     const uint64_t* in_off, const uint64_t* out_off, uint64_t* off, uint32_t* count, const EnvBuild& b,
                     cudaStream_t st);
// Test and A/B hooks that override launch decisions of the library, read from the process environment by
// read_launch_overrides() once per API call, so that a process can change them between calls.  The defaults leave
// every decision to the library.  No other code of the library reads the environment.
struct LaunchOverrides {
    bool no_tiles = false;        // LOCOHD_NO_TILES (non-zero integer): job lists never take score_tile_kernel
    int tile_teams = 0;           // LOCOHD_TILE_TEAMS: lowers TileGeometry::teams when in [1, teams)
    int tile_rep = -1;            // LOCOHD_TILE_REP: lowers TileGeometry::rep_n when in [0, rep_n)
    unsigned tile_run = 0;        // LOCOHD_TILE_RUN (1 ... 4096): longest run of units a team claims (0: kTileRun)
    long long tile_slice = -1;    // LOCOHD_TILE_SLICE: anchors per slice of a tile launch, 0 = tile-major order (a
                                  // value <= 0); -1: not set, the slice follows from the L2 budget
    double tile_slice_mb = 0.0;   // LOCOHD_TILE_SLICE_MB (> 0): that L2 budget in MB (0: the default)
    bool legacy_gather = false;   // LOCOHD_LEGACY_GATHER (any value not starting with '0'): environments are built
                                  // with the multi-kernel gather
};
LaunchOverrides read_launch_overrides();
int launch_score(const ScoreArgs& args, const KParams& p, unsigned max_a, unsigned max_b, double mean_a, double mean_b,
                 const LaunchOverrides& ov, cudaStream_t st);
// Launch geometry of score_tile_kernel for environments of at most max_a / max_b members (teams = 0: the kernel does
// not apply; below 6 teams the pair kernel is the better one and job lists are not tiled).  The one place that decides
// it: launch_tiles, the tile eligibility of locohd_score_jobs_stats and locohd_tile_geometry read it.
struct TileGeometry {
    int teams;        // teams of four warps per CTA (LaunchOverrides::tile_teams lowers it)
    int cp;           // count rows per warp: 8 (C <= 8) or 16 (C <= 16), the instantiation score_tile_kernel<cp, ...>
    int rep_n;        // replicated head of the count-indexed tables, 0 = unreplicated (always 0 for cp 16;
                      // LaunchOverrides::tile_rep lowers it)
    int table_n;      // entries of each table
    int stage_keys;   // keys a team stages per unit
    int team_bytes;   // shared memory per team
};
TileGeometry tile_geometry(const KParams& p, unsigned max_a, unsigned max_b, int key_is_w, const LaunchOverrides& ov);
// One side of the pairs of a gradient call: environment `first` + p of `env` is that side of pair p.  The set was built
// with keep_indices or from rows, so `dist` / `idx` hold the exact distances and the members' indices (inside their
// structure, or the column inside their row).
struct GradSide {
    EnvView env;
    const double* dist;
    const uint32_t* idx;
    uint64_t first;
};
// Gradients of the scores of n_pairs pairs (score_grad_kernel).  Where each event's dS/dt goes is the kernel's
// GradTarget: the coordinates of a from_primitives call (one set passed as both sides, side[s].first = {0, n_pairs};
// the kernel reads that set through side[0]) or the entries of two row sets (from_dmxs / from_coords,
// side[s].first = 0).
struct GradArgs {
    GradSide side[2];
    uint64_t n_pairs;
    const uint32_t* wf_idx;         // per pair or nullptr
    const double* pair_weights;     // upstream gradient g_p per pair or nullptr (all 1)
    double* out;                    // [n_pairs] scores
    // GradTarget::kCoords
    const double* xyz;              // raw [n_prims][3] of the structure set
    const uint64_t* prim_off;       // [n_structs + 1]
    uint64_t n_structs;
    const uint32_t* anchor_struct;  // [2 n_pairs]
    const uint32_t* anchor_prim;    // [2 n_pairs]
    double* grad[2];                // [n_prims of structure s][3], zeroed by the caller: sum_p g_p dS_p / dxyz
    // GradTarget::kEntries: g_p dS_p / dt of entry (row p, column c) of side s at entry_grad[s][entry_off[s][p] + c];
    // every entry of every row is written (0 for the anchor, t = 0 and non-finite t)
    const uint64_t* entry_off[2];   // [n_pairs]
    double* entry_grad[2];
};
enum class GradTarget { kCoords, kEntries };
// returns the number of launches, or -1 when the per-warp state of C categories does not fit shared memory
int launch_score_grad(const GradArgs& g, const KParams& p, GradTarget target, cudaStream_t st);
// grad[i] = sum_j (G[i][j] + G[j][i]) (x_i - x_j) / t_ij over the n points xyz, G dense [n][n] (from_coords_grad)
int launch_coords_chain(const double* xyz, const double* G, uint64_t n, double* grad, cudaStream_t st);
int launch_wf_density(const WfDev* wf, uint64_t n, const double* x, double* out, int* err, cudaStream_t st);
int launch_job_means(const double* scores, const uint64_t* job_pair_off, uint64_t n_jobs, double* means,
                     cudaStream_t st);
int launch_widen_xyz(const float* in, double* out, uint64_t n3, cudaStream_t st);
// centroids of n_frames frames of one topology (f32 sequential mean per primitive) -> f64 coordinates
int launch_centroids(const float* atoms, uint64_t n_atoms, uint64_t n_frames, const uint32_t* seg_start,
                     const uint32_t* atom_index, uint64_t n_prims, double* xyz_out, int* err, cudaStream_t st);
int launch_validate_wf_idx(const uint32_t* wf_idx, uint64_t n, uint32_t n_wf, int* err, cudaStream_t st);
// per-anchor mean / population std over n_jobs uniform jobs of n anchors; scratch: two arrays of n doubles
int launch_anchor_stats(const double* scores, uint64_t n, uint64_t n_jobs, double* sum_scratch, double* m2_scratch,
                        double* mean_out, double* std_out, cudaStream_t st);
int launch_anchor_lists(const KParams& p, const uint8_t* seq_a, uint64_t len_a, const double* da, const uint8_t* seq_b,
                        uint64_t len_b, const double* db, uint32_t wf_idx, double* out, cudaStream_t st);
int launch_wf_points(const WfDev* wf, uint64_t n, const double* x, double* out, int* err, cudaStream_t st);
int launch_sd_run(int kind, double q0, double q1, int C, uint64_t n, const double* p1, const double* p2, double* out,
                  cudaStream_t st);
int launch_fp64_peak(double* scratch, int blocks, int iters, cudaStream_t st);

}  // namespace locohd
