/* ============================================================================
 * locohd_b200.h — C ABI of the B200-native LoCoHD per-anchor scoring path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no Python / torch
 * types.  The entry points are what a host binding for the reference's hot path
 * would bind (the rayon loop and kd-tree of /root/reference/src/locohd.rs are
 * replaced; its `#[pymethods]` keep their Python signatures in the host layer,
 * see INTEGRATION.md).  Each function cites the reference interface it serves.
 *
 * Conventions
 *  - Every function returns a locohd_status (0 = ok).  After a failure
 *    `locohd_last_error(ctx)` holds a message (ctx may be NULL for failures of
 *    `locohd_ctx_create`).
 *  - Array arguments may live in host memory OR in device memory of the
 *    context's GPU (unified virtual addressing decides); host arrays are only
 *    borrowed for the duration of the call.  Output arrays likewise.
 *  - Categories (primitive types) and tags are interned by the caller:
 *    category id in [0, n_categories), LOCOHD_UNKNOWN_CATEGORY for a name the
 *    LoCoHD instance does not know (pmf.rs:34-45 makes that an error only when
 *    such a primitive is met inside an environment); tags are arbitrary u32 ids
 *    shared by both structures and by the tag-pair table.
 *  - There is no CPU fallback: without a CUDA device every call fails.
 * ==========================================================================*/
#ifndef LOCOHD_B200_H
#define LOCOHD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LOCOHD_ABI_VERSION 2
#define LOCOHD_UNKNOWN_CATEGORY 0xFFFFu
#define LOCOHD_MAX_CATEGORIES 255

typedef enum locohd_status {
    LOCOHD_OK = 0,
    LOCOHD_ERR_LEN_MISMATCH = 1,     /* locohd.rs:70-73 */
    LOCOHD_ERR_FIRST_NOT_ZERO = 2,   /* locohd.rs:74-77 */
    LOCOHD_ERR_UNKNOWN_CATEGORY = 3, /* pmf.rs:38-42 */
    LOCOHD_ERR_ZERO_NORM = 4,        /* pmf.rs:70-76 */
    LOCOHD_ERR_NEGATIVE_POINT = 5,   /* weight_function.rs:97-100 */
    LOCOHD_ERR_NAN = 6,              /* reference panics: partial_cmp().unwrap(), utils.rs:28 */
    LOCOHD_ERR_EMPTY_ENV = 7,        /* reference panics: dists_a[0] on an empty Vec, locohd.rs:74 */
    LOCOHD_ERR_INDEX = 8,            /* reference panics: prim_seq[anchor_idx], locohd.rs:521 */
    LOCOHD_ERR_DMX_SHAPE = 9,        /* locohd.rs:420-428 */
    LOCOHD_ERR_BAD_PARAM = 10,       /* constructor-level validation (locohd.rs:305-346, weight_function.rs:24-89, ...) */
    LOCOHD_ERR_CUDA = 100,           /* CUDA runtime failure; message holds cudaGetErrorString */
    LOCOHD_ERR_NO_DEVICE = 101,
    LOCOHD_ERR_UNSUPPORTED = 102
} locohd_status;

typedef enum locohd_wf_kind {    /* weight_function.rs:29-90 */
    LOCOHD_WF_HYPER_EXP = 0,     /* cdfs.rs:5-21   params a_1..a_n, b_1..b_n */
    LOCOHD_WF_DAGUM = 1,         /* cdfs.rs:27-29  params a, b, p */
    LOCOHD_WF_UNIFORM = 2,       /* cdfs.rs:39-45  params x_min, x_max */
    LOCOHD_WF_KUMARASWAMY = 3    /* cdfs.rs:56-63  params x_min, x_max, a, b */
} locohd_wf_kind;

typedef enum locohd_sd_kind {    /* pmf/statistical_distances.rs:80-86 */
    LOCOHD_SD_HELLINGER = 0,     /* params: exponent */
    LOCOHD_SD_KOLMOGOROV_SMIRNOV = 1,
    LOCOHD_SD_KULLBACK_LEIBLER = 2, /* params: epsilon */
    LOCOHD_SD_RENYI = 3          /* params: alpha, epsilon */
} locohd_sd_kind;

typedef enum locohd_tpr_kind {   /* tag_pairing_rule.rs:5-21 */
    LOCOHD_TPR_WITHOUT_LIST = 0, /* accept_same */
    LOCOHD_TPR_WITH_LIST = 1     /* tag_pairs, accepted_pairs, ordered */
} locohd_tpr_kind;

#define LOCOHD_MAX_WF_PARAMS 16

typedef struct locohd_weight_function {
    int32_t kind;                          /* locohd_wf_kind */
    int32_t n_params;                      /* <= LOCOHD_MAX_WF_PARAMS */
    double params[LOCOHD_MAX_WF_PARAMS];
} locohd_weight_function;

/* State of one LoCoHD instance (locohd.rs:42-55), already validated/defaulted by the host
 * (LoCoHD::build, locohd.rs:289-389).  Validation is repeated here and reported as
 * LOCOHD_ERR_BAD_PARAM. */
typedef struct locohd_params {
    int32_t n_categories;                  /* 1 .. LOCOHD_MAX_CATEGORIES */
    const double* category_weights;        /* [n_categories], all > 0 */
    int32_t sd_kind;                       /* locohd_sd_kind */
    double sd_params[2];
    int32_t n_weight_functions;            /* >= 1; index 0 is the default for wf_idx == NULL */
    const locohd_weight_function* weight_functions;
    int32_t tpr_kind;                      /* locohd_tpr_kind */
    int32_t tpr_accept_same;               /* WITHOUT_LIST */
    int32_t tpr_accepted_pairs;            /* WITH_LIST */
    int32_t tpr_ordered;                   /* WITH_LIST */
    uint64_t n_tag_pairs;                  /* WITH_LIST */
    const uint64_t* tag_pairs;             /* (anchor_tag << 32) | neighbour_tag, any order */
} locohd_params;

typedef enum locohd_prof_group {
    LOCOHD_PROF_CELLS = 0,   /* K0 build_cells_kernel */
    LOCOHD_PROF_COUNT = 1,   /* K1a env_tile_kernel<false>: upper-bound sizes (fused gather: of a 1/16 sample, only
                                for calls above 32 768 anchors without a remembered store size) */
    LOCOHD_PROF_SCAN = 2,    /* scan of the environment sizes (multi-kernel fallback only) */
    LOCOHD_PROF_FILL = 3,    /* K1 env_fused_kernel, once per attempt: gather + sort + packing (fallback: K1b
                                env_tile_kernel<true>) */
    LOCOHD_PROF_SCORE = 4,   /* K2 score_fast_kernel / score_kernel */
    LOCOHD_PROF_OTHER = 5,   /* anchor ordering, conversions, validation, means, row copies, ... */
    LOCOHD_PROF_SORT = 6,    /* K1c env_sort_kernel (multi-kernel fallback only): per-environment sort, CDF, packing */
    LOCOHD_PROF_GROUPS = 7
} locohd_prof_group;

typedef struct locohd_ctx locohd_ctx;            /* one GPU + one stream + one LoCoHD parameter set */
typedef struct locohd_structs locohd_structs;    /* device-resident set of primitive structures */
typedef struct locohd_envset locohd_envset;      /* device-resident sorted environments of a list of anchors */
typedef struct locohd_graph locohd_graph;        /* device-resident sparse result: pairs whose score is within a bound */

/* A run of anchor pairs with identity pairing: pair p (0 <= p < n) scores environment
 * (a_first + p) of env-set A against environment (b_first + p) of env-set B. */
typedef struct locohd_job {
    uint64_t a_first;
    uint64_t b_first;
    uint64_t n;
} locohd_job;

/* ---- context ------------------------------------------------------------------------- */
int locohd_abi_version(void);
int locohd_device_count(void);
/* Replaces the rayon pool of LoCoHD::build (locohd.rs:372-383): one context = one GPU. */
int locohd_ctx_create(int device, locohd_ctx** out);
void locohd_ctx_destroy(locohd_ctx* ctx);
const char* locohd_last_error(const locohd_ctx* ctx);
/* LoCoHD::build state (locohd.rs:289-389). May be called again to change parameters. */
int locohd_ctx_set_params(locohd_ctx* ctx, const locohd_params* params);
/* The cudaStream_t all work of this context is enqueued on (for CUDA-event timing). */
void* locohd_ctx_stream(locohd_ctx* ctx);
/* Wait for the stream and surface any device-side error (unknown category, bad index, ...). */
int locohd_ctx_synchronize(locohd_ctx* ctx);
/* Kernel launches issued by this context since creation (benchmark accounting). */
uint64_t locohd_ctx_launch_count(const locohd_ctx* ctx);
/* How many of them were the tile scoring kernel (locohd_score_jobs[_stats] on job lists whose jobs share runs of
 * environments, e.g. the all-vs-all ensemble of compare_ensembles.py:250-296 listed in 4 x 4 blocks). */
uint64_t locohd_ctx_tile_launches(const locohd_ctx* ctx);
/* How many of those were the wide form, one CTA per 32 x 32 tile of jobs and one lane per anchor pair: taken when
 * the list fills such tiles to at least 80 % and their stage fits shared memory, unless LOCOHD_WIDE_TILES=0 is set in
 * the environment (the 4 x 4 tiles then score the list). */
uint64_t locohd_ctx_wide_launches(const locohd_ctx* ctx);
/* Per-kernel timing with CUDA events on the context stream (benchmark roofline accounting).  While enabled every
 * kernel group is bracketed by a pair of events; locohd_ctx_profile_read waits for the stream, adds the elapsed
 * times per group to ms[k] / launches[k] (k < LOCOHD_PROF_GROUPS, see locohd_prof_group) and clears the records. */
int locohd_ctx_profile_enable(locohd_ctx* ctx, int on);
int locohd_ctx_profile_read(locohd_ctx* ctx, double* ms, uint64_t* launches);
/* Sustained FP64 FMA rate of the device (TFLOP/s, 2 flops per FMA) from a register-resident FMA kernel:
 * the denominator of the FP64 roofline (MEASURED_PEAKS.json has no FP64 entry). */
int locohd_measure_fp64_tflops(locohd_ctx* ctx, double* out_tflops);
/* Pinned host memory for callers that want asynchronous copies. */
int locohd_host_alloc(uint64_t bytes, void** out);
void locohd_host_free(void* p);

/* ---- structures (Vec<PrimitiveAtom>, locohd.rs:480-481; primitive_atom.rs:4-16) ------- */
/* n_structs structures concatenated: structure s owns primitives [prim_offsets[s], prim_offsets[s+1]).
 * xyz is [n_prims][3] f64, category [n_prims] u16, tag [n_prims] u32.  Coordinates must be finite. */
int locohd_structs_create(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* prim_offsets, const double* xyz,
                          const uint16_t* category, const uint32_t* tag, locohd_structs** out);
/* Same with f32 coordinates on the wire (half the upload): Bio.PDB and MDAnalysis positions are float32 and the
 * centroids of atom_converter_utils.py:117,126 stay float32, so for such callers the f32 -> f64 widening done on the
 * device is exact and the results are identical to passing the widened values to locohd_structs_create. */
int locohd_structs_create_f32(locohd_ctx* ctx, uint64_t n_structs, const uint64_t* prim_offsets, const float* xyz,
                              const uint16_t* category, const uint32_t* tag, locohd_structs** out);
void locohd_structs_destroy(locohd_structs* s);
/* Replace the coordinates of an existing set in place (trajectory frames: same topology). */
int locohd_structs_update_xyz(locohd_structs* s, const double* xyz);
int locohd_structs_update_xyz_f32(locohd_structs* s, const float* xyz);
/* Primitive assignment for a compiled topology on the device (PrimitiveAssigner.assign_primitive_structure,
 * loco_hd/atom_converter_utils.py:92-131, re-run per frame by trajectory_analyzer.py:34-74,112): structures
 * [first_struct, first_struct + n_frames) get new coordinates, primitive p of frame f = the f32 mean (sequential sum
 * in the given order, then one f32 division - what np.mean(atom_coords, axis=0) computes) of the atoms
 * atom_index[segment_start[p] .. segment_start[p + 1]) of atom_xyz[f] ([n_frames][n_atoms][3] f32).  Every updated
 * structure must have n_prims primitives; categories and tags stay as created. */
int locohd_structs_update_from_atoms(locohd_structs* s, uint64_t first_struct, uint64_t n_frames, uint64_t n_atoms,
                                     const float* atom_xyz, uint64_t n_prims, const uint32_t* segment_start,
                                     const uint32_t* atom_index, uint64_t n_atom_refs);
/* Forget the cached cell lists so that the next locohd_envset_build rebuilds them (the reference rebuilds its
 * kd-trees on every from_primitives call, locohd.rs:504-510; benchmarks use this to time that step too). */
void locohd_structs_drop_cells(locohd_structs* s);

/* ---- environments (kd-tree build + env_from_idx, locohd.rs:504-542) -------------------- */
/* For anchor e: structure anchor_struct[e] (NULL = structure 0), primitive anchor_prim[e] (index inside
 * that structure).  Builds the cell list for `threshold` if needed, gathers every primitive with
 * box test and d^2 < r^2 (strict) that is the anchor itself or passes the tag rule, and sorts each
 * environment by distance.  keep_indices != 0 also keeps the primitive index of every member
 * (needed by locohd_envset_dump only). */
int locohd_envset_build(locohd_ctx* ctx, locohd_structs* s, uint64_t n_anchors, const uint32_t* anchor_struct,
                        const uint32_t* anchor_prim, double threshold, int keep_indices, locohd_envset** out);
/* Environments given directly as distance rows (from_dmxs, locohd.rs:410-446: every row is an anchor, the
 * environment is the whole row, no cutoff, no tag rule): dmx is row-major [n_rows][row_len], category
 * [row_len] is shared by all rows.  Rows are sorted on the device (utils.rs:25-39). */
int locohd_envset_from_rows(locohd_ctx* ctx, uint64_t n_rows, uint64_t row_len, const double* dmx,
                            const uint16_t* category, locohd_envset** out);
/* The same for rows of different lengths (the reference takes Vec<Vec<f64>>: row r is co-sorted with the first len_r
 * entries of the category sequence, utils.rs:25-39): row r = values[row_offsets[r] .. row_offsets[r + 1]); category
 * holds n_categories_given entries and every row must be at most that long (the reference panics otherwise). */
int locohd_envset_from_ragged_rows(locohd_ctx* ctx, uint64_t n_rows, const uint64_t* row_offsets, const double* values,
                                   const uint16_t* category, uint64_t n_categories_given, locohd_envset** out);
/* from_coords (locohd.rs:463-476 + utils.rs:10-22): rows are Euclidean distances of every point to every point. */
int locohd_envset_from_coords(locohd_ctx* ctx, uint64_t n_points, const double* xyz, const uint16_t* category,
                              locohd_envset** out);
void locohd_envset_destroy(locohd_envset* e);
uint64_t locohd_envset_size(const locohd_envset* e);         /* number of environments */
uint64_t locohd_envset_total_members(const locohd_envset* e);/* sum of environment sizes */
/* Debug / parity: copy out offsets [n+1], and (any may be NULL) distances, categories, primitive indices
 * of all members in sorted order (arrays of locohd_envset_total_members entries). */
int locohd_envset_dump(locohd_ctx* ctx, const locohd_envset* e, uint64_t* offsets, double* distances,
                       uint16_t* categories, uint32_t* prim_indices);

/* ---- scoring (stat_dist_integral, locohd.rs:61-226) ------------------------------------ */
/* Explicit pairs: pairs is [n_pairs][2] (environment index in A, environment index in B).
 * wf_idx (NULL = weight function 0 for all) selects the weight function per pair
 * (keys_to_weight_functions, locohd.rs:230-283).  out_scores [n_pairs] f64. */
int locohd_score_pairs(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_pairs,
                       const uint32_t* pairs, const uint32_t* wf_idx, double* out_scores);
/* Runs of identity-paired environments (structure-pair / frame batches).  Scores are written job after
 * job (sum of jobs[j].n entries).  If out_job_means != NULL the per-job mean score is written there too. */
int locohd_score_jobs(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_jobs,
                      const locohd_job* jobs, const uint32_t* wf_idx, double* out_scores, double* out_job_means);
/* locohd_score_jobs plus the reductions the reference's callers compute from the scores next (all optional, NULL =
 * not wanted; the per-anchor ones need jobs of one common size n and give n values):
 *   out_job_means     mean over the anchors of every job        np.mean(lchd_scores), casp14_extend_with_locohd.py:88,
 *                                                               lchd_dmx entries, compare_ensembles.py:293
 *   out_anchor_means  mean of anchor p over the jobs            np.mean(lchd_by_atom, axis=0), compare_ensembles.py:299
 *   out_anchor_stds   population std of anchor p over the jobs  np.std(all_points[1:], axis=0), trajectory_analyzer.py:310
 * With out_scores == NULL the per-anchor scores never leave the device. */
int locohd_score_jobs_stats(locohd_ctx* ctx, const locohd_envset* a, const locohd_envset* b, uint64_t n_jobs,
                            const locohd_job* jobs, const uint32_t* wf_idx, double* out_scores, double* out_job_means,
                            double* out_anchor_means, double* out_anchor_stds);
/* Every environment of a range of A against every environment of a range of B (an extension: the reference scores
 * listed pairs only; kras_scan.py:47-52 lists one anchor against every anchor, clustering and nearest-site searches
 * need the whole matrix).  Row i = environment a_first + i of A (i < n_a), column j = environment b_first + j of B
 * (j < n_b), all with weight function wf_idx: M[i][j] is the score locohd_score_pairs gives for the pair
 * (a_first + i, b_first + j).
 *   out_scores      [n_a][n_b] M, row-major, or NULL.
 *   k               0: no k-nearest output; 1 .. 32: per row the k smallest M[i][j] in ascending order - equal scores
 *                   by smaller j, NaN after +inf (a deterministic function of M) - into out_knn_scores [n_a][k] and
 *                   out_knn_index [n_a][k] (u32 column j, relative to b_first); either may be NULL, not both.
 *   skip_self       leaves out the column of the row's own environment (a_first + i == b_first + j); needs a == b.
 * Rows are scored in chunks of whole rows whose scores fit a fixed scratch budget (256 MB; LOCOHD_CROSS_ROWS in the
 * environment lowers the rows per chunk), so with out_scores == NULL the matrix never leaves the device and device
 * memory stays bounded whatever n_a is.  The tile kernel scores the matrix when locohd_score_jobs_stats would tile a
 * job list of these sets (one weight function, Hellinger-2, unit category weights, at most 16 categories, >= 6 teams
 * at the sets' largest environments, LOCOHD_NO_TILES unset; counted by locohd_ctx_tile_launches); otherwise the pair
 * kernel scores explicit pairs.  Errors: a range outside its set LOCOHD_ERR_INDEX; no output, k out of range (above
 * 32, above the columns a row has left, 0 with a k-nearest output or non-zero without one), skip_self with two sets
 * LOCOHD_ERR_BAD_PARAM; a bad wf_idx as in locohd_score_pairs; unknown categories and empty environments as in
 * locohd_score_jobs.  Outputs may be host or device memory. */
int locohd_score_cross(locohd_ctx* ctx, const locohd_envset* a, uint64_t a_first, uint64_t n_a, const locohd_envset* b,
                       uint64_t b_first, uint64_t n_b, uint32_t wf_idx, int skip_self, double* out_scores, uint32_t k,
                       double* out_knn_scores, uint32_t* out_knn_index);
/* Every unordered pair of one range once (an extension, for clustering within one env-set: scipy.cluster.hierarchy
 * .linkage and scipy.spatial.distance.squareform take this vector).  For 0 <= i < j < n, out_scores[n i - i (i + 1) / 2
 * + (j - i - 1)] is the score locohd_score_pairs gives for the pair (first + i, first + j) with weight function
 * wf_idx: scipy's pdist order, n (n - 1) / 2 entries.  Each entry is bit-identical to M[i][j] of
 * locohd_score_cross(s, first, n, s, first, n, ...), which scores both triangles: this call scores one, half the work
 * and half the output.  Only symmetric statistical distances are accepted (Hellinger with any exponent,
 * Kolmogorov-Smirnov); Kullback-Leibler and Renyi give LOCOHD_ERR_BAD_PARAM - use locohd_score_cross for them.
 * Route as in locohd_score_cross (the tile kernel, counted by locohd_ctx_tile_launches, or explicit pairs on the pair
 * kernel).  Rows are scored in chunks of whole blocks of 4 rows whose scores fit the 256 MB scratch (a device output
 * takes the whole triangle in one launch of the tile kernel; LOCOHD_CROSS_ROWS in the environment lowers the rows per
 * chunk); a chunk is one contiguous slice of out_scores, host or device memory.  Errors: a range outside the set
 * LOCOHD_ERR_INDEX; an asymmetric distance, out_scores NULL with n >= 2, a bad wf_idx LOCOHD_ERR_BAD_PARAM; unknown
 * categories and empty environments as in locohd_score_jobs.  n < 2 writes nothing. */
int locohd_score_condensed(locohd_ctx* ctx, const locohd_envset* s, uint64_t first, uint64_t n, uint32_t wf_idx,
                           double* out_scores);
/* Threshold graphs (an extension, for density clustering, connected components of similar sites and near-duplicate
 * counts without the dense matrix): every pair whose score s satisfies s <= max_score, as a CSR graph that stays on
 * the device until locohd_graph_copy.  NaN scores are never in the graph, +inf is when max_score is +inf, a NaN
 * max_score is LOCOHD_ERR_BAD_PARAM.  Rows ascend, columns ascend within a row, and every stored score is
 * bit-identical to the same entry of locohd_score_cross (locohd_score_within) or locohd_score_condensed
 * (locohd_score_within_condensed) on the same range and route; the result is the same on every call.
 * locohd_score_within: rows = n_a, row i holds the columns j (u32, relative to b_first) with M[i][j] <= max_score, M
 * the matrix of locohd_score_cross; range, skip_self, wf_idx checks, route and chunks as there (LOCOHD_CROSS_ROWS
 * lowers the rows per chunk).  locohd_score_within_condensed: rows = cols = n, row i holds only the columns j > i (the
 * upper triangle) of the range against itself; symmetric distances only, as locohd_score_condensed.  Both score in
 * chunks of the 256 MB scratch and read back one count per chunk; the graph storage grows geometrically and ends at
 * 8 (rows + 1) + 12 nnz bytes.  Empty ranges give an empty graph of `rows` rows.  On any error *out is NULL; a failed
 * allocation of the graph storage is LOCOHD_ERR_CUDA with the entries reached in the message.  The graph keeps its
 * context's device memory until locohd_graph_destroy, which must come before locohd_ctx_destroy. */
int locohd_score_within(locohd_ctx* ctx, const locohd_envset* a, uint64_t a_first, uint64_t n_a, const locohd_envset* b,
                        uint64_t b_first, uint64_t n_b, uint32_t wf_idx, int skip_self, double max_score,
                        locohd_graph** out);
int locohd_score_within_condensed(locohd_ctx* ctx, const locohd_envset* s, uint64_t first, uint64_t n, uint32_t wf_idx,
                                  double max_score, locohd_graph** out);
/* rows, cols and stored entries of a graph (any output may be NULL) */
int locohd_graph_shape(const locohd_graph* g, uint64_t* rows, uint64_t* cols, uint64_t* nnz);
/* Copies indptr [rows + 1] (u64), indices [nnz] (u32) and scores [nnz] (f64) out of the graph: any may be NULL, each
 * host or device memory; scipy.sparse.csr_matrix((scores, indices, indptr), shape=(rows, cols)) takes them. */
int locohd_graph_copy(locohd_ctx* ctx, const locohd_graph* g, uint64_t* indptr, uint32_t* indices, double* scores);
void locohd_graph_destroy(locohd_graph* g);
/* Planning query, no device needed: position `unit` of a launch of locohd_score_condensed on a range of n environments,
 * for the chunk of row blocks [row_block0, row_block0 + row_blocks) (a row block: 4 rows; ceil(n / 4) blocks) -> the
 * block of 4 x 4 pairs scored there, *out_row_block <= *out_col_block.  Units run column block major: first the
 * column blocks of the chunk's own rows (a triangle, row blocks row_block0 .. column block), then every further column
 * block with all row blocks of the chunk, row blocks ascending within a column block.  LOCOHD_ERR_BAD_PARAM for a
 * chunk outside the blocks or a unit out of range. */
int locohd_condensed_unit(uint64_t n, uint64_t row_block0, uint64_t row_blocks, uint64_t unit, uint64_t* out_row_block,
                          uint64_t* out_col_block);
/* Planning query, no device needed: how locohd_score_jobs[_stats] would group this job list for the tile kernel (jobs
 * that share runs of environments are scored tile by tile: up to 4 runs of A against up to 4 runs of B staged once per
 * anchor).  *out_tiles = tiles the list groups into (in list order if that tiles well, else regrouped by the ranks of
 * the runs), *out_rows = tile rows in use, *out_pays = 1 if the grouping passes the fill criteria (equal job sizes,
 * >= 60 % of the row cells used, >= 3 rows per tile).  Whether a call then takes the tile kernel also depends on the
 * instance (Hellinger-2, unit category weights, one weight function) and on the environment sizes. */
int locohd_plan_job_tiles(uint64_t n_jobs, const locohd_job* jobs, uint64_t* out_tiles, uint64_t* out_rows, int* out_pays);
/* Planning query, no device needed: position `unit` of a tile launch of n_tiles tiles with n_anchors anchors per job
 * -> the (tile, anchor) scored there.  The tile kernel visits all tiles for one slice of `slice` consecutive anchors
 * before the next slice starts, so that the environments of a slice stay in L2 while the tiles pass over them
 * (slice = 0 or >= n_anchors: tile-major order; the library picks the slice from the size of the environment store,
 * LOCOHD_TILE_SLICE / LOCOHD_TILE_SLICE_MB in the environment override it).  LOCOHD_ERR_BAD_PARAM for a unit out of
 * range. */
int locohd_tile_unit(uint64_t n_tiles, uint64_t n_anchors, uint64_t slice, uint64_t unit, uint64_t* out_tile,
                     uint64_t* out_anchor);
/* Planning query, no device needed: the launch geometry of the tile kernel for an instance of n_categories categories
 * in the configuration the tile kernel requires (Hellinger-2, unit category weights, one weight function) and
 * environment sets whose largest environments hold max_a / max_b members.  *teams = teams of four warps per CTA (0: the
 * tile kernel does not apply; locohd_score_jobs[_stats] takes it only from 6 teams on), *cp = count rows per warp (8 for
 * n_categories <= 8, else 16), *rep_n = head of the count-indexed tables replicated per bank pair (0: unreplicated),
 * *table_n = entries per table.  LOCOHD_TILE_TEAMS / LOCOHD_TILE_REP in the environment lower teams / rep_n, as they do
 * for a launch.  cp, rep_n and table_n may be NULL. */
int locohd_tile_geometry(int n_categories, uint32_t max_a, uint32_t max_b, int* teams, int* cp, int* rep_n,
                         int* table_n);
/* from_anchors (locohd.rs:392-406): one pair of caller-ordered environments, walked in the reference's
 * exact three-way-merge order (the lists are NOT required to be sorted, as in the reference). */
int locohd_score_anchor_lists(locohd_ctx* ctx, const uint16_t* seq_a, uint64_t len_a, const double* dists_a,
                              uint64_t dlen_a, const uint16_t* seq_b, uint64_t len_b, const double* dists_b,
                              uint64_t dlen_b, uint32_t wf_idx, double* out_score);

/* ---- one-call drop-in for LoCoHD::from_primitives (locohd.rs:479-567) ------------------- */
/* Host (or device) arrays in, scores out: upload, cell lists, environments, scoring, download.
 * anchors is [n_pairs][2] (primitive index in A, primitive index in B). */
int locohd_from_primitives(locohd_ctx* ctx, uint64_t n_a, const double* xyz_a, const uint16_t* cat_a,
                           const uint32_t* tag_a, uint64_t n_b, const double* xyz_b, const uint16_t* cat_b,
                           const uint32_t* tag_b, uint64_t n_pairs, const uint32_t* anchors,
                           const uint32_t* wf_idx, double threshold, double* out_scores);
/* The same call with the coordinate gradients of the scores (an extension: the reference has none).
 * out_grad_a [n_a][3] and out_grad_b [n_b][3] are overwritten with sum_p g_p dS_p/dxyz, g_p = pair_weights[p]
 * (NULL: all 1).  out_scores [n_pairs] may be NULL.  The gradient is the one-sided derivative in the walk's order
 * (distance, then A before B, then store order) where distances tie; membership changes at the threshold are not
 * differentiated.  Scores are deterministic; gradients are summed with FP64 atomics and may differ in the last bits
 * from call to call.  Any argument may be host or device memory. */
int locohd_from_primitives_grad(locohd_ctx* ctx, uint64_t n_a, const double* xyz_a, const uint16_t* cat_a,
                                const uint32_t* tag_a, uint64_t n_b, const double* xyz_b, const uint16_t* cat_b,
                                const uint32_t* tag_b, uint64_t n_pairs, const uint32_t* anchors,
                                const uint32_t* wf_idx, double threshold, const double* pair_weights,
                                double* out_scores, double* out_grad_a, double* out_grad_b);
/* from_dmxs (ragged rows, as locohd_envset_from_ragged_rows, per side) with the gradient of the scores with respect to
 * every entry: out_grad_s has row_offsets_s[n_rows] entries in the layout of values_s (an extension: the reference has
 * none).  Row r of A is scored against row r of B; entry (r, c) of side s receives g_r dS_r/d values_s[r][c],
 * g_r = pair_weights[r] (NULL: all 1).  Each row is sorted stably; its first entry is the anchor (distance 0) and
 * the others are events in merged order (distance, then A before B, then store order); an event's entry receives
 * g_r w(t) (H_{k-1} - H_k), w = dW/dt.  The anchor's entry, entries at t = 0 and non-finite entries (+inf bans) get
 * exactly 0; where distances tie the result is the one-sided derivative in that order.  Every entry is written by
 * one plain store, so scores and gradients are deterministic.  Validation and errors are those of from_dmxs
 * (locohd_envset_from_ragged_rows per side, the weight-function indices of locohd_score_jobs).  out_scores [n_rows]
 * may be NULL; any argument may be host or device memory. */
int locohd_from_rows_grad(locohd_ctx* ctx, uint64_t n_rows,
                          const uint64_t* row_offsets_a, const double* values_a, const uint16_t* category_a, uint64_t n_categories_a,
                          const uint64_t* row_offsets_b, const double* values_b, const uint16_t* category_b, uint64_t n_categories_b,
                          const uint32_t* wf_idx, const double* pair_weights,
                          double* out_scores, double* out_grad_a, double* out_grad_b);
/* from_coords with coordinate gradients: out_grad_s is [n_points][3], overwritten with sum_r g_r dS_r/dxyz_s.  The
 * entry gradients G_s[i][j] of locohd_from_rows_grad on the Euclidean rows t_ij = |x_j - x_i| give
 * grad_i = sum_j (G_s[i][j] + G_s[j][i]) (x_i - x_j) / t_ij, summed in a fixed order: deterministic.  Every point is in
 * every environment, so no member crosses a cutoff and the score is continuous in the coordinates (kinks: ties and
 * the weight function's own).  Memory: besides the 20 n^2 bytes per side of the row environments that from_coords
 * builds, 8 n^2 bytes per side of scratch for G.  Validation and errors are those of locohd_envset_from_coords; any
 * argument may be host or device memory. */
int locohd_from_coords_grad(locohd_ctx* ctx, uint64_t n_points, const double* xyz_a, const uint16_t* cat_a,
                            const double* xyz_b, const uint16_t* cat_b, const uint32_t* wf_idx,
                            const double* pair_weights, double* out_scores, double* out_grad_a, double* out_grad_b);

/* ---- leaf math on the device (parity checks of the FP64 device functions) --------------- */
/* WeightFunction::integral_point over n points (weight_function.rs:95-116). */
int locohd_wf_integral_points(locohd_ctx* ctx, const locohd_weight_function* wf, uint64_t n, const double* x,
                              double* out);
/* The density w(x) = dW/dx of the weight function over n points (the derivative of integral_point). */
int locohd_wf_density_points(locohd_ctx* ctx, const locohd_weight_function* wf, uint64_t n, const double* x,
                             double* out);
/* StatisticalDistance::run on n pairs of already-normalised vectors [n][n_categories]
 * (statistical_distances.rs:123-142); uses sd_kind/sd_params given here, not the context's. */
int locohd_sd_run(locohd_ctx* ctx, int32_t sd_kind, const double* sd_params, int32_t n_categories, uint64_t n,
                  const double* p1, const double* p2, double* out);

#ifdef __cplusplus
}
#endif
#endif /* LOCOHD_B200_H */
