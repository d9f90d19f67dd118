// locohd_kernels.cu — hand-written sm_100a kernels of the LoCoHD per-anchor scoring path.
//
// Pipeline (all FP64 where the reference is FP64; no tensor cores: there is no dense contraction):
//   K0   build_cells_kernel     one CTA per structure: bounding box, cell grid (edge r / 2 along y and z, r / 8 along
//                               x), counting sort of the primitives into cell order
//                               (replaces KdTree::build_by_ordered_float, locohd.rs:504-510)
//   Ka   anchor_slot_* kernels  put the requested anchors into cell order: neighbouring anchors are processed
//                               together and read the same candidate rows
//   K1   env_fused_kernel       one persistent WARP per anchor: row pruning, exact FP64 gather with the kd-tree
//                               predicate + tag rule, register bitonic sort, sqrt, CDF, key packing, store
//                               (kdtree.within_radius + filter + euclidean_distance + sort_together,
//                               locohd.rs:514-542, utils.rs:1-39); env_tile_kernel<false> on a 1/16 sample sizes
//                               the store beforehand
//   K2   score_fast_kernel /    one warp per anchor pair: merge-path split of the two sorted environments over the
//        score_kernel           32 lanes, per-lane category counts by warp prefix sums, per-lane walk that
//                               accumulates dW * H (stat_dist_integral, locohd.rs:61-226, as a flat prefix scan)
//   K2t  score_tile_kernel      job lists whose jobs share runs of environments (all-vs-all ensembles): a team of four
//                               warps per (4 x 4 tile of structure pairs, anchor) stages the 8 environments once and
//                               scores the 16 anchor pairs with 8 lanes each
//   fallback gather (environments the fused kernel cannot take, rows of from_dmxs / from_coords):
//   K1a  env_tile_kernel<false> one THREAD per anchor: FP32 prefilter over the candidate cells, counts the
//                               survivors (upper bound of the environment size) -> scan -> store offsets
//   K1b  env_tile_kernel<true>  same traversal; survivors are re-tested in FP64, (distance, category) is written
//                               unsorted into the store
//   K1c  env_sort_kernel<CAP>   one warp per environment: bucket sort by distance in shared memory, CDF, packing
// plus the small kernels around them (scans, row copies, the exact-order sequential walk of from_anchors,
// leaf-math probes).
#include "locohd_kernels.cuh"

#include <cfloat>
#include <cmath>
#include <cstdlib>

namespace locohd {

namespace {

constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ void raise(int* err, int code) { atomicCAS(err, 0, code); }

// ------------------------------------------------------------------------------------------------
// small utility kernels
// ------------------------------------------------------------------------------------------------
__global__ void convert_categories_kernel(const uint16_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n,
                                          int C) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const unsigned c = in[i];
        out[i] = (c < (unsigned)C) ? (uint8_t)c : kUnknownCat8;
    }
}

__global__ void validate_xyz_kernel(const double* __restrict__ xyz, uint64_t n3, int* err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3 && !isfinite(xyz[i])) raise(err, LOCOHD_ERR_NAN);
}

// ------------------------------------------------------------------------------------------------
// Exclusive scan of u32 values into u64 offsets (three kernels: tile sums, scan of the sums, apply).
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanPer = 8;
constexpr int kScanTile = kScanThreads * kScanPer;

template <int THREADS = kScanThreads>
__device__ __forceinline__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long* total) {
    __shared__ unsigned long long wsum[THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    unsigned long long base = 0, tot = 0;
    for (int w = 0; w < THREADS / 32; ++w) {
        if (w < wid) base += wsum[w];
        tot += wsum[w];
    }
    __syncthreads();
    if (total) *total = tot;
    return base + incl - v;
}

__device__ __forceinline__ unsigned scan_value(unsigned v, int round_even) { return round_even ? (v + 1u) & ~1u : v; }

__global__ void __launch_bounds__(kScanThreads) scan_tile_sums_kernel(const uint32_t* __restrict__ values, uint64_t n,
                                                                      int round_even,
                                                                      uint64_t* __restrict__ block_sums,
                                                                      ScanStats* stats) {
    const uint64_t t0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanPer;
    unsigned long long sum = 0;
    unsigned mx = 0;
    for (int q = 0; q < kScanPer; ++q) {
        const uint64_t i = t0 + q;
        if (i < n) {
            const unsigned c = values[i];
            sum += scan_value(c, round_even);
            mx = max(mx, c);
        }
    }
    unsigned long long tot;
    block_exclusive_scan(sum, &tot);
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(kFull, mx, o));
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(&stats->max_value, mx);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(kScanThreads) scan_block_sums_kernel(uint64_t* block_sums, uint64_t n_blocks,
                                                                       ScanStats* stats) {
    unsigned long long carry = 0;
    for (uint64_t b0 = 0; b0 < n_blocks; b0 += kScanThreads) {
        const uint64_t i = b0 + threadIdx.x;
        const unsigned long long v = (i < n_blocks) ? block_sums[i] : 0ull;
        unsigned long long tot;
        const unsigned long long ex = block_exclusive_scan(v, &tot);
        if (i < n_blocks) block_sums[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) stats->total = carry;
}

__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(const uint32_t* __restrict__ values, uint64_t n,
                                                                  int round_even,
                                                                  const uint64_t* __restrict__ block_sums,
                                                                  uint64_t* __restrict__ off) {
    const uint64_t t0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanPer;
    unsigned loc[kScanPer];
    unsigned long long sum = 0;
    for (int q = 0; q < kScanPer; ++q) {
        const uint64_t i = t0 + q;
        loc[q] = (i < n) ? scan_value(values[i], round_even) : 0u;
        sum += loc[q];
    }
    unsigned long long run = block_sums[blockIdx.x] + block_exclusive_scan(sum, nullptr);
    for (int q = 0; q < kScanPer; ++q) {
        const uint64_t i = t0 + q;
        if (i < n) off[i] = run;
        run += loc[q];
        if (i + 1 == n) off[n] = run;
    }
}

// ------------------------------------------------------------------------------------------------
// K0: cell list.  One CTA (256 threads) per structure; cell edge = half the radius (search +-2 cells), enlarged
// when the structure would need more than max(2 N, 8) cells.
// ------------------------------------------------------------------------------------------------
constexpr int kCellThreads = 512;   // latency-bound passes over one structure: more threads, more loads in flight
constexpr int kMaxCellsAxis = 1024;

__device__ __forceinline__ int cell_coord(double rel, double inv_cell, int n) {
    int c = (int)(rel * inv_cell);
    return min(max(c, 0), n - 1);
}

// SMEM: cell counters / cursors of structures whose grid fits the dynamic shared memory live there (shared-memory
// atomics, one scan pass); larger grids use the global arrays.
template <bool SMEM>
__global__ void __launch_bounds__(kCellThreads) build_cells_kernel(StructsView s, double threshold, int smem_words) {
    extern __shared__ uint32_t sm_cells[];
    __shared__ double red[6][kCellThreads / 32];
    __shared__ StructMeta sm_meta;
    __shared__ unsigned long long sh_carry;

    const uint64_t sid = blockIdx.x;
    const uint64_t base = s.prim_off[sid];
    const uint32_t n = (uint32_t)(s.prim_off[sid + 1] - base);
    const double* xyz = s.xyz + 3 * base;
    uint32_t* cell_start = s.cell_start + cell_base(base, sid);
    uint32_t* cell_fill = s.cell_fill + cell_base(base, sid);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

    // ---- bounding box
    double mn[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mx[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
    for (uint32_t i = tid; i < n; i += kCellThreads) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double v = xyz[3 * (uint64_t)i + k];
            mn[k] = fmin(mn[k], v);
            mx[k] = fmax(mx[k], v);
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        for (int o = 16; o; o >>= 1) {
            mn[k] = fmin(mn[k], __shfl_xor_sync(kFull, mn[k], o));
            mx[k] = fmax(mx[k], __shfl_xor_sync(kFull, mx[k], o));
        }
        if (lane == 0) { red[k][wid] = mn[k]; red[3 + k][wid] = mx[k]; }
    }
    __syncthreads();
    if (tid == 0) {
        double lo[3], hi[3];
        for (int k = 0; k < 3; ++k) {
            lo[k] = red[k][0]; hi[k] = red[3 + k][0];
            for (int w = 1; w < kCellThreads / 32; ++w) { lo[k] = fmin(lo[k], red[k][w]); hi[k] = fmax(hi[k], red[3 + k][w]); }
        }
        if (n == 0) { lo[0] = lo[1] = lo[2] = 0.0; hi[0] = hi[1] = hi[2] = 0.0; }
        const double ext[3] = {hi[0] - lo[0], hi[1] - lo[1], hi[2] - lo[2]};
        const double emax = fmax(ext[0], fmax(ext[1], ext[2]));
        const long long max_cells = max(2ll * (long long)n, 8ll);
        // cell edge slightly larger than half the radius: with reach = floor(r / edge * (1 + 1e-6)) + 1 rounding can
        // never push a member of the environment outside the visited cells
        double inv_cell = 2.0 / (threshold * (1.0 + 1e-6));
        if (!(inv_cell > 0.0) || !isfinite(inv_cell)) inv_cell = 0.0;  // infinite radius: a single cell
        StructMeta m;
        int xf = 4;   // x refinement: x cells of r / 8 as long as the grid stays within its bounds
        for (int it = 0; it < 200; ++it) {
            m.nx = (int)fmin(ext[0] * inv_cell * xf, 1.0e6) + 1;
            m.ny = (int)fmin(ext[1] * inv_cell, 1.0e6) + 1;
            m.nz = (int)fmin(ext[2] * inv_cell, 1.0e6) + 1;
            if ((long long)m.nx * m.ny * m.nz <= max_cells && m.nx <= kMaxCellsAxis && m.ny <= kMaxCellsAxis &&
                m.nz <= kMaxCellsAxis)
                break;
            if (xf > 1) xf >>= 1; else inv_cell *= 0.8;
        }
        if ((long long)m.nx * m.ny * m.nz > max_cells) { inv_cell = 0.0; xf = 1; m.nx = m.ny = m.nz = 1; }
        const double inv_cell_x = inv_cell * xf;
        m.ox = lo[0]; m.oy = lo[1]; m.oz = lo[2];
        m.inv_cell = inv_cell;
        m.inv_cell_x = inv_cell_x;
        // radius in cells.  A member lies less than `span` cells from its anchor along every axis, the anchor sits
        // at a fractional position < 1 inside its own cell, so the cell index differs by at most floor(span) + 1;
        // the default edge (r / 2 * (1 + 1e-6)) gives span = 1.999998 -> reach 2 (5 x 5 rows of 5 cells).
        const double span = threshold * inv_cell * (1.0 + 1e-9);   // 1e-9: rounding of the product near an integer
        m.reach = (inv_cell > 0.0 && isfinite(span)) ? (int)fmin(span, 2.0e6) + 1 : 0;
        if (inv_cell == 0.0) m.reach = 0;
        const double span_x = threshold * inv_cell_x * (1.0 + 1e-9);
        m.reach_x = (inv_cell_x > 0.0 && isfinite(span_x)) ? (int)fmin(span_x, 2.0e6) + 1 : 0;
        m.pad0 = 0;
        {   // the anchor-independent form of the fused gather's thin-shell bound: the structure's largest |coordinate|
            // stands in for the anchor's (a larger value only sends more candidates to the box test, never fewer)
            double qmax = threshold;
            for (int k = 0; k < 3; ++k) qmax = fmax(qmax, fmax(fabs(lo[k]), fabs(hi[k])));
            const double r_safe = threshold - 8.9e-16 * (qmax + threshold);
            m.r2_safe = (r_safe > 0.0 && isfinite(r_safe)) ? r_safe * r_safe * (1.0 - 1e-15)
                                                          : (isinf(threshold) ? __dmul_rn(threshold, threshold) : 0.0);
        }
        // FP32 prefilter: relative coordinates are rounded to f32 (error <= emax * 2^-24 each); the bound below
        // is generous (see DESIGN.md "prefilter margin").
        const double delta = 4.0 * emax * 5.9604644775390625e-8;
        const double tr = threshold + 2.0 * delta;
        const double t2 = tr * tr * (1.0 + 1e-6);
        float tf = (t2 < 3.0e38) ? (float)t2 : INFINITY;
        if (isfinite(tf)) tf = nextafterf(tf, INFINITY);
        m.thr2f = tf;
        // Row pruning of the fused gather works on the f32 relative coordinates.  A cell edge evaluated in f32
        // ((float)index * cellf) and an f32 coordinate are each within 2.5e-7 * (emax + cell + r) =: D of the exact
        // values, so a row that holds a member has a y-z gap below r + 2 D, and the x half-width
        // sqrt((r + 2 D)^2 - gap^2) covers the member (DESIGN.md, "row pruning").
        if (inv_cell > 0.0 && isfinite(threshold) && isfinite(emax)) {
            const double cell = 1.0 / inv_cell;
            const double D = 2.5e-7 * (emax + cell + threshold) * 1.001;
            const double pr = (threshold + 2.0 * D) * (1.0 + 1e-5);
            m.cellf = (float)cell;
            m.inv_cellxf = (float)inv_cell_x;
            m.prune_r = (pr < 1.0e18) ? nextafterf((float)pr, INFINITY) : 0.f;
            if (!(m.prune_r > 0.f) || !isfinite(m.cellf) || !isfinite(m.inv_cellxf)) { m.cellf = 0.f; m.prune_r = 0.f; }
        } else {
            m.cellf = 0.f; m.inv_cellxf = 0.f; m.prune_r = 0.f;
        }
        sm_meta = m;
        s.meta[sid] = m;
        sh_carry = 0;
    }
    __syncthreads();
    const StructMeta m = sm_meta;
    const int ncell = m.nx * m.ny * m.nz;
    const bool in_smem = SMEM && ncell + 1 <= smem_words;   // uniform over the CTA
    uint32_t* cnt = in_smem ? sm_cells : cell_start;
    for (int c = tid; c <= ncell; c += kCellThreads) cnt[c] = 0;
    __syncthreads();

    // ---- histogram
    for (uint32_t i = tid; i < n; i += kCellThreads) {
        const double x = xyz[3 * (uint64_t)i], y = xyz[3 * (uint64_t)i + 1], z = xyz[3 * (uint64_t)i + 2];
        const int cx = cell_coord(x - m.ox, m.inv_cell_x, m.nx);
        const int cy = cell_coord(y - m.oy, m.inv_cell, m.ny);
        const int cz = cell_coord(z - m.oz, m.inv_cell, m.nz);
        atomicAdd(&cnt[(cz * m.ny + cy) * m.nx + cx], 1u);
    }
    __syncthreads();

    uint32_t* fill;
    if (in_smem) {
        // ---- exclusive scan in shared memory: a contiguous run of cells per thread, one block scan of the run sums
        const int per = (ncell + kCellThreads - 1) / kCellThreads;
        const int c_lo = min(tid * per, ncell), c_hi = min(c_lo + per, ncell);
        unsigned long long sum = 0;
        for (int c = c_lo; c < c_hi; ++c) sum += cnt[c];
        unsigned long long run = block_exclusive_scan<kCellThreads>(sum, nullptr);
        for (int c = c_lo; c < c_hi; ++c) {
            const uint32_t v = cnt[c];
            cnt[c] = (uint32_t)run;          // from here on: the fill cursor of the cell
            cell_start[c] = (uint32_t)run;
            run += v;
        }
        if (tid == 0) cell_start[ncell] = n;
        fill = cnt;
    } else {
        // ---- exclusive scan over the cells in global memory, kCellThreads cells per round
        for (int c0 = 0; c0 < ncell; c0 += kCellThreads) {
            const int c = c0 + tid;
            const unsigned long long v = (c < ncell) ? cell_start[c] : 0u;
            unsigned long long tot;
            const unsigned long long ex = block_exclusive_scan<kCellThreads>(v, &tot);
            const unsigned long long carry = sh_carry;
            if (c < ncell) {
                cell_start[c] = (uint32_t)(carry + ex);
                cell_fill[c] = (uint32_t)(carry + ex);
            }
            __syncthreads();
            if (tid == 0) sh_carry = carry + tot;
            __syncthreads();
        }
        if (tid == 0) cell_start[ncell] = n;
        fill = cell_fill;
    }
    __syncthreads();

    // ---- scatter into cell order
    for (uint32_t i = tid; i < n; i += kCellThreads) {
        const double x = xyz[3 * (uint64_t)i], y = xyz[3 * (uint64_t)i + 1], z = xyz[3 * (uint64_t)i + 2];
        const int cx = cell_coord(x - m.ox, m.inv_cell_x, m.nx);
        const int cy = cell_coord(y - m.oy, m.inv_cell, m.ny);
        const int cz = cell_coord(z - m.oz, m.inv_cell, m.nz);
        const uint32_t pos = atomicAdd(&fill[(cz * m.ny + cy) * m.nx + cx], 1u);
        PrimRec r;
        r.x = x; r.y = y; r.z = z;
        r.tag = s.tag[base + i];
        r.cat = s.cat[base + i];
        s.pd[base + pos] = r;
        s.porig[base + pos] = i;
        s.pf[base + pos] = make_float4((float)(x - m.ox), (float)(y - m.oy), (float)(z - m.oz),
                                       __uint_as_float(r.tag));
        s.sorted_pos[base + i] = pos;
    }
}

// ------------------------------------------------------------------------------------------------
// Tag rule
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool tag_pair_in_table(const KParams& p, uint32_t a, uint32_t b) {
    const uint64_t key = ((uint64_t)a << 32) | b;
    uint64_t lo = 0, hi = p.n_tag_pairs;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        const uint64_t v = __ldg(p.tag_pairs + mid);
        if (v < key) lo = mid + 1; else hi = mid;
    }
    return lo < p.n_tag_pairs && __ldg(p.tag_pairs + lo) == key;
}

// TagPairingRule::pair_accepted on interned ids (tag_pairing_rule.rs:49-76); pair = (anchor.tag, neighbour.tag)
__device__ __forceinline__ bool tag_rule_accepts(const KParams& p, uint32_t anchor_tag, uint32_t other_tag) {
    if (p.tpr_kind == LOCOHD_TPR_WITHOUT_LIST) {
        const bool same = anchor_tag == other_tag;
        return p.tpr_accept_same ? same : !same;
    }
    bool acc = tag_pair_in_table(p, anchor_tag, other_tag);
    if (!p.tpr_ordered) acc = acc || tag_pair_in_table(p, other_tag, anchor_tag);
    return p.tpr_accepted_pairs ? acc : !acc;
}

// ------------------------------------------------------------------------------------------------
// Ka: anchors in cell order.  slot = global cell-sorted position of the anchor's primitive.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool anchor_slot(const StructsView& s, const uint32_t* anchor_struct,
                                            const uint32_t* anchor_prim, uint64_t e, int* err, uint64_t* slot) {
    const uint64_t sid = anchor_struct ? anchor_struct[e] : 0;
    const uint32_t prim = anchor_prim[e];
    if (sid >= s.n_structs) { raise(err, LOCOHD_ERR_INDEX); return false; }
    const uint64_t base = s.prim_off[sid];
    if (prim >= s.prim_off[sid + 1] - base) { raise(err, LOCOHD_ERR_INDEX); return false; }  // locohd.rs:521 panics
    *slot = base + s.sorted_pos[base + prim];
    return true;
}

__global__ void anchor_slot_count_kernel(StructsView s, KParams p, uint64_t n_env,
                                         const uint32_t* __restrict__ anchor_struct,
                                         const uint32_t* __restrict__ anchor_prim, uint32_t* slot_cnt) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_env) return;
    uint64_t slot = 0;
    anchor_slot(s, anchor_struct, anchor_prim, e, p.err, &slot);  // invalid anchors go to slot 0 (the call fails)
    atomicAdd(&slot_cnt[slot], 1u);
}

__global__ void anchor_slot_scatter_kernel(StructsView s, KParams p, uint64_t n_env,
                                           const uint32_t* __restrict__ anchor_struct,
                                           const uint32_t* __restrict__ anchor_prim, uint32_t* slot_cnt,
                                           const uint64_t* __restrict__ slot_off, uint32_t* __restrict__ order,
                                           uint2* __restrict__ order_rec) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_env) return;
    uint64_t slot = 0;
    const bool ok = anchor_slot(s, anchor_struct, anchor_prim, e, p.err, &slot);
    const uint32_t k = atomicSub(&slot_cnt[slot], 1u) - 1u;
    const uint64_t pos = slot_off[slot] + k;
    order[pos] = (uint32_t)e;
    if (order_rec) {   // (structure, cell-sorted position) next to the order: the gather needs one load per anchor
        const uint32_t sid = anchor_struct ? anchor_struct[e] : 0u;
        order_rec[pos] = ok ? make_uint2(sid, (uint32_t)(slot - s.prim_off[sid])) : make_uint2(0xFFFFFFFFu, 0u);
    }
}

// Small calls keep the caller's anchor order (no counting sort: five launches less; the locality it buys only
// matters when thousands of anchors share candidate rows).
__global__ void anchor_identity_kernel(StructsView s, KParams p, uint64_t n_env, const uint32_t* __restrict__ anchor_struct,
                                       const uint32_t* __restrict__ anchor_prim, uint32_t* __restrict__ order,
                                       uint2* __restrict__ order_rec) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_env) return;
    uint64_t slot = 0;
    const bool ok = anchor_slot(s, anchor_struct, anchor_prim, e, p.err, &slot);
    order[e] = (uint32_t)e;
    const uint32_t sid = anchor_struct ? anchor_struct[e] : 0u;
    order_rec[e] = ok ? make_uint2(sid, (uint32_t)(slot - s.prim_off[sid])) : make_uint2(0xFFFFFFFFu, 0u);
}

// ------------------------------------------------------------------------------------------------
// K1a / K1b: one thread per anchor, anchors taken in cell order.
//   Every lane walks the candidate cells of its own anchor (rows of 2*reach+1 cells are contiguous in the
//   cell-sorted arrays); neighbouring lanes sit in the same or adjacent cells, so their float4 loads hit the same
//   lines.  FILL: every FP32 survivor is re-tested at once in FP64 — box test + ((dx^2 + dy^2) + dz^2) < r^2 with
//   unfused arithmetic, the kd-tree crate's predicate and operation order; the anchor itself is always kept,
//   others must pass the tag rule (locohd.rs:521-528).  Lanes of a warp look at the same candidate at the same
//   time, so the 32-byte exact record is one broadcast load.
// ------------------------------------------------------------------------------------------------
constexpr int kTileThreads = 128;

template <bool FILL>
__global__ void __launch_bounds__(kTileThreads) env_tile_kernel(StructsView s, KParams p, uint64_t n_env,
                                                                const uint32_t* __restrict__ order,
                                                                const uint32_t* __restrict__ anchor_struct,
                                                                const uint32_t* __restrict__ anchor_prim,
                                                                double threshold, uint32_t* __restrict__ ub,
                                                                EnvBuild b, uint32_t stride,
                                                                unsigned long long* sample_sum) {
    // stride > 1 (count mode only): every stride-th group of 32 consecutive anchors is visited (a warp keeps
    // neighbouring anchors, so its lanes walk the same candidate rows) and the sizes are summed into *sample_sum
    const int tid = threadIdx.x;
    const uint64_t t0 = (uint64_t)blockIdx.x * kTileThreads + tid;
    const uint64_t t = (t0 >> 5) * 32 * stride + (t0 & 31);
    bool active = t < n_env;
    const uint64_t e = active ? order[t] : 0;
    uint64_t base = 0;
    uint32_t jpos = 0;
    StructMeta m;
    m.nx = m.ny = m.nz = 1; m.reach = 0; m.inv_cell = 0.0; m.ox = m.oy = m.oz = 0.0; m.thr2f = 0.f;
    m.cellf = m.prune_r = m.inv_cellxf = 0.f; m.inv_cell_x = 0.0; m.reach_x = 0; m.pad0 = 0; m.r2_safe = 0.0;
    const uint32_t* cell_start = s.cell_start;
    if (active) {
        const uint64_t sid = anchor_struct ? anchor_struct[e] : 0;
        const uint32_t prim = anchor_prim[e];
        if (sid >= s.n_structs || prim >= s.prim_off[sid + 1] - s.prim_off[sid]) {
            raise(p.err, LOCOHD_ERR_INDEX);
            active = false;
        } else {
            base = s.prim_off[sid];
            jpos = s.sorted_pos[base + prim];
            m = s.meta[sid];
            cell_start = s.cell_start + cell_base(base, sid);
        }
    }
    PrimRec q;
    q.x = q.y = q.z = 0.0; q.tag = 0; q.cat = 0;
    float4 qf = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active) { q = s.pd[base + jpos]; qf = s.pf[base + jpos]; }
    const uint32_t qtag = __float_as_uint(qf.w);
    const double r2 = __dmul_rn(threshold, threshold);
    const int cx = cell_coord(q.x - m.ox, m.inv_cell_x, m.nx);
    const int cy = cell_coord(q.y - m.oy, m.inv_cell, m.ny);
    const int cz = cell_coord(q.z - m.oz, m.inv_cell, m.nz);
    const int x0 = max(cx - m.reach_x, 0), x1 = min(cx + m.reach_x, m.nx - 1);
    int reach = active ? m.reach : 0;
    for (int o = 16; o; o >>= 1) reach = max(reach, __shfl_xor_sync(kFull, reach, o));   // warp-uniform loop bounds

    const float4* pf = s.pf + base;
    const PrimRec* pd = s.pd + base;
    const uint64_t off = (FILL && active) ? b.off[e] : 0;
    const uint32_t cap = (FILL && active) ? b.ub[e] : 0;
    uint32_t cnt = 0;
    const double lox = q.x - threshold, hix = q.x + threshold;
    const double loy = q.y - threshold, hiy = q.y + threshold;
    const double loz = q.z - threshold, hiz = q.z + threshold;
    // Below r2_safe the box test cannot fail: |dx| < r - margin with margin >= the rounding error of q + r
    // (4 ulp of the larger of |q| and r).  Only the thin shell above it pays for the six extra compares.
    const double qmax = fmax(fmax(fabs(q.x), fabs(q.y)), fmax(fabs(q.z), threshold));
    const double r_safe = threshold - 8.9e-16 * (qmax + threshold);
    const double r2_safe = (r_safe > 0.0 && isfinite(r_safe)) ? r_safe * r_safe * (1.0 - 1e-15) : (isinf(threshold) ? r2 : 0.0);

    for (int dz = -reach; dz <= reach; ++dz) {
        for (int dy = -reach; dy <= reach; ++dy) {
            const int zz = cz + dz, yy = cy + dy;
            uint32_t j = 0, end = 0;
            if (active && abs(dz) <= m.reach && abs(dy) <= m.reach && zz >= 0 && zz < m.nz && yy >= 0 && yy < m.ny) {
                const int row = (zz * m.ny + yy) * m.nx;
                j = __ldg(cell_start + row + x0);
                end = __ldg(cell_start + row + x1 + 1);
            }
            for (; j < end; ++j) {
                const float4 c = __ldg(pf + j);
                const float dx = c.x - qf.x, dyf = c.y - qf.y, dzf = c.z - qf.z;
                const float d2f = dx * dx + dyf * dyf + dzf * dzf;
                if (d2f <= m.thr2f) {
                    if (!FILL) {
                        ++cnt;
                    } else {
                        const PrimRec r = pd[j];
                        const double ex = r.x - q.x, ey = r.y - q.y, ez = r.z - q.z;
                        const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
                        bool acc = d2 < r2;
                        if (acc && !(d2 < r2_safe)) {
                            // within rounding distance of the sphere: the crate's per-axis box test can still reject
                            acc = !(r.x < lox) && !(r.x > hix) && !(r.y < loy) && !(r.y > hiy) && !(r.z < loz) &&
                                  !(r.z > hiz);
                        }
                        if (acc && j != jpos) acc = tag_rule_accepts(p, qtag, __float_as_uint(c.w));
                        if (acc) {
                            if (cnt < cap) {
                                b.key[off + cnt] = (uint64_t)__double_as_longlong(d2);  // sqrt in the sort kernel
                                b.cat[off + cnt] = (uint8_t)r.cat;
                                if (b.idx) b.idx[off + cnt] = s.porig[base + j];
                            }
                            ++cnt;
                        }
                    }
                }
            }
        }
    }
    if (FILL) {
        if (active) {
            if (cnt > cap) raise(p.err, LOCOHD_ERR_CUDA);  // the FP32 count is an upper bound by construction
            b.count[e] = min(cnt, cap);
        }
    } else if (sample_sum) {
        unsigned v = active ? cnt : 0u;
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
        if ((tid & 31) == 0 && v) atomicAdd(sample_sum, (unsigned long long)v);
    } else if (active) {
        ub[e] = cnt;
    } else if (t < n_env) {
        ub[e] = 0;
    }
}

__device__ __forceinline__ uint32_t smem_u32_early(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float rsqrt_approx(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// f64 bits of W (or of the distance) with the low mantissa byte replaced by the category
__device__ __forceinline__ uint64_t pack_key(double w, uint32_t cat) {
    w = w + 0.0;                 // -0.0 -> +0.0
    w = fmax(w, 0.0);            // a CDF that rounds to a tiny negative value must not set the sign bit
    return ((uint64_t)__double_as_longlong(w) & ~kCatMask) | (uint64_t)(cat & 0xFFu);
}

// ------------------------------------------------------------------------------------------------
// K1 (fused): one persistent WARP per anchor does the whole of env_from_idx (locohd.rs:514-542) in one pass:
//   rows      lane r < 25 owns one of the (2 reach + 1)^2 <= 25 candidate rows of the anchor (reach <= 2 always:
//             cells are never smaller than r / 2): rows farther than r in the y-z plane are dropped, the x range of
//             the others is cut to sqrt(r^2 - gap^2), in f32 with conservative margins (build_cells_kernel)
//   gather    lanes over the flat concatenation of the rows (coalesced 32-byte records, the next round is loaded
//             while the current one is tested); the row of a flat index comes from a bitmap of the row starts
//             + popc, no search loop.  Exact membership: the kd-tree crate's predicate in FP64 with unfused
//             arithmetic (as env_tile_kernel<true>) + tag rule; members are ballot-compacted into shared memory:
//             squared distance, category and a 32-bit sort key = 23-bit fixed-point squared distance << 9 | slot.
//             (No FP32 prefilter here: with a warp per anchor every lane tests a different candidate, the FP64
//             instructions are issued once per round either way.)
//   sort      warp bitonic network on the 32-bit keys in registers (4, 8 or 16 per lane; min/max and shuffles, no
//             shared-memory atomics; stages run as loops to keep the code small), then neighbours with equal
//             fixed-point distance are checked against the exact values (rare serial repair)
//   store     sqrt (utils.rs:1-8), CDF (specialised by WFK), key packing; coalesced stores into a chunk of the store
//             the warp reserved with one atomicAdd per kFusedChunk entries.
// CAP (512 or 1024) bounds the members of an environment.  Environments that do not fit, or a store that turns out
// too small, raise the overflow word: the host retries with the larger CAP and finally rebuilds the call with the
// exact multi-kernel path.
// ------------------------------------------------------------------------------------------------
template <bool DEBUG, int CAP>
struct FusedLayout {
    static constexpr int kD2Off = 0;                              // f64 [CAP] exact squared distances
    static constexpr int kKeyOff = kD2Off + 8 * CAP;              // u32 [CAP] sort keys
    static constexpr int kRowOff = kKeyOff + 4 * CAP;             // i32 [32] row delta (start - flat prefix)
    static constexpr int kMaskWords = CAP / 8;                    // row-start bits of up to 4 CAP candidates
    static constexpr int kMaskOff = kRowOff + 4 * 32;             // u32 [kMaskWords]
    static constexpr int kCatOff = kMaskOff + 4 * kMaskWords;     // u8 [CAP]
    static constexpr int kIdxOff = kCatOff + CAP;                 // u32 [CAP] (DEBUG)
    static constexpr int kBytes = (kIdxOff + (DEBUG ? 4 * CAP : 0) + 15) & ~15;
};
// sort key = fixed-point squared distance << SB | slot, SB = log2(CAP) slot bits
template <int CAP> struct FusedKey {
    static constexpr int SB = CAP == 512 ? 9 : 10;
    static constexpr uint32_t kSlotMask = (1u << SB) - 1u;
    static constexpr double kScale = (double)((1u << (32 - SB)) - 16u);   // d2 < r2 -> fixed point < 2^(32-SB) - 15
};

// ascending compare-exchange of two registers of one lane
__device__ __forceinline__ void cex(uint32_t& a, uint32_t& c) {
    const uint32_t lo = min(a, c), hi = max(a, c);
    a = lo;
    c = hi;
}

// Ascending bitonic sort of 32 * PER distinct keys, element g = lane * PER + r, in the formulation whose first stage
// of every merge compares g with g ^ (size - 1) (mirror) and the others g with g ^ stride: every compare-exchange
// puts the smaller key at the lower index, so in-lane stages are plain min / max pairs and a cross-lane exchange is
// SHFL + ISETP.XOR + SEL (keep mine iff (mine < other) != I-am-the-upper-lane).  Merges that span lanes run as
// (not unrolled) loops to keep the code small.
template <int PER>
__device__ __forceinline__ void warp_bitonic(uint32_t (&k)[PER], int lane) {
    // merges inside a lane: static network
#pragma unroll
    for (int size = 2; size <= PER; size <<= 1) {
#pragma unroll
        for (int r = 0; r < PER; ++r)
            if ((r & (size >> 1)) == 0) cex(k[r], k[r ^ (size - 1)]);
#pragma unroll
        for (int stride = size >> 2; stride > 0; stride >>= 1) {
#pragma unroll
            for (int r = 0; r < PER; ++r)
                if ((r & stride) == 0) cex(k[r], k[r | stride]);
        }
    }
    // merges across lanes: lsz = lanes per merged run
#pragma unroll 1
    for (int lsz = 2; lsz <= 32; lsz <<= 1) {
        {   // mirror stage: element r of this lane meets element PER - 1 - r of lane ^ (lsz - 1)
            const bool upper = (lane & (lsz >> 1)) != 0;
            uint32_t x[PER];
#pragma unroll
            for (int r = 0; r < PER; ++r) x[r] = __shfl_xor_sync(kFull, k[PER - 1 - r], lsz - 1);
#pragma unroll
            for (int r = 0; r < PER; ++r) k[r] = ((k[r] < x[r]) != upper) ? k[r] : x[r];
        }
#pragma unroll 1
        for (int lm = lsz >> 2; lm > 0; lm >>= 1) {
            const bool upper = (lane & lm) != 0;
#pragma unroll
            for (int r = 0; r < PER; ++r) {
                const uint32_t x = __shfl_xor_sync(kFull, k[r], lm);
                k[r] = ((k[r] < x) != upper) ? k[r] : x;
            }
        }
#pragma unroll
        for (int stride = PER >> 1; stride > 0; stride >>= 1) {
#pragma unroll
            for (int r = 0; r < PER; ++r)
                if ((r & stride) == 0) cex(k[r], k[r | stride]);
        }
    }
}

// Sorts key32[0, M) in place.  Returns (warp-uniform) whether two neighbours of the sorted order share their
// fixed-point distance (key >> SB): only then does the caller compare exact distances.
template <int PER, int SB>
__device__ __noinline__ bool fused_sort(uint32_t* key32, uint32_t M, int lane) {
    // A lane owns PER consecutive keys: 16-byte accesses (4 wavefronts per warp instruction; word accesses at a
    // stride of PER words would be 8-way bank conflicts).  Entries from M on are padding on the way in and are
    // written back as such (nothing reads key32 beyond M afterwards; 32 * PER <= CAP).
    uint32_t k[PER];
    uint4* key4 = reinterpret_cast<uint4*>(key32) + lane * (PER / 4);
#pragma unroll
    for (int q = 0; q < PER / 4; ++q) {
        const uint4 v = key4[q];
        k[4 * q] = v.x; k[4 * q + 1] = v.y; k[4 * q + 2] = v.z; k[4 * q + 3] = v.w;
    }
#pragma unroll
    for (int r = 0; r < PER; ++r)
        if ((uint32_t)(lane * PER + r) >= M) k[r] = 0xFFFFFFFFu;
    __syncwarp();
    warp_bitonic<PER>(k, lane);
    bool tie = false;
    const uint32_t next0 = __shfl_down_sync(kFull, k[0], 1);   // first key of the next lane
#pragma unroll
    for (int r = 0; r < PER; ++r) {
        const uint32_t g = (uint32_t)(lane * PER + r);
        const uint32_t nb = (r + 1 < PER) ? k[(r + 1) % PER] : next0;
        tie |= (g + 1 < M) && ((k[r] >> SB) == (nb >> SB)) && (r + 1 < PER || lane < 31);
    }
#pragma unroll
    for (int q = 0; q < PER / 4; ++q) key4[q] = make_uint4(k[4 * q], k[4 * q + 1], k[4 * q + 2], k[4 * q + 3]);
    __syncwarp();
    return __any_sync(kFull, tie);
}

// serial repair of groups with equal fixed-point distance (order by exact squared distance, category, slot)
template <int SB>
__device__ __noinline__ void fused_repair(uint32_t* key32, const double* d2s, const uint8_t* cats, uint32_t M) {
    constexpr uint32_t kMask = (1u << SB) - 1u;
    for (uint32_t g = 1; g < M; ++g) {
        const uint32_t kg = key32[g];
        const uint32_t sg = kg & kMask;
        const double dg = d2s[sg];
        const uint32_t cg = cats[sg];
        uint32_t u = g;
        while (u > 0) {
            const uint32_t kf = key32[u - 1];
            if ((kf >> SB) != (kg >> SB)) break;
            const uint32_t sf = kf & kMask;
            const double df = d2s[sf];
            const uint32_t cf = cats[sf];
            if (df < dg || (df == dg && (cf < cg || (cf == cg && sf < sg)))) break;
            key32[u] = kf;
            --u;
        }
        key32[u] = kg;
    }
}

// WFK: 0 uniform, 1 kumaraswamy with small integer exponents, 2 anything else (wf_cdf, or plain distances),
// 3 kumaraswamy with the exponents (2, 5) of the reference's own parametrisation (tests/test_locohd.py:42) fixed at
// compile time: the run-time switch of powi_small cost 151 warp instructions per environment (profiles/r4g_k1_lines.md).
// The parameters of variants 0 and 1 are read once per kernel into registers (FusedWf): left in global memory the
// compiler reloads them in every round of the store loop (they may alias the stores) and the loop waits on them.
struct FusedWf {
    double p0, p1, inv_range;
    int int_a, int_b;
};
template <int WFK>
__device__ __forceinline__ double fused_weight(const WfDev& wf, const FusedWf& f, double d, int key_is_w) {
    if (WFK == 0) {
        const double z = (d - f.p0) * f.inv_range;
        return (d < f.p0) ? 0.0 : ((d > f.p1) ? 1.0 : z);
    } else if (WFK == 1) {
        const double z = (d - f.p0) * f.inv_range;
        const double u = 1.0 - powi_small(z, f.int_a);
        const double v = 1.0 - powi_small(u, f.int_b);
        return (d < f.p0) ? 0.0 : ((d > f.p1) ? 1.0 : v);
    } else if (WFK == 3) {   // the same operations powi_small performs for e = 2 and e = 5
        const double z = (d - f.p0) * f.inv_range;
        const double u = 1.0 - z * z;
        const double u2 = u * u;
        const double v = 1.0 - u2 * u2 * u;
        return (d < f.p0) ? 0.0 : ((d > f.p1) ? 1.0 : v);
    } else {
        return key_is_w ? wf_cdf(wf, d) : d;
    }
}

// Distance from the exact squared distance.  Parity dumps (EXACT) take the IEEE square root; otherwise the value only
// feeds W(d) / the packed key, and MUFU.RSQ (f32 seed) + two coupled Newton steps in FP64 (~1e-16 relative, a third of
// the instructions) is used inside the f32 exponent range.
template <bool EXACT>
__device__ __forceinline__ double fused_distance(double d2) {
    if (EXACT) return sqrt(d2);
    // d2 < r^2 < 1e30 here (host check).  Below 1e-30 (distances under 1e-15) the seed is clamped: the result is then
    // only a monotone value of the same vanishing size, which is all W(d) needs there; 0 stays exactly 0.
    const double g = (double)rsqrt_approx(fmaxf((float)d2, 1e-30f));
    double sq = d2 * g, hh = 0.5 * g;
    double r = fma(-sq, hh, 0.5);
    sq = fma(sq, r, sq); hh = fma(hh, r, hh);
    r = fma(-sq, hh, 0.5);
    return fma(sq, r, sq);
}

template <int WFK, bool DEBUG, int CAP, bool LIST>
__global__ void __launch_bounds__(fused_warps(CAP, DEBUG) * 32, CAP == 512 ? 1 : 16 / fused_warps(CAP, DEBUG)) env_fused_kernel(StructsView s, KParams p, uint64_t n_env,
                                                                     const uint32_t* __restrict__ order,
                                                                     const uint32_t* __restrict__ anchor_struct,
                                                                     const uint32_t* __restrict__ anchor_prim,
                                                                     double threshold, EnvBuild b, FusedStats* stats,
                                                                     uint64_t capacity) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using L = FusedLayout<DEBUG, CAP>;
    using K = FusedKey<CAP>;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned char* smem = smem_raw + (size_t)wib * L::kBytes;
    double* d2s = reinterpret_cast<double*>(smem + L::kD2Off);
    uint32_t* key32 = reinterpret_cast<uint32_t*>(smem + L::kKeyOff);
    int* row_delta = reinterpret_cast<int*>(smem + L::kRowOff);
    uint32_t* row_mask = reinterpret_cast<uint32_t*>(smem + L::kMaskOff);
    uint8_t* cats = smem + L::kCatOff;
    uint32_t* sidx = reinterpret_cast<uint32_t*>(smem + L::kIdxOff);
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned le_mask = lt_mask | (1u << lane);

    const double r2 = __dmul_rn(threshold, threshold);
    const double qscale = K::kScale / r2;   // the host sends radii with r^2 >= 1e30 (or infinite) to the multi-kernel path
    constexpr bool simple_rule = !LIST;   // WithoutList rule: a tag comparison; WithList: table look-ups (own instantiation)
    const bool accept_same = p.tpr_accept_same != 0;
    const WfDev& wf = p.wfs[0];
    FusedWf fwf;
    fwf.p0 = wf.p[0]; fwf.p1 = wf.p[1]; fwf.inv_range = wf.inv_range; fwf.int_a = wf.int_a; fwf.int_b = wf.int_b;
    const bool fix_monotone = (WFK == 2) && b.key_is_w && !wf.monotone;
    const int key_is_w = b.key_is_w;
    uint64_t chunk_pos = 0, chunk_end = 0;   // warp-uniform: the reserved part of the store
    unsigned max_m = 0;

    // Every CTA takes a contiguous block of the cell-ordered anchors and its warps draw the next anchor from a
    // shared cursor: at any time the warps of a CTA hold consecutive anchors (they do not drift apart as with a
    // fixed stride), read overlapping candidate rows (L1 hits) and finish together.
    // (a 32-bit offset and a plain atom.shared.add: the 64-bit shared-memory atomicAdd is a compare-and-swap loop, and
    //  the compiler wraps an atomicAdd under `if (lane == 0)` into its warp-aggregation sequence - ~30 instructions per
    //  environment together)
    __shared__ unsigned int cta_cursor;
    const uint64_t per_block = (n_env + gridDim.x - 1) / gridDim.x;
    const uint64_t t_begin = min(n_env, (uint64_t)blockIdx.x * per_block);
    const uint64_t t_end = min(n_env, (uint64_t)(blockIdx.x + 1) * per_block);
    const uint32_t t_count = (uint32_t)min(t_end - t_begin, (uint64_t)0xFFFFFFFFu);   // the host keeps per_block below 2^32
    if (threadIdx.x == 0) cta_cursor = 0u;
    __syncthreads();
    const uint32_t cursor_addr = smem_u32_early(&cta_cursor);
#pragma unroll 1
    for (;;) {
        __syncwarp();
        uint32_t tk = 0;
        if (lane == 0) asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(tk) : "r"(cursor_addr) : "memory");
        tk = __shfl_sync(kFull, tk, 0);
        if (tk >= t_count) break;
        const uint64_t t = t_begin + tk;
        const uint64_t e = order[t];
        const uint2 rec = b.order_rec[t];   // (structure, cell-sorted position), written with the anchor order
        const uint64_t sid = rec.x;
        if (rec.x == 0xFFFFFFFFu) {   // anchor index out of range (locohd.rs:521 panics)
            if (lane == 0) { raise(p.err, LOCOHD_ERR_INDEX); b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }
        const uint64_t base = s.prim_off[sid];
        const uint32_t jpos = rec.y;
        const StructMeta m = s.meta[sid];
        const uint32_t* cell_start = s.cell_start + cell_base(base, sid);
        const PrimRec* pd = s.pd + base;
        const PrimRec q = pd[jpos];
        const float4 qf = __ldg(s.pf + base + jpos);
        const uint32_t qtag = __float_as_uint(qf.w);
        if (m.reach > 2) {   // cannot happen (cells are never smaller than r / 2); leave it to the multi-kernel path
            if (lane == 0) { atomicOr(&stats->overflow, 2u); b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }

        // ---- candidate rows: lane r < W * W owns row (dy, dz)
        uint32_t my_len = 0, my_pre = 0;
        {
            const int W = 2 * m.reach + 1;
            const int cx = cell_coord(q.x - m.ox, m.inv_cell_x, m.nx);
            const int cy = cell_coord(q.y - m.oy, m.inv_cell, m.ny);
            const int cz = cell_coord(q.z - m.oz, m.inv_cell, m.nz);
            uint32_t start = 0;
            if (lane < W * W) {
                const int dzi = (lane * 13) >> 6;   // lane / 5 for lane < 25
                const int dz5 = (W == 5) ? dzi : ((W == 3) ? (lane * 11) >> 5 : 0);   // lane / W
                const int dyi = lane - dz5 * W - m.reach, dzz = dz5 - m.reach;
                const int yy = cy + dyi, zz = cz + dzz;
                if (yy >= 0 && yy < m.ny && zz >= 0 && zz < m.nz) {
                    int x0 = max(cx - m.reach_x, 0), x1 = min(cx + m.reach_x, m.nx - 1);
                    bool keep = true;
                    if (m.prune_r > 0.f) {
                        float gy = 0.f, gz = 0.f;
                        if (dyi > 0) gy = (float)yy * m.cellf - qf.y;
                        else if (dyi < 0) gy = qf.y - (float)(yy + 1) * m.cellf;
                        if (dzz > 0) gz = (float)zz * m.cellf - qf.z;
                        else if (dzz < 0) gz = qf.z - (float)(zz + 1) * m.cellf;
                        gy = fmaxf(gy, 0.f); gz = fmaxf(gz, 0.f);
                        const float h2 = m.prune_r * m.prune_r - (gy * gy + gz * gz);
                        if (h2 < 0.f) keep = false;
                        else {
                            const float hx = sqrtf(h2) * 1.00001f;
                            const float lo = (qf.x - hx) * m.inv_cellxf - 2e-3f, hi = (qf.x + hx) * m.inv_cellxf + 2e-3f;
                            x0 = max(x0, (int)floorf(fmaxf(lo, 0.f)));
                            x1 = min(x1, (int)fminf(hi, 2.0e6f));
                        }
                    }
                    if (keep && x0 <= x1) {
                        const int row = (zz * m.ny + yy) * m.nx;
                        start = __ldg(cell_start + row + x0);
                        my_len = __ldg(cell_start + row + x1 + 1) - start;
                    }
                }
            }
            uint32_t incl = my_len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += v;
            }
            my_pre = incl - my_len;
            const unsigned nonempty = __ballot_sync(kFull, my_len > 0);
            if (my_len > 0) row_delta[__popc(nonempty & lt_mask)] = (int)start - (int)my_pre;
        }
        const uint32_t T = __shfl_sync(kFull, my_pre + my_len, 31);
        if (T > 32u * L::kMaskWords) {   // more candidates than the row-start bitmap covers: multi-kernel path
            if (lane == 0) { atomicOr(&stats->overflow, 16u); b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }
        // bitmap of the flat positions at which a row starts: one shared-memory read per round locates the rows
        for (uint32_t w = lane; w <= (T >> 5) && w < (uint32_t)L::kMaskWords; w += 32) row_mask[w] = 0;
        __syncwarp();
        if (my_len > 0) atomicOr(&row_mask[my_pre >> 5], 1u << (my_pre & 31u));
        __syncwarp();

        // ---- candidates: lanes over the flat concatenation of the rows; exact membership with the kd-tree crate's
        //      predicate (unfused FP64, as env_tile_kernel<true>) + tag rule; members ballot-compacted.
        //      The record of the next round is requested before the current one is tested.
        const double r2_safe = m.r2_safe;   // per structure (build_cells_kernel): ~40 instructions per environment less than from the anchor
        uint32_t M = 0;
        {
            int row_base = -1;   // compacted row of the last candidate of the previous round
            // flat index -> cell-sorted position: row = rows started up to my position (bitmap + popc), no search
            auto locate = [&](uint32_t i0) -> uint32_t {
                const unsigned starts = row_mask[i0 >> 5];
                const int row = row_base + __popc(starts & le_mask);
                row_base += __popc(starts);
                const uint32_t i = i0 + lane;
                return (i < T) ? (uint32_t)((int)i + row_delta[row]) : 0xFFFFFFFFu;
            };
            // one round: 32 candidates, one per lane
            // Lanes past the end of the list test the anchor's own record with `valid` false (no branch around the
            // loads or the arithmetic); members beyond CAP are not stored (the environment is rejected after the loop).
            auto test = [&](bool valid, uint32_t j, const PrimRec& r, uint32_t rtag) {
                const double ex = r.x - q.x, ey = r.y - q.y, ez = r.z - q.z;
                const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
                bool acc = valid && d2 < r2;
                // Within rounding distance of the sphere the crate's per-axis box test can still reject.  The thin
                // shell is hit by about one candidate in 1e14: a warp-uniform branch (one vote) instead of a
                // divergent region around every test.
                if (__any_sync(kFull, acc && !(d2 < r2_safe))) {
                    if (acc && !(d2 < r2_safe))
                        acc = !(r.x < q.x - threshold) && !(r.x > q.x + threshold) && !(r.y < q.y - threshold) &&
                              !(r.y > q.y + threshold) && !(r.z < q.z - threshold) && !(r.z > q.z + threshold);
                }
                if (simple_rule) acc = acc && (((rtag == qtag) == accept_same) || j == jpos);
                else if (acc && j != jpos) acc = tag_rule_accepts(p, qtag, rtag);
                const unsigned mask = __ballot_sync(kFull, acc);
                const uint32_t slot = M + __popc(mask & lt_mask);
                if (acc && slot < (uint32_t)CAP) {   // members beyond CAP are only counted: the environment is redone
                    d2s[slot] = d2;
                    cats[slot] = (uint8_t)r.cat;
                    key32[slot] = ((uint32_t)(d2 * qscale) << K::SB) | slot;
                    if (DEBUG) sidx[slot] = __ldg(s.porig + base + j);
                }
                M += __popc(mask);
            };
            // two rounds per iteration: both records are requested before either is tested
#pragma unroll 1
            for (uint32_t i0 = 0; i0 < T; i0 += 64) {
                const uint32_t l0 = locate(i0);
                const bool second = i0 + 32 < T;
                const uint32_t l1 = second ? locate(i0 + 32) : 0xFFFFFFFFu;
                const bool v0 = l0 != 0xFFFFFFFFu, v1 = l1 != 0xFFFFFFFFu;
                const uint32_t j0 = v0 ? l0 : jpos, j1 = v1 ? l1 : jpos;
                const PrimRec r0 = pd[j0];
                const PrimRec r1 = pd[j1];
                test(v0, j0, r0, r0.tag);
                if (second) test(v1, j1, r1, r1.tag);
            }
        }
        __syncwarp();
        if (M > (uint32_t)CAP) {
            if (lane == 0) { atomicOr(&stats->overflow, 8u); b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }
        if (M == 0) {   // cannot happen for r > 0 (the anchor is a member); keep the store consistent anyway
            if (lane == 0) { b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }
        // ---- sort
        bool ties;
        if (M <= 128) ties = fused_sort<4, K::SB>(key32, M, lane);
        else if (M <= 256) ties = fused_sort<8, K::SB>(key32, M, lane);
        else if (CAP == 512 || M <= 512) ties = fused_sort<16, K::SB>(key32, M, lane);
        else ties = fused_sort<CAP == 512 ? 16 : 32, K::SB>(key32, M, lane);
        if (ties) {   // equal fixed-point distances (rare): order by the exact (distance, category)
            bool viol = false;
            for (uint32_t g = lane; g + 1 < M; g += 32) {
                const uint32_t ka = key32[g], kb = key32[g + 1];
                if ((ka >> K::SB) == (kb >> K::SB)) {
                    const uint32_t sa = ka & K::kSlotMask, sb = kb & K::kSlotMask;
                    const double da = d2s[sa], db = d2s[sb];
                    viol |= (da > db) || (da == db && cats[sa] > cats[sb]);
                }
            }
            if (__any_sync(kFull, viol)) {
                if (lane == 0) fused_repair<K::SB>(key32, d2s, cats, M);
                __syncwarp();
            }
        }

        // ---- reserve the store range
        const uint32_t Mpad = (M + 1u) & ~1u;
        if (chunk_pos + Mpad > chunk_end) {
            unsigned long long got = 0;
            if (lane == 0) got = atomicAdd(&stats->cursor, (unsigned long long)kFusedChunk);
            got = __shfl_sync(kFull, got, 0);
            chunk_pos = got; chunk_end = got + kFusedChunk;
        }
        if (chunk_end > capacity) {
            if (lane == 0) { atomicOr(&stats->overflow, 1u); b.count[e] = 0; b.off_out[e] = 0; }
            continue;
        }
        const uint64_t off = chunk_pos;
        chunk_pos += Mpad;
        max_m = max(max_m, M);

        // ---- sqrt, CDF, packing, coalesced store
        uint64_t carry = 0;
        for (uint32_t g0 = 0; g0 < Mpad; g0 += 32) {
            const uint32_t g = g0 + lane;
            uint64_t packed = 0;
            if (g < M) {
                const uint32_t slot = key32[g] & K::kSlotMask;
                const double d = fused_distance<DEBUG>(d2s[slot]);   // utils.rs:1-8
                packed = pack_key(fused_weight<WFK>(wf, fwf, d, key_is_w), cats[slot]);
                if (DEBUG) { b.dist[off + g] = d; b.idx[off + g] = sidx[slot]; }
            }
            if (fix_monotone) {
                uint64_t wbits = packed & ~kCatMask;
                for (int o = 1; o < 32; o <<= 1) {
                    const uint64_t v = __shfl_up_sync(kFull, wbits, o);
                    if (lane >= o) wbits = max(wbits, v);
                }
                wbits = max(wbits, carry);
                carry = __shfl_sync(kFull, wbits, 31);
                if (g < M) packed = wbits | (packed & kCatMask);
            }
            if (g < Mpad) b.key[off + g] = packed;
        }
        if (lane == 0) { b.off_out[e] = off; b.count[e] = M; }
    }
    if (lane == 0 && max_m) atomicMax(&stats->max_count, max_m);
}

// ------------------------------------------------------------------------------------------------
// K1c: per-warp bucket sort of one environment, in place in the store.
//   (1) every member goes to a bucket that is a monotone function of its distance, (2) buckets are laid out by a
//   warp prefix sum, (3) every lane insertion-sorts a few (mostly 0-2 member) buckets; `perm` then lists the
//   members in ascending order, and they are written back with coalesced stores as packed keys:
//   f64 bits of W(d) (or of d) with the low mantissa byte replaced by the category.
// ------------------------------------------------------------------------------------------------
constexpr int kSortWarps = 4;

template <int CAP, bool DEBUG>
struct SortLayout {
    static constexpr int NB = CAP > 1024 ? 1024 : CAP;  // buckets
    static constexpr int kKeyOff = 0;                           // f64 [CAP]
    static constexpr int kIdxOff = kKeyOff + 8 * CAP;           // u32 [CAP] (DEBUG)
    static constexpr int kEndOff = kIdxOff + (DEBUG ? 4 * CAP : 0);  // u32 [NB]
    static constexpr int kBktOff = kEndOff + 4 * NB;            // u16 [CAP]
    static constexpr int kPermOff = kBktOff + 2 * CAP;          // u16 [CAP]
    static constexpr int kCatOff = kPermOff + 2 * CAP;          // u8 [CAP]
    static constexpr int kBytes = (kCatOff + CAP + 15) & ~15;
};

template <int CAP, bool DEBUG>
__global__ void __launch_bounds__(kSortWarps * 32) env_sort_kernel(KParams p, EnvBuild b, uint32_t min_m,
                                                                   double scale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using L = SortLayout<CAP, DEBUG>;
    constexpr int NB = L::NB;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint64_t e = (uint64_t)blockIdx.x * kSortWarps + wib;
    if (e >= b.n_env) return;
    const uint32_t M = b.count[e];
    if (M <= min_m || M > (uint32_t)CAP) return;
    unsigned char* smem = smem_raw + (size_t)wib * L::kBytes;
    double* key = reinterpret_cast<double*>(smem + L::kKeyOff);
    uint32_t* sidx = reinterpret_cast<uint32_t*>(smem + L::kIdxOff);
    uint32_t* bend = reinterpret_cast<uint32_t*>(smem + L::kEndOff);
    uint16_t* bkt = reinterpret_cast<uint16_t*>(smem + L::kBktOff);
    uint16_t* perm = reinterpret_cast<uint16_t*>(smem + L::kPermOff);
    uint8_t* scat = smem + L::kCatOff;
    const uint64_t off = b.off[e];
    uint64_t* gkey = b.key + off;

    // ---- load
    bool bad = false;
    double kmax = 0.0;
    for (uint32_t i = lane; i < M; i += 32) {
        const double d = __longlong_as_double((long long)gkey[i]);
        bad |= isnan(d);
        if (isfinite(d)) kmax = fmax(kmax, d);
        key[i] = d;
        scat[i] = b.cat[off + i];
        if (DEBUG) sidx[i] = b.idx[off + i];
    }
    if (__any_sync(kFull, bad)) { raise(p.err, LOCOHD_ERR_NAN); return; }  // partial_cmp().unwrap() panics (utils.rs:28)
    if (!(scale > 0.0)) {   // rows mode: bucket scale from the largest finite distance
        for (int o = 16; o; o >>= 1) kmax = fmax(kmax, __shfl_xor_sync(kFull, kmax, o));
        scale = (kmax > 0.0) ? (1.0 - 1e-9) / kmax : 0.0;
    }
    for (int q = lane; q < NB; q += 32) bend[q] = 0;
    __syncwarp();
    // ---- bucket = NB * (d * scale)^2: members of a spherical environment grow like d^2 per unit distance
    //      (keys that are already squared distances come with scale = 1 / r^2 and are used linearly)
    for (uint32_t i = lane; i < M; i += 32) {
        const float x = (float)(key[i] * scale);       // monotone in the key; NaN only for inf * 0
        const float f = (b.key_is_sq ? x : x * fabsf(x)) * (float)NB;
        int q = (int)fminf(f, (float)(NB - 1));        // fminf(NaN, y) = y: infinities land in the last bucket
        q = max(q, 0);
        bkt[i] = (uint16_t)q;
        atomicAdd(&bend[q], 1u);
    }
    __syncwarp();
    {   // exclusive prefix over the buckets, NB/32 consecutive buckets per lane; bend[q] := start of bucket q
        constexpr int PER = NB / 32;
        uint32_t sum = 0;
#pragma unroll 8
        for (int q = 0; q < PER; ++q) sum += bend[lane * PER + q];
        uint32_t incl = sum;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += v;
        }
        uint32_t run = incl - sum;
#pragma unroll 8
        for (int q = 0; q < PER; ++q) {
            const uint32_t v = bend[lane * PER + q];
            bend[lane * PER + q] = run;
            run += v;
        }
    }
    __syncwarp();
    for (uint32_t i = lane; i < M; i += 32) {   // scatter; afterwards bend[q] = end of bucket q
        const uint32_t pos = atomicAdd(&bend[bkt[i]], 1u);
        perm[pos] = (uint16_t)i;
    }
    __syncwarp();
    // ---- insertion sort inside every bucket; order = (distance, category, slot)
    for (int q = lane; q < NB; q += 32) {
        const uint32_t s0 = q ? bend[q - 1] : 0u, s1 = bend[q];
        for (uint32_t t = s0 + 1; t < s1; ++t) {
            const uint16_t en = perm[t];
            const double k = key[en];
            const uint32_t c = scat[en];
            uint32_t u = t;
            while (u > s0) {
                const uint16_t f = perm[u - 1];
                const double kf = key[f];
                const uint32_t cf = scat[f];
                if (kf < k || (kf == k && (cf < c || (cf == c && f < en)))) break;
                perm[u] = f;
                --u;
            }
            perm[u] = en;
        }
    }
    __syncwarp();
    if (b.check_first_zero && key[perm[0]] != 0.0) { raise(p.err, LOCOHD_ERR_FIRST_NOT_ZERO); return; }  // locohd.rs:74-77
    // ---- write back in ascending order (coalesced): packed keys, plus plain distances / indices for parity dumps
    const WfDev& wf = p.wfs[0];
    const bool fix_monotone = b.key_is_w && !wf.monotone;
    uint64_t carry = 0;
    for (uint32_t pos0 = 0; pos0 < M; pos0 += 32) {
        const uint32_t pos = pos0 + lane;
        uint64_t packed = 0;
        if (pos < M) {
            const uint32_t en = perm[pos];
            const double d = b.key_is_sq ? sqrt(key[en]) : key[en];   // utils.rs:1-8
            const double w = b.key_is_w ? ((d < 0.0) ? 0.0 : wf_cdf(wf, d)) : d;
            packed = pack_key(w, scat[en]);
            if (b.dist) b.dist[off + pos] = d;
            if (DEBUG) b.idx[off + pos] = sidx[en];
        }
        if (fix_monotone) {
            // pow/exp based CDFs are not guaranteed to be monotone to the last bit: keep the weights non-decreasing
            uint64_t wbits = packed & ~kCatMask;
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t v = __shfl_up_sync(kFull, wbits, o);
                if (lane >= o) wbits = max(wbits, v);
            }
            wbits = max(wbits, carry);
            carry = __shfl_sync(kFull, wbits, 31);
            packed = wbits | (packed & kCatMask);
        }
        if (pos < M) gkey[pos] = packed;
    }
}

// In-place ascending bitonic network for environments that exceed every shared-memory class (min always to the
// lower index, so the virtual +inf padding above M never moves).  One CTA per such environment.
constexpr int kBigThreads = 256;
__global__ void __launch_bounds__(kBigThreads) env_sort_big_kernel(KParams p, EnvBuild b, uint32_t min_m) {
    __shared__ unsigned long long sh_carry;
    const uint64_t e = blockIdx.x;
    const uint32_t M = b.count[e];
    if (M <= min_m) return;
    const uint64_t off = b.off[e];
    double* d = reinterpret_cast<double*>(b.key + off);
    uint8_t* c = b.cat + off;
    uint32_t* ix = b.idx ? b.idx + off : nullptr;
    bool bad = false;
    for (uint32_t i = threadIdx.x; i < M; i += kBigThreads) {
        if (b.key_is_sq) d[i] = sqrt(d[i]);
        bad |= isnan(d[i]);
    }
    if (__syncthreads_or(bad)) { if (threadIdx.x == 0) raise(p.err, LOCOHD_ERR_NAN); return; }
    uint32_t n2 = 1;
    while (n2 < M) n2 <<= 1;
    auto cex = [&](uint32_t i, uint32_t q) {
        if (q < M) {
            const double di = d[i], dq = d[q];
            const uint8_t ci = c[i], cq = c[q];
            if (dq < di || (dq == di && cq < ci)) {
                d[i] = dq; d[q] = di;
                c[i] = cq; c[q] = ci;
                if (ix) { const uint32_t u = ix[i]; ix[i] = ix[q]; ix[q] = u; }
            }
        }
    };
    for (uint32_t k = 2; k <= n2; k <<= 1) {
        const uint32_t h = k >> 1;
        for (uint32_t t = threadIdx.x; t < n2 / 2; t += kBigThreads) {
            const uint32_t i = (t / h) * k + (t % h);
            cex(i, i ^ (k - 1));
        }
        __syncthreads();
        for (uint32_t j = h >> 1; j >= 1; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < n2 / 2; t += kBigThreads) {
                const uint32_t i = (t / j) * (2 * j) + (t % j);
                cex(i, i + j);
            }
            __syncthreads();
        }
    }
    if (b.check_first_zero && d[0] != 0.0) { if (threadIdx.x == 0) raise(p.err, LOCOHD_ERR_FIRST_NOT_ZERO); return; }
    // ---- pack (sequential carry keeps non-monotone CDFs non-decreasing)
    const WfDev& wf = p.wfs[0];
    const bool fix_monotone = b.key_is_w && !wf.monotone;
    if (threadIdx.x == 0) sh_carry = 0;
    __syncthreads();
    for (uint32_t i0 = 0; i0 < M; i0 += kBigThreads) {
        const uint32_t i = i0 + threadIdx.x;
        uint64_t packed = 0;
        if (i < M) {
            const double v = d[i];
            if (b.dist) b.dist[off + i] = v;
            const double w = b.key_is_w ? ((v < 0.0) ? 0.0 : wf_cdf(wf, v)) : v;
            packed = pack_key(w, c[i]);
        }
        if (fix_monotone) {
            __shared__ unsigned long long tile[kBigThreads];
            tile[threadIdx.x] = packed & ~kCatMask;
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned long long run = sh_carry;
                for (int t = 0; t < kBigThreads; ++t) { run = max(run, tile[t]); tile[t] = run; }
                sh_carry = run;
            }
            __syncthreads();
            packed = tile[threadIdx.x] | (packed & kCatMask);
            __syncthreads();
        }
        if (i < M) b.key[off + i] = packed;
    }
}

// ------------------------------------------------------------------------------------------------
// Rows as environments (from_dmxs / from_coords): every row is copied unsorted into the store and then sorted by
// the same kernels.  Distance of point i to point j exactly as utils.rs:1-22 (the diagonal is 0).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double row_distance(const double* xyz, uint64_t i, uint64_t j) {
    if (i == j) return 0.0;
    const double ex = xyz[3 * i] - xyz[3 * j], ey = xyz[3 * i + 1] - xyz[3 * j + 1], ez = xyz[3 * i + 2] - xyz[3 * j + 2];
    return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez)));
}

// Row r starts at in_off[r] of the input and at out_off[r] of the store (ragged rows, utils.rs:25-39: row r is
// co-sorted with the first len_r categories), or, without offsets, holds row_len entries and starts at r * row_len of
// the input and at r * row_stride of the store.  With xyz the entries are the distances of point r to the points.
__global__ void rows_copy_kernel(const double* __restrict__ values, const double* __restrict__ xyz,
                                 const uint8_t* __restrict__ cat, uint64_t n_rows, uint64_t row_len,
                                 const uint64_t* __restrict__ in_off, const uint64_t* __restrict__ out_off,
                                 uint64_t* off, uint32_t* count, EnvBuild b) {
    const uint64_t row_stride = (row_len + 1) & ~1ull;
    for (uint64_t row = blockIdx.y; row < n_rows; row += gridDim.y) {
        const uint64_t i0 = in_off ? in_off[row] : row * row_len;
        const uint64_t len = in_off ? in_off[row + 1] - i0 : row_len;
        const uint64_t o0 = out_off ? out_off[row] : row * row_stride;
        if (blockIdx.x == 0 && threadIdx.x == 0) { off[row] = o0; count[row] = (uint32_t)len; }
        for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < len; j += (uint64_t)gridDim.x * blockDim.x) {
            const double d = xyz ? row_distance(xyz, row, j) : values[i0 + j];
            b.key[o0 + j] = (uint64_t)__double_as_longlong(d);
            b.cat[o0 + j] = cat[j];
            if (b.idx) b.idx[o0 + j] = (uint32_t)j;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2: scoring.  One warp per anchor pair (persistent warps stride over the pairs).
// ------------------------------------------------------------------------------------------------
// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) of one environment into a warp's stage, completion on an mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LOCOHD_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LOCOHD_DONE;\n"
        "bra LOCOHD_WAIT;\n"
        "LOCOHD_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

constexpr uint64_t kSentinel = ~0ull;   // staged behind either list of the fast kernel: above every key
constexpr int kScoreMaxWarps = 8;
// fast kernel: one large CTA per SM shares a single copy of the tables.  The W-keyed instantiations need 50 registers
// (32 warps fit the register file); the distance-keyed ones (several weight functions) need up to 72: 28 warps.
__host__ __device__ constexpr int score_fast_max_warps(bool key_is_w, bool weighted) { return weighted ? 24 : (key_is_w ? 32 : 28); }
constexpr uint64_t kWMask = ~kCatMask;

// per-lane values and counts of the generic kernel + the warp's mbarrier (16 bytes at the end)
__host__ __device__ inline int score_state_bytes(int C) { return (((2 * C * 32 * 8 + 2 * C * 32 * 4) + 15) & ~15) + 16; }
__host__ __device__ inline int fast_state_bytes(int CP) { return CP * 32 * 4 + 16; }   // counts + the warp's mbarrier
constexpr int kFastWeightBytes = 128;   // 16 category weights behind the tables of the fast kernel

struct PairEnvs {
    bool ok;
    uint64_t oa, ob;
    uint32_t Ma, Mb;
};

// Resolves pair -> (environment of A, environment of B) in explicit or job mode and validates it (warp-uniform).
__device__ __forceinline__ PairEnvs resolve_pair(const ScoreArgs& a, uint64_t pair, int* err) {
    PairEnvs r;
    r.ok = false;
    uint64_t ea, eb;
    if (a.pairs) {
        ea = a.pairs[2 * pair];
        eb = a.pairs[2 * pair + 1];
    } else {
        uint64_t job, within;
        if (a.uniform_n) {
            if (((pair | a.uniform_n) >> 32) == 0) {   // 32-bit division: ~40 instructions fewer than the 64-bit one
                const uint32_t q = (uint32_t)pair / (uint32_t)a.uniform_n;
                job = q;
                within = (uint32_t)pair - q * (uint32_t)a.uniform_n;
            } else {
                job = pair / a.uniform_n;
                within = pair - job * a.uniform_n;
            }
        } else {
            uint64_t lo = 0, hi = a.n_jobs;  // last job with job_pair_off[job] <= pair
            while (hi - lo > 1) {
                const uint64_t mid = (lo + hi) >> 1;
                if (__ldg(a.job_pair_off + mid) <= pair) lo = mid; else hi = mid;
            }
            job = lo;
            within = pair - __ldg(a.job_pair_off + job);
        }
        ea = a.jobs[job].a_first + within;
        eb = a.jobs[job].b_first + within;
    }
    if (ea >= a.a.n_env || eb >= a.b.n_env) { raise(err, LOCOHD_ERR_INDEX); return r; }
    r.oa = a.a.off[ea]; r.ob = a.b.off[eb];
    r.Ma = a.a.count[ea]; r.Mb = a.b.count[eb];
    if (r.Ma == 0 || r.Mb == 0) { raise(err, LOCOHD_ERR_EMPTY_ENV); return r; }  // locohd.rs:74 panics upstream
    r.ok = true;
    return r;
}

// merge-path split: number of A events among the first `diag` merged events (A precedes B on ties; the category
// byte does not take part in the order)
__device__ __forceinline__ uint32_t merge_path(const uint64_t* kA, const uint64_t* kB, uint32_t na, uint32_t nb,
                                               uint32_t diag) {
    uint32_t lo = diag > nb ? diag - nb : 0, hi = min(diag, na);
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if ((kA[mid] & kWMask) <= (kB[diag - 1 - mid] & kWMask)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ double key_value(uint64_t k) { return __longlong_as_double((long long)(k & kWMask)); }

// Generic kernel: any C <= 255, any statistical distance, category weights, per-pair weight functions, environments
// of any size (read from global memory when they do not fit the shared-memory stage).
template <bool HELL2>
__global__ void __launch_bounds__(kScoreMaxWarps * 32) score_kernel(ScoreArgs a, KParams P, int warps_per_block,
                                                                    int per_warp_bytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (wib >= warps_per_block) return;
    const int C = P.C;
    unsigned char* mine = smem_raw + (size_t)wib * per_warp_bytes;
    double* val = reinterpret_cast<double*>(mine);                         // [2C][32]
    uint32_t* cnt = reinterpret_cast<uint32_t*>(mine + 2 * C * 32 * 8);    // [2C][32]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(mine + score_state_bytes(C) - 16);
    uint64_t* stage = reinterpret_cast<uint64_t*>(mine + score_state_bytes(C));
    const bool key_is_w = a.a.key_is_w != 0;
    if (lane == 0) { mbar_init(mbar, 1); fence_proxy_async(); }
    __syncwarp();
    unsigned mbar_parity = 0;

    for (uint64_t pair = (uint64_t)blockIdx.x * warps_per_block + wib; pair < a.n_pairs;
         pair += (uint64_t)gridDim.x * warps_per_block) {
        __syncwarp();
        const PairEnvs pe = resolve_pair(a, pair, P.err);
        if (!pe.ok) continue;
        const uint32_t Ma = pe.Ma, Mb = pe.Mb;
        const uint32_t Ma_pad = (Ma + 1) & ~1u, Mb_pad = (Mb + 1) & ~1u;
        if (a.only_unstaged && (int)(Ma_pad + Mb_pad) <= a.only_unstaged) continue;  // the fast kernel scored it
        const uint64_t* kA = a.a.key + pe.oa;
        const uint64_t* kB = a.b.key + pe.ob;
        if ((int)(Ma_pad + Mb_pad) <= a.stage_cap) {   // staged by two TMA bulk copies, as in the fast kernel
            if (lane == 0) {
                fence_proxy_async();
                mbar_expect_tx(mbar, (Ma_pad + Mb_pad) * 8u);
                bulk_g2s(stage, kA, Ma_pad * 8u, mbar);
                bulk_g2s(stage + Ma_pad, kB, Mb_pad * 8u, mbar);
            }
            mbar_wait(mbar, mbar_parity);
            mbar_parity ^= 1u;
            kA = stage; kB = stage + Ma_pad;
        }
        const uint64_t keyA0 = kA[0], keyB0 = kB[0];
        if (!key_is_w && ((keyA0 & kWMask) != 0 || (keyB0 & kWMask) != 0)) { raise(P.err, LOCOHD_ERR_FIRST_NOT_ZERO); continue; }
        const uint32_t catA0 = (uint32_t)(keyA0 & kCatMask), catB0 = (uint32_t)(keyB0 & kCatMask);
        const uint64_t key0 = max(keyA0 & kWMask, keyB0 & kWMask);   // anchors: W(0) or distance 0
        kA += 1; kB += 1;                                            // events = members after the anchor
        const uint32_t na = Ma - 1, nb = Mb - 1;
        const uint32_t E = na + nb;
        const uint32_t Q = (E + 31) / 32;

        // ---- merge-path split: lane l owns merged events [l*Q, (l+1)*Q)
        const uint32_t diag = min(E, (uint32_t)lane * Q);
        uint32_t i = merge_path(kA, kB, na, nb, diag), j = diag - i;
        uint32_t i1 = __shfl_down_sync(kFull, i, 1), j1 = __shfl_down_sync(kFull, j, 1);
        if (lane == 31) { i1 = na; j1 = nb; }

        // ---- category counts before my chunk: per-lane histogram, then exclusive prefix over the lanes
        for (int r = 0; r < 2 * C; ++r) cnt[r * 32 + lane] = 0;
        bool unknown = (catA0 >= (uint32_t)C) || (catB0 >= (uint32_t)C);
        for (uint32_t x = i; x < i1; ++x) {
            const uint32_t c = (uint32_t)(kA[x] & kCatMask);
            if (c < (uint32_t)C) cnt[c * 32 + lane] += 1; else unknown = true;
        }
        for (uint32_t x = j; x < j1; ++x) {
            const uint32_t c = (uint32_t)(kB[x] & kCatMask);
            if (c < (uint32_t)C) cnt[(C + c) * 32 + lane] += 1; else unknown = true;
        }
        if (__any_sync(kFull, unknown)) { raise(P.err, LOCOHD_ERR_UNKNOWN_CATEGORY); continue; }  // pmf.rs:38-42
        for (int r = 0; r < 2 * C; ++r) {
            const uint32_t v = cnt[r * 32 + lane];
            uint32_t incl = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += u;
            }
            uint32_t ex = incl - v;
            if (r == (int)catA0 || r == C + (int)catB0) ex += 1;   // anchors (locohd.rs:82-84)
            cnt[r * 32 + lane] = ex;
        }

        // ---- state: HELL2 keeps sqrt(weighted count); the generalised Hellinger distance (exponent e != 2) keeps
        //      (weighted count)^(1/e), so that one event costs one root instead of 2 C; the other distances keep the
        //      weighted count itself and scale it by 1 / norm when they are evaluated
        const bool hell_e = !HELL2 && P.sd_kind == LOCOHD_SD_HELLINGER;
        const double inv_e = hell_e ? 1.0 / P.sd_p0 : 0.0;
        auto root_e = [&](double x) -> double { return x > 0.0 ? exp(inv_e * log(x)) : 0.0; };   // x^(1/e), x = w * count
        double normA = 0.0, normB = 0.0;
        uint32_t totA = 0, totB = 0;
        for (int r = 0; r < C; ++r) {
            const uint32_t ka = cnt[r * 32 + lane], kb = cnt[(C + r) * 32 + lane];
            const double w = P.cat_w[r];
            normA += (double)ka * w; normB += (double)kb * w;
            totA += ka; totB += kb;
            if (HELL2) {
                const double sw = P.cat_sw[r];
                val[r * 32 + lane] = (ka < (uint32_t)kSqrtTableSize ? __ldg(P.sqrt_tbl + ka) : sqrt((double)ka)) * sw;
                val[(C + r) * 32 + lane] = (kb < (uint32_t)kSqrtTableSize ? __ldg(P.sqrt_tbl + kb) : sqrt((double)kb)) * sw;
            } else if (hell_e) {
                val[r * 32 + lane] = root_e((double)ka * w);
                val[(C + r) * 32 + lane] = root_e((double)kb * w);
            } else {
                val[r * 32 + lane] = (double)ka * w;
                val[(C + r) * 32 + lane] = (double)kb * w;
            }
        }
        // per-side scale of the values above: norm^(-1/e) for the generalised Hellinger distance, 1 / norm otherwise
        auto side_scale = [&](double norm) -> double { return hell_e ? exp(-inv_e * log(norm)) : 1.0 / norm; };
        double iA = HELL2 ? 0.0 : side_scale(normA), iB = HELL2 ? 0.0 : side_scale(normB);
        auto inv_sqrt_norm = [&](double norm, uint32_t tot) -> double {
            if (P.unit_w && tot < (uint32_t)kSqrtTableSize) return __ldg(P.rsqrt_tbl + tot);
            return 1.0 / sqrt(norm);
        };
        double rA = HELL2 ? inv_sqrt_norm(normA, totA) : 0.0;
        double rB = HELL2 ? inv_sqrt_norm(normB, totB) : 0.0;

        auto stat_dist = [&]() -> double {
            if (HELL2) {
                // (1/2 * sum (sqrt(p_i) - sqrt(q_i))^2)^(1/2) in difference form (statistical_distances.rs:4-10, e = 2);
                // both products are rounded before the subtraction (no FMA contraction): identical compositions
                // must give exactly 0, as they do upstream
                double acc = 0.0;
                for (int r = 0; r < C; ++r) {
                    const double u = __dmul_rn(val[r * 32 + lane], rA) - __dmul_rn(val[(C + r) * 32 + lane], rB);
                    acc = fma(u, u, acc);
                }
                return sqrt(0.5 * acc);
            } else if (hell_e) {
                // (1/2 sum |p_i^(1/e) - q_i^(1/e)|^e)^(1/e) with p_i^(1/e) = (w_i a_i)^(1/e) * normA^(-1/e)
                // (statistical_distances.rs:4-10); identical compositions give exactly 0 (both sides do the same operations)
                double dist = 0.0;
                for (int r = 0; r < C; ++r) {
                    const double t = fabs(__dmul_rn(val[r * 32 + lane], iA) - __dmul_rn(val[(C + r) * 32 + lane], iB));
                    if (t > 0.0) dist += exp(P.sd_p0 * log(t));
                }
                return dist > 0.0 ? exp(inv_e * log(0.5 * dist)) : 0.0;
            } else {
                auto va = [&](int r) { return val[r * 32 + lane]; };
                auto vb = [&](int r) { return val[(C + r) * 32 + lane]; };
                return sd_scaled(P.sd_kind, P.sd_p0, P.sd_p1, C, va, vb, iA, iB);
            }
        };

        const WfDev& wf = P.wfs[a.wf_idx ? min(a.wf_idx[pair], (uint32_t)(P.n_wf - 1)) : 0u];   // range checked by validate_wf_idx_kernel
        auto weight = [&](uint64_t k) -> double { return key_is_w ? key_value(k) : wf_cdf(wf, key_value(k)); };
        uint64_t kprev = key0;
        if (i > 0) kprev = kA[i - 1] & kWMask;
        if (j > 0) kprev = max(kprev, kB[j - 1] & kWMask);
        double wprev = weight(kprev);
        double h = stat_dist();
        double acc = 0.0;

        // ---- walk my chunk
        uint64_t ra = (i < i1) ? kA[i] : 0, rb = (j < j1) ? kB[j] : 0;
        while (i < i1 || j < j1) {
            const bool takeA = (i < i1) && (!(j < j1) || (ra & kWMask) <= (rb & kWMask));
            const uint64_t raw = takeA ? ra : rb;
            const uint32_t c = (uint32_t)(raw & kCatMask);
            const double w = weight(raw);
            acc = fma(w - wprev, h, acc);
            wprev = w;
            const int row = (takeA ? 0 : C) + (int)c;
            const uint32_t k = cnt[row * 32 + lane] + 1;
            cnt[row * 32 + lane] = k;
            const double wc = P.cat_w[c];
            if (HELL2) {
                val[row * 32 + lane] = (k < (uint32_t)kSqrtTableSize ? __ldg(P.sqrt_tbl + k) : sqrt((double)k)) * P.cat_sw[c];
            } else if (hell_e) {
                val[row * 32 + lane] = root_e((double)k * wc);
            } else {
                val[row * 32 + lane] = (double)k * wc;
            }
            if (takeA) {
                normA += wc; totA += 1;
                if (HELL2) rA = inv_sqrt_norm(normA, totA); else iA = side_scale(normA);
                ++i;
                if (i < i1) ra = kA[i];
            } else {
                normB += wc; totB += 1;
                if (HELL2) rB = inv_sqrt_norm(normB, totB); else iB = side_scale(normB);
                ++j;
                if (j < j1) rb = kB[j];
            }
            h = stat_dist();
        }
        // ---- tail to infinity (locohd.rs:165-171, 204-221): owned by the last lane, whose state is final
        if (lane == 31) acc = fma(wf.w_inf - wprev, h, acc);
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
        if (lane == 0) a.out[pair] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Coordinate gradients (locohd_from_primitives_grad).  With the non-anchor members of both environments in merged
// order at distances t_1 <= ... <= t_K and H_k the statistical distance after event k,
//     S = sum_k (W(t_k) - W(t_{k-1})) H_{k-1} + (W(inf) - W(t_K)) H_K,   dS/dt_k = w(t_k) (H_{k-1} - H_k),
// so the walk of score_kernel yields the gradient without a derivative of H.  Events are merged by the exact
// distances of the keep_indices store (A before B on ties), W and w are evaluated there, and dt/dx_member =
// (x_member - x_anchor) / t = -dt/dx_anchor.  Membership changes at the threshold are not differentiated.
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline int grad_state_bytes(int C) { return ((2 * C * 32 * 8 + 2 * C * 32 * 4) + 15) & ~15; }

// merge-path split of score_kernel on exact distances
__device__ __forceinline__ uint32_t merge_path_dist(const double* dA, const double* dB, uint32_t na, uint32_t nb,
                                                    uint32_t diag) {
    uint32_t lo = diag > nb ? diag - nb : 0, hi = min(diag, na);
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (dA[mid] <= dB[diag - 1 - mid]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// The walk is the same for both targets; GradTarget decides where an event's dS/dt goes and what bounds the members'
// indices (the structure's primitives, or the row's length).
template <GradTarget T>
__global__ void __launch_bounds__(kScoreMaxWarps * 32) score_grad_kernel(GradArgs g, KParams P, int warps_per_block) {
    constexpr bool kEntries = T == GradTarget::kEntries;
    // The store that holds the B sides: the coordinate target scores the pairs of one environment set, which
    // from_primitives_grad passes as both sides, and reading it through side[0] alone keeps one set of store pointers
    // live (that instantiation's registers and spills are those of the single-set kernel it replaced).
    constexpr int kStoreB = kEntries ? 1 : 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (wib >= warps_per_block) return;
    const int C = P.C;
    unsigned char* mine = smem_raw + (size_t)wib * grad_state_bytes(C);
    double* val = reinterpret_cast<double*>(mine);                         // [2C][32]
    uint32_t* cnt = reinterpret_cast<uint32_t*>(mine + 2 * C * 32 * 8);    // [2C][32]

    for (uint64_t pair = (uint64_t)blockIdx.x * warps_per_block + wib; pair < g.n_pairs;
         pair += (uint64_t)gridDim.x * warps_per_block) {
        __syncwarp();
        const uint64_t env[2] = {g.side[0].first + pair, g.side[1].first + pair};
        uint32_t M[2];
        uint64_t off[2], sid[2], base[2], nprim[2];   // kEntries: nprim = the row's length
        uint32_t anchor[2];
        double xa[2][3];
        bool bad = false;
        for (int s = 0; s < 2; ++s) {
            off[s] = g.side[s * kStoreB].env.off[env[s]];
            M[s] = g.side[s * kStoreB].env.count[env[s]];
            if (kEntries) {
                nprim[s] = M[s];
                bad |= M[s] > 0 && g.side[s].idx[off[s]] >= M[s];
                continue;
            }
            sid[s] = g.anchor_struct[env[s]];
            const uint32_t ap = g.anchor_prim[env[s]];
            anchor[s] = ap;
            bad |= sid[s] >= g.n_structs;
            if (bad) break;
            base[s] = g.prim_off[sid[s]];
            nprim[s] = g.prim_off[sid[s] + 1] - base[s];
            bad |= ap >= nprim[s];
            if (bad) break;
            for (int k = 0; k < 3; ++k) xa[s][k] = g.xyz[3 * (base[s] + ap) + k];
        }
        if (bad) { raise(P.err, LOCOHD_ERR_INDEX); continue; }
        if (M[0] == 0 || M[1] == 0) { raise(P.err, LOCOHD_ERR_EMPTY_ENV); continue; }
        const uint64_t* kA = g.side[0].env.key + off[0] + 1;   // events = members after the anchor
        const uint64_t* kB = g.side[kStoreB].env.key + off[1] + 1;
        const double* dA = g.side[0].dist + off[0] + 1;
        const double* dB = g.side[kStoreB].dist + off[1] + 1;
        const uint32_t* xA = g.side[0].idx + off[0] + 1;
        const uint32_t* xB = g.side[kStoreB].idx + off[1] + 1;
        const uint32_t catA0 = (uint32_t)(g.side[0].env.key[off[0]] & kCatMask);
        const uint32_t catB0 = (uint32_t)(g.side[kStoreB].env.key[off[1]] & kCatMask);
        const double t0 = fmax(g.side[0].dist[off[0]], g.side[kStoreB].dist[off[1]]);
        const uint32_t na = M[0] - 1, nb = M[1] - 1;
        const uint32_t E = na + nb;
        const uint32_t Q = (E + 31) / 32;

        // ---- merge-path split: lane l owns merged events [l*Q, (l+1)*Q)
        const uint32_t diag = min(E, (uint32_t)lane * Q);
        uint32_t i = merge_path_dist(dA, dB, na, nb, diag), j = diag - i;
        uint32_t i1 = __shfl_down_sync(kFull, i, 1), j1 = __shfl_down_sync(kFull, j, 1);
        if (lane == 31) { i1 = na; j1 = nb; }

        // ---- category counts before my chunk (as in score_kernel)
        for (int r = 0; r < 2 * C; ++r) cnt[r * 32 + lane] = 0;
        bool unknown = (catA0 >= (uint32_t)C) || (catB0 >= (uint32_t)C);
        bool bad_idx = false;
        for (uint32_t x = i; x < i1; ++x) {
            const uint32_t c = (uint32_t)(kA[x] & kCatMask);
            if (c < (uint32_t)C) cnt[c * 32 + lane] += 1; else unknown = true;
            bad_idx |= xA[x] >= nprim[0];
        }
        for (uint32_t x = j; x < j1; ++x) {
            const uint32_t c = (uint32_t)(kB[x] & kCatMask);
            if (c < (uint32_t)C) cnt[(C + c) * 32 + lane] += 1; else unknown = true;
            bad_idx |= xB[x] >= nprim[1];
        }
        if (__any_sync(kFull, unknown)) { raise(P.err, LOCOHD_ERR_UNKNOWN_CATEGORY); continue; }
        if (__any_sync(kFull, bad_idx)) { raise(P.err, LOCOHD_ERR_INDEX); continue; }
        for (int r = 0; r < 2 * C; ++r) {
            const uint32_t v = cnt[r * 32 + lane];
            uint32_t incl = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += u;
            }
            uint32_t ex = incl - v;
            if (r == (int)catA0 || r == C + (int)catB0) ex += 1;   // anchors
            cnt[r * 32 + lane] = ex;
        }

        // ---- state: the Hellinger distance keeps (weighted count)^(1/e) for any exponent, the others the weighted
        //      count (score_kernel's generic branches)
        const bool hell = P.sd_kind == LOCOHD_SD_HELLINGER;
        const double inv_e = hell ? 1.0 / P.sd_p0 : 0.0;
        auto root_e = [&](double x) -> double { return x > 0.0 ? exp(inv_e * log(x)) : 0.0; };
        auto side_scale = [&](double norm) -> double { return hell ? exp(-inv_e * log(norm)) : 1.0 / norm; };
        double norm[2] = {0.0, 0.0};
        for (int r = 0; r < C; ++r) {
            const uint32_t ka = cnt[r * 32 + lane], kb = cnt[(C + r) * 32 + lane];
            const double w = P.cat_w[r];
            norm[0] += (double)ka * w; norm[1] += (double)kb * w;
            val[r * 32 + lane] = hell ? root_e((double)ka * w) : (double)ka * w;
            val[(C + r) * 32 + lane] = hell ? root_e((double)kb * w) : (double)kb * w;
        }
        double iA = side_scale(norm[0]), iB = side_scale(norm[1]);
        auto stat_dist = [&]() -> double {
            if (hell) {
                double dist = 0.0;
                for (int r = 0; r < C; ++r) {
                    const double t = fabs(__dmul_rn(val[r * 32 + lane], iA) - __dmul_rn(val[(C + r) * 32 + lane], iB));
                    if (t > 0.0) dist += exp(P.sd_p0 * log(t));
                }
                return dist > 0.0 ? exp(inv_e * log(0.5 * dist)) : 0.0;
            }
            auto va = [&](int r) { return val[r * 32 + lane]; };
            auto vb = [&](int r) { return val[(C + r) * 32 + lane]; };
            return sd_scaled(P.sd_kind, P.sd_p0, P.sd_p1, C, va, vb, iA, iB);
        };

        const WfDev& wf = P.wfs[g.wf_idx ? min(g.wf_idx[pair], (uint32_t)(P.n_wf - 1)) : 0u];   // range checked on entry
        const double gp = g.pair_weights ? g.pair_weights[pair] : 1.0;
        double tprev = t0;
        if (i > 0) tprev = dA[i - 1];
        if (j > 0) tprev = fmax(tprev, dB[j - 1]);
        double wprev = wf_cdf(wf, tprev);
        double h = stat_dist();
        double acc = 0.0;
        double ganc[2][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};   // the anchors' shares

        // ---- walk my chunk
        while (i < i1 || j < j1) {
            const bool takeA = (i < i1) && (!(j < j1) || dA[i] <= dB[j]);
            const int s = takeA ? 0 : 1;
            const uint32_t x = takeA ? i : j;
            const double t = takeA ? dA[x] : dB[x];
            const uint32_t c = (uint32_t)((takeA ? kA[x] : kB[x]) & kCatMask);
            const uint32_t m = takeA ? xA[x] : xB[x];
            const double w = wf_cdf(wf, t);
            acc = fma(w - wprev, h, acc);
            wprev = w;
            const int row = s * C + (int)c;
            const uint32_t k = cnt[row * 32 + lane] + 1;
            cnt[row * 32 + lane] = k;
            const double wc = P.cat_w[c];
            val[row * 32 + lane] = hell ? root_e((double)k * wc) : (double)k * wc;
            norm[s] += wc;
            if (takeA) { iA = side_scale(norm[0]); ++i; } else { iB = side_scale(norm[1]); ++j; }
            const double hn = stat_dist();
            if (kEntries) {
                // every entry is written: the anchor's, t = 0 and non-finite t (+inf bans) give exactly 0
                const bool live = gp != 0.0 && t > 0.0 && isfinite(t);
                g.entry_grad[s][g.entry_off[s][pair] + m] = live ? gp * wf_pdf(wf, t) * (h - hn) : 0.0;
            } else if (gp != 0.0 && t > 0.0) {   // a member on top of its anchor has no direction: it contributes 0
                const double coef = gp * wf_pdf(wf, t) * (h - hn) / t;
                double* gm = g.grad[sid[s]] + 3 * (uint64_t)m;
                const double* xm = g.xyz + 3 * (base[s] + m);
                for (int q = 0; q < 3; ++q) {
                    const double v = coef * (xm[q] - xa[s][q]);
                    atomicAdd(gm + q, v);
                    ganc[s][q] -= v;
                }
            }
            h = hn;
        }
        // ---- tail to infinity: owned by the last lane, whose state is final
        if (lane == 31) acc = fma(wf.w_inf - wprev, h, acc);
        for (int o = 16; o; o >>= 1) {
            acc += __shfl_xor_sync(kFull, acc, o);
            for (int s = 0; s < 2; ++s)
                for (int q = 0; q < 3; ++q) ganc[s][q] += __shfl_xor_sync(kFull, ganc[s][q], o);
        }
        if (lane == 0) {
            g.out[pair] = acc;
            if (kEntries) {
                for (int s = 0; s < 2; ++s) g.entry_grad[s][g.entry_off[s][pair] + g.side[s].idx[off[s]]] = 0.0;
            } else if (gp != 0.0) {
                for (int s = 0; s < 2; ++s) {
                    for (int q = 0; q < 3; ++q) atomicAdd(g.grad[sid[s]] + 3 * (uint64_t)anchor[s] + q, ganc[s][q]);
                }
            }
        }
    }
}

// Chain rule of from_coords_grad: G[i][j] = g_i dS_i/dt_ij of row i (score_grad_kernel<kEntries>), and t_ij enters
// row i and row j, so grad_i = sum_j (G[i][j] + G[j][i]) (x_i - x_j) / t_ij.  One warp per point; lane l takes
// j = l, l + 32, ... and a fixed shuffle tree sums the lanes, so the result does not depend on scheduling.  t_ij is
// recomputed as in rows_copy_kernel (row_distance(i, j) and row_distance(j, i) are bitwise equal); t = 0 contributes 0,
// as do its G entries.
__global__ void __launch_bounds__(256) coords_chain_kernel(const double* __restrict__ xyz, const double* __restrict__ G,
                                                           uint64_t n, double* __restrict__ grad) {
    const int lane = threadIdx.x & 31;
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n;
         i += ((uint64_t)gridDim.x * blockDim.x) >> 5) {
        const double xi = xyz[3 * i], yi = xyz[3 * i + 1], zi = xyz[3 * i + 2];
        double gx = 0.0, gy = 0.0, gz = 0.0;
        for (uint64_t j = lane; j < n; j += 32) {
            const double t = row_distance(xyz, i, j);
            if (!(t > 0.0)) continue;
            const double c = (G[i * n + j] + G[j * n + i]) / t;
            gx = fma(c, xi - xyz[3 * j], gx);
            gy = fma(c, yi - xyz[3 * j + 1], gy);
            gz = fma(c, zi - xyz[3 * j + 2], gz);
        }
        for (int o = 16; o; o >>= 1) {
            gx += __shfl_xor_sync(kFull, gx, o);
            gy += __shfl_xor_sync(kFull, gy, o);
            gz += __shfl_xor_sync(kFull, gz, o);
        }
        if (lane == 0) { grad[3 * i] = gx; grad[3 * i + 1] = gy; grad[3 * i + 2] = gz; }
    }
}

// Fast kernel: Hellinger-2, unit category weights, C <= CP (8 or 16), both environments staged in shared memory.
//
// With unit weights the compositions are count_r / n, so
//     H^2 = 1/2 sum_r (sqrt(a_r / nA) - sqrt(b_r / nB))^2 = 1 - D / sqrt(nA nB),   D = sum_r sqrt(a_r) sqrt(b_r),
// and one event changes a single term of D: D += (sqrt(k + 1) - sqrt(k)) * sqrt(other count of that category).
// Each lane therefore keeps (D, nA, nB, #categories whose two counts differ) in registers, the counts of a category
// share one 32-bit shared-memory word, and sqrt / delta-sqrt / rsqrt come from shared-memory tables.
// The expanded form loses digits when H^2 is tiny, so
//   * identical counts give H = 0 exactly (as upstream, and as the difference form does),
//   * H^2 < kSmallH2 (only reachable for environments of thousands of members, or proportional compositions) is
//     recomputed in the difference form sum_r (sqrt(a_r) rA - sqrt(b_r) rB)^2 from the counts,
//   * D is rebuilt from the counts at the start of every lane's chunk (at most 64 events), so rounding cannot drift.
// Error of the fast branch: |dH| <= ~5e-16 / (2 * sqrt(kSmallH2)) = 2.5e-12 (bar: 1e-9 on the score).
// With KEY_IS_W the environments already hold W(distance).  Pairs that do not fit the stage are left to score_kernel.
// (Measured and dropped in round 2, profiles/r5c_k2_lanes_per_pair.md: 16 or 8 lanes per pair, i.e. two or four pairs
//  per warp with a stage each.  The set-up is then issued once for two pairs - 1 503 instead of 1 949 warp instructions
//  and 455 instead of 523 shared-memory wavefronts per pair - but a stage per pair leaves 18 warps per SM and a warp
//  needs ~6 cycles per instruction (fixed-latency and shared-memory dependencies): issue slots 63 % busy instead of
//  82 %, 12.3 ms against 11.6 ms.)
constexpr double kSmallH2 = 1e-8;
constexpr float kSmallH2f = 1e-8f;   // the same bound, tested on (float)h2 - the seed's input (tile kernel)

// sqrt of a double in [1e-8, ~1]: MUFU.RSQ (f32) seed + one coupled Newton step in FP64, relative error
// 1.5 * 2^-44 = 8.5e-14.  Used for H itself (nothing amplifies the error; bar 1e-9 on the score); IEEE sqrt costs
// ~30 instructions per event, this one 7.
__device__ __forceinline__ double sqrt_unit(double v) {
    const double g = (double)rsqrt_approx((float)v);
    const double s0 = v * g;
    const double r = fma(-s0, 0.5 * g, 0.5);
    return fma(s0, r, s0);
}

// 2 sqrt(v) for v in [1e-8, ~1]: the seed and Newton step of sqrt_unit with the factor 1/2 left out,
// s0 (3 - g s0) = 2 sqrt(v) (1 - 1.5 e^2 + ...) for a seed g of relative error e - the same error bound, one DMUL fewer.
__device__ __forceinline__ double twice_sqrt_unit(double v) {
    const double g = (double)rsqrt_approx((float)v);
    const double s0 = v * g;
    return s0 * fma(-s0, g, 3.0);
}

// 1 / sqrt(x) for a positive, normal double: MUFU.RSQ64H seed (rsqrt.approx.f64, 2^-22 relative) and two Newton steps
// (~2e-16 relative).  Straight-line code: the library rsqrt() carries a slow path behind a call, which costs the
// weighted walk its registers.
__device__ __forceinline__ double rsqrt_pos(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x * y, y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-x * y, y, 1.0);
    return fma(0.5 * y, e, y);
}

// Shared-memory accesses by 32-bit shared-space address (walk loop of the fast kernel: no generic -> shared
// conversions, immediate offsets).  Tables and staged keys are read-only during the walk: plain asm, free to schedule;
// the count words are read-modify-written: volatile with a memory clobber.
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint64_t lds_u64(uint32_t addr) {
    uint64_t v;
    asm("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32_rmw(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u32_rmw(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// WEIGHTED: category weights other than 1 (LoCoHD(category_weights=...), pmf.rs:47-63; pisces_random_pairs.py:32-41 runs
// Hellinger-2 with such weights).  With p_r = w_r a_r / NA, NA = sum_r w_r a_r:
//     H^2 = 1 - D / sqrt(NA NB),   D = sum_r w_r sqrt(a_r) sqrt(b_r),
// so the incremental update only gains a factor w_c, and 1 / sqrt(NA) comes from rsqrt() instead of a table indexed by
// an integer total.  (Weighted counts enter as count * w; upstream adds w repeatedly: <= 1e-13, documented deviation.)
template <int CP, bool KEY_IS_W, bool WEIGHTED>
__global__ void __launch_bounds__(score_fast_max_warps(KEY_IS_W, WEIGHTED) * 32) score_fast_kernel(ScoreArgs a, KParams P, int warps_per_block,
                                                                  int per_warp_bytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int table_n = a.table_n;
    double* s_sqrt = reinterpret_cast<double*>(smem_raw);   // sqrt(k)
    double* s_dsq = s_sqrt + table_n;                       // sqrt(k + 1) - sqrt(k)   (exact: Sterbenz)
    double* s_rsqrt = s_dsq + table_n;                      // sqrt(k / (k + 1)), the factor that takes 1 / sqrt(k)
                                                            // to 1 / sqrt(k + 1)
    double* s_w = s_rsqrt + table_n;                        // [16] category weights (WEIGHTED)
    for (int k = threadIdx.x; k < table_n; k += blockDim.x) {
        const double s0 = P.sqrt_tbl[k], s1 = P.sqrt_tbl[k + 1];
        s_sqrt[k] = s0;
        s_dsq[k] = s1 - s0;
        s_rsqrt[k] = sqrt((double)k / (double)(k + 1));
    }
    if (threadIdx.x < 16) s_w[threadIdx.x] = (WEIGHTED && (int)threadIdx.x < P.C) ? P.cat_w[threadIdx.x] : 1.0;
    __syncthreads();
    if (wib >= warps_per_block) return;
    const int C = P.C;
    unsigned char* mine = smem_raw + (size_t)3 * table_n * 8 + kFastWeightBytes + (size_t)wib * per_warp_bytes;
    uint32_t* cnt = reinterpret_cast<uint32_t*>(mine);                       // [CP][32]: A count | B count << 16
    uint64_t* mbar = reinterpret_cast<uint64_t*>(mine + CP * 32 * 4);
    uint64_t* stage = reinterpret_cast<uint64_t*>(mine + fast_state_bytes(CP));
    if (lane == 0) { mbar_init(mbar, 1); fence_proxy_async(); }
    __syncwarp();
    unsigned mbar_parity = 0;
    // Shared-space addresses used by the walk.  They pass through an identity shuffle once so that ptxas keeps them
    // in registers: left alone it rematerialises them (S2R, LDC, IMAD ... ~12 instructions) in every walk iteration.
    const uint32_t sq_base = __shfl_sync(kFull, smem_u32(s_sqrt), lane);
    const uint32_t dsq_base = __shfl_sync(kFull, smem_u32(s_dsq), lane);
    const uint32_t ratio_base = __shfl_sync(kFull, smem_u32(s_rsqrt), lane);
    const uint32_t cnt_lane = __shfl_sync(kFull, smem_u32(cnt + lane), lane);
    auto sqrt_of = [&](uint32_t k) -> double { return s_sqrt[k]; };
    auto rsqrt_of = [&](uint32_t k) -> double { return __ldg(P.rsqrt_tbl + k); };   // chunk start and the small-H^2 path only

    // Work distribution: warps claim runs of kScoreRun consecutive pairs from a global cursor.  All resident warps
    // then work at one moving frontier of the pair list, so consecutive jobs that share a structure find its
    // environments in L2.  (A fixed stride per warp lets the SMs drift apart by hundreds of jobs over a launch of
    // 10^9 pairs: the ~10^2 uses of an environment spread over that many job times and it is evicted between them -
    // ncu r5h: 2.0 KB of DRAM reads per pair in job order where 1.5 KB are unavoidable.)
    uint64_t run_pos = 0, run_end = 0;
    for (;;) {
        __syncwarp();
        if (run_pos == run_end) {
            unsigned long long got = 0;
            if (lane == 0) got = atomicAdd(a.cursor, (unsigned long long)a.run);
            got = __shfl_sync(kFull, got, 0);
            if (got >= a.n_pairs) break;
            run_pos = got;
            run_end = min((uint64_t)got + a.run, a.n_pairs);
        }
        const uint64_t pair = run_pos++;
        const PairEnvs pe = resolve_pair(a, pair, P.err);
        if (!pe.ok) continue;
        const uint32_t Ma = pe.Ma, Mb = pe.Mb;
        const uint32_t Ma_pad = (Ma + 1) & ~1u, Mb_pad = (Mb + 1) & ~1u;
        if ((int)(Ma_pad + Mb_pad) > a.stage_cap) continue;   // left to the generic kernel (second pass)
        // Both environments come in as TMA bulk copies (environments start at even offsets and are padded to even
        // sizes: 16-byte granules); the warp waits on its mbarrier.  No LDG / STS instructions, no shared-memory
        // wavefronts on the LSU pipe for the staging.
        // A sentinel (all ones: above every key) follows either list in the stage, so the walk needs no bounds.
        const uint32_t Ma_st = (Ma + 2) & ~1u;   // even, >= Ma + 1: B starts behind A's sentinel
        if (lane == 0) {
            fence_proxy_async();   // the previous pair's reads of the stage come before the asynchronous writes
            mbar_expect_tx(mbar, (Ma_pad + Mb_pad) * 8u);
            bulk_g2s(stage, a.a.key + pe.oa, Ma_pad * 8u, mbar);
            bulk_g2s(stage + Ma_st, a.b.key + pe.ob, Mb_pad * 8u, mbar);
        }
        mbar_wait(mbar, mbar_parity);
        mbar_parity ^= 1u;
        if (lane == 0) { stage[Ma] = kSentinel; stage[Ma_st + Mb] = kSentinel; }
        __syncwarp();
        const uint64_t* kA = stage;
        const uint64_t* kB = stage + Ma_st;
        const uint64_t keyA0 = kA[0], keyB0 = kB[0];
        if (!KEY_IS_W && ((keyA0 & kWMask) != 0 || (keyB0 & kWMask) != 0)) { raise(P.err, LOCOHD_ERR_FIRST_NOT_ZERO); continue; }
        const uint32_t catA0 = (uint32_t)(keyA0 & kCatMask), catB0 = (uint32_t)(keyB0 & kCatMask);
        const uint64_t key0 = max(keyA0 & kWMask, keyB0 & kWMask);
        kA += 1; kB += 1;
        const uint32_t na = Ma - 1, nb = Mb - 1;
        const uint32_t E = na + nb;
        const uint32_t Q = (E + 31) / 32;
        const uint32_t diag = min(E, (uint32_t)lane * Q);
        uint32_t i = merge_path(kA, kB, na, nb, diag), j = diag - i;
        uint32_t i1 = __shfl_down_sync(kFull, i, 1), j1 = __shfl_down_sync(kFull, j, 1);
        if (lane == 31) { i1 = na; j1 = nb; }

        // ---- per-lane histogram of my chunk, exclusive prefix over the lanes, anchors added.  The chunk counts live
        //      in registers - 8-bit fields, 8 categories per 64-bit word and side; a lane owns at most 64 events - so
        //      the only shared-memory traffic of this step is the final store of the prefixes.
        constexpr int HW = CP / 8;   // 64-bit words per side
        unsigned long long hA[HW], hB[HW];
#pragma unroll
        for (int w = 0; w < HW; ++w) { hA[w] = 0; hB[w] = 0; }
        bool unknown = (catA0 >= (uint32_t)C) || (catB0 >= (uint32_t)C);
        for (uint32_t x = i; x < i1; ++x) {
            const uint32_t c = reinterpret_cast<const uint8_t*>(kA + x)[0];
            unknown |= c >= (uint32_t)C;
            const unsigned long long one = 1ull << (8u * (c & 7u));
#pragma unroll
            for (int w = 0; w < HW; ++w) hA[w] += (HW == 1 || (int)((c >> 3) & (HW - 1)) == w) ? one : 0ull;
        }
        for (uint32_t x = j; x < j1; ++x) {
            const uint32_t c = reinterpret_cast<const uint8_t*>(kB + x)[0];
            unknown |= c >= (uint32_t)C;
            const unsigned long long one = 1ull << (8u * (c & 7u));
#pragma unroll
            for (int w = 0; w < HW; ++w) hB[w] += (HW == 1 || (int)((c >> 3) & (HW - 1)) == w) ? one : 0ull;
        }
        if (__any_sync(kFull, unknown)) { raise(P.err, LOCOHD_ERR_UNKNOWN_CATEGORY); continue; }  // pmf.rs:38-42
#pragma unroll
        for (int r = 0; r < CP; ++r) {
            const uint32_t v = (uint32_t)((hA[r >> 3] >> (8 * (r & 7))) & 0xFFu) |
                               ((uint32_t)((hB[r >> 3] >> (8 * (r & 7))) & 0xFFu) << 16);
            uint32_t incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += u;
            }
            uint32_t ex = incl - v;
            if (r == (int)catA0) ex += 1u;          // anchors (locohd.rs:82-84)
            if (r == (int)catB0) ex += 0x10000u;
            cnt[r * 32 + lane] = ex;
        }

        uint32_t totA = 0, totB = 0;
        int mism = 0;
        double D = 0.0, rA = 0.0, rB = 0.0;
        double NA = 0.0, NB = 0.0;   // WEIGHTED: weighted totals
        // (re)build D, the totals and the mismatch count from the counts
        auto rebuild = [&]() {
            totA = 0; totB = 0; mism = 0; D = 0.0; NA = 0.0; NB = 0.0;
#pragma unroll
            for (int r = 0; r < CP; ++r) {
                const uint32_t word = cnt[r * 32 + lane];
                const uint32_t ka = word & 0xffffu, kb = word >> 16;
                totA += ka; totB += kb;
                mism += (ka != kb) ? 1 : 0;
                if (WEIGHTED) {
                    const double w = s_w[r];
                    NA = fma(w, (double)ka, NA); NB = fma(w, (double)kb, NB);
                    D = fma(w * sqrt_of(ka), sqrt_of(kb), D);
                } else {
                    D = fma(sqrt_of(ka), sqrt_of(kb), D);
                }
            }
            if (WEIGHTED) { rA = rsqrt_pos(NA); rB = rsqrt_pos(NB); }
            else { rA = rsqrt_of(totA); rB = rsqrt_of(totB); }
        };
        // difference form from the counts (small H^2 only)
        auto exact_h2 = [&]() -> double {
            double acc = 0.0;
#pragma unroll
            for (int r = 0; r < CP; ++r) {
                const uint32_t word = cnt[r * 32 + lane];
                const double u = __dmul_rn(sqrt_of(word & 0xffffu), rA) - __dmul_rn(sqrt_of(word >> 16), rB);
                acc = WEIGHTED ? fma(s_w[r] * u, u, acc) : fma(u, u, acc);
            }
            return 0.5 * acc;
        };
        auto stat_dist = [&]() -> double {
            if (mism == 0) return 0.0;                       // identical counts: exactly 0
            const double h2 = fma(-__dmul_rn(rA, rB), D, 1.0);
            if (h2 < kSmallH2) return sqrt(exact_h2());
            return sqrt_unit(h2);
        };
        rebuild();

        const WfDev& wf = P.wfs[(!KEY_IS_W && a.wf_idx) ? min(a.wf_idx[pair], (uint32_t)(P.n_wf - 1)) : 0u];
        auto weight = [&](uint64_t k) -> double { return KEY_IS_W ? key_value(k) : wf_cdf(wf, key_value(k)); };
        uint64_t kprev = key0;
        if (i > 0) kprev = kA[i - 1] & kWMask;
        if (j > 0) kprev = max(kprev, kB[j - 1] & kWMask);
        double wprev = weight(kprev);
        double h = stat_dist();
        double acc = 0.0;

        // The first nev events of the merge that starts at (i, j) are exactly my chunk (same comparison as the
        // merge-path split: A before B on ties); the sentinels end the lists.
        const uint32_t nev = (i1 - i) + (j1 - j);
        // The tables cover every count (launch_score sizes them to the stage).  Per-lane state: shared-space addresses
        // of the next key of either list (pa, pb); the index into the ratio table advances in step with them, so it is
        // a constant offset (dA, dB) from the key address; R = rA * rB is carried as a product and updated by one table
        // factor (<= 64 events per chunk: <= 64 roundings, ~1e-14 relative - H >= 1e-4 here, bar 1e-9).
        uint32_t pa = smem_u32(kA + i), pb = smem_u32(kB + j);
        const uint32_t dA = ratio_base + 8u * totA - pa, dB = ratio_base + 8u * totB - pb;
        double R = __dmul_rn(rA, rB);
        uint64_t ra = lds_u64(pa), rb = lds_u64(pb);
        for (uint32_t it = 0; it < nev; ++it) {   // (unrolled by 2: 5.58 -> 5.60 ms on config 2, profiles/r6z - this kernel sits on the shared-memory pipe)
            const bool takeA = ra <= (rb | kCatMask);   // == (ra & kWMask) <= (rb & kWMask)
            const uint64_t raw = takeA ? ra : rb;
            const double w = weight(raw);
            acc = fma(w - wprev, h, acc);
            wprev = w;
            uint32_t ca;   // cnt_lane + category * 128 (one IMAD; the compiler's shift + mask + add are three)
            asm("mad.lo.u32 %0, %1, 128, %2;" : "=r"(ca) : "r"((uint32_t)raw & 0xFFu), "r"(cnt_lane));
            const uint32_t word = lds_u32_rmw(ca);
            const uint32_t ka = word & 0xffffu, kb = word >> 16;
            const uint32_t mine_k = takeA ? ka : kb, other_k = takeA ? kb : ka;
            sts_u32_rmw(ca, word + (takeA ? 1u : 0x10000u));
            mism += (mine_k == other_k ? 1 : 0) - (mine_k + 1u == other_k ? 1 : 0);
            const uint32_t pk = takeA ? pa : pb;
            if (WEIGHTED) {
                const double wc = s_w[(uint32_t)raw & 0xFFu];
                D = fma(wc * lds_f64(dsq_base + 8u * mine_k), lds_f64(sq_base + 8u * other_k), D);
                NA += takeA ? wc : 0.0;
                NB += takeA ? 0.0 : wc;
                const double rnew = rsqrt_pos(takeA ? NA : NB);
                rA = takeA ? rnew : rA;
                rB = takeA ? rB : rnew;
                R = rA * rB;
            } else {
                D = fma(lds_f64(dsq_base + 8u * mine_k), lds_f64(sq_base + 8u * other_k), D);
                R *= lds_f64(pk + (takeA ? dA : dB));
            }
            const uint64_t nxt = lds_u64(pk + 8u);
            pa = takeA ? pk + 8u : pa;
            pb = takeA ? pb : pk + 8u;
            ra = takeA ? nxt : ra;
            rb = takeA ? rb : nxt;
            const double h2 = fma(-R, D, 1.0);
            // (measured and dropped, profiles/r4d: sum |a_r - b_r| instead of the mismatch count and an integer test
            //  of h2's high word - fewer instructions, 1-2 % slower: the kernel is bound by the shared-memory pipe)
            h = (mism == 0) ? 0.0 : sqrt_unit(h2);       // identical counts: exactly 0
            if (mism != 0 && h2 < kSmallH2) {            // rare: difference form from the counts
                if (!WEIGHTED) {
                    rA = rsqrt_of((pa + dA - ratio_base) >> 3);
                    rB = rsqrt_of((pb + dB - ratio_base) >> 3);
                }
                h = sqrt(exact_h2());
            }
        }
        if (lane == 31) acc = fma(wf.w_inf - wprev, h, acc);
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
        if (lane == 0) a.out[pair] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Tile kernel: the all-vs-all ensemble (compare_ensembles.py:250-296) and every other job list in which runs of
// environments meet several partners.  Unit of work = (tile, anchor): the <= 4 environments of env-set A and <= 4 of
// env-set B that the tile's jobs use at this anchor are staged ONCE (<= 8 bulk copies on one mbarrier) and scored as
// <= 16 anchor pairs by a team of 4 warps - warp r owns row r, 8 lanes per pair.  Against one pair per warp:
//   * 0.5 instead of 2 staged environments per pair: a quarter of the L2 -> shared-memory traffic, and 8 teams
//     (32 warps) still fit one SM although four pairs share a warp (a stage per pair leaves 9 warps, profiles/r5c);
//   * the straight-line set-up of a pair (merge-path split, prefix scans, D from the counts, reduction: ~1 000 of the
//     1 860 warp instructions of score_fast_kernel) is issued once for four pairs; prefix scans and the reduction
//     take 3 shuffle steps instead of 5.
// The arithmetic per event is that of score_fast_kernel<CP, true, false> (same tables, same expanded form, same
// small-H^2 fallback, exact 0 for identical counts); a lane's chunk is E / 8 events instead of E / 32 (the host caps
// E at 1024: <= 128 roundings of R and D per chunk, ~3e-14 relative).  One CTA per SM (tables staged once), teams
// synchronise on named barriers.  The walk is bound by its instruction count (profiles/r6w, r6x, r7a), so its event is
// kept short (49 SASS instructions in <8, true>, profiles/r11a_tile_walk.md): count words hold 8 count (the table
// offset, one add-min per look-up), identical compositions are found from sum |a_r - b_r| inside the small-H^2 branch
// only, and the walk carries 2 H (twice_sqrt_unit).
// ncu (profiles/r6b): 1 214 warp instructions and 375 shared-memory wavefronts per pair (1 949 / 523 for one pair per
// warp); the shared-memory data pipe is 92 % busy and is the wall - 245 of the 375 wavefronts are the four scattered
// 8-byte reads of the walk (next key 73, ratio table 70, the two sqrt tables 51 each; a half-warp of 14 active lanes
// into 16 bank pairs takes ~2.7 wavefronts where 1 is ideal).
// Measured and dropped on this kernel (profiles/r6c): R = 1 / sqrt(nA nB) by MUFU.RSQ + one Newton step instead of
// the ratio-table read (-70 wavefronts, +7 instructions per event and a longer dependent chain: 136.6 -> 141.5 ms on
// the 200-structure ensemble); lanes dealt to the four pairs of a row in proportion to their event counts (12 % fewer
// walk iterations per warp, but the wavefronts follow the lane-events, not the iterations: 137.6 -> 140.6 ms);
// 7 / 6 teams per SM run 1.3 % / 4.4 % slower than 8; cp.async.bulk.prefetch.L2 of the next unit's environments one unit
// ahead (134.0 -> 136.2 ms, profiles/r6o).
constexpr int kTileLanes = 8;                          // lanes per anchor pair
constexpr int kTeamThreads = kTileDim * kTileDim * kTileLanes;   // 128: warp r = row r, lane >> 3 = column
constexpr int kTileMaxTeams = 8;
constexpr int kTileCtrlBytes = 128;
constexpr int kTileRepMax = 64;                        // at most this many table entries are replicated per bank pair
constexpr int kTileRun = 8;                            // consecutive units (anchors of one tile) a team claims at once
static_assert(kTeamThreads == 128 && kTileLanes * kTileDim == 32, "a warp covers one row of the tile");
__host__ __device__ inline int tile_team_bytes(int CP, int stage_keys) {
    return CP * kTeamThreads * 4 + kTileCtrlBytes + stage_keys * 8;
}

struct TileCtrl {         // written by the team's loader warp between the two team barriers of an iteration
    uint64_t mbar;
    uint32_t tile[2];     // tile and anchor (inside the jobs of the tile) of the current unit and of the next one:
    uint32_t p[2];        // written by fetch() one iteration ahead, slot = iteration & 1
    uint32_t state;       // 0 = score, 1 = skip (an error was raised), 2 = no units left
    uint32_t pad;
    uint32_t start[2 * kTileDim];   // stage position of rows 0..3, columns 0..3
    uint32_t M[2 * kTileDim];       // their sizes (0: absent)
};
static_assert(sizeof(TileCtrl) <= kTileCtrlBytes, "control block");

__device__ __forceinline__ void team_barrier(int team) {
    asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(kTeamThreads) : "memory");
}

template <int CP, bool REP>
__global__ void __launch_bounds__(kTileMaxTeams * kTeamThreads, 1) score_tile_kernel(ScoreArgs a, KParams P, int teams,
                                                                                      int team_bytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int table_n = a.table_n;
    // Tables.  The two count-indexed ones (sqrt(k), sqrt(k + 1) - sqrt(k)) are "mixed" when REP: entries k < rep_n
    // exist once per bank pair (entry k of copy c at word 16 k + c; lane l reads copy l & 15, so these reads are
    // conflict-free whatever the counts of the 32 lanes are: 2 wavefronts per warp read instead of 3.8), the entries
    // from rep_n on follow unreplicated.  Word index of entry k for copy c: k + min(15 k + c, 15 rep_n) - one IMAD,
    // one min and one add, no branch.  The host picks rep_n from the shared memory the teams leave over.
    const int rep_n = REP ? a.rep_n : 0;
    const int mix_n = 15 * rep_n + table_n;
    double* s_ratio = reinterpret_cast<double*>(smem_raw);   // sqrt(k / (k + 1)), indexed by a side's total
    double* s_sqrt = s_ratio + table_n;                      // sqrt(k)
    double* s_dsq = s_sqrt + mix_n;                          // sqrt(k + 1) - sqrt(k)   (exact: Sterbenz)
    for (int x = threadIdx.x; x < table_n; x += blockDim.x) s_ratio[x] = sqrt((double)x / (double)(x + 1));
    for (int x = threadIdx.x; x < mix_n; x += blockDim.x) {
        const int e = x < 16 * rep_n ? x >> 4 : x - 15 * rep_n;
        const double s0 = P.sqrt_tbl[e], s1 = P.sqrt_tbl[e + 1];
        s_sqrt[x] = s0;
        s_dsq[x] = s1 - s0;
    }
    __syncthreads();
    const int team = wib >> 2, row = wib & 3;
    if (team >= teams) return;
    const int C = P.C;
    unsigned char* mine = smem_raw + (size_t)(table_n + 2 * mix_n) * 8 + (size_t)team * team_bytes;
    uint32_t* cnt = reinterpret_cast<uint32_t*>(mine) + row * CP * 32;   // [CP][32] per warp: 8 A | 8 B << 16 (8 count:
                                                                         // the byte offset of the count's table entry)
    TileCtrl* ctrl = reinterpret_cast<TileCtrl*>(mine + CP * kTeamThreads * 4);
    uint64_t* stage = reinterpret_cast<uint64_t*>(mine + CP * kTeamThreads * 4 + kTileCtrlBytes);
    const bool loader = row == 0;
    if (loader && lane == 0) { mbar_init(&ctrl->mbar, 1); fence_proxy_async(); }
    unsigned flags = 0;   // bit 0: parity of the team's mbarrier, bit 1: control-block slot of the NEXT fetch
    const uint32_t sq_base = __shfl_sync(kFull, smem_u32(s_sqrt), lane);
    const uint32_t dsq_base = __shfl_sync(kFull, smem_u32(s_dsq), lane);
    const uint32_t ratio_base = __shfl_sync(kFull, smem_u32(s_ratio), lane);
    const uint32_t cnt_lane = __shfl_sync(kFull, smem_u32(cnt + lane), lane);
    // shared-space address of entry e of a count-indexed table, from e8 = 8 e (the count words hold 8 count):
    // base + 8 e + min(120 e + 8 copy, 120 rep_n) = min(16 e8 + base + 8 copy, e8 + base + 120 rep_n) - one shift-add
    // and one add-min (VIADDMNMX) per look-up
    const uint32_t copy8 = 8u * (lane & 15), cap8 = 120u * (uint32_t)rep_n;
    const uint32_t sq_copy = __shfl_sync(kFull, sq_base + copy8, lane), sq_cap = __shfl_sync(kFull, sq_base + cap8, lane);
    const uint32_t dsq_copy = __shfl_sync(kFull, dsq_base + copy8, lane), dsq_cap = __shfl_sync(kFull, dsq_base + cap8, lane);
    auto sq_addr = [&](uint32_t e8) -> uint32_t { return REP ? min(16u * e8 + sq_copy, e8 + sq_cap) : sq_base + e8; };
    auto dsq_addr = [&](uint32_t e8) -> uint32_t { return REP ? min(16u * e8 + dsq_copy, e8 + dsq_cap) : dsq_base + e8; };
    // warp = row of the tile, 8 lanes per column.  (Measured and dropped, profiles/r6p: warp w scoring the pairs
    // (r, (r + w) mod 4) - a Latin square, equal event totals for the four warps, where ncu shows 19.6 % of the warp time
    // in the team barrier waiting for the row with the largest A_r - 134.9 -> 139.5 ms: the 32 lanes of a row share
    // one A list, lanes at the same place of their chunks read the same or neighbouring words.)
    // Lane order: the column is the fast index (lane = 4 chunk + column): the four lanes that sit at the same place of
    // their chunks of the shared A list are neighbours in one half-warp and read the same or adjacent words (keys of
    // A, ratio-table entries).  Against lane = 8 column + chunk: 134.7 -> 133.8 ms (profiles/r6q).
    constexpr int lstep = kTileDim;   // lane distance between consecutive chunks of a pair
    const int sub = lane >> 2;
    const int prow = row, pcol = lane & (kTileDim - 1);
    const uint64_t n = a.uniform_n, n_units = a.n_tiles * n;
    const WfDev& wf = P.wfs[0];

    // Loader lanes 0..7 of warp 0 hold the descriptor of the NEXT unit: it is fetched one iteration ahead, right
    // after the team was released into the current unit, so the loads (tile -> offset, size, an odd last member) run
    // under the scoring of the current unit.  Units are claimed in runs of kTileRun consecutive anchors with one
    // atomicAdd: the descriptors of a run share their cache lines, and the teams of all SMs still work at one
    // moving frontier of the unit list.
    uint64_t run_pos = 0, run_end = 0;   // loader warp, uniform
    uint64_t nx_unit = 0, nx_off = 0, nx_last = 0;
    uint32_t nx_M = 0;
    bool nx_present = false;
    auto fetch = [&]() {
        if (run_pos == run_end) {
            unsigned long long got = 0;
            if (lane == 0) got = atomicAdd(a.cursor, (unsigned long long)a.run);
            got = __shfl_sync(kFull, got, 0);
            run_pos = min((uint64_t)got, n_units);
            run_end = min((uint64_t)got + a.run, n_units);
        }
        const uint64_t u = run_pos;
        if (run_pos < run_end) ++run_pos;
        nx_unit = u; nx_off = 0; nx_M = 0; nx_last = 0; nx_present = false;
        if (u < n_units && lane < 2 * kTileDim) {
            uint64_t tile, p;
            // unit -> (tile, anchor) in the sliced order (TileOrder, locohd_kernels.cuh); the team reads them from the
            // control block's slot of the unit's iteration (two slots: this fetch runs while the current unit is scored)
            if (((n_units | n) >> 32) == 0) { uint32_t t32, p32; tile_unit<uint32_t>(a.order, (uint32_t)u, &t32, &p32); tile = t32; p = p32; }
            else tile_unit<uint64_t>(a.order, u, &tile, &p);
            if (lane == 0) { ctrl->tile[(flags >> 1) & 1u] = (uint32_t)tile; ctrl->p[(flags >> 1) & 1u] = (uint32_t)p; }
            const ScoreTile& T = a.tiles[tile];
            const uint64_t first = lane < kTileDim ? __ldg(T.a_first + lane) : __ldg(T.b_first + (lane - kTileDim));
            if (first != kTileNone) {
                const EnvView& v = lane < kTileDim ? a.a : a.b;
                nx_off = __ldg(v.off + first + p);
                nx_M = __ldg(v.count + first + p);
                if (nx_M & 1u) nx_last = __ldg(v.key + nx_off + nx_M - 1);
                nx_present = true;
            }
        }
    };
    if (loader) fetch();

    for (;;) {
        const uint32_t slot = (flags >> 1) & 1u;   // where fetch() left this unit's tile and anchor
        flags ^= 2u;
        team_barrier(team);   // every warp of the team is done with the stage of the previous unit
        if (loader) {
            const uint64_t u = nx_unit;
            uint32_t state = 0;
            if (u >= n_units) state = 2;
            else {
                if (__any_sync(kFull, nx_present && nx_M == 0)) { raise(P.err, LOCOHD_ERR_EMPTY_ENV); state = 1; }  // locohd.rs:74 panics upstream
                // slot of an environment: its members, the sentinel, padded to an even number of keys
                const uint32_t slot = nx_present ? ((nx_M + 2u) & ~1u) : 0u;
                uint32_t incl = slot;
#pragma unroll
                for (int o = 1; o < 2 * kTileDim; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(kFull, incl, o);
                    if (lane >= o) incl += t;
                }
                const uint32_t start = incl - slot;
                // The even part of an environment comes as one bulk copy (16-byte granules); an odd last member was
                // fetched with the descriptor and is stored by hand, so the sentinel behind it is never overwritten
                // by the copy.
                const uint32_t bytes = (state == 0 && nx_present) ? (nx_M & ~1u) * 8u : 0u;
                uint32_t total = bytes;
#pragma unroll
                for (int o = 1; o < 2 * kTileDim; o <<= 1) total += __shfl_xor_sync(kFull, total, o);
                if (state == 0) {
                    const EnvView& v = lane < kTileDim ? a.a : a.b;
                    if (lane == 0) { fence_proxy_async(); mbar_expect_tx(&ctrl->mbar, total); }
                    __syncwarp();
                    if (lane < 2 * kTileDim && nx_present) {
                        if (bytes) { fence_proxy_async(); bulk_g2s(stage + start, v.key + nx_off, bytes, &ctrl->mbar); }
                        if (nx_M & 1u) stage[start + nx_M - 1] = nx_last;
                        stage[start + nx_M] = kSentinel;
                    }
                }
                if (lane < 2 * kTileDim) { ctrl->start[lane] = start; ctrl->M[lane] = (state == 0 && nx_present) ? nx_M : 0u; }
            }
            if (lane == 0) ctrl->state = state;
        }
        team_barrier(team);   // descriptor, hand-copied members and sentinels are visible
        const uint32_t state = ctrl->state;
        if (state == 2) break;
        if (loader) fetch();
        if (state == 1) continue;
        const uint64_t out_first = __ldg(a.tiles[ctrl->tile[slot]].out_first + prow * kTileDim + pcol);
        const uint32_t Ma = ctrl->M[prow], Mb = ctrl->M[kTileDim + pcol];
        const uint32_t p = ctrl->p[slot];
        const bool valid = out_first != kTileNone && Ma != 0 && Mb != 0;
        const uint64_t* kA = stage + (valid ? ctrl->start[prow] : 0u);
        const uint64_t* kB = stage + (valid ? ctrl->start[kTileDim + pcol] : 0u);
        mbar_wait(&ctrl->mbar, flags & 1u);
        flags ^= 1u;
        if (!__any_sync(kFull, valid)) continue;

        const uint64_t keyA0 = kA[0], keyB0 = kB[0];
        const uint32_t catA0 = (uint32_t)(keyA0 & kCatMask), catB0 = (uint32_t)(keyB0 & kCatMask);
        const uint64_t key0 = max(keyA0 & kWMask, keyB0 & kWMask);
        kA += 1; kB += 1;
        const uint32_t na = valid ? Ma - 1 : 0u, nb = valid ? Mb - 1 : 0u;
        const uint32_t E = na + nb;
        const uint32_t Q = (E + kTileLanes - 1) / kTileLanes;
        const uint32_t diag = min(E, (uint32_t)sub * Q);
        const uint32_t i = merge_path(kA, kB, na, nb, diag), j = diag - i;
        uint32_t i1 = __shfl_down_sync(kFull, i, lstep), j1 = __shfl_down_sync(kFull, j, lstep);
        if (sub == kTileLanes - 1) { i1 = na; j1 = nb; }

        // per-lane histogram of my chunk (8-bit fields: a chunk has at most 128 events), exclusive prefix over the 8
        // lanes of the pair, anchors added; D and sum_r |a_r - b_r| are built from the prefixes while they are in
        // registers
        constexpr int HW = CP / 8;
        unsigned long long hA[HW], hB[HW];
#pragma unroll
        for (int w = 0; w < HW; ++w) { hA[w] = 0; hB[w] = 0; }
        bool unknown = valid && ((catA0 >= (uint32_t)C) || (catB0 >= (uint32_t)C));
        if constexpr (HW == 1) {
            // No test per event: the increment of a category >= 8 is shifted out of the word (shl.b64 clamps the shift
            // amount), one in [C, 8) lands in a field that has to stay empty - both are found after the loops, from the
            // sum of the fields (<= 128 events per chunk: no carry between them) and the fields from C on.
            auto bump = [](unsigned long long& hh, uint32_t c) {
                unsigned long long one;
                asm("shl.b64 %0, %1, %2;" : "=l"(one) : "l"(1ull), "r"(8u * c));
                hh += one;
            };
            for (uint32_t x = i; x < i1; ++x) bump(hA[0], reinterpret_cast<const uint8_t*>(kA + x)[0]);
            for (uint32_t x = j; x < j1; ++x) bump(hB[0], reinterpret_cast<const uint8_t*>(kB + x)[0]);
            const unsigned long long hs = hA[0] + hB[0];
            const uint32_t counted = (uint32_t)((hs * 0x0101010101010101ull) >> 56);
            unknown |= counted != (i1 - i) + (j1 - j);
            unknown |= C < 8 && (hs >> (8 * C)) != 0ull;
        } else {
            for (uint32_t x = i; x < i1; ++x) {
                const uint32_t c = reinterpret_cast<const uint8_t*>(kA + x)[0];
                unknown |= c >= (uint32_t)C;
                const unsigned long long one = 1ull << (8u * (c & 7u));
#pragma unroll
                for (int w = 0; w < HW; ++w) hA[w] += ((int)((c >> 3) & (HW - 1)) == w) ? one : 0ull;
            }
            for (uint32_t x = j; x < j1; ++x) {
                const uint32_t c = reinterpret_cast<const uint8_t*>(kB + x)[0];
                unknown |= c >= (uint32_t)C;
                const unsigned long long one = 1ull << (8u * (c & 7u));
#pragma unroll
                for (int w = 0; w < HW; ++w) hB[w] += ((int)((c >> 3) & (HW - 1)) == w) ? one : 0ull;
            }
        }
        if (__any_sync(kFull, unknown)) { raise(P.err, LOCOHD_ERR_UNKNOWN_CATEGORY); continue; }  // pmf.rs:38-42
        uint32_t l1 = 0;   // sum_r |a_r - b_r|: 0 <=> identical compositions
        double D = 0.0;
#pragma unroll
        for (int r = 0; r < CP; ++r) {
            const uint32_t v = (uint32_t)((hA[r >> 3] >> (8 * (r & 7))) & 0xFFu) |
                               ((uint32_t)((hB[r >> 3] >> (8 * (r & 7))) & 0xFFu) << 16);
            uint32_t incl = v;
#pragma unroll
            for (int o = 1; o < kTileLanes; o <<= 1) {
                const uint32_t u = __shfl_up_sync(kFull, incl, o * lstep);
                if (sub >= o) incl += u;
            }
            uint32_t ex = incl - v;
            if (r == (int)catA0) ex += 1u;          // anchors (locohd.rs:82-84)
            if (r == (int)catB0) ex += 0x10000u;
            cnt[r * 32 + lane] = 8u * ex;   // <= 1024 members a side (tile_geometry): 8 count fits 16 bits
            const uint32_t ka = ex & 0xffffu, kb = ex >> 16;
            l1 += ka > kb ? ka - kb : kb - ka;
            D = fma(lds_f64(sq_addr(8u * ka)), lds_f64(sq_addr(8u * kb)), D);
        }
        const uint32_t totA = i + 1u, totB = j + 1u;   // members of either side before my chunk, anchors included
        double rA = __ldg(P.rsqrt_tbl + totA), rB = __ldg(P.rsqrt_tbl + totB);
        // 4 H^2 in the difference form from the counts (small H^2 only)
        auto exact_4h2 = [&]() -> double {
            double s = 0.0;
#pragma unroll
            for (int r = 0; r < CP; ++r) {
                const uint32_t word = cnt[r * 32 + lane];
                const double u = __dmul_rn(lds_f64(sq_addr(word & 0xffffu)), rA) - __dmul_rn(lds_f64(sq_addr(word >> 16)), rB);
                s = fma(u, u, s);
            }
            return 2.0 * s;
        };
        uint64_t kprev = key0;
        if (i > 0) kprev = kA[i - 1] & kWMask;
        if (j > 0) kprev = max(kprev, kB[j - 1] & kWMask);
        double wprev = key_value(kprev);
        double R = __dmul_rn(rA, rB);
        // The walk carries h = 2 H (twice_sqrt_unit saves a multiply per event) and halves the sum at the end: scaling
        // by 2 is exact, the sum is the one of H itself.
        double h;
        {
            const double h2 = fma(-R, D, 1.0);
            h = (l1 == 0) ? 0.0 : (h2 < kSmallH2 ? sqrt(exact_4h2()) : twice_sqrt_unit(h2));
        }
        double acc = 0.0;
        const uint32_t nev = (i1 - i) + (j1 - j);
        uint32_t pa = smem_u32(kA + i), pb = smem_u32(kB + j);
        const uint32_t dA = ratio_base + 8u * totA - pa, dB = ratio_base + 8u * totB - pb;
        uint64_t ra = lds_u64(pa), rb = lds_u64(pb);
        // Identical compositions: an event moves sum_r |a_r - b_r| by +1 (my count of the category was >= the other
        // side's) or -1, so after k events the sum is l1 - k + 2 #{events with mine >= other}.  The walk keeps
        // m = l1 - 1 + 2 #{...} (one predicated add per event) and compares only where H^2 is tiny: there, after the
        // event taken with `left` events to go (k = nev - left + 1), m + left == nev <=> identical <=> H = 0 exactly.
        // Identical compositions are frequent in ensembles of near-copies; their h2 is a rounding residue below 1e-8,
        // so they take the branch of the small-H^2 case instead of a test and a select on every event (6 -> 2
        // instructions of bookkeeping per event against the count of differing categories).
        uint32_t m = l1 - 1u;
        // unrolled by 2: no register rotation of the carried key / weight and half the loop overhead, 130.8 -> 126.9 ms
        // on the 200-structure ensemble (profiles/r6x); by 4: 128.7 ms (profiles/r6y)
#pragma unroll 2
        for (uint32_t left = nev; left != 0; --left) {
            const bool takeA = ra <= (rb | kCatMask);   // == (ra & kWMask) <= (rb & kWMask)
            const uint64_t raw = takeA ? ra : rb;
            const double w = key_value(raw);
            acc = fma(w - wprev, h, acc);
            wprev = w;
            uint32_t ca;   // cnt_lane + category * 128
            asm("mad.lo.u32 %0, %1, 128, %2;" : "=r"(ca) : "r"((uint32_t)raw & 0xFFu), "r"(cnt_lane));
            const uint32_t word = lds_u32_rmw(ca);
            const uint32_t ka = word & 0xffffu, kb = word >> 16;
            const uint32_t mine_k = takeA ? ka : kb, other_k = takeA ? kb : ka;
            sts_u32_rmw(ca, word + (takeA ? 8u : 0x80000u));
            // a predicated add in place (left to itself, ptxas adds into a new register and selects: two instructions)
            asm("{\n\t.reg .pred p;\n\tsetp.ge.u32 p, %1, %2;\n\t@p add.u32 %0, %0, 2;\n\t}" : "+r"(m) : "r"(mine_k), "r"(other_k));
            const uint32_t pk = takeA ? pa : pb;
            D = fma(lds_f64(dsq_addr(mine_k)), lds_f64(sq_addr(other_k)), D);
            R *= lds_f64(pk + (takeA ? dA : dB));
            const uint64_t nxt = lds_u64(pk + 8u);
            pa = takeA ? pk + 8u : pa;
            pb = takeA ? pb : pk + 8u;
            ra = takeA ? nxt : ra;
            rb = takeA ? rb : nxt;
            const double h2 = fma(-R, D, 1.0);
            h = twice_sqrt_unit(h2);
            if ((float)h2 < kSmallH2f) {   // h2 < 1e-8 (or negative): identical counts (exactly 0) or rare (difference form)
                if (m + left == nev) {
                    h = 0.0;
                } else {
                    rA = __ldg(P.rsqrt_tbl + ((pa + dA - ratio_base) >> 3));
                    rB = __ldg(P.rsqrt_tbl + ((pb + dB - ratio_base) >> 3));
                    h = sqrt(exact_4h2());
                }
            }
        }
        if (sub == kTileLanes - 1) acc = fma(wf.w_inf - wprev, h, acc);   // tail to infinity: the last chunk's state is final
#pragma unroll
        for (int o = kTileLanes / 2; o; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o * lstep);
        if (sub == 0 && valid) a.out[out_first + p] = 0.5 * acc;
    }
}

__global__ void job_means_kernel(const double* __restrict__ scores, const uint64_t* __restrict__ job_pair_off,
                                 uint64_t n_jobs, double* __restrict__ means) {
    const int lane = threadIdx.x & 31;
    const uint64_t job = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (job >= n_jobs) return;
    const uint64_t b = job_pair_off[job], e = job_pair_off[job + 1];
    double s = 0.0;
    for (uint64_t i = b + lane; i < e; i += 32) s += scores[i];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
    if (lane == 0) means[job] = (e > b) ? s / (double)(e - b) : 0.0;
}

// ------------------------------------------------------------------------------------------------
// f32 wire format, per-frame centroids, weight-function index check, per-anchor statistics over jobs
// ------------------------------------------------------------------------------------------------
// Coordinates that arrive as f32 (Bio.PDB / MDAnalysis positions, atom_converter_utils.py:117,126) are widened on
// the device: f32 -> f64 is exact, the upload is half the bytes.
__global__ void widen_xyz_kernel(const float* __restrict__ in, double* __restrict__ out, uint64_t n3) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3) out[i] = (double)in[i];
}

// PrimitiveAssigner.assign_primitive_structure for a compiled topology (atom_converter_utils.py:92-131): primitive
// p of every frame = np.mean of its atoms' f32 coordinates, i.e. a sequential f32 sum in atom order followed by
// an f32 division by the atom count (numpy reduces axis 0 of a [k, 3] float32 array row by row).  One thread per
// (frame, primitive); the result is widened to the f64 coordinates of the structure set.
__global__ void centroid_kernel(const float* __restrict__ atoms, uint64_t n_atoms, uint64_t n_frames,
                                const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ atom_index,
                                uint64_t n_prims, double* __restrict__ xyz_out, int* err) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_frames * n_prims) return;
    const uint64_t f = t / n_prims, p = t - f * n_prims;
    const uint32_t s0 = seg_start[p], s1 = seg_start[p + 1];
    const float* fa = atoms + 3 * f * n_atoms;
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (uint32_t k = s0; k < s1; ++k) {
        const uint32_t a = atom_index[k];
        if (a >= n_atoms) { raise(err, LOCOHD_ERR_INDEX); return; }
        sx = __fadd_rn(sx, fa[3 * (uint64_t)a]);
        sy = __fadd_rn(sy, fa[3 * (uint64_t)a + 1]);
        sz = __fadd_rn(sz, fa[3 * (uint64_t)a + 2]);
    }
    const float cnt = (float)(s1 - s0);   // an empty segment gives 0 / 0 = NaN, as np.mean of nothing does
    xyz_out[3 * t] = (double)__fdiv_rn(sx, cnt);
    xyz_out[3 * t + 1] = (double)__fdiv_rn(sy, cnt);
    xyz_out[3 * t + 2] = (double)__fdiv_rn(sz, cnt);
}

__global__ void validate_wf_idx_kernel(const uint32_t* __restrict__ wf_idx, uint64_t n, uint32_t n_wf, int* err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && wf_idx[i] >= n_wf) raise(err, LOCOHD_ERR_BAD_PARAM);
}

// Per-anchor statistics over uniform jobs (scores is [n_jobs][n]): mean and population standard deviation of
// anchor p over the jobs - np.mean(lchd_by_atom, axis=0) (compare_ensembles.py:299) and
// np.std(all_points[1:], axis=0) (trajectory_analyzer.py:310).  Two passes like numpy's (mean, then squared
// deviations); grid.y splits the jobs, partial sums meet in double atomics.
constexpr int kStatThreads = 256;
__global__ void __launch_bounds__(kStatThreads) anchor_sum_kernel(const double* __restrict__ scores, uint64_t n,
                                                                 uint64_t n_jobs, double* __restrict__ sum) {
    const uint64_t p = (uint64_t)blockIdx.x * kStatThreads + threadIdx.x;
    if (p >= n) return;
    double acc = 0.0;
    for (uint64_t j = blockIdx.y; j < n_jobs; j += gridDim.y) acc += scores[j * n + p];
    atomicAdd(sum + p, acc);
}
__global__ void __launch_bounds__(kStatThreads) anchor_dev_kernel(const double* __restrict__ scores, uint64_t n,
                                                                 uint64_t n_jobs, const double* __restrict__ sum,
                                                                 double* __restrict__ m2) {
    const uint64_t p = (uint64_t)blockIdx.x * kStatThreads + threadIdx.x;
    if (p >= n) return;
    const double mean = sum[p] / (double)n_jobs;
    double acc = 0.0;
    for (uint64_t j = blockIdx.y; j < n_jobs; j += gridDim.y) {
        const double d = scores[j * n + p] - mean;
        acc = fma(d, d, acc);
    }
    atomicAdd(m2 + p, acc);
}
__global__ void anchor_finish_kernel(uint64_t n, uint64_t n_jobs, const double* __restrict__ sum,
                                     const double* __restrict__ m2, double* __restrict__ mean_out,
                                     double* __restrict__ std_out) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    if (mean_out) mean_out[p] = sum[p] / (double)n_jobs;
    if (std_out) std_out[p] = sqrt(m2[p] / (double)n_jobs);
}

// ------------------------------------------------------------------------------------------------
// from_anchors: one caller-ordered pair, walked by a single thread in the reference's exact statement order
// (locohd.rs:61-226), so unsorted inputs behave as they do upstream.
// ------------------------------------------------------------------------------------------------
struct SeqWalk {
    const KParams& P;
    const WfDev& wf;
    double pmf1[LOCOHD_MAX_CATEGORIES], pmf2[LOCOHD_MAX_CATEGORIES];
    int status;
    __device__ SeqWalk(const KParams& P_, const WfDev& wf_) : P(P_), wf(wf_), status(0) {
        for (int r = 0; r < P.C; ++r) { pmf1[r] = 0.0; pmf2[r] = 0.0; }
    }
    __device__ void update(double* pmf, uint32_t c) {  // pmf.rs:47-63
        if (c >= (uint32_t)P.C) { if (!status) status = LOCOHD_ERR_UNKNOWN_CATEGORY; return; }
        pmf[c] += P.cat_w[c];
    }
    __device__ double distance() {  // pmf.rs:65-88
        double n1 = 0.0, n2 = 0.0;
        for (int r = 0; r < P.C; ++r) n1 += pmf1[r];
        for (int r = 0; r < P.C; ++r) n2 += pmf2[r];
        if (n1 == 0.0 || n2 == 0.0) { if (!status) status = LOCOHD_ERR_ZERO_NORM; return 0.0; }
        auto p1 = [&](int r) { return pmf1[r] / n1; };
        auto p2 = [&](int r) { return pmf2[r] / n2; };
        return sd_run(P.sd_kind, P.sd_p0, P.sd_p1, P.C, p1, p2);
    }
    __device__ double range(double from, double to) {  // weight_function.rs:95-120
        if (to < 0.0 || from < 0.0) { if (!status) status = LOCOHD_ERR_NEGATIVE_POINT; return 0.0; }
        return wf_cdf(wf, to) - wf_cdf(wf, from);
    }
};

__global__ void anchor_lists_kernel(KParams P, const uint8_t* __restrict__ sa, uint64_t len_a,
                                    const double* __restrict__ da, const uint8_t* __restrict__ sb, uint64_t len_b,
                                    const double* __restrict__ db, uint32_t wf_idx, double* out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (da[0] != 0.0 || db[0] != 0.0) { raise(P.err, LOCOHD_ERR_FIRST_NOT_ZERO); return; }
    SeqWalk w(P, P.wfs[wf_idx]);
    w.update(w.pmf1, sa[0]);
    w.update(w.pmf2, sb[0]);
    uint64_t ia = 0, ib = 0;
    double integral = 0.0, buffer = 0.0;
    while (ia < len_a - 1 && ib < len_b - 1 && !w.status) {
        const double h = w.distance();
        double nd;
        if (da[ia + 1] < db[ib + 1]) { ++ia; w.update(w.pmf1, sa[ia]); nd = da[ia]; }
        else if (da[ia + 1] > db[ib + 1]) { ++ib; w.update(w.pmf2, sb[ib]); nd = db[ib]; }
        else if (da[ia + 1] == db[ib + 1]) { ++ia; ++ib; w.update(w.pmf1, sa[ia]); w.update(w.pmf2, sb[ib]); nd = da[ia]; }
        else { w.status = LOCOHD_ERR_NAN; break; }
        integral += w.range(buffer, nd) * h;
        buffer = nd;
    }
    if (!w.status) {
        if (ib < len_b - 1) {
            double h = w.distance();
            ++ib;
            integral += w.range(da[len_a - 1], db[ib]) * h;
            w.update(w.pmf2, sb[ib]);
            while (ib < len_b - 1 && !w.status) {
                ++ib;
                h = w.distance();
                integral += w.range(db[ib - 1], db[ib]) * h;
                w.update(w.pmf2, sb[ib]);
            }
            h = w.distance();
            integral += w.range(db[len_b - 1], INFINITY) * h;
        } else if (ia < len_a - 1) {
            double h = w.distance();
            ++ia;
            integral += w.range(db[len_b - 1], da[ia]) * h;
            w.update(w.pmf1, sa[ia]);
            while (ia < len_a - 1 && !w.status) {
                ++ia;
                h = w.distance();
                integral += w.range(da[ia - 1], da[ia]) * h;
                w.update(w.pmf1, sa[ia]);
            }
            h = w.distance();
            integral += w.range(da[len_a - 1], INFINITY) * h;
        } else {
            const double h = w.distance();
            integral += w.range(da[len_a - 1], INFINITY) * h;
        }
    }
    if (w.status) { raise(P.err, w.status); return; }
    *out = integral;
}

// ------------------------------------------------------------------------------------------------
// leaf-math probes
// ------------------------------------------------------------------------------------------------
__global__ void wf_points_kernel(const WfDev* wf, uint64_t n, const double* __restrict__ x, double* __restrict__ out,
                                 int* err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    if (v < 0.0) { raise(err, LOCOHD_ERR_NEGATIVE_POINT); return; }  // weight_function.rs:97-100
    out[i] = wf_cdf(*wf, v);
}

__global__ void wf_density_kernel(const WfDev* wf, uint64_t n, const double* __restrict__ x, double* __restrict__ out,
                                  int* err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    if (v < 0.0) { raise(err, LOCOHD_ERR_NEGATIVE_POINT); return; }
    out[i] = wf_pdf(*wf, v);
}

__global__ void sd_run_kernel(int kind, double q0, double q1, int C, uint64_t n, const double* __restrict__ p1,
                              const double* __restrict__ p2, double* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* a = p1 + i * C;
    const double* b = p2 + i * C;
    out[i] = sd_run(kind, q0, q1, C, [&](int r) { return a[r]; }, [&](int r) { return b[r]; });
}

// FP64 FMA peak probe: 8 independent register-resident chains per thread.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 12345.678) out[0] = s;  // never true; keeps the chains alive
}

inline unsigned blocks_for(uint64_t n, unsigned per) { return (unsigned)((n + per - 1) / per); }

}  // namespace

// ================================================================================================
// launchers
// ================================================================================================
int launch_convert_categories(const uint16_t* in, uint8_t* out, uint64_t n, int C, cudaStream_t st) {
    if (!n) return 0;
    convert_categories_kernel<<<blocks_for(n, 256), 256, 0, st>>>(in, out, n, C);
    return 1;
}

int launch_validate_xyz(const double* xyz, uint64_t n3, int* err, cudaStream_t st) {
    if (!n3) return 0;
    validate_xyz_kernel<<<blocks_for(n3, 256), 256, 0, st>>>(xyz, n3, err);
    return 1;
}

int launch_build_cells(const StructsView& s, double threshold, uint64_t max_prims, cudaStream_t st) {
    if (!s.n_structs) return 0;
    // a structure has at most max(2 N, 8) cells (+ the end marker)
    const uint64_t words = (2 * max_prims > 8 ? 2 * max_prims : 8) + 1;
    if (words * 4 <= 160 * 1024) {
        const int smem = (int)(words * 4);
        cudaFuncSetAttribute(build_cells_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        build_cells_kernel<true><<<(unsigned)s.n_structs, kCellThreads, smem, st>>>(s, threshold, (int)words);
    } else {
        build_cells_kernel<false><<<(unsigned)s.n_structs, kCellThreads, 0, st>>>(s, threshold, 0);
    }
    return 1;
}

uint64_t scan_scratch_entries(uint64_t n) { return (n + kScanTile - 1) / kScanTile + 1; }

int launch_scan(const uint32_t* values, uint64_t n, int round_even, uint64_t* off, uint64_t* scratch, ScanStats* stats,
                cudaStream_t st) {
    cudaMemsetAsync(stats, 0, sizeof(ScanStats), st);
    if (!n) { cudaMemsetAsync(off, 0, sizeof(uint64_t), st); return 0; }
    const unsigned nb = blocks_for(n, kScanTile);
    scan_tile_sums_kernel<<<nb, kScanThreads, 0, st>>>(values, n, round_even, scratch, stats);
    scan_block_sums_kernel<<<1, kScanThreads, 0, st>>>(scratch, nb, stats);
    scan_apply_kernel<<<nb, kScanThreads, 0, st>>>(values, n, round_even, scratch, off);
    return 3;
}

int launch_anchor_order(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* anchor_struct,
                        const uint32_t* anchor_prim, uint64_t n_prims, uint32_t* slot_cnt, uint64_t* slot_off,
                        uint64_t* scan_scratch, ScanStats* stats, uint32_t* order, uint2* order_rec, cudaStream_t st) {
    if (!n_env) return 0;
    if (n_env <= kIdentityOrderMax) {
        anchor_identity_kernel<<<blocks_for(n_env, 256), 256, 0, st>>>(s, p, n_env, anchor_struct, anchor_prim, order, order_rec);
        return 1;
    }
    cudaMemsetAsync(slot_cnt, 0, (n_prims + 1) * sizeof(uint32_t), st);
    anchor_slot_count_kernel<<<blocks_for(n_env, 256), 256, 0, st>>>(s, p, n_env, anchor_struct, anchor_prim, slot_cnt);
    int n = 1 + launch_scan(slot_cnt, n_prims + 1, 0, slot_off, scan_scratch, stats, st);
    anchor_slot_scatter_kernel<<<blocks_for(n_env, 256), 256, 0, st>>>(s, p, n_env, anchor_struct, anchor_prim,
                                                                      slot_cnt, slot_off, order, order_rec);
    return n + 1;
}

int launch_env_count(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* order,
                     const uint32_t* anchor_struct, const uint32_t* anchor_prim, double threshold, uint32_t* ub,
                     cudaStream_t st) {
    if (!n_env) return 0;
    EnvBuild none{};
    env_tile_kernel<false><<<blocks_for(n_env, kTileThreads), kTileThreads, 0, st>>>(
        s, p, n_env, order, anchor_struct, anchor_prim, threshold, ub, none, 1u, nullptr);
    return 1;
}

int launch_env_sample(const StructsView& s, const KParams& p, uint64_t n_env, const uint32_t* order,
                      const uint32_t* anchor_struct, const uint32_t* anchor_prim, double threshold, uint32_t stride,
                      unsigned long long* sum, cudaStream_t st) {
    if (!n_env) return 0;
    EnvBuild none{};
    const uint64_t n_vis = ((n_env + 32ull * stride - 1) / (32ull * stride)) * 32;   // whole groups of 32 anchors
    env_tile_kernel<false><<<blocks_for(n_vis, kTileThreads), kTileThreads, 0, st>>>(
        s, p, n_env, order, anchor_struct, anchor_prim, threshold, nullptr, none, stride, sum);
    return 1;
}

// WFK of a parameter block: 0 uniform, 1 integer-exponent kumaraswamy, 2 generic / plain distances
static int fused_wfk(const KParams& p, const WfDev* host_wf, int key_is_w) {
    (void)p;
    if (!key_is_w || !host_wf) return 2;
    if (host_wf->kind == LOCOHD_WF_UNIFORM) return 0;
    if (host_wf->kind == LOCOHD_WF_KUMARASWAMY && host_wf->int_a == 2 && host_wf->int_b == 5) return 3;
    if (host_wf->kind == LOCOHD_WF_KUMARASWAMY && host_wf->int_a >= 0 && host_wf->int_b >= 0) return 1;
    return 2;
}

template <int WFK, bool DEBUG, int CAP, bool LIST>
static unsigned fused_grid_t(uint64_t n_env) {
    const int smem = FusedLayout<DEBUG, CAP>::kBytes * fused_warps(CAP, DEBUG);
    cudaFuncSetAttribute(env_fused_kernel<WFK, DEBUG, CAP, LIST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, env_fused_kernel<WFK, DEBUG, CAP, LIST>, fused_warps(CAP, DEBUG) * 32, smem);
    if (occ < 1) occ = 1;
    const uint64_t need = (n_env + fused_warps(CAP, DEBUG) - 1) / fused_warps(CAP, DEBUG);
    const uint64_t cap = (uint64_t)sms * occ;
    return (unsigned)(need < cap ? need : cap);
}

template <int WFK, bool DEBUG, int CAP, bool LIST>
static void fused_launch_t(const StructsView& s, const KParams& p, const uint32_t* anchor_struct,
                           const uint32_t* anchor_prim, double threshold, const EnvBuild& b, FusedStats* stats,
                           uint64_t capacity, unsigned grid, cudaStream_t st) {
    const int smem = FusedLayout<DEBUG, CAP>::kBytes * fused_warps(CAP, DEBUG);
    env_fused_kernel<WFK, DEBUG, CAP, LIST><<<grid, fused_warps(CAP, DEBUG) * 32, smem, st>>>(s, p, b.n_env, b.order, anchor_struct,
                                                                            anchor_prim, threshold, b, stats, capacity);
}

// dispatch over (CDF specialisation, parity arrays, members per environment, kind of tag rule)
#define LOCOHD_FUSED_DISPATCH2(CALL, W, D, C)                                             \
    if (p.tpr_kind == LOCOHD_TPR_WITHOUT_LIST) { CALL(W, D, C, false); } else { CALL(W, D, C, true); }
#define LOCOHD_FUSED_DISPATCH(CALL)                                                                        \
    switch ((fused_wfk(p, host_wf, key_is_w) * 2 + (debug ? 1 : 0)) * 2 + (cap > 512 ? 1 : 0)) {          \
        case 0: LOCOHD_FUSED_DISPATCH2(CALL, 0, false, 512) break;                                        \
        case 1: LOCOHD_FUSED_DISPATCH2(CALL, 0, false, 1024) break;                                       \
        case 2: LOCOHD_FUSED_DISPATCH2(CALL, 0, true, 512) break;                                         \
        case 3: LOCOHD_FUSED_DISPATCH2(CALL, 0, true, 1024) break;                                        \
        case 4: LOCOHD_FUSED_DISPATCH2(CALL, 1, false, 512) break;                                        \
        case 5: LOCOHD_FUSED_DISPATCH2(CALL, 1, false, 1024) break;                                       \
        case 6: LOCOHD_FUSED_DISPATCH2(CALL, 1, true, 512) break;                                         \
        case 7: LOCOHD_FUSED_DISPATCH2(CALL, 1, true, 1024) break;                                        \
        case 8: LOCOHD_FUSED_DISPATCH2(CALL, 2, false, 512) break;                                        \
        case 9: LOCOHD_FUSED_DISPATCH2(CALL, 2, false, 1024) break;                                       \
        case 10: LOCOHD_FUSED_DISPATCH2(CALL, 2, true, 512) break;                                        \
        case 11: LOCOHD_FUSED_DISPATCH2(CALL, 2, true, 1024) break;                                       \
        case 12: LOCOHD_FUSED_DISPATCH2(CALL, 3, false, 512) break;                                       \
        case 13: LOCOHD_FUSED_DISPATCH2(CALL, 3, false, 1024) break;                                      \
        case 14: LOCOHD_FUSED_DISPATCH2(CALL, 3, true, 512) break;                                        \
        default: LOCOHD_FUSED_DISPATCH2(CALL, 3, true, 1024) break;                                       \
    }

unsigned fused_grid(const KParams& p, const WfDev* host_wf, int key_is_w, bool debug, int cap, uint64_t n_env) {
    unsigned g = 1;
#define LOCOHD_CALL(W, D, C, L) g = fused_grid_t<W, D, C, L>(n_env)
    LOCOHD_FUSED_DISPATCH(LOCOHD_CALL)
#undef LOCOHD_CALL
    return g;
}

int launch_env_fused(const StructsView& s, const KParams& p, const WfDev* host_wf, const uint32_t* anchor_struct,
                     const uint32_t* anchor_prim, double threshold, const EnvBuild& b, int cap, FusedStats* stats,
                     uint64_t capacity, unsigned grid, cudaStream_t st) {
    if (!b.n_env) return 0;
    const int key_is_w = b.key_is_w;
    const bool debug = b.idx != nullptr;
#define LOCOHD_CALL(W, D, C, L) fused_launch_t<W, D, C, L>(s, p, anchor_struct, anchor_prim, threshold, b, stats, capacity, grid, st)
    LOCOHD_FUSED_DISPATCH(LOCOHD_CALL)
#undef LOCOHD_CALL
    return 1;
}

int launch_env_fill(const StructsView& s, const KParams& p, const uint32_t* anchor_struct, const uint32_t* anchor_prim,
                    double threshold, const EnvBuild& b, cudaStream_t st) {
    if (!b.n_env) return 0;
    env_tile_kernel<true><<<blocks_for(b.n_env, kTileThreads), kTileThreads, 0, st>>>(
        s, p, b.n_env, b.order, anchor_struct, anchor_prim, threshold, nullptr, b, 1u, nullptr);
    return 1;
}

template <int CAP, bool DEBUG>
static int launch_sort_class(const KParams& p, const EnvBuild& b, uint32_t min_m, double scale, cudaStream_t st) {
    const int smem = SortLayout<CAP, DEBUG>::kBytes * kSortWarps;
    cudaFuncSetAttribute(env_sort_kernel<CAP, DEBUG>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    env_sort_kernel<CAP, DEBUG><<<blocks_for(b.n_env, kSortWarps), kSortWarps * 32, smem, st>>>(p, b, min_m, scale);
    return 1;
}

template <bool DEBUG>
static int launch_env_sort_t(const KParams& p, const EnvBuild& b, unsigned max_count, double scale, cudaStream_t st) {
    int n = 0;
    n += launch_sort_class<256, DEBUG>(p, b, 0, scale, st);
    if (max_count > 256) n += launch_sort_class<512, DEBUG>(p, b, 256, scale, st);
    if (max_count > 512) n += launch_sort_class<1024, DEBUG>(p, b, 512, scale, st);
    if (max_count > 1024) n += launch_sort_class<2048, DEBUG>(p, b, 1024, scale, st);
    if (max_count > 2048) {
        env_sort_big_kernel<<<(unsigned)b.n_env, kBigThreads, 0, st>>>(p, b, 2048);
        ++n;
    }
    return n;
}

int launch_env_sort(const KParams& p, const EnvBuild& b, unsigned max_count, double threshold, cudaStream_t st) {
    if (!b.n_env) return 0;
    // gather mode: distances are below the threshold; rows mode (threshold <= 0): scale from the data
    double scale = 0.0;
    if (threshold > 0.0 && std::isfinite(threshold * threshold))
        scale = b.key_is_sq ? (1.0 - 1e-9) / (threshold * threshold) : (1.0 - 1e-9) / threshold;
    return b.idx ? launch_env_sort_t<true>(p, b, max_count, scale, st) : launch_env_sort_t<false>(p, b, max_count, scale, st);
}

int launch_rows_copy(const double* values, const double* xyz, const uint8_t* cat, uint64_t n_rows, uint64_t row_len,
                     const uint64_t* in_off, const uint64_t* out_off, uint64_t* off, uint32_t* count, const EnvBuild& b,
                     cudaStream_t st) {
    if (!n_rows || !row_len) return 0;
    dim3 grid((unsigned)((row_len + 255) / 256), (unsigned)(n_rows > 32768 ? 32768 : n_rows));
    if (grid.x > 64) grid.x = 64;
    rows_copy_kernel<<<grid, 256, 0, st>>>(values, xyz, cat, n_rows, row_len, in_off, out_off, off, count, b);
    return 1;
}

template <class K>
static unsigned persistent_grid(K kernel, int threads, int smem, uint64_t n_pairs, int warps) {
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem);
    if (occ < 1) occ = 1;
    const uint64_t need = (n_pairs + warps - 1) / warps;
    // Large launches: exactly the resident CTAs, so that at any time they work on one contiguous window of pairs
    // (stride = the resident set) - consecutive jobs that share a structure then find its environments in L2.
    // With 8 times as many CTAs the first wave strode over the whole job list and every pair re-read both
    // environments from DRAM (ncu r5f: 3.0 KB per pair on the 1000-structure ensemble).  Small launches keep the
    // oversubscription, which evens out the tail.
    const uint64_t resident = (uint64_t)sms * occ;
    const uint64_t cap = need >= 64 * resident ? resident : resident * 8;   // (the fast kernel claims its pairs dynamically)
    return (unsigned)(need < cap ? need : cap);
}

template <class K>
static int launch_score_kernel(K kernel, const ScoreArgs& a, const KParams& p, int warps, int per_warp, int smem,
                               cudaStream_t st) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const unsigned grid = persistent_grid(kernel, warps * 32, smem, a.n_pairs, warps);
    if (a.cursor) cudaMemsetAsync(a.cursor, 0, sizeof(unsigned long long), st);
    ScoreArgs b = a;
    const uint64_t per_warp_pairs = a.n_pairs / ((uint64_t)grid * warps * 4) ;
    b.run = (unsigned)(per_warp_pairs < 1 ? 1 : (per_warp_pairs > (uint64_t)kScoreRun ? (uint64_t)kScoreRun : per_warp_pairs));
    kernel<<<grid, warps * 32, smem, st>>>(b, p, warps, per_warp);
    return 1;
}

static int launch_generic(const ScoreArgs& args, const KParams& p, unsigned stage_want, int only_unstaged,
                          cudaStream_t st) {
    ScoreArgs a = args;
    const int budget = 100 * 1024;
    const int state = score_state_bytes(p.C);
    int cap = (int)(stage_want > 2048u ? 2048u : stage_want);
    int per_warp = state + cap * 8;
    if (per_warp > budget) { cap = 0; per_warp = state; }
    if (per_warp > 220 * 1024) return -1;
    int warps = budget / per_warp;
    if (warps > kScoreMaxWarps) warps = kScoreMaxWarps;
    if (warps < 1) warps = 1;
    a.stage_cap = cap;
    a.only_unstaged = only_unstaged;
    const int smem = per_warp * warps;
    return p.hell2 ? launch_score_kernel(score_kernel<true>, a, p, warps, per_warp, smem, st)
                   : launch_score_kernel(score_kernel<false>, a, p, warps, per_warp, smem, st);
}

template <int CP, bool KEY_IS_W>
static int launch_fast(const ScoreArgs& a, const KParams& p, int warps, int per_warp, int smem, cudaStream_t st) {
    return p.unit_w ? launch_score_kernel(score_fast_kernel<CP, KEY_IS_W, false>, a, p, warps, per_warp, smem, st)
                    : launch_score_kernel(score_fast_kernel<CP, KEY_IS_W, true>, a, p, warps, per_warp, smem, st);
}

LaunchOverrides read_launch_overrides() {
    const auto env = [](const char* name) { return std::getenv(name); };
    LaunchOverrides o;
    if (const char* v = env("LOCOHD_NO_TILES")) o.no_tiles = std::atoi(v) != 0;
    if (const char* v = env("LOCOHD_TILE_TEAMS")) o.tile_teams = std::atoi(v);
    if (const char* v = env("LOCOHD_TILE_REP")) o.tile_rep = std::atoi(v);
    if (const char* v = env("LOCOHD_TILE_RUN")) { const int r = std::atoi(v); if (r >= 1 && r <= 4096) o.tile_run = (unsigned)r; }
    if (const char* v = env("LOCOHD_TILE_SLICE")) { const long long s = std::atoll(v); o.tile_slice = s < 0 ? 0 : s; }
    if (const char* v = env("LOCOHD_TILE_SLICE_MB")) { const double mb = std::atof(v); if (mb > 0.0) o.tile_slice_mb = mb; }
    if (const char* v = env("LOCOHD_LEGACY_GATHER")) o.legacy_gather = v[0] && v[0] != '0';
    return o;
}

TileGeometry tile_geometry(const KParams& p, unsigned max_a, unsigned max_b, int key_is_w, const LaunchOverrides& ov) {
    TileGeometry g{};
    if (!(p.hell2 && p.unit_w && p.C >= 1 && p.C <= 16 && key_is_w)) return g;   // the configuration of score_fast_kernel<CP, true, false>
    if (max_a < 1 || max_b < 1 || max_a + max_b > 1024u) return g;   // chunks of at most 128 events per lane
    const unsigned need = (max_a > max_b ? max_a : max_b) + 2u;
    g.table_n = (int)((need + 63u) & ~63u);
    g.cp = p.C <= 8 ? 8 : 16;
    g.stage_keys = kTileDim * (int)((max_a + 2u) & ~1u) + kTileDim * (int)((max_b + 2u) & ~1u);
    g.team_bytes = tile_team_bytes(g.cp, g.stage_keys);
    const int budget = 227 * 1024 - 3 * g.table_n * 8;
    int teams = budget / g.team_bytes;
    if (teams > kTileMaxTeams) teams = kTileMaxTeams;
    if (ov.tile_teams >= 1 && ov.tile_teams < teams) teams = ov.tile_teams;
    // what the teams leave over replicates the head of the two count-indexed tables (240 bytes per entry); only the
    // 8-row instantiation has the replicated form
    int rep_n = teams > 0 && g.cp == 8 ? (budget - teams * g.team_bytes) / 240 : 0;
    if (rep_n > kTileRepMax) rep_n = kTileRepMax;
    if (rep_n < 16) rep_n = 0;
    if (ov.tile_rep >= 0 && ov.tile_rep < rep_n) rep_n = ov.tile_rep;
    g.teams = teams;
    g.rep_n = rep_n;
    return g;
}

// Anchors per slice of the unit order (TileOrder): as many as keep the environments of one slice of every structure
// inside a budget of L2 (126 MB on a B200, in two halves; 32 MB leaves room for the scores written and for the tile
// descriptors), a multiple of the run length so that a claimed run stays inside one tile.  0 = tile-major order
// (the whole store fits the budget, or LaunchOverrides::tile_slice = 0).
static uint64_t tile_slice(const ScoreArgs& a, double mean_a, double mean_b, const LaunchOverrides& ov) {
    const uint64_t n = a.uniform_n;
    if (ov.tile_slice >= 0) return (uint64_t)ov.tile_slice >= n ? 0 : (uint64_t)ov.tile_slice;
    const double budget = (ov.tile_slice_mb > 0.0 ? ov.tile_slice_mb : 32.0) * 1048576.0;
    const bool same = a.a.key == a.b.key && a.a.off == a.b.off;
    const double store = 8.0 * ((double)a.a.n_env * (mean_a + 1.0) + (same ? 0.0 : (double)a.b.n_env * (mean_b + 1.0)));
    if (n == 0 || store <= budget) return 0;
    const double per_anchor = store / (double)n;           // bytes of environments per anchor index, all structures
    uint64_t s = (uint64_t)(budget / per_anchor);
    s = s / kTileRun * kTileRun;
    if (s < (uint64_t)kTileRun) s = kTileRun;
    return s >= n ? 0 : s;
}

static int launch_tiles(const ScoreArgs& args, const KParams& p, unsigned max_a, unsigned max_b, double mean_a, double mean_b,
                        const LaunchOverrides& ov, cudaStream_t st) {
    ScoreArgs a = args;
    const TileGeometry g = tile_geometry(p, max_a, max_b, a.a.key_is_w, ov);
    const int teams = g.teams, team_bytes = g.team_bytes;
    if (teams < 1) return -1;
    a.table_n = g.table_n;
    a.stage_cap = g.stage_keys;
    a.rep_n = g.rep_n;
    const bool rep = a.rep_n > 0;
    const int smem = (g.table_n + 2 * (15 * a.rep_n + g.table_n)) * 8 + teams * team_bytes;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const uint64_t units = a.n_tiles * a.uniform_n;
    const uint64_t need = (units + teams - 1) / teams;
    const unsigned grid = (unsigned)(need < (uint64_t)sms ? need : (uint64_t)sms);   // persistent: teams claim units from the cursor
    cudaMemsetAsync(a.cursor, 0, sizeof(unsigned long long), st);
    const uint64_t per_team = units / ((uint64_t)grid * teams * 4);   // short launches: shorter runs even out the tail
    const uint64_t max_run = ov.tile_run ? ov.tile_run : kTileRun;
    a.run = (unsigned)(per_team < 1 ? 1 : (per_team > max_run ? max_run : per_team));
    a.order = make_tile_order(a.n_tiles, a.uniform_n, tile_slice(a, mean_a, mean_b, ov));
    auto go = [&](auto kernel) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        kernel<<<grid, teams * kTeamThreads, smem, st>>>(a, p, teams, team_bytes);
    };
    if (g.cp == 8) { if (rep) go(score_tile_kernel<8, true>); else go(score_tile_kernel<8, false>); }
    else go(score_tile_kernel<16, false>);
    return 1;
}

int launch_score(const ScoreArgs& args, const KParams& p, unsigned max_a, unsigned max_b, double mean_a, double mean_b,
                 const LaunchOverrides& ov, cudaStream_t st) {
    if (!args.n_pairs) return 0;
    if (args.tiles) return launch_tiles(args, p, max_a, max_b, mean_a, mean_b, ov, st);
    const unsigned pad_max = ((max_a + 1) & ~1u) + ((max_b + 1) & ~1u);
    const bool key_is_w = args.a.key_is_w != 0;
    const bool fast = p.hell2 && p.C <= 16;   // Hellinger-2 with or without category weights
    if (!fast) return launch_generic(args, p, pad_max, 0, st);

    ScoreArgs a = args;
    const int CP = p.C <= 8 ? 8 : 16;
    // stage: everything when the largest pair is small, else what a typical pair needs (the rest goes to the
    // generic kernel in a second pass)
    unsigned stage = pad_max;
    if (stage > 1024u) {
        stage = (unsigned)(1.5 * (mean_a + mean_b)) + 64u;
        stage = (stage + 63u) & ~63u;
        if (stage > 2048u) stage = 2048u;
        if (stage > pad_max) stage = pad_max;
    }
    int n = 0;
    // tables: counts never exceed the environment sizes, and a staged pair's counts and totals are below stage - 1
    static_assert(2048 + 1 < kSqrtTableSize, "the table fill reads sqrt_tbl[k + 1] for k < the largest stage");
    const unsigned need = (max_a > max_b ? max_a : max_b) + 2u;
    const unsigned table_n = ((need < stage ? need : stage) + 63u) & ~63u;
    a.table_n = (int)table_n;
    a.stage_cap = (int)stage;
    a.only_unstaged = 0;
    const int tables = 3 * (int)table_n * 8 + kFastWeightBytes;
    const int per_warp = fast_state_bytes(CP) + ((int)stage + 4) * 8;   // + the two sentinels and their padding
    const int budget = 220 * 1024;  // one CTA per SM: the tables are staged once, the rest goes to the warps' stages
    int warps = (budget - tables) / per_warp;
    if (warps > score_fast_max_warps(key_is_w, !p.unit_w)) warps = score_fast_max_warps(key_is_w, !p.unit_w);
    if (warps < 1) warps = 1;
    const int smem = tables + per_warp * warps;
    if (CP == 8) n += key_is_w ? launch_fast<8, true>(a, p, warps, per_warp, smem, st)
                               : launch_fast<8, false>(a, p, warps, per_warp, smem, st);
    else n += key_is_w ? launch_fast<16, true>(a, p, warps, per_warp, smem, st)
                       : launch_fast<16, false>(a, p, warps, per_warp, smem, st);
    if (pad_max > stage) {
        const int m = launch_generic(args, p, 0, (int)stage, st);
        if (m < 0) return m;
        n += m;
    }
    return n;
}

int launch_job_means(const double* scores, const uint64_t* job_pair_off, uint64_t n_jobs, double* means,
                     cudaStream_t st) {
    if (!n_jobs) return 0;
    job_means_kernel<<<blocks_for(n_jobs * 32, 256), 256, 0, st>>>(scores, job_pair_off, n_jobs, means);
    return 1;
}

int launch_widen_xyz(const float* in, double* out, uint64_t n3, cudaStream_t st) {
    if (!n3) return 0;
    widen_xyz_kernel<<<blocks_for(n3, 256), 256, 0, st>>>(in, out, n3);
    return 1;
}

int launch_centroids(const float* atoms, uint64_t n_atoms, uint64_t n_frames, const uint32_t* seg_start,
                     const uint32_t* atom_index, uint64_t n_prims, double* xyz_out, int* err, cudaStream_t st) {
    if (!n_frames || !n_prims) return 0;
    centroid_kernel<<<blocks_for(n_frames * n_prims, 128), 128, 0, st>>>(atoms, n_atoms, n_frames, seg_start, atom_index,
                                                                       n_prims, xyz_out, err);
    return 1;
}

int launch_validate_wf_idx(const uint32_t* wf_idx, uint64_t n, uint32_t n_wf, int* err, cudaStream_t st) {
    if (!n || !wf_idx) return 0;
    validate_wf_idx_kernel<<<blocks_for(n, 256), 256, 0, st>>>(wf_idx, n, n_wf, err);
    return 1;
}

int launch_anchor_stats(const double* scores, uint64_t n, uint64_t n_jobs, double* sum_scratch, double* m2_scratch,
                        double* mean_out, double* std_out, cudaStream_t st) {
    if (!n || !n_jobs) return 0;
    cudaMemsetAsync(sum_scratch, 0, n * sizeof(double), st);
    const unsigned bx = blocks_for(n, kStatThreads);
    // enough CTAs to fill the machine; every CTA column walks its share of the jobs
    uint64_t splits = (148ull * 16 + bx - 1) / bx;
    if (splits > n_jobs) splits = n_jobs;
    if (splits > 65535) splits = 65535;
    if (splits < 1) splits = 1;
    const dim3 grid(bx, (unsigned)splits);
    int launches = 2;
    anchor_sum_kernel<<<grid, kStatThreads, 0, st>>>(scores, n, n_jobs, sum_scratch);
    if (std_out) {
        cudaMemsetAsync(m2_scratch, 0, n * sizeof(double), st);
        anchor_dev_kernel<<<grid, kStatThreads, 0, st>>>(scores, n, n_jobs, sum_scratch, m2_scratch);
        ++launches;
    }
    anchor_finish_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, n_jobs, sum_scratch, m2_scratch, mean_out, std_out);
    return launches;
}

int launch_anchor_lists(const KParams& p, const uint8_t* seq_a, uint64_t len_a, const double* da, const uint8_t* seq_b,
                        uint64_t len_b, const double* db, uint32_t wf_idx, double* out, cudaStream_t st) {
    anchor_lists_kernel<<<1, 32, 0, st>>>(p, seq_a, len_a, da, seq_b, len_b, db, wf_idx, out);
    return 1;
}

int launch_wf_points(const WfDev* wf, uint64_t n, const double* x, double* out, int* err, cudaStream_t st) {
    if (!n) return 0;
    wf_points_kernel<<<blocks_for(n, 256), 256, 0, st>>>(wf, n, x, out, err);
    return 1;
}

int launch_wf_density(const WfDev* wf, uint64_t n, const double* x, double* out, int* err, cudaStream_t st) {
    if (!n) return 0;
    wf_density_kernel<<<blocks_for(n, 256), 256, 0, st>>>(wf, n, x, out, err);
    return 1;
}

template <GradTarget T>
static int launch_score_grad_t(const GradArgs& g, const KParams& p, cudaStream_t st) {
    const int per_warp = grad_state_bytes(p.C);
    if (per_warp > 220 * 1024) return -1;
    int warps = (100 * 1024) / per_warp;
    if (warps > kScoreMaxWarps) warps = kScoreMaxWarps;
    if (warps < 1) warps = 1;
    const int smem = per_warp * warps;
    cudaFuncSetAttribute(score_grad_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const unsigned grid = persistent_grid(score_grad_kernel<T>, warps * 32, smem, g.n_pairs, warps);
    score_grad_kernel<T><<<grid, warps * 32, smem, st>>>(g, p, warps);
    return 1;
}

int launch_score_grad(const GradArgs& g, const KParams& p, GradTarget target, cudaStream_t st) {
    if (!g.n_pairs) return 0;
    return target == GradTarget::kEntries ? launch_score_grad_t<GradTarget::kEntries>(g, p, st)
                                          : launch_score_grad_t<GradTarget::kCoords>(g, p, st);
}

int launch_coords_chain(const double* xyz, const double* G, uint64_t n, double* grad, cudaStream_t st) {
    if (!n) return 0;
    coords_chain_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(xyz, G, n, grad);   // one warp per point
    return 1;
}

int launch_fp64_peak(double* scratch, int blocks, int iters, cudaStream_t st) {
    fp64_peak_kernel<<<blocks, 256, 0, st>>>(scratch, iters, 0.999999, 1e-9);
    return 1;
}

int launch_sd_run(int kind, double q0, double q1, int C, uint64_t n, const double* p1, const double* p2, double* out,
                  cudaStream_t st) {
    if (!n) return 0;
    sd_run_kernel<<<blocks_for(n, 128), 128, 0, st>>>(kind, q0, q1, C, n, p1, p2, out);
    return 1;
}

}  // namespace locohd
