// kernels.h — launcher declarations shared by the C-ABI layer (fdcm_api.cu)
#pragma once
#include <cuda.h>   // CUtensorMap (types only: the driver entry point is resolved at run time)

#include "common.cuh"
#include "../../include/fdcm_b200.h"

namespace fdcm {

// ---- dt3_kernels.cu ----
void launch_raster(const float* d_lines, const int32_t* d_bins, int n_lines, const MapDims& dm, uint32_t* d_mask, cudaStream_t s);
// literal Felzenszwalb pass; src_kind: 0 = the plane itself, 1 = the 1-bit edge mask (column pass only), 2 = explicit u16 distances
void launch_dt_pass_literal(int src_kind, bool along_rows, const void* d_src, float* d_planes, const MapDims& dm, void* d_stack,
                            cudaStream_t s);
void launch_transpose_square(float* d_planes, const MapDims& dm, cudaStream_t s);
void launch_sqrt(float* d_planes, const MapDims& dm, cudaStream_t s);
void launch_propagate(float* d_planes, const MapDims& dm, const PropParams& pp, bool sqrt_first, cudaStream_t s);

// ---- integral_tma.cu: lineIntegral as one persistent TMA-fed kernel ----
struct IntegralPlanDev {
    const int4* items4;          // (plane, first chain of the strip, first tile, end tile: where the strip meets the image), heaviest first
    int n_items;
    int* counter;                // work counter, zero before the launch
    CUtensorMap map_y, map_x;    // the planes with the y-major / x-major box shapes
};
size_t integral_tma_smem_bytes();
int integral_strip_chains();
int integral_tile_steps();
bool integral_tma_encode(const void* planes, const MapDims& dm, CUtensorMap* map_y, CUtensorMap* map_x);
void launch_integral_tma(float* d_planes, const MapDims& dm, const IntegralParams& ip, const IntegralPlanDev& plan, int n_sms,
                         cudaStream_t s);

// ---- dt_band_kernels.cu (exact regime, lane-per-row formulation) ----
int dt_band_count(const MapDims& dm);
size_t dt_band_info_bytes(const MapDims& dm);
size_t dt_band_spill_bytes(const MapDims& dm, int maxdepth);
void launch_dt_col_band(const uint32_t* d_mask, const MapDims& dm, void* d_info, cudaStream_t s);
// d_info (band records) or d_g (explicit u16 rows, tests) feeds the envelope build; exactly one of them is non-null
// [row_lo, row_hi]: rows that can hold edge pixels (only used to order the bands in the grid)
// which: 0 = every band, 1 = only the bands overlapping the scene rows [row_lo, row_hi], 2 = only the other (far) bands
void launch_dt_row_envelope(const void* d_info, const uint16_t* d_g, const MapDims& dm, void* d_ws, int win_lo, int win_hi, int row_lo,
                            int row_hi, int which, cudaStream_t s);
void dt_band_scene_rows(const MapDims& dm, int row_lo, int row_hi, int* y0, int* y1);
void launch_dt_row_fill(float* d_planes, const MapDims& dm, void* d_ws, int win_lo, int win_hi, cudaStream_t s);
// fill fused with propagateOrientation (and the L2 sqrt): the distance-transform planes never reach HBM
bool dt_fill_propagate_supported(const MapDims& dm);
// image rows [ya0, ya1) and [yb0, yb1); the resolve pass rewrites the envelope arrays in place and must precede the fused fill
void launch_dt_resolve(const MapDims& dm, void* d_ws, int win_lo, int win_hi, int ya0, int ya1, int yb0, int yb1, cudaStream_t s);
void launch_dt_fill_propagate(float* d_planes, const MapDims& dm, void* d_ws, int win_lo, int win_hi, const PropParams& pp,
                              bool sqrt_first, int ya0, int ya1, int yb0, int yb1, cudaStream_t s);

// L1: row call straight from the band records (exact at any size), stand-alone or fused with propagateOrientation
void launch_dt_row_l1_band(const void* d_info, float* d_planes, const MapDims& dm, cudaStream_t s);
void launch_dt_l1_propagate(const void* d_info, float* d_planes, const MapDims& dm, const PropParams& pp, cudaStream_t s);
size_t dt_band_smem_bytes(const MapDims& dm);
// parity hook of the fused fill's square root (integers 0 .. 2^24 and FLT_MAX against the IEEE sqrtf)
cudaError_t run_sqrt_check(unsigned long long* h_bad, uint32_t* h_first, cudaStream_t s);

// ---- search_kernels.cu ----
struct MapView {                 // read-only view of a built feature map
    const float* planes;
    MapDims dm;
    float shift_x, shift_y;      // sceneTranslation (dt3cpu.h:56)
};

struct TemplatesView {
    const float4* lines;         // all template lines, CSR by offsets
    const int32_t* offsets;      // n_tmpl + 1
    const int32_t* argsort;      // per template: line indices by descending length (std::sort order)
    const float* line_len;       // per line length
    const float* denom;          // per template penalty denominator (or nullptr)
    int32_t n_tmpl;
    int32_t max_lines;           // longest template
};

struct SceneView {
    const float4* lines;         // original (un-shifted) scene lines
    const float* sorted_len;     // lengths, descending (std::sort order of the reference comparator)
    const int32_t* sorted_idx;   // scene line index of each sorted entry
    int32_t n;
};

struct SearchLaunch {
    int32_t max_tmpl_lines, max_scene_lines, batch;
    int32_t tmpl_idx_base;
    const int64_t* hyp_off;      // n_tmpl + 1 prefix of hypothesis counts
    int64_t n_hyp;
    const int32_t* perm;         // processing order: slot i handles hypothesis perm[i] (nullptr: identity)
    const int4* hyp_ready;       // hypotheses already decoded by the ordering pass (tmpl + base, tmpl line, scene line, rev)
    const float2* direct_align;  // optimize() entry point: hypothesis h = template h as given (identity transform)
                                 // with alignment vector direct_align[h]; nullptr for the fused search
};

struct SearchOutputs {
    fdcm_match* rec;             // n_hyp records
    uint8_t* valid;              // n_hyp flags (0 = nullopt)
    int4* hyp;                   // n_hyp (tmpl, tmpl_line, scene_line, rev)
    unsigned long long* counters;// [0] evaluations, [1] lookups, [2] valid
};

// spatial ordering of the hypotheses (locality of the map gathers): keys + radix sort -> permutation
// Cell of the spatial hypothesis order (search_key_kernel).  The hypotheses are processed cell row by cell row, x fastest:
// the map rows a cell row reaches (its own height + twice the template radius, all D planes) slide through the L2 once per
// cell row, so tall cells re-read the map fewer times, as long as the window (rows reached x columns of the cells in
// flight) still fits the L2.  Measured on config 3 (1080p, D = 30, templates reaching +-270 px), search kernel alone, cell
// height 128 -> 1.174 ms, 256 -> 1.149, 336 -> 1.157, 352 -> 1.053, 368 -> 1.076, 384 -> 1.071, 400 -> 1.073, 416 -> 1.148,
// 448 -> 1.102, 480 -> 1.125, 512 -> 1.145, 640 -> 1.051, 720 -> 1.067, one row of 32-px columns -> 1.090: tall beats short,
// with +-4 % of scene-dependent scatter on top (a height derived from the L2 size, the depth and the template diagonal was
// tried and landed on 480: the scatter is larger than what such a model resolves, so the height is a constant).
constexpr int kSearchCellW = 128, kSearchCellH = 384;
size_t search_order_temp_bytes(int64_t n_hyp);
void launch_search_order(const TemplatesView& tv, const SceneView& sv, const SearchLaunch& sl, uint32_t* d_keys, uint32_t* d_keys_out,
                         int32_t* d_idx, int32_t* d_perm, void* d_temp, size_t temp_bytes, float minx, float miny, int cells_x,
                         int key_bits, int4* d_hyp, cudaStream_t s);

// Every warp stages the aligned longest template of the set in shared memory: a block runs 4, 2 or 1 warps, whichever
// fits smem_optin (the device's cudaDevAttrMaxSharedMemoryPerBlockOptin).  search_max_template_lines(smem_optin) is the
// longest template one warp can take; launch_search returns cudaErrorInvalidValue above it.
int search_max_template_lines(int smem_optin);
cudaError_t launch_search(const MapView& map, const SlopeTableDev& table, const TemplatesView& tv, const SceneView& sv,
                          const SearchLaunch& sl, const SearchOutputs& out, int smem_optin, cudaStream_t s);
// the line search over a scale grid (fdcm_search_scales): after launch_search on the copies, every valid record is remapped
// in place to its original template and scaled pose, and its grid scale goes to rec_scale (the selection's angle test)
struct ScaleRemapLaunch {
    fdcm_match* rec;             // n_hyp records of the copy search
    const uint8_t* valid;        // n_hyp flags
    float* rec_scale;            // n_hyp grid scales, written for the valid records
    int64_t n_hyp;
    int32_t scales, tmpl_idx_base;
    float scale[FDCM_DENSE_MAX_SCALES];   // s_k
};
void launch_search_scale_remap(const ScaleRemapLaunch& p, cudaStream_t s);

// top-K smallest (score, index) among valid records; returns via d_out (k records) and d_n_out
void launch_topk(const fdcm_match* d_rec, const uint8_t* d_valid, int64_t n, int k, float* d_ws_score, int64_t* d_ws_idx,
                 int ws_blocks, fdcm_match* d_out, int* d_n_out, cudaStream_t s);
int topk_ws_blocks(int64_t n);
// multi-GPU: merge of the all-gathered per-rank top-k lists; k invalid records for an empty shard
void launch_topk_merge(const fdcm_match* d_gathered, int n_cand, int k, fdcm_match* d_out, int* d_n_out, cudaStream_t s);
void launch_topk_invalid(fdcm_match* d_out, int k, int* d_n_out, cudaStream_t s);

// distinct top-K (fdcm_search_select): selection over the records / valid flags the search kernel left in HBM
struct SelectLaunch {
    const fdcm_match* rec;       // n_hyp records, valid ones written by the search
    const uint8_t* valid;        // n_hyp flags
    const int64_t* hyp_off;      // n_tmpl + 1: the hypotheses of template t are [hyp_off[t], hyp_off[t+1])
    const float2* anchors;       // n_tmpl template anchors (bounding-box centres)
    int64_t n_hyp;
    int32_t n_tmpl, tmpl_idx_base;
    int32_t top_k;
    int32_t cap;                 // max_per_template (0: none)
    int32_t radius_on, any_angle;
    float r2, cos_thr;           // radius * radius, (float)cos((double)max_angle)
    const float* rec_scale;      // n_hyp grid scales of the scaled dense search (angle test cos_thr * (s_a * s_b)), or nullptr
};
constexpr int kSelectMaxAcross = FDCM_SELECT_MAX_ACROSS;   // accepted list of the across-template walk (shared memory)
// bytes of CUB scratch the select sorts need for n_hyp (< 2^31) hypotheses
size_t select_temp_bytes(int64_t n_hyp);
// 1. one order-preserving key per hypothesis (score, NaN as +inf; 0xFFFFFFFF for an invalid one) and its stable radix sort
//    with the hypothesis index as value (vals_in receives the identity).  by_template: 64-bit keys (template << 32 | key),
//    so that the hypotheses of template t keep their range [hyp_off[t], hyp_off[t+1]) in (score, h) order; otherwise the
//    high half is 0: one global (score, h) order.
void launch_select_sort(const SelectLaunch& p, bool by_template, uint64_t* keys_in, uint64_t* keys_out, int32_t* vals_in,
                        int32_t* vals_out, void* d_temp, size_t temp_bytes, cudaStream_t s);
// 2a. across_templates == 0: one warp walks each template's sorted range and writes the key of every accepted hypothesis to
//     surv_keys (0xFFFFFFFF elsewhere); acc: n_hyp x 16 B of accepted anchors, read only with a radius
void launch_select_greedy(const SelectLaunch& p, const uint64_t* sorted_keys, const int32_t* sorted_h, uint32_t* surv_keys, float4* acc,
                          cudaStream_t s);
// 3a. the first top_k survivors in (score, h) order: stable sort of surv_keys (values: the identity in vals_in), gather
void launch_select_topk(const SelectLaunch& p, const uint32_t* surv_keys, uint32_t* keys_out, const int32_t* vals_in, int32_t* vals_out,
                        void* d_temp, size_t temp_bytes, fdcm_match* d_out, int* d_n_out, cudaStream_t s);
// 2b. across_templates != 0 (top_k <= kSelectMaxAcross): one block walks the global order, accepted list in shared memory
void launch_select_walk(const SelectLaunch& p, const uint64_t* sorted_keys, const int32_t* sorted_h, fdcm_match* d_out, int* d_n_out,
                        cudaStream_t s);
// d_out[0, top_k) + *d_n_out are written like the top-K kernels' (unused slots: tmpl_idx -1, score +inf).

// pose refinement (fdcm_refine_matches / fdcm_search_refine; rules in include/fdcm_b200.h)
constexpr int kRefineSide = 2 * FDCM_REFINE_MAX_STEPS + 1;
struct RefineLevel {             // host-computed table of one level
    float ci[kRefineSide], si[kRefineSide];   // index i + rot_steps
    float h;                     // trans_step * 2^-level
};
struct RefineState { float c[6]; float raw; int32_t valid; };   // running centre C, its raw score, any valid pose yet
struct RefineLaunch {
    const fdcm_match* in;        // the matches (tmpl_idx, transform M)
    const int* d_n;              // number of matches on the device (fused path), or nullptr: n
    int32_t n;                   // slots (the grid covers n matches)
    const float4* lines;         // template set
    const int32_t* offsets;
    const float2* anchors;
    const float* denom;          // per template penalty denominator, or nullptr
    int32_t tmpl_idx_base;
    int32_t n_r, n_t;
    RefineState* state;          // n
    unsigned long long* keys;    // n: (score bits << 32 | walk order << 1 | score is NaN) of the level's best, ~0 when none
};
// the pose of a grid point with rotation index i (cos ci, sin si) around the anchor (ax, ay) of C, before dx / dy
struct RefineRot { float r0, r1, r3, r4, bx, by; };
__host__ __device__ inline RefineRot refine_rotation(const float* c, float ax, float ay, int i, float ci, float si) {
    if (i == 0) return RefineRot{c[0], c[1], c[3], c[4], c[2], c[5]};
    const float px = (c[0] * ax + c[1] * ay) + c[2], py = (c[3] * ax + c[4] * ay) + c[5];
    const float ux = c[2] - px, uy = c[5] - py;
    return RefineRot{ci * c[0] - si * c[3], ci * c[1] - si * c[4], si * c[0] + ci * c[3], si * c[1] + ci * c[4],
                     (ci * ux - si * uy) + px, (si * ux + ci * uy) + py};
}
void launch_refine_init(const RefineLaunch& p, cudaStream_t s);
// one level: one block per (match, rotation), one thread per translation (k, j); atomicMin of the key per match
cudaError_t launch_refine_eval(const MapView& map, const SlopeTableDev& table, const RefineLaunch& p, const RefineLevel& lv,
                               int max_lines, int smem_optin, cudaStream_t s);
// the level's argmin becomes the centre; out != nullptr (last level): writes the refined matches
void launch_refine_advance(const RefineLaunch& p, const RefineLevel& lv, fdcm_match* out, cudaStream_t s);

// dense pose-grid search (fdcm_search_dense; rules in include/fdcm_b200.h)
struct DenseLaunch {
    const float4* lines;         // template set
    const int32_t* offsets;
    const float2* anchors;
    const float2* rot;           // (c_r, s_r) of every rotation; scaled: (a_kr, b_kr) at k * rotations + r
    const float* denom;          // per template penalty denominator, or nullptr; scaled: per (t, k) at t * scales + k
    int32_t n_tmpl, rotations, tmpl_idx_base;
    int32_t scales;              // 1 for the unscaled search
    const float* scale;          // scaled: the s_k, or nullptr
    float* rec_scale;            // scaled: n_rec grid scales of the records, written for the valid ones (or nullptr)
    int32_t lo_x, lo_y, stride;  // grid point (u, v) is the map pixel (lo_x + u stride, lo_y + v stride)
    int32_t nx, ny;              // grid points per row / column
    int32_t cell, cells_x, cells_y;
    int32_t band;                // cell rows per block of the evaluation kernel
    int32_t n_bands;             // ceil(cells_y / band)
    int64_t n_rec;               // n_tmpl * scales * rotations * cells_y * cells_x
    unsigned long long* keys;    // n_rec: (score bits << 32 | grid index << 1 | score is NaN) of the cell's best, ~0 when none
    fdcm_match* rec;             // n_rec records and valid flags (the search's record buffers)
    uint8_t* valid;
};
// translation of the grid pose whose anchor lands on map pixel (gx, gy): the same arithmetic on the host and the device
__host__ __device__ inline float dense_tx(float c, float s, float ax, float ay, int gx, float shift_x) {
    return ((float)gx - shift_x) - (c * ax - s * ay);
}
__host__ __device__ inline float dense_ty(float c, float s, float ax, float ay, int gy, float shift_y) {
    return ((float)gy - shift_y) - (s * ax + c * ay);
}
__host__ __device__ inline void dense_pose(float c, float s, float ax, float ay, int gx, int gy, float shift_x, float shift_y, float* P) {
    P[0] = c; P[1] = -s; P[2] = dense_tx(c, s, ax, ay, gx, shift_x);
    P[3] = s; P[4] = c;  P[5] = dense_ty(c, s, ax, ay, gy, shift_y);
}
// one block per (template, scale, rotation, band of cell rows); atomicMin of the key per record.  keys must hold ~0 on entry.
cudaError_t launch_dense_eval(const MapView& map, const SlopeTableDev& table, const DenseLaunch& p, int max_lines, int smem_optin,
                              cudaStream_t s);
// keys -> records and valid flags (the winning pose recomputed from its grid index, the penalty applied)
void launch_dense_finish(const MapView& map, const DenseLaunch& p, cudaStream_t s);

// ---- coverage_kernels.cu: match verification (fdcm_match_coverage / the coverage filter; rules in include/fdcm_b200.h) ----
// the dilated edge mask of (radius, tol), the mask's layout; d_tmp: scratch of the mask's size
void launch_coverage_dilate(const uint32_t* d_mask, const MapDims& dm, int radius, int tol, uint32_t* d_tmp, uint32_t* d_dil,
                            cudaStream_t s);
struct CoverageLaunch {
    const uint32_t* dil;         // dilated mask [D][H][wwords]
    MapDims dm;
    float shift_x, shift_y;
    const fdcm_match* rec;       // n matches
    int64_t n;
    const float4* lines;         // template set
    const int32_t* offsets;
    int32_t n_tmpl, tmpl_idx_base;
    float* coverage;             // standalone: n coverages (valid == nullptr)
    uint8_t* valid;              // filter: the records' flags, cleared below min_coverage (coverage == nullptr)
    float min_coverage;
};
// one warp per match
void launch_coverage_eval(const CoverageLaunch& p, const SlopeTableDev& table, cudaStream_t s);

// ---- fit_kernels.cu: pose fit (fdcm_fit_matches; rules in include/fdcm_b200.h) ----
constexpr int kFitCell = 16;     // side of a cell of the scene-line grid, in map pixels
// samples of a template line (rule 2): the same arithmetic on the host (fdcm_fit_samples) and the device
__host__ __device__ inline int fit_line_samples(float x1, float y1, float x2, float y2, float step) {
    const float dx = x2 - x1, dy = y2 - y1;
    const float len = sqrtf(dx * dx + dy * dy);
    if (!(len > 0.f)) return 0;
    const int n = (int)ceilf(len / step) + 1;
    return n < 2 ? 2 : n;
}
__host__ __device__ inline void fit_sample(float x1, float y1, float x2, float y2, int i, int n, double& sx, double& sy) {
    const double f = (double)i / (double)(n - 1);
    sx = (double)x1 + ((double)x2 - (double)x1) * f;
    sy = (double)y1 + ((double)y2 - (double)y1) * f;
}
// the scene-line grid of (map, max_distance): cells gx x gy; the lines of cell c are items[off[c] .. off[c + 1])
size_t fit_grid_scan_bytes(int n_cells);
// pass 0: per-cell counts into cnt (zeroed, n_cells + 1 entries); then an exclusive scan of cnt into off
void launch_fit_grid_count(const float4* d_lines, int n_lines, float max_distance, int gx, int gy, unsigned long long* d_cnt,
                           unsigned long long* d_off, void* d_temp, size_t temp_bytes, cudaStream_t s);
// pass 1: the line indices into items; d_cursor: n_cells zeroed counters
void launch_fit_grid_fill(const float4* d_lines, int n_lines, float max_distance, int gx, int gy, const unsigned long long* d_off,
                          unsigned long long* d_cursor, int32_t* d_items, cudaStream_t s);
struct FitLaunch {
    MapView map;
    const float4* scene;         // the build scene's lines in map coordinates, and their bins
    const int32_t* scene_bins;
    const unsigned long long* cell_off;   // gx * gy + 1
    const int32_t* cell_items;
    int32_t gx, gy;
    const fdcm_match* in;        // n matches
    int64_t n;
    const float4* lines;         // template set
    const int32_t* offsets;
    const float2* anchors;
    const float* denom;          // per template penalty denominator, or nullptr
    int32_t tmpl_idx_base;
    fdcm_fit_params prm;
    fdcm_match* out;             // n records
    fdcm_fit_stats* stats;       // n entries
    int32_t scaled;              // 0: the rigid fit; 1: the scaled fit within [min_scale, max_scale]
    float min_scale, max_scale;
};
// one warp per match; the rigid and the scaled fit are two instantiations of one kernel
void launch_fit_eval(const FitLaunch& p, const SlopeTableDev& table, cudaStream_t s);

void launch_evaluate(const MapView& map, const SlopeTableDev& table, const float4* d_lines, const int32_t* d_toff,
                     const float2* d_transl, const int32_t* d_troff, const int32_t* d_owner, int64_t n_scores,
                     float* d_scores, cudaStream_t s);
void launch_classify(const SlopeTableDev& table, const float4* d_lines, int n, int32_t* d_bins, cudaStream_t s);

}   // namespace fdcm
