/* fdcm_b200.h — C ABI of the B200-native OpenFDCM hot paths (libfdcm_b200.so).
 *
 * Drop-in boundary for the two data-parallel hot paths of Innoptech/OpenFDCM v0.10.0:
 *   (1) the DT3 feature-map build      (reference: buildCpuFeaturemap, matching/featuremaps/dt3cpu.h:174-234)
 *   (2) template search / optimise / match (reference: search<DefaultMatch>, matching/src/matchstrategies/defaultmatch.cpp:32-89)
 * Everything behind this header is hand-written sm_100a CUDA; there is NO CPU fallback: every
 * compute entry point returns FDCM_ERR_CUDA when no device is usable.
 *
 * Conventions
 *   - line arrays are packed float32 records [x1,y1,x2,y2] (the column-major memory image of the
 *     reference's `LineArray = Eigen::Matrix<float,4,-1>`, core/math.h:66);
 *   - 2x3 transforms are row-major [r00 r01 tx r10 r11 ty] (values of core::Mat23, math.h:64);
 *   - plain pointers + sizes, caller owns every host buffer, the library owns opaque handles;
 *   - every function returns an fdcm_status; fdcm_last_error() gives the message (thread-local);
 *   - nothing throws across this boundary; empty inputs are not errors (empty scene -> empty map,
 *     like dt3cpu.h:180-181; no templates -> no matches, like defaultmatch.cpp:40-41).
 *
 * `path:line` citations are relative to the reference tree.
 */
#ifndef FDCM_B200_H
#define FDCM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDCM_B200_ABI_VERSION 3

typedef enum fdcm_status {
    FDCM_OK = 0,
    FDCM_ERR_INVALID = 1,      /* bad argument */
    FDCM_ERR_CUDA = 2,         /* CUDA runtime failure / no device */
    FDCM_ERR_NOMEM = 3,        /* host or device allocation failed */
    FDCM_ERR_OUT_OF_RANGE = 4, /* penalize: tmpl_idx outside templatelengths (exponentialpenalty.cpp:47-62) */
    FDCM_ERR_CAPACITY = 5      /* output buffer too small; *n_out holds the required count */
} fdcm_status;

/* core::Distance (core/imgproc.h:148) — same numeric values */
typedef enum fdcm_distance { FDCM_L2 = 0, FDCM_L2_SQUARED = 1, FDCM_L1 = 2 } fdcm_distance;

/* Dt3CpuParameters (dt3cpu.h:34-42) + the runtime distance of PyDt3CpuParameters (python/src/matching.cpp:51-60) */
typedef struct fdcm_dt3_params {
    int32_t depth;      /* number of orientation planes, 1..64 (reference default 30) */
    float dt3_coeff;    /* orientation propagation coefficient (default 5) */
    float padding;      /* padding ratio (default 2.2) */
    int32_t distance;   /* fdcm_distance */
} fdcm_dt3_params;

/* matching::Match (matchstrategy.h:35-44): 32-byte POD */
typedef struct fdcm_match {
    int32_t tmpl_idx;
    float score;
    float transform[6];
} fdcm_match;

typedef enum fdcm_penalty_kind { FDCM_PENALTY_NONE = 0, FDCM_PENALTY_DEFAULT = 1, FDCM_PENALTY_EXPONENTIAL = 2 } fdcm_penalty_kind;

/* DefaultSearch(max_tmpl_lines, max_scene_lines) (searchstrategies/defaultsearch.h:53-66),
 * BatchOptimize(batch_size) (optimizestrategies/batchoptimize.h:8-23; batch_size == 0 selects the
 * step-1 DefaultOptimize rules, defaultoptimize.cpp:49-64), optional fused penalty
 * (penaltystrategies/{default,exponential}penalty.cpp) and top-K (sortMatches(matches, n), matchstrategy.h:52-55). */
typedef struct fdcm_search_params {
    int32_t max_tmpl_lines;
    int32_t max_scene_lines;
    int32_t batch_size;
    int32_t penalty_kind;   /* fdcm_penalty_kind */
    float penalty_tau;
    int32_t top_k;          /* 0 = every match in hypothesis order (the reference's search() result);
                               >0 = the top_k best (ascending score, ties by hypothesis order) */
    int32_t tmpl_idx_base;  /* added to tmpl_idx in the emitted matches (template sharding keeps global indices) */
    /* ConcentricRangeStrategy (searchstrategies/concentricrange.h:35-60): when concentric != 0 only the scene lines whose
     * centre lies at a radius in (low_radius - eps, high_radius) of (center_x, center_y) take part in the search */
    int32_t concentric;
    float center_x, center_y, low_radius, high_radius;
} fdcm_search_params;

typedef struct fdcm_dt3_info {
    int32_t depth;
    int32_t width, height;          /* feature size (dt3cpu.h:57 getFeatureSize) */
    int32_t pitch;                  /* row pitch of the device planes, in floats */
    float scene_translation[2];     /* dt3cpu.h:56 getSceneTranslation */
    int32_t distance;
    int32_t device;
    int32_t n_scene_lines;
    int32_t exact_dt_path;          /* 1: integer-exact fast DT path (side <= 2897), 0: literal general path */
} fdcm_dt3_info;

/* counters of the last search on a feature map (SURVEY.md §8d) */
typedef struct fdcm_search_stats {
    int64_t n_hypotheses;
    int64_t n_valid;        /* hypotheses with a value (not nullopt) */
    int64_t n_evaluations;  /* candidate translations scored */
    int64_t n_lookups;      /* feature-map gathers = 2 * lines * evaluations */
} fdcm_search_stats;

typedef struct fdcm_dt3 fdcm_dt3;               /* device feature map: [depth][height][pitch] fp32 planes */
typedef struct fdcm_templates fdcm_templates;   /* device-resident template set */
typedef struct fdcm_comm fdcm_comm;             /* multi-GPU communicator of one rank (one process per GPU, NCCL) */
typedef struct fdcm_scene_batch fdcm_scene_batch;   /* double-buffered maps + build stream of a multi-scene batch */

const char* fdcm_last_error(void);
int32_t fdcm_abi_version(void);
fdcm_status fdcm_device_count(int32_t* n);
/* Run every kernel of this library on a caller-owned CUDA stream (e.g. torch's current stream) of `device`;
 * NULL restores the library's own stream.  The change applies to later calls; work already queued on a map (an
 * asynchronous rebuild or rerun) stays ordered before every later call on that map, whatever stream that call uses. */
fdcm_status fdcm_set_stream(int32_t device, void* cuda_stream);

/* ---- hot path 1: feature map -------------------------------------------------------------- */
/* buildCpuFeaturemap<D>(scene, params, pool) (dt3cpu.h:174-234). Blocking. `stage`: 0 = full map,
 * 1 = stop after the distance transforms, 2 = stop after propagateOrientation (parity tests only). */
fdcm_status fdcm_dt3_build(const float* scene_xyxy, int32_t n_lines, const fdcm_dt3_params* params, int32_t device,
                           int32_t stage, fdcm_dt3** out);
/* Same map object, new scene: reuses the device allocations when the new map fits. */
fdcm_status fdcm_dt3_rebuild(fdcm_dt3* map, const float* scene_xyxy, int32_t n_lines);
/* fdcm_dt3_rebuild without the final wait: returns once the build kernels are queued on the current stream; they are
 * ordered before any later call on this map, on any stream (the map records an event that every call waits on).  Lets
 * host-side preparation of the following search overlap the device build. */
fdcm_status fdcm_dt3_rebuild_async(fdcm_dt3* map, const float* scene_xyxy, int32_t n_lines);
/* Re-run the build kernels on the scene lines already resident on the device (kernel-only timing). */
fdcm_status fdcm_dt3_rerun(fdcm_dt3* map);
/* fdcm_dt3_rerun without the final wait (ordered before any later call on this map, on any stream). */
fdcm_status fdcm_dt3_rerun_async(fdcm_dt3* map);
fdcm_status fdcm_dt3_retain(fdcm_dt3* map);
fdcm_status fdcm_dt3_release(fdcm_dt3* map);
fdcm_status fdcm_dt3_get_info(const fdcm_dt3* map, fdcm_dt3_info* info);
/* the `depth` angle keys in plane order (dt3cpu.h:188-190) */
fdcm_status fdcm_dt3_angles(const fdcm_dt3* map, float* keys);
/* Dt3Cpu::getDt3Map()[angle_i] as a dense row-major height x width image (python: get_dt3_map) */
fdcm_status fdcm_dt3_download_plane(const fdcm_dt3* map, int32_t plane, float* dst);
/* rasterised edge mask of plane i (1 = edge pixel), height x width bytes (drawLines, core/drawing.h:111-125) */
fdcm_status fdcm_dt3_download_mask(const fdcm_dt3* map, int32_t plane, uint8_t* dst);
/* orientation plane of each scene line (classifyLines, dt3cpu.h:123-134) */
fdcm_status fdcm_dt3_scene_bins(const fdcm_dt3* map, int32_t* bins);
/* raw device pointer of the planes (for zero-copy consumers, e.g. torch.from_blob / NCCL broadcast).  Reads through it
 * are the caller's to order: after an asynchronous rebuild or rerun, read on the stream it was queued on or synchronise. */
fdcm_status fdcm_dt3_device_ptr(const fdcm_dt3* map, void** planes, uint64_t* n_bytes);

/* minmaxTranslation<Dt3Cpu>(featuremap, tmpl, align_vec) (dt3cpu.cpp:119-124, :30-75) */
fdcm_status fdcm_dt3_minmax_translation(const fdcm_dt3* map, const float* tmpl_xyxy, int32_t n_lines,
                                        const float align_vec[2], float out_min_max[2]);
/* evaluate<Dt3Cpu>(featuremap, templates, translations) (dt3cpu.cpp:126-179).
 * templates: CSR (tmpl_lines, tmpl_offsets[n_tmpl+1]); translations: CSR of (x,y) pairs
 * (translations, transl_offsets[n_tmpl+1]); scores: transl_offsets[n_tmpl] floats. */
fdcm_status fdcm_dt3_evaluate(const fdcm_dt3* map, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                              const float* translations, const int32_t* transl_offsets, float* scores);
/* closestOrientation (dt3cpu.h:93-114) of arbitrary lines against this map's planes, computed on the
 * device through the slope-threshold table (parity hook for the bin assignment of template lines) */
fdcm_status fdcm_dt3_classify(const fdcm_dt3* map, const float* lines_xyxy, int32_t n_lines, int32_t* bins);

/* ---- hot path 2: search ------------------------------------------------------------------- */
/* Upload a template set once (templates are typically static across scenes). */
fdcm_status fdcm_templates_create(const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl, int32_t device,
                                  fdcm_templates** out);
fdcm_status fdcm_templates_release(fdcm_templates* t);
/* getTemplateLengths (core/math.h:319-324) */
fdcm_status fdcm_templates_lengths(const fdcm_templates* t, float* lengths);

/* search(DefaultMatch, DefaultSearch, BatchOptimize|DefaultOptimize, featuremap, templates, scene)
 * (defaultmatch.cpp:32-89) [+ penalize + sort/top-k]. `scene_xyxy` is the ORIGINAL scene
 * (un-shifted), as in the reference; n_scene == 0 yields no matches (defaultmatch.cpp:40) and
 * n_scene == FDCM_SCENE_RESIDENT (scene_xyxy ignored) searches the scene the map was built from, which is
 * already resident on the device.  out: capacity records; *n_out = number written (or required
 * when FDCM_ERR_CAPACITY).
 * Template size limit: the search kernel keeps the aligned copy of the longest template of the set in shared memory,
 * 16 L + round_up(L, 16) bytes per hypothesis in flight and at least one per block.  On a device with S bytes of opt-in
 * shared memory per block (cudaDevAttrMaxSharedMemoryPerBlockOptin; 232448 on a B200) the longest template may have
 * L lines with 16 L + round_up(L, 16) <= S: 13673 lines on a B200.  A set holding a longer template fails with
 * FDCM_ERR_INVALID (the message states the limit); so do fdcm_optimize and fdcm_search_scenes.  Templates of up to
 * S / 68 lines (3418 on a B200) run 4 hypotheses per block, longer ones 2 or 1. */
#define FDCM_SCENE_RESIDENT (-1)
fdcm_status fdcm_search(const fdcm_dt3* map, const fdcm_templates* templates, const float* scene_xyxy, int32_t n_scene,
                        const fdcm_search_params* params, fdcm_match* out, int64_t capacity, int64_t* n_out);
/* ---- distinct top-K (beyond the reference) -------------------------------------------------
 * Many hypotheses of one template converge on the same pose, so a plain top-K is mostly repeats.  The *_select entry
 * points run the search like fdcm_search (top_k > 0, penalty, ConcentricRange and tmpl_idx_base as there) and then
 * select on the device, from the valid matches ordered by ascending (score, hypothesis index), NaN as +inf:
 * walk that order with an accepted list A (empty at first) and accept a candidate b iff
 *   |A| < top_k, and
 *   max_per_template == 0 or A holds fewer than max_per_template matches of b's template, and
 *   radius == 0 or no a in A with near(a, b) has (across_templates || a's template == b's template);
 * the result is A in acceptance order.  max_per_template == 0 and radius == 0 give exactly fdcm_search's top-K.
 * near(a, b), in fp32 without contraction: the anchor of a template is the centre of the bounding box of its 2L end
 * points ((min + max) * 0.5f per axis; (0, 0) for an empty template), the anchor of a match with transform T is
 * ((T0*ax + T1*ay) + T2, (T3*ax + T4*ay) + T5); near holds iff dx*dx + dy*dy <= radius*radius for the difference of the
 * two anchors and either max_angle >= 3.14159274f or Ta0*Tb0 + Ta3*Tb3 >= (float)cos((double)max_angle) (a reversed
 * hypothesis carries -R, a rotation by pi).
 * Cost: with across_templates == 0 every template is walked by its own warp (each rule only involves matches of one
 * template, so this is the global walk); with across_templates != 0 one thread block walks the sorted list, worst case
 * H x top_k anchor tests for H hypotheses, and top_k may not exceed FDCM_SELECT_MAX_ACROSS (the accepted list lives in
 * shared memory).  Invalid parameters (top_k < 1, max_per_template < 0, radius negative or not finite, max_angle
 * negative or NaN, that bound) fail with FDCM_ERR_INVALID. */
#define FDCM_SELECT_MAX_ACROSS 1024
typedef struct fdcm_select_params {      /* 16 bytes */
    int32_t max_per_template;   /* > 0: at most this many matches of one template; 0: no cap */
    float radius;               /* > 0: suppression radius (pixels) between match anchors; 0: no suppression */
    float max_angle;            /* radians; with radius > 0, suppress only within this rotation; >= pi: any rotation */
    int32_t across_templates;   /* 0: a match suppresses matches of its own template only; 1: of every template */
} fdcm_select_params;
fdcm_status fdcm_search_select(const fdcm_dt3* map, const fdcm_templates* templates, const float* scene_xyxy, int32_t n_scene,
                               const fdcm_search_params* params, const fdcm_select_params* select,
                               fdcm_match* out, int64_t capacity, int64_t* n_out);
/* anchors of n_tmpl templates (CSR like fdcm_template_lengths), n_tmpl (x, y) pairs; host only */
fdcm_status fdcm_template_anchors(const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl, float* anchors_xy);

/* ---- pose refinement (beyond the reference) -----------------------------------------------------
 * A search match aligns one template line with one scene line, so its rotation is that scene line's direction and its
 * translation moves along that line only.  Refinement walks a coarse-to-fine grid of rotations and 2-D translations
 * around each match and keeps the pose with the lowest evaluate<Dt3Cpu> score over all template lines.
 * It minimises that score and nothing else.  At sub-pixel and 0.01 rad scales the score is not lowest at the true pose
 * (a noise-free instance scores far lower a pixel or 0.01 rad away), so refinement was measured to INCREASE the error
 * against known poses, also when started at the exact pose (DESIGN.md section 4).
 * Rules, in fp32 without contraction, in the order written.  For a match with transform M = (m0..m5) and template t:
 *   1. Centre.  The walk starts with C = M.  At every level the rotation centre is p = C applied to the anchor a of t
 *      (fdcm_template_anchors): px = (c0*ax + c1*ay) + c2, py = (c3*ax + c4*ay) + c5.
 *   2. Grid of level l (0-based): i in [-rot_steps, rot_steps], k and j in [-trans_steps, trans_steps];
 *      ci = (float)cos((double)i * ((double)rot_step / 2^l)), si likewise with sin (host C library);
 *      h = trans_step * 2^-l, dx = (float)j * h, dy = (float)k * h.
 *   3. Candidate P.  i != 0: P0 = ci*c0 - si*c3, P1 = ci*c1 - si*c4, P3 = si*c0 + ci*c3, P4 = si*c1 + ci*c4,
 *      ux = c2 - px, uy = c5 - py, P2 = ((ci*ux - si*uy) + px) + dx, P5 = ((si*ux + ci*uy) + py) + dy.
 *      i == 0 keeps C's rotation: P = (c0, c1, c2 + dx, c3, c4, c5 + dy).  The grid point (0, 0, 0) is C itself.
 *   4. Score of P: evaluate<Dt3Cpu>(map, {R_P tmpl}, {(P2, P5)}) (fdcm_dt3_evaluate): end point (x, y) -> (P0*x + P1*y,
 *      P3*x + P4*y); orientation bin from the slope of the rotated line; lookups (int)(r + (shift + P2)); Eigen's sum
 *      order.  P is valid iff no entry of P and no rotated end point is NaN and every rotated end point has
 *      0 <= rx + (shift_x + P2) <= W - 1 and 0 <= ry + (shift_y + P5) <= H - 1 (an empty template: any P without NaN).
 *      Invalid poses are neither evaluated nor read.
 *   5. Walk.  The grid points by ascending i*i + k*k + j*j (the centre first), equal distances in ascending (i, k, j).
 *      A valid candidate replaces the running best iff there is none yet or its score is lower (NaN as +inf, strict: ties
 *      keep the earlier candidate, so the centre wins ties and a plateau of equal scores resolves to its point nearest
 *      the centre).  The best of level l is the centre of level l + 1; a level without a valid pose keeps C.
 *   6. Result.  tmpl_idx unchanged; the transform is the final best pose; the score is its raw score, divided by the
 *      search's penalty denominator (host powf of the template length) when a penalty is given.  No valid pose at any
 *      level: transform M, score NaN.  Output i is the refinement of input i (not re-sorted; fdcm_sort_matches re-ranks).
 * Invalid parameters (levels < 1, rot_steps or trans_steps outside 0..FDCM_REFINE_MAX_STEPS, a negative or non-finite
 * step, a null refine pointer, a template longer than the search accepts) fail with FDCM_ERR_INVALID; a tmpl_idx -
 * tmpl_idx_base outside the template set fails with FDCM_ERR_OUT_OF_RANGE.
 * Cost per level and match: (2 rot_steps + 1)(2 trans_steps + 1)^2 poses of 2 L map gathers each. */
#define FDCM_REFINE_MAX_STEPS 15
typedef struct fdcm_refine_params {      /* 20 bytes */
    int32_t levels;             /* >= 1: coarse-to-fine levels; steps halve at every level */
    int32_t rot_steps;          /* n_r: rotations i * rot_step / 2^l, i in [-n_r, n_r] */
    float rot_step;             /* radians */
    int32_t trans_steps;        /* n_t: translations (j, k) * trans_step / 2^l, j, k in [-n_t, n_t] */
    float trans_step;           /* pixels */
} fdcm_refine_params;
/* refine n host matches (search output or from elsewhere) against a map and a resident template set; n == 0 is no error */
fdcm_status fdcm_refine_matches(const fdcm_dt3* map, const fdcm_templates* templates, int32_t tmpl_idx_base, int32_t penalty_kind,
                                float penalty_tau, const fdcm_refine_params* refine, const fdcm_match* in, int64_t n,
                                fdcm_match* out);
/* fdcm_search (top_k > 0) or, with select != NULL, fdcm_search_select, then refinement of the selected matches on the
 * device and one download: byte-identical to fdcm_refine_matches applied to their output */
fdcm_status fdcm_search_refine(const fdcm_dt3* map, const fdcm_templates* templates, const float* scene_xyxy, int32_t n_scene,
                               const fdcm_search_params* params, const fdcm_select_params* select,
                               const fdcm_refine_params* refine, fdcm_match* out, int64_t capacity, int64_t* n_out);
/* the candidate transforms of one level (0 <= level < levels) in grid order, 6 floats each,
 * (2 rot_steps + 1)(2 trans_steps + 1)^2 of them; host-only parity hook */
fdcm_status fdcm_refine_poses(const float transform[6], const float anchor[2], const fdcm_refine_params* refine, int32_t level,
                              float* out);

/* ---- dense pose-grid search (beyond the reference) ----------------------------------------------
 * The search above only poses a template where one of its longest lines lies on one of the scene's longest lines, so a
 * broken, merged or missing scene line leaves no hypothesis.  The dense search scores every template at a grid of
 * rotations about its anchor and translations that put the anchor on a grid of map pixels, keeps the best pose of every
 * cell of the grid and passes those records through the search's top-K or distinct selection, then optionally refinement.
 * The grid is finite: before refinement a pose is off by up to stride / 2 px and rot_step / 2 rad, and like refinement
 * it minimises the evaluate<Dt3Cpu> score, which is not lowest at the true pose at sub-pixel scales.
 * Rules, in fp32 without contraction.  Map W x H, scene translation shift = (shift_x, shift_y), templates t = 0..T-1:
 *   1. Rotations r = 0..rotations-1: theta_r = (double)rot_start + r * (double)rot_step, c_r = (float)cos(theta_r),
 *      s_r = (float)sin(theta_r) (host C library).
 *   2. Grid.  Map-pixel range [lo_x, hi_x] x [lo_y, hi_y]: [0, W-1] x [0, H-1], or with roi_on and roi = (x0, y0, x1, y1)
 *      in scene coordinates lo_x = max(0, ceil(x0 + shift_x)), hi_x = min(W-1, floor(x1 + shift_x)) evaluated in double,
 *      y likewise.  Grid point (u, v) is the map pixel (gx, gy) = (lo_x + u stride, lo_y + v stride), for every such
 *      point inside the range: nx = (hi_x - lo_x) / stride + 1 per row (0 when lo_x > hi_x), ny likewise.  Grid index
 *      g = v nx + u (row-major).
 *   3. Pose with anchor a (fdcm_template_anchors): qx = (float)gx - shift_x, qy = (float)gy - shift_y,
 *      P = (c, -s, qx - (c*ax - s*ay), s, c, qy - (s*ax + c*ay)).  When c == 1 and s == 0 the end points are used exactly
 *      as given, without a multiply (-s * y would turn the zero dx of a vertical line negative and flip its orientation
 *      bin), so the theta = 0 slice is fdcm_dt3_evaluate of the template itself.
 *   4. Score and validity: refinement rule 4 (rotated end points (P0*x + P1*y, P3*x + P4*y), orientation bin from the
 *      rotated slope, lookups (int)(r + (shift + P2)), Eigen's sum order; valid iff nothing is NaN and the rotated end
 *      points lie inside the map); invalid poses are never read.  An empty template has no valid pose.
 *   5. Cells.  Grid point (u, v) is in cell (cu, cv) = (u / cell, v / cell); cells_x = ceil(nx / cell), cells_y likewise.
 *      Record h = ((t * rotations + r) * cells_y + cv) * cells_x + cu is valid iff its cell has a valid pose; its pose is
 *      the valid pose of the cell with the lowest raw score (NaN as +inf), ties to the lowest grid index; its score is the
 *      raw score, divided by the search's penalty denominator of t (host powf of the template length) when a penalty is
 *      given (the argmin is taken on the raw score); tmpl_idx = t + tmpl_idx_base.
 *   6. Output: the valid records like fdcm_search's hypothesis records: the top_k best in (score, h) order, or with select
 *      the walk of fdcm_search_select; then with refine the refinement of those, byte-identical to fdcm_refine_matches of
 *      the unrefined output.
 * Invalid parameters fail with FDCM_ERR_INVALID: rotations outside 1..FDCM_DENSE_MAX_ROTATIONS, stride < 1, cell < 1,
 * rot_start or rot_step not finite, a region not finite or with x0 > x1 or y0 > y1, top_k < 1, a record count of 2^31
 * or more (T * rotations * cells_y * cells_x), a template longer than the search accepts, and the select and refine
 * parameters fdcm_search_refine rejects.  An empty map, an empty template set or a grid without points (a region outside
 * the map) give no matches.  Cost: T * rotations * nx * ny poses of up to 2 L map gathers each; the dense search is
 * meant for template sets of hundreds, not thousands. */
#define FDCM_DENSE_MAX_ROTATIONS 4096
typedef struct fdcm_dense_params {       /* 40 bytes */
    int32_t rotations;          /* 1..FDCM_DENSE_MAX_ROTATIONS */
    float rot_start;            /* radians */
    float rot_step;             /* radians */
    int32_t stride;             /* >= 1: map pixels between grid points */
    int32_t cell;               /* >= 1: grid points per cell side; every cell keeps its best pose */
    int32_t roi_on;             /* 0: the whole map; 1: the region roi */
    float roi[4];               /* x0, y0, x1, y1 in scene coordinates (inclusive) */
} fdcm_dense_params;
fdcm_status fdcm_search_dense(const fdcm_dt3* map, const fdcm_templates* templates, const fdcm_dense_params* dense, int32_t penalty_kind,
                              float penalty_tau, int32_t top_k, int32_t tmpl_idx_base, const fdcm_select_params* select,
                              const fdcm_refine_params* refine, fdcm_match* out, int64_t capacity, int64_t* n_out);
/* the transforms of rotation `rotation` in grid order, 6 floats each (*n_out = nx * ny; FDCM_ERR_CAPACITY when that exceeds
 * capacity), and grid_wh = (nx, ny), for a map of W x H with scene translation shift; host-only parity hook */
fdcm_status fdcm_dense_poses(const fdcm_dense_params* dense, const float anchor[2], const float shift[2], int32_t width, int32_t height,
                             int32_t rotation, float* out, int64_t capacity, int64_t* n_out, int32_t grid_wh[2]);

/* optimize(optimizer, templates, alignments, featuremap) (matching/optimizestrategy.h:62-64; BatchOptimize:
 * batchoptimize.cpp:6-123, batch_size == 0: DefaultOptimize, defaultoptimize.cpp:6-93).  The templates are used
 * as given (already aligned); alignments: n_tmpl (x,y) pairs.  Outputs per template: has_value (0 = nullopt),
 * score and translation[2] (OptimalTranslation, optimizestrategy.h:34-38). */
fdcm_status fdcm_optimize(const fdcm_dt3* map, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                          const float* alignments, int32_t batch_size, uint8_t* has_value, float* scores,
                          float* translations);
/* one-shot variant taking host templates (uploads, searches, frees) */
fdcm_status fdcm_search_host(const fdcm_dt3* map, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                             const float* scene_xyxy, int32_t n_scene, const fdcm_search_params* params,
                             fdcm_match* out, int64_t capacity, int64_t* n_out);
/* the hypothesis list of the last fdcm_search on this map: 4 ints per hypothesis
 * (tmpl_idx, tmpl_line_idx, scene_line_idx, reversed) in hypothesis order (parity hook) */
fdcm_status fdcm_search_last_hypotheses(const fdcm_dt3* map, int32_t* out, int64_t capacity, int64_t* n_out);
fdcm_status fdcm_search_last_stats(const fdcm_dt3* map, fdcm_search_stats* stats);

/* establishSearchStrategy<DefaultSearch> for one template (defaultsearch.cpp:29-49): pairs of
 * (tmpl_line_idx, scene_line_idx); host-side helper mirroring the SearchStrategy concept. */
fdcm_status fdcm_default_search(const float* tmpl_xyxy, int32_t n_tmpl_lines, const float* scene_xyxy, int32_t n_scene,
                                int32_t max_tmpl_lines, int32_t max_scene_lines, int32_t* out_pairs, int32_t capacity,
                                int32_t* n_out);

/* establishSearchStrategy<ConcentricRangeStrategy> for one template (concentricrange.cpp:29-60) */
fdcm_status fdcm_concentric_search(const float* tmpl_xyxy, int32_t n_tmpl_lines, const float* scene_xyxy, int32_t n_scene,
                                   int32_t max_tmpl_lines, int32_t max_scene_lines, float center_x, float center_y,
                                   float low_radius, float high_radius, int32_t* out_pairs, int32_t capacity, int32_t* n_out);

/* Parity hook: run the horizontal L2^2 pass (second _distanceTransformColumnPassL2 call, core/imgproc.h:91-130)
 * on n_rows arbitrary rows of u16 vertical distances g (0xFFFF = FLT_MAX), f = g*g.  literal = 1 selects the
 * literal stack kernel (the path of maps with side > 2897), 2 the exact-regime band kernels (envelope + fill).
 * out: n_rows x n floats (squared distances). */
fdcm_status fdcm_debug_dt_rows(const uint16_t* g_rows, int32_t n_rows, int32_t n, int32_t literal, int32_t device, float* out);

/* Parity hook: the fused fill + propagate kernel takes the square root of the L2 transform (core/imgproc.h:191-192) with
 * rsqrt.approx + one Newton step instead of the general IEEE routine.  Its inputs are integers 0 .. 2^24 and FLT_MAX;
 * this call compares the two on every one of them on the device.  n_mismatches must come back 0. */
fdcm_status fdcm_debug_sqrt_check(int32_t device, int64_t* n_mismatches, uint32_t* first_mismatch);

/* Orientation bins (closestOrientation, dt3cpu.h:93-114, for the `depth` keys of dt3cpu.h:188-190) of n lines,
 * computed on the host two ways: with libm atanf (what the reference does) and through the slope-threshold
 * table the device kernels use.  Host-only parity hook: the two outputs must be identical. */
fdcm_status fdcm_orientation_bins(int32_t depth, const float* lines_xyxy, int32_t n_lines, int32_t* bins_atanf,
                                  int32_t* bins_table);

/* penalize (penaltystrategies/{default,exponential}penalty.cpp) and sort_matches
 * (python/src/matching.cpp:302-307) on host match lists — O(#matches) host helpers */
fdcm_status fdcm_penalize(int32_t penalty_kind, float tau, fdcm_match* matches, int64_t n, const float* lengths,
                          int64_t n_lengths);
fdcm_status fdcm_sort_matches(fdcm_match* matches, int64_t n);
/* getTemplateLengths without a device */
fdcm_status fdcm_template_lengths(const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl, float* lengths);

/* ---- multi-scene batches (BASELINE config 5: many scenes x one template set) ---------------------------------------
 * What a caller of the reference writes as `for scene: fm = build_cpu_featuremap(scene); search(...); penalize; sort`
 * (notebooks/pose_extimation_example.ipynb).  Scenes are CSR: scene_lines + scene_offsets[n_scenes + 1].  For every scene the
 * batch builds its DT3 map and runs the fused search -> penalize -> top-k of `params->top_k` (> 0) records against the
 * resident template set; two internal maps alternate so that the build of scene s+1 runs on a second stream under the
 * search of scene s.  out: n_scenes x top_k records (scene-major), n_out[s] = records written for scene s. */
fdcm_status fdcm_scene_batch_create(const fdcm_dt3_params* params, int32_t device, fdcm_scene_batch** out);
fdcm_status fdcm_scene_batch_destroy(fdcm_scene_batch* batch);
fdcm_status fdcm_search_scenes(fdcm_scene_batch* batch, const float* scene_lines, const int32_t* scene_offsets, int32_t n_scenes,
                               const fdcm_templates* templates, const fdcm_search_params* params, fdcm_match* out, int32_t* n_out);
/* the same with the distinct top-K selection of fdcm_search_select in every scene */
fdcm_status fdcm_search_scenes_select(fdcm_scene_batch* batch, const float* scene_lines, const int32_t* scene_offsets, int32_t n_scenes,
                                      const fdcm_templates* templates, const fdcm_search_params* params,
                                      const fdcm_select_params* select, fdcm_match* out, int32_t* n_out);

/* ---- multi-GPU (SURVEY.md 8e): one process per GPU, templates sharded by tmpl_idx, NCCL over NVLink ------------
 * The reference has no distributed code; these entry points are what a multi-GPU host (C++ or Python) calls instead of
 * looping search() over template blocks.  NCCL is resolved at run time (dlopen of libnccl.so.2); without it every
 * fdcm_comm_* call returns FDCM_ERR_CUDA.  Bootstrap like NCCL itself: rank 0 creates the id, the application ships the
 * 128 bytes to the other ranks (MPI, a file, torch.distributed ...), every rank calls fdcm_comm_init. */
#define FDCM_COMM_ID_BYTES 128
fdcm_status fdcm_comm_unique_id(uint8_t id[FDCM_COMM_ID_BYTES]);
fdcm_status fdcm_comm_init(const uint8_t id[FDCM_COMM_ID_BYTES], int32_t rank, int32_t world, int32_t device, fdcm_comm** out);
fdcm_status fdcm_comm_destroy(fdcm_comm* comm);
fdcm_status fdcm_comm_info(const fdcm_comm* comm, int32_t* rank, int32_t* world);
/* contiguous block [begin, end) of `n_items` templates (or scenes) owned by `rank`: global tmpl_idx = begin + local index */
fdcm_status fdcm_comm_shard(int32_t n_items, int32_t rank, int32_t world, int32_t* begin, int32_t* end);
/* fdcm_search (top_k > 0) of this rank's template shard (params->tmpl_idx_base = first global index of the shard), then
 * the exchange on the device: ncclAllGather of the k x 32-byte top-K buffer on the compute stream, an R*k -> k merge
 * kernel (ascending score, ties by rank then position = global hypothesis order), one download.  Every rank returns the
 * same global top-k.  Collective: every rank must call it, also with an empty shard. */
fdcm_status fdcm_comm_search_topk(fdcm_comm* comm, const fdcm_dt3* map, const fdcm_templates* shard, const float* scene_xyxy,
                                  int32_t n_scene, const fdcm_search_params* params, fdcm_match* out, int64_t capacity,
                                  int64_t* n_out);
/* fdcm_comm_search_topk with the distinct top-K selection of fdcm_search_select.  Only across_templates == 0: each rank's
 * accepted list is then the global one restricted to its templates, so the same exchange yields the global result;
 * across_templates != 0 fails with FDCM_ERR_INVALID (suppression across ranks does not decompose). */
fdcm_status fdcm_comm_search_select(fdcm_comm* comm, const fdcm_dt3* map, const fdcm_templates* shard, const float* scene_xyxy,
                                    int32_t n_scene, const fdcm_search_params* params, const fdcm_select_params* select,
                                    fdcm_match* out, int64_t capacity, int64_t* n_out);
/* the same with this rank's shard given as host templates (like fdcm_search_host: uploaded into a reusable device set) */
fdcm_status fdcm_comm_search_host_topk(fdcm_comm* comm, const fdcm_dt3* map, const float* tmpl_lines, const int32_t* tmpl_offsets,
                                       int32_t n_tmpl, const float* scene_xyxy, int32_t n_scene, const fdcm_search_params* params,
                                       fdcm_match* out, int64_t capacity, int64_t* n_out);
/* fdcm_dt3_rebuild on every rank with the kernels run on `root` only and the planes sent by ncclBroadcast (collective):
 * the alternative to every rank building the scene's map itself; bench.py measures both. */
fdcm_status fdcm_comm_rebuild_broadcast(fdcm_comm* comm, fdcm_dt3* map, const float* scene_xyxy, int32_t n_lines, int32_t root);
/* worker threads of the host-side template preparation (std::sort per template); 0 = default.  fdcm_comm_init sets
 * cores / world when it is still at the default so that the ranks of one host do not oversubscribe it. */
fdcm_status fdcm_set_host_threads(int32_t n);

/* ---- per-kernel timing (CUDA events on the launching stream; feeds bench.py's roofline) ------ */
fdcm_status fdcm_profile_enable(int32_t on);
fdcm_status fdcm_profile_reset(void);
/* n-th recorded kernel: name, total ms, launches, algorithmic bytes per launch (last launch) */
fdcm_status fdcm_profile_get(int32_t index, char* name, int32_t name_cap, double* total_ms, int64_t* launches,
                             double* bytes_per_launch);
fdcm_status fdcm_profile_count(int32_t* n);
/* number of kernels this library launched since process start */
int64_t fdcm_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FDCM_B200_H */
