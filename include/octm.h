/*
 * octm.h -- C ABI of the B200 (sm_100a) OCT segmentation-metric kernels.
 *
 * Drop-in boundary for the evaluation-metric suite of
 * ZhangHH233/Retinal_OCT_Image_Segmentation_via_Deep_Learning (directory Metrics/).  The
 * reference has no FFI: its boundary is 17 Python functions f(y_true, y_pred) -> scalar.  The
 * Python modules under retinal_oct_image_segmentation_via_deep_learning_b200/Metrics keep those
 * names and signatures and call the entry points below through ctypes (see INTEGRATION.md for
 * the stub a reference maintainer would add).
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer owned by the caller; the library never allocates,
 *     frees or synchronises; scratch comes from a caller workspace sized by a *_workspace_bytes
 *     query; every launch goes on the caller's cudaStream_t, passed as void*.
 *   - label maps are uint8 [n_items][H][W], C-contiguous, values < K (2 <= K <= 16); a value >= K
 *     is undefined behaviour for the fast kernels (checked only by octm_validate_labels_u8).
 *   - return value: OCTM_OK or a negative OCTM_ERR_*; octm_last_error() gives the thread-local
 *     message of the last failure.  The one positive status is OCTM_PACK_WIDE_LABEL of the host packer.
 *   - outputs are fully overwritten (no pre-zeroing needed) unless stated otherwise.
 */
#ifndef OCTM_H_
#define OCTM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCTM_ABI_VERSION 1

#if defined(__GNUC__)
#define OCTM_API __attribute__((visibility("default")))
#else
#define OCTM_API
#endif

#define OCTM_OK 0
#define OCTM_ERR_INVALID (-1)     /* bad pointer / shape / K */
#define OCTM_ERR_UNSUPPORTED (-2) /* shape outside what the kernels handle */
#define OCTM_ERR_LAUNCH (-3)      /* CUDA launch or attribute call failed */
#define OCTM_ERR_WORKSPACE (-4)   /* workspace too small */

/* element types of floating-point inputs (scores, probabilities, soft boundary positions) */
#define OCTM_DTYPE_F32 0
#define OCTM_DTYPE_F16 1
#define OCTM_DTYPE_BF16 2
#define OCTM_DTYPE_F64 3
#define OCTM_DTYPE_I32 4

#define OCTM_MAX_CLASSES 16
#define OCTM_NO_SEED 0xFFFFFFFFu

OCTM_API int octm_abi_version(void);
OCTM_API const char* octm_last_error(void);

/* Number of launches of this library's kernels since load (all entry points, this process). */
OCTM_API uint64_t octm_launch_count(void);

/* Per-kernel device timing for benchmarks.  octm_profile_enable(1) clears earlier records and makes every kernel
 * launch of the library record two CUDA events on its launch stream; octm_profile_enable(0) stops and clears.
 * octm_profile_report synchronises with the recorded launches and writes one line per kernel,
 * "<kernel> <launches> <total ms>\n", in first-launch order, NUL-terminated and truncated to cap bytes;
 * it returns the size the full report needs.  Off by default; not meant for timed regions. */
OCTM_API int octm_profile_enable(int on);
OCTM_API size_t octm_profile_report(char* buf, size_t cap);

/* ---------------------------------------------------------------------------------------------
 * K1  confusion matrix.  counts[i][t][p] = #{pixels of item i with y_true == t and y_pred == p}.
 * One K x K uint64 matrix per item replaces the reference's per-class recomputation of
 *   np.sum(y_true * y_pred), np.sum((1 - y_true) * (1 - y_pred)), ...
 * (Metrics/ConfusionMatrix_based_metrics.py:14-17, 30-32, 45-47, 60-62;
 *  Metrics/Region_based_metrics.py:13-15, 28-30, 43-45, 58-60; binary-mask forms of
 *  Metrics/PixelError_based_metrics.py:14-17, Metrics/Contour_based_metrics.py:68-71 and
 *  Metrics/Biomarker_based_metrics.py:34-38).  item_elems = H*W; items need not be 2-D here. */
OCTM_API int octm_confusion_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items,
                      int64_t item_elems, int num_classes, uint64_t* counts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  column (A-scan) scan.  For every item and column x:
 *   thickness_c(x) = #{y : L[y][x] == c}          (np.sum(mask, axis=0),
 *                                                  Metrics/Biomarker_based_metrics.py:14-15)
 *   boundary  b_k(x) = #{y : L[y][x] < k}, k=1..K-1 (build-defined, SURVEY.md 8a-D)
 * Outputs (any may be NULL):
 *   thick_absdiff[i][c]   = sum_x |thickness_c^true(x) - thickness_c^pred(x)|   int64 [n][K]
 *                           (numerator of thickness_difference, Biomarker_based_metrics.py:18-21)
 *   bnd_sq[i][k-1]        = sum_x (b_k^true(x) - b_k^pred(x))^2                 int64 [n][K-1]
 *   bnd_abs[i][k-1]       = sum_x |b_k^true(x) - b_k^pred(x)|                   int64 [n][K-1]
 *                           (numerators of mean_squared_error / mad on boundary arrays,
 *                            PixelError_based_metrics.py:14-17, Contour_based_metrics.py:68-71)
 *   bnd_true / bnd_pred   = b_k(x)                                              int32 [n][K-1][W] */
OCTM_API int octm_column_scan_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                        int num_classes, int64_t* thick_absdiff, int64_t* bnd_sq, int64_t* bnd_abs,
                        int32_t* bnd_true, int32_t* bnd_pred, void* stream);

/* K3  boundary-position error on caller-supplied boundary arrays int32 [n][Kb][W]
 * (e.g. positions produced by a layer model): sum_sq[i][k], sum_abs[i][k] as int64 [n][Kb]. */
OCTM_API int octm_boundary_error_i32(const int32_t* bnd_true, const int32_t* bnd_pred, int64_t n_items,
                            int num_boundaries, int W, int64_t* sum_sq, int64_t* sum_abs, void* stream);

/* K3 on CONTINUOUS boundary positions (the soft-argmax rows LayerEngine.get_layer_positions produces,
 * SOTAS/Layers_Segment/SD_Layer_Net/layer_engine.py:46-47): float64 sums of (a-b)^2 and |a-b| per
 * (item, boundary) row, i.e. the numerators of mean_squared_error (PixelError_based_metrics.py:14-17) and
 * mad (Contour_based_metrics.py:68-71) on float arrays [n][Kb][W] of dtype OCTM_DTYPE_*. */
OCTM_API int octm_boundary_error_float(const void* bnd_true, const void* bnd_pred, int dtype, int64_t n_items,
                              int num_boundaries, int64_t W, double* sum_sq, double* sum_abs, void* stream);

/* Topology violations of boundary positions [n][Kb][W] (layer_engine.py:74-76, relu(pos[k] - pos[k+1])):
 * sum_violation double [n][Kb-1], n_violations uint32 [n][Kb-1] (columns where boundary k lies below k+1). */
OCTM_API int octm_topology_violations_float(const void* positions, int dtype, int64_t n_items, int num_boundaries,
                                   int64_t W, double* sum_violation, uint32_t* n_violations, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused label pass: K1 + K2 + K3 + contour seeds in ONE read of both label tensors.
 *   counts, thick_absdiff, bnd_sq, bnd_abs, bnd_true, bnd_pred : as above, any may be NULL
 *   first_pos  uint32 [n][2][K] : raster index (y*W + x) of the first pixel of class c in y_true
 *                                 ([i][0][c]) and y_pred ([i][1][c]); OCTM_NO_SEED if absent.
 *                                 This is what locates contour [0] (see octm_contour2d_u8). */
OCTM_API int octm_label_pass_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                       int num_classes, uint64_t* counts, int64_t* thick_absdiff, int64_t* bnd_sq,
                       int64_t* bnd_abs, int32_t* bnd_true, int32_t* bnd_pred, uint32_t* first_pos,
                       void* stream);

/* The full pass (all outputs above required except the boundary rows) plus a per-item certificate of LAYERING:
 *   unsorted  uint32 [n] : bit 0 / bit 1 set when some column of y_true / y_pred is not non-decreasing from top to
 *                          bottom (0 = every A-scan of both maps crosses the classes in order).  For an item with
 *                          unsorted == 0 every class contour is a function of the boundary rows alone, which is what
 *                          lets octm_contour2d_metrics_u8 measure it without reading the label maps again.
 *                          Items taller than 500 rows are reported as unsorted (not certified). */
OCTM_API int octm_label_pass_sorted_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                              int num_classes, uint64_t* counts, int64_t* thick_absdiff, int64_t* bnd_sq,
                              int64_t* bnd_abs, int32_t* bnd_true, int32_t* bnd_pred, uint32_t* first_pos,
                              uint32_t* unsorted, void* stream);

/* Which implementation octm_label_pass_u8 / K1 / K2 would use for this shape:
 * 1 = TMA-staged column-strip kernel (K <= 8, W % 16 == 0), 2 = warp-per-strip run-length kernel (K <= 16, W % 4 == 0,
 * 4-byte aligned maps), 0 = byte-wise generic kernel. */
OCTM_API int octm_label_pass_path(int H, int W, int num_classes, const void* y_true, const void* y_pred);

/* What the suite's kernels assume about the stream of label maps -- a speed heuristic, never a difference in results:
 * 0 = follow the data (default: every certified label pass reports how many maps its certificate rejected; the next calls
 * assume a noisy stream once that was more than a fifth), 1 = assume clean (seeds from the column totals + a rescan of
 * rejected maps; confusion matrices from the boundary rows + a per-pixel histogram of the rejected items, when the call
 * asks for the boundary rows; contour stage: boundary-row pass first), 2 = assume noisy (seeds tracked per pixel and the
 * confusion histogram taken in the label pass; contour stage: the rejected maps' contours are verified against the label
 * pixels first so that the fast pass can measure them).
 * Returns the previous policy (any other argument: just reports it). */
OCTM_API int octm_label_pass_seed_policy(int policy);

/* max label over the whole tensor -> *max_label (device uint32); for input validation. */
OCTM_API int octm_validate_labels_u8(const uint8_t* labels, int64_t n_elems, uint32_t* max_label, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Contour metrics (2-D): hausdorff_distance, hausdorff_distance_95, assd of
 * Metrics/Contour_based_metrics.py:5-56, per item and class, on masks (L == c).
 * Semantics reproduced literally: only contour [0] of skimage.measure.find_contours(mask, 0.5)
 * (the iso-contour through the raster-first mixed 2x2 square; a closed contour repeats one
 * vertex).  Vertices live on the doubled lattice (2H-1) x (2W-1); all distances are exact integer
 * squared lattice distances D2, so a reference distance is sqrt(D2 / 4.0) bit-exactly.
 *
 * Per (item i, class c); direction 0 = "for each pred vertex, nearest true vertex" (d1 of the
 * reference), direction 1 = "for each true vertex, nearest pred vertex" (d2):
 *   n_pts     uint32 [n][K][2]    vertices of contour [0] of y_true ([0]) / y_pred ([1]) incl. the
 *                                 closing repeat; 0 = mask has no contour (reference: IndexError)
 *   flags     uint32 [n][K]       OCTM_CF_* bits
 *   max_sq    uint32 [n][K][2]    max D2 per direction
 *   p95_sq    uint32 [n][K][2][2] the two order statistics D2[lo], D2[lo+1] that numpy's linear
 *                                 95th percentile interpolates, lo = floor(0.95*(m-1)) computed
 *                                 as numpy does; m = number of query vertices of the direction
 *   sum_dist  double [n][K][2]    sum over query vertices of sqrt(D2 / 4.0)
 * max_pts bounds the vertices kept per contour (workspace); longer contours set an overflow flag
 * and their outputs are invalid -- the host retries those items with a larger bound. */
#define OCTM_CF_TRUE_CLOSED 1u
#define OCTM_CF_PRED_CLOSED 2u
#define OCTM_CF_TRUE_OVERFLOW 4u
#define OCTM_CF_PRED_OVERFLOW 8u

OCTM_API size_t octm_contour2d_workspace_bytes(int64_t n_items, int H, int W, int num_classes, int max_pts);

OCTM_API int octm_contour2d_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                      int num_classes, const uint32_t* first_pos /* from the label pass, or NULL */,
                      int max_pts, uint32_t* n_pts, uint32_t* flags, uint32_t* max_sq,
                      uint32_t* p95_sq, double* sum_dist, void* workspace, size_t workspace_bytes,
                      void* stream);

/* The same metrics for callers that ran octm_label_pass_sorted_u8 first (the batched suite does): first_pos, the
 * boundary rows bnd_true / bnd_pred [n][K-1][W] and the label pass's layering certificate `unsorted` [n] are handed in
 * (bnd_* and unsorted may be NULL: everything then goes through vertex lists like octm_contour2d_u8).
 * On an item whose columns are all in class order, contour [0] of a class mask is a height function over the columns
 * exactly when a few inequalities between neighbouring boundary rows hold; such pairs are verified AND measured from
 * the boundary rows in shared memory: neither the label maps nor any vertex list are touched again.  Everything else
 * (blobs, broken or touching layers, stray pixels) is verified against the label pixels, walked, and searched through
 * vertex lists.  Identical outputs either way.
 * workspace: 2 * round_up(n * K * 2 * max_pts * 4, 256) + 256 bytes (vertices, d2, one counter). */
OCTM_API int octm_contour2d_metrics_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                              int num_classes, const uint32_t* first_pos, const int32_t* bnd_true,
                              const int32_t* bnd_pred, const uint32_t* unsorted, int max_pts, uint32_t* n_pts,
                              uint32_t* flags, uint32_t* max_sq, uint32_t* p95_sq, double* sum_dist, void* workspace,
                              size_t workspace_bytes, void* stream);

/* The two stages of the above, exposed for tests and for callers that want the vertices.
 *   verts   uint32 [n][K][2][max_pts]  packed (y2 << 16 | x2) doubled-lattice vertices of contour [0]: the
 *                                      polyline's vertices, each once, in an unspecified order except
 *                                      that the closing repeat, if any, is the last entry.  With the
 *                                      label pass's boundary rows (bnd_true / bnd_pred) layered maps
 *                                      are not walked: their contours are verified and emitted in
 *                                      parallel (left to right); without them every contour is walked.
 *   d2      uint32 [n][K][2][max_pts]  per-query-vertex D2: [i][c][d][j] = squared distance from vertex j
 *                                      of map 1-d to the nearest vertex of map d.  Required.  With
 *                                      keep_d2 == 0 it is scratch and its contents are unspecified on
 *                                      return (the search kernel counts most units' distances in
 *                                      shared memory instead of storing them); keep_d2 != 0 stores all. */
OCTM_API int octm_first_pos_u8(const uint8_t* labels, int64_t n_items, int64_t item_elems, int num_classes,
                      uint32_t* first_pos /* [n][K] */, void* stream);
OCTM_API int octm_contour2d_trace_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H,
                            int W, int num_classes, const uint32_t* first_pos,
                            const int32_t* bnd_true /* [n][K-1][W] from octm_label_pass_u8, or NULL */,
                            const int32_t* bnd_pred, int max_pts,
                            uint32_t* verts, uint32_t* n_pts, uint32_t* flags, void* stream);
OCTM_API int octm_contour2d_distance(const uint32_t* verts, const uint32_t* n_pts, int64_t n_items,
                            int num_classes, int max_pts, int H, int W /* shape the vertices were traced on */,
                            uint32_t* max_sq, uint32_t* p95_sq, double* sum_dist, uint32_t* d2, int keep_d2,
                            void* stream);

/* ---------------------------------------------------------------------------------------------
 * Contour distances with a physical pixel spacing.  spacing is a HOST array {sy, sx}: the pixel size along rows (H,
 * axial) and along columns (W, lateral), in any unit.  Same vertex lists (octm_contour2d_trace_u8 or
 * octm_contour2d_all_vertices_u8), units and directions as octm_contour2d_distance; with wy = sy * sy, wx = sx * sx a
 * vertex pair at lattice offset (a, b) is q = fl(fl(wy * a^2) + fl(wx * b^2)) in float64, in that order, and
 *   d2       double [n][K][2][max_pts]  per query vertex, the minimum of q over the source set.  Required; with
 *                                       keep_d2 == 0 it is scratch (short lists are kept in shared memory instead)
 *   max_sq   double [n][K][2]           the largest d2
 *   p95_sq   double [n][K][2][2]        the d2 of ranks floor((m - 1) * 0.95) and the next one (the same at the end)
 *   sum_dist double [n][K][2]           sum of sqrt(d2 / 4.0), in a fixed order
 * Distance = sqrt(d2 / 4.0) in the units of the spacing; at {1, 1} d2 equals the integer D2 and every statistic the
 * pixel one (sum_dist up to its summation order).  Bit-reproducible run to run.  Every argument is checked before any
 * CUDA call: both spacings finite and > 0, their squares normal doubles, q of the image diagonal finite. */
OCTM_API int octm_contour2d_distance_spacing(const uint32_t* verts, const uint32_t* n_pts, int64_t n_items,
                                    int num_classes, int max_pts, int H, int W, const double* spacing /* HOST [2] */,
                                    double* max_sq, double* p95_sq, double* sum_dist, double* d2, int keep_d2,
                                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * All-contour distances (build-defined, no reference counterpart): hausdorff / hd95 / assd over EVERY contour of
 * each class mask instead of contour [0] only -- the whole boundary, as MONAI, medpy and surface-distance measure it.
 * Per (item i, class c, map m) the vertex set is
 *   V(i, c, m) = doubled-lattice midpoints of every crack between two 4-adjacent pixels of the image exactly one of
 *                which is class c  (= unique(concatenate(find_contours(L == c, 0.5))) * 2)
 * each vertex ONCE: no closing repeats.  Lattice row 2y holds the cracks (y, x) | (y, x + 1) at x2 = 2x + 1, row
 * 2y + 1 the cracks (y, x) | (y + 1, x) at x2 = 2x.  Outputs as for octm_contour2d_u8 with these sets in place of
 * contour [0]: direction 0 queries every pred vertex against the true set, direction 1 the other way.
 *   verts   uint32 [n][K][2][max_pts]  packed (y2 << 16 | x2), in raster order of the doubled lattice (y2, then x2):
 *                                      deterministic, so sum_dist is bit-reproducible
 *   n_pts   uint32 [n][K][2]           |V| EXACTLY, also when it exceeds max_pts (then only the first max_pts
 *                                      vertices are stored and the OCTM_CF_*_OVERFLOW bit is set: redo the item with
 *                                      max_pts >= n_pts).  0 = class absent from the map or filling it (metrics NaN).
 *   flags   uint32 [n][K]              OCTM_CF_*_OVERFLOW only; the *_CLOSED bits are never set.
 * |V| <= (H - 1) * W + H * (W - 1) (every crack).  One read of each label map emits all K classes. */
OCTM_API int octm_contour2d_all_vertices_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                   int num_classes, int max_pts, uint32_t* verts, uint32_t* n_pts,
                                   uint32_t* flags, void* stream);
/* One call: octm_contour2d_all_vertices_u8 + octm_contour2d_distance; max_sq / p95_sq / sum_dist as for
 * octm_contour2d_u8.  workspace >= octm_contour2d_workspace_bytes(n_items, H, W, num_classes, max_pts). */
OCTM_API int octm_contour2d_all_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                          int num_classes, int max_pts, uint32_t* n_pts, uint32_t* flags, uint32_t* max_sq,
                          uint32_t* p95_sq, double* sum_dist, void* workspace, size_t workspace_bytes,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Normalized surface Dice at tolerance tau (build-defined, no reference counterpart; MONAI compute_surface_dice,
 * surface-distance compute_surface_dice_at_tolerance): the share of both boundaries that lies within tau of the other.
 * The surfaces are the all-contour vertex sets V_t, V_p of octm_contour2d_all_vertices_u8, whatever contour mode the
 * other metrics use.  Per (item i, class c) and integer threshold T_j (squared doubled-lattice distance; for a
 * tolerance of tau pixels, T = max{D : sqrt(D / 4.0) <= tau}, the expression every contour distance here is reported
 * through):
 *   n_surf    uint32 [n][K][2]             (|V_t|, |V_p|), as n_pts of octm_contour2d_all_vertices_u8
 *   n_within  uint32 [n][K][2][n_thresholds]  [..][0][j] = #{v in V_p : min_{u in V_t} |v - u|^2 <= T_j} (pred -> true,
 *                                          direction 0 as elsewhere), [..][1][j] the same for V_t against V_p
 *   NSD_j = (n_within[..][0][j] + n_within[..][1][j]) / (|V_t| + |V_p|): NaN when both sets are empty, 0 when one is.
 * thresholds_sq is a HOST array of parameters, not data (the exception to the device-pointer rule): 1 to
 * OCTM_SURFACE_DICE_MAX_TOL values in ascending order, each <= OCTM_SURFACE_DICE_MAX_SQ (tau <= 8 px), read before the
 * call returns.  Counts are exact (no workspace, no overflow); one read of each label map. */
#define OCTM_SURFACE_DICE_MAX_TOL 4
#define OCTM_SURFACE_DICE_MAX_SQ 256      /* T(8 px) */
OCTM_API int octm_surface_dice_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                  int num_classes, const uint32_t* thresholds_sq /* HOST array, ascending */,
                                  int n_thresholds, uint32_t* n_surf /* [n][K][2] */,
                                  uint32_t* n_within /* [n][K][2][n_thresholds] */, void* stream);
/* The same counts with a pixel spacing {sy, sx} (HOST array, as octm_contour2d_distance_spacing) and 1 to
 * OCTM_SURFACE_DICE_MAX_TOL tolerances (HOST array, any order, in the units of the spacing): a vertex is within tau when
 * sqrt(q / 4.0) <= tau for q = fl(fl(wy * a^2) + fl(wx * b^2)) of its nearest source vertex.  The library turns each tau
 * into the exact column reach of every lattice row offset; the reach is limited to 16 lattice rows and 16 lattice columns,
 * i.e. tau < min(sqrt(fl(wy * 289) / 4.0), sqrt(fl(wx * 289) / 4.0)) (just below 8.5 at {1, 1}); a larger tau returns
 * OCTM_ERR_INVALID with the largest one allowed in octm_last_error(). */
OCTM_API int octm_surface_dice_spacing_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                          int num_classes, const double* spacing /* HOST [2] */,
                                          const double* tolerances /* HOST [n_tolerances] */, int n_tolerances,
                                          uint32_t* n_surf /* [n][K][2] */,
                                          uint32_t* n_within /* [n][K][2][n_tolerances] */, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Connected components per class (build-defined, no reference counterpart; scipy.ndimage.label, skimage.measure.label).
 * Per (item i, class c, map m: 0 = y_true, 1 = y_pred; o the other map), connectivity 4 or 8:
 *   n_comp  uint32 [n][K][2]   number of connected components of (L_m == c)
 *   n_hit   uint32 [n][K][2]   how many of them share at least one pixel with (L_o == c): detected (m = 0), matched (m = 1)
 * Labels >= num_classes belong to no class and are never counted.  Counts are exact with no upper bound (no workspace,
 * no overflow, no host synchronisation); each (item, map) is one row-streaming union-find over runs of equal labels. */
OCTM_API int octm_components_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                int num_classes, int connectivity /* 4 or 8 */,
                                uint32_t* n_comp /* [n][K][2] */, uint32_t* n_hit /* [n][K][2] */, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Boundary rows -> label maps (SURVEY.md 8f-4: the layer datasets catalogued in the reference's
 * Datasets.md:3-26 annotate boundary curves, while Metrics/*.py score masks).  The inverse of the label
 * pass's boundary rows on layered maps:
 *   labels[i][y][x] = #{ k : b_k(i, x) <= y }
 *   boundaries  [n][num_boundaries][W] of dtype OCTM_DTYPE_I32 or OCTM_DTYPE_F32, any order per column, any
 *               value (outside [0, H]: the layer is empty / fills the column); NaN = boundary absent
 *   labels      uint8 [n][H][W], values 0 .. num_boundaries (<= 15) */
OCTM_API int octm_labels_from_boundaries(const void* boundaries, int dtype, int64_t n_items, int num_boundaries,
                                int H, int W, uint8_t* labels, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Layer thickness per en-face sector of OCT volumes (build-defined, no reference counterpart; the ETDRS grid of clinical
 * OCT reports).  Reads the boundary rows b_k(x) = #{y : L[y][x] < k} of octm_label_pass_u8 (b_0 = 0, b_K = H): they are
 * counts, so for ANY label map with values < K the thickness of the classes first .. last in A-scan x is
 * b_{last+1}(x) - b_first(x).  Items [v * items_per_volume, (v + 1) * items_per_volume) form volume v.
 *   bnd_true, bnd_pred  int32 [n][K-1][W]   boundary rows of y_true / y_pred (undefined for maps with a label >= K)
 *   region   uint8 [n][W]                   region of every A-scan: 0 .. n_regions - 1; any other value (255) = none
 *   groups   HOST int32 [n_groups][2]       (first, last) class of each group, 0 <= first <= last <= K - 1
 *   sums     int64 [n / items_per_volume][n_groups][n_regions][5]   per (volume, group, region), over its A-scans:
 *                                           count, sum t, sum p, sum |t - p|, sum (t - p)^2, with t / p the group
 *                                           thickness of y_true / y_pred in pixels.  Fully overwritten; exact integers
 *                                           (the order of the device atomics does not matter: bit-reproducible)
 *   thick    int32 [n][2][n_groups][W]      t ([i][0]) and p ([i][1]) of every A-scan, whatever its region; or NULL
 * Every argument is checked before any CUDA call: shapes, 2 <= K <= 16, n % items_per_volume == 0, 1 <= n_regions <= 16,
 * 1 <= n_groups <= 16 and the group bounds, items_per_volume * W * H^2 < 2^53 (every sum exact in int64 and in a float64
 * all-reduce), at most 65535 volumes; device pointers other than thick may be NULL only when n_items == 0. */
OCTM_API int octm_sector_thickness_i32(const int32_t* bnd_true, const int32_t* bnd_pred, int64_t n_items,
                                       int num_classes, int H, int W, int items_per_volume, const uint8_t* region,
                                       int n_regions, const int32_t* groups /* HOST [n_groups][2] */, int n_groups,
                                       int64_t* sums, int32_t* thick, void* stream);

/* ---------------------------------------------------------------------------------------------
 * 3-D surface-distance metrics (BASELINE config 5; the reference's contour metrics are 2-D only, this is
 * their build-defined 3-D counterpart): per class, distances between the SURFACES of the class regions of
 * two label volumes [D0][D1][D2] by an exact separable squared Euclidean distance transform (Meijster).
 *   surface(mask) = voxels of the mask with a 6-neighbour outside it (outside the volume = outside)
 *   unit u = class * 2 + direction; direction 0: every surface voxel of y_pred -> nearest surface voxel of
 *   y_true, direction 1 the other way.  Units [unit_begin, unit_end) are computed (multi-GPU: disjoint
 *   ranges per rank), outputs of the others are left untouched:
 *   n_pts    uint32 [K][2]     surface voxels of y_true ([c][0], written by direction 1) / y_pred ([c][1]) that
 *                              have a finite distance; 0 when either surface is empty
 *   max_sq   uint32 [K][2], p95_sq uint32 [K][2][2], sum_dist double [K][2]: as for octm_contour2d_u8, but on
 *                              the unit lattice (distance = sqrt(D2), not sqrt(D2 / 4))
 * Limits: D0, D1 <= 2048, D2 <= 65534, squared diagonal < 2^28. */
OCTM_API size_t octm_surface3d_workspace_bytes(int D0, int D1, int D2);
OCTM_API int octm_surface3d_u8(const uint8_t* y_true, const uint8_t* y_pred, int D0, int D1, int D2, int num_classes,
                      int unit_begin, int unit_end, uint32_t* n_pts, uint32_t* max_sq, uint32_t* p95_sq,
                      double* sum_dist, void* workspace, size_t workspace_bytes, void* stream);

/* The same surfaces, units and directions in physical units, plus normalized-surface-Dice counts.
 *   spacing    double [3]: voxel spacing along D0, D1, D2 (finite, > 0, each square a normal double, the squared
 *              diagonal of the volume finite).  With w_i = spacing[i]^2 the squared distance
 *              to a source voxel at integer offset (a, b, c) is d2 = w0*a^2 + (w1*b^2 + w2*c^2), float64, in that order
 *   tolerances double [num_tolerances], 0 <= num_tolerances <= 4, each finite and >= 0, in the units of spacing; a
 *              query voxel is within tau when sqrt(d2) <= tau (float64)
 *   n_pts      uint32 [K][2] as octm_surface3d_u8 (0 when either surface is empty)
 *   max_sq     double [K][2], p95_sq double [K][2][2] (order statistics of d2 at ranks floor((m-1)*0.95) and the next),
 *   sum_dist   double [K][2] (sum of sqrt(d2)); all bit-reproducible from run to run
 *   n_surf     uint32 [K][2] surface voxels of y_true / y_pred, counted even when the other surface is empty
 *   n_within   uint32 [K][2][num_tolerances] query voxels within each tolerance, per direction
 *   n_surf and n_within may be null only when num_tolerances == 0.
 * Unit (c, dir) writes only n_pts[c][1 - dir], n_surf[c][1 - dir] and its own [c][dir] entries.  Never uses the
 * near-field path.  Limits: D0, D1 <= 2048, D2 <= 65534; workspace 16 B per voxel and a little more. */
OCTM_API size_t octm_surface3d_spacing_workspace_bytes(int D0, int D1, int D2);
OCTM_API int octm_surface3d_spacing_u8(const uint8_t* y_true, const uint8_t* y_pred, int D0, int D1, int D2,
                      int num_classes, int unit_begin, int unit_end, const double* spacing,
                      const double* tolerances, int num_tolerances, uint32_t* n_pts, double* max_sq,
                      double* p95_sq, double* sum_dist, uint32_t* n_surf, uint32_t* n_within,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Front end: model scores -> uint8 label map, argmax over the class dimension (what a user does between
 * a model's forward() and the metric functions; every model of the reference returns
 * (B, num_classes, H, W), e.g. SOTAS/Lesions_Segment/ReLayNet_2017.py:106-108).
 *   scores        [n][K][plane_elems] (channels_last = 0, NCHW) or [n][plane_elems][K] (channels_last = 1)
 *   dtype         OCTM_DTYPE_F32 / F16 / BF16
 *   labels        uint8 [n][plane_elems]; first maximal class wins ties, NaN counts as maximal
 *                 (numpy / torch argmax semantics) */
OCTM_API int octm_argmax_labels(const void* scores, int dtype, int64_t n_items, int num_classes,
                       int64_t plane_elems, int channels_last, uint8_t* labels, void* stream);

/* ---------------------------------------------------------------------------------------------
 * auc_score (Metrics/ConfusionMatrix_based_metrics.py:65-84): area under the ROC curve of a score map
 * against a binary truth mask, per item -- sklearn.metrics.roc_auc_score(y_true.flatten(),
 * y_pred.flatten()) with ties between scores counted one half (exact 64-bit rank sums, one division).
 *   y_true   uint8 [n][item_elems]   two distinct values: the larger one is the positive class
 *   scores   [n][item_elems] of dtype OCTM_DTYPE_F32 / F16 / BF16 / F64
 *   auc      double [n]
 * As in the reference (`except ValueError: return 0.0`): more than two label values, or NaN / inf
 * scores, give 0.0.  A single-class (or empty) y_true gives single_class_value: NaN reproduces
 * scikit-learn >= 1.6 (warns), 0.0 the older versions (raise).  Scratch: octm_auc_workspace_bytes. */
OCTM_API size_t octm_auc_workspace_bytes(int64_t n_items, int64_t item_elems, int dtype);
OCTM_API int octm_auc_u8(const uint8_t* y_true, const void* scores, int dtype, int64_t n_items, int64_t item_elems,
                double single_class_value, double* auc, void* workspace, size_t workspace_bytes,
                void* stream);

/* ---------------------------------------------------------------------------------------------
 * Transfer encoding for host-resident label maps (K <= 16): two labels per byte across PCIe.
 *   octm_host_pack_nibbles   HOST function: dst[i] = src[2i] | src[2i+1] << 4 for n_labels labels
 *                            (dst holds (n_labels + 1) / 2 bytes), on `threads` host threads (<= 0: all cores).
 *                            A data-format conversion only; no metric arithmetic runs on the host.
 *                            Returns OCTM_PACK_WIDE_LABEL (not an error) when some src byte is >= 16: such a
 *                            label has no 4-bit code, dst does not encode src, and the caller must send src as
 *                            it is (a transfer encoding must never change a result).
 *   octm_unpack_nibbles_u8   device kernel: the inverse, packed (device) -> labels uint8 [n_labels] (device). */
#define OCTM_PACK_WIDE_LABEL 1    /* octm_host_pack_nibbles: a label >= 16 was seen, dst is not usable */
OCTM_API int octm_host_pack_nibbles(const uint8_t* src, uint8_t* dst, size_t n_labels, int threads);
OCTM_API int octm_unpack_nibbles_u8(const uint8_t* packed, int64_t n_labels, uint8_t* labels, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Float64 epilogue on the device.  class_metrics[i][c][m] (double [n][K][OCTM_NUM_CLASS_METRICS]) holds
 * the value the reference function OCTM_M_* returns for the masks (y_true == c, y_pred == c) of
 * item i, evaluated from the exact integers above with the reference's operation order
 * (ConfusionMatrix_based_metrics.py:14-62, Region_based_metrics.py:13-60,
 *  PixelError_based_metrics.py:14-35, Biomarker_based_metrics.py:18-38,
 *  Contour_based_metrics.py:22,39,56,68-71).  Contour metrics are NaN where a mask has no contour
 * (the reference raises IndexError) or when n_pts is NULL.
 *   boundary_metrics double [n][K-1][3] = mean_squared_error, root_mean_squared_error, mad of the
 *                                         boundary rows b_k (may be NULL)
 *   totals           double [octm_totals_len(K)] = this batch's dataset-level partial sums in the
 *                    layout [n_items | cm K*K | thick K | bnd_sq K-1 | bnd_abs K-1 | contour_items K |
 *                    sum hd K | sum hd95 K | sum assd K | n_overflow_items | n_bad_label_items |
 *                    max hd K | OR of contour flags] (may be NULL; written for n_items == 0 as well);
 *                    integer fields are exact below 2^53.  The first octm_totals_sum_len(K) entries are what
 *                    the multi-GPU all-reduce sums: n_overflow_items = items with an OCTM_CF_*_OVERFLOW flag,
 *                    n_bad_label_items = items whose confusion counts do not add up to H * W (the label pass
 *                    drops every pixel pair with a label >= K instead of aliasing it into another class). */
#define OCTM_M_ACCURACY 0
#define OCTM_M_SENSITIVITY 1
#define OCTM_M_CM_PRECISION 2
#define OCTM_M_SPECIFICITY 3
#define OCTM_M_DICE 4
#define OCTM_M_IOU 5
#define OCTM_M_REGION_PRECISION 6
#define OCTM_M_RECALL 7
#define OCTM_M_MSE 8
#define OCTM_M_RMSE 9
#define OCTM_M_MAD 10
#define OCTM_M_VASCULARITY 11
#define OCTM_M_THICKNESS_DIFF 12
#define OCTM_M_HAUSDORFF 13
#define OCTM_M_HAUSDORFF95 14
#define OCTM_M_ASSD 15
#define OCTM_NUM_CLASS_METRICS 16

OCTM_API int octm_totals_len(int num_classes);
OCTM_API int octm_totals_sum_len(int num_classes);
OCTM_API int octm_derive_metrics(const uint64_t* counts, const int64_t* thick_absdiff, const int64_t* bnd_sq,
                        const int64_t* bnd_abs, const uint32_t* n_pts, const uint32_t* max_sq,
                        const uint32_t* p95_sq, const double* sum_dist, const uint32_t* contour_flags,
                        int64_t n_items, int H, int W, int num_classes, double* class_metrics,
                        double* boundary_metrics, double* totals, void* stream);
/* octm_derive_metrics with a pixel spacing {sy, sx} (HOST array): max_sq / p95_sq are the float64 squared distances of
 * octm_contour2d_distance_spacing, and the thickness and boundary errors scale with the row spacing:
 * thickness (sum / W) * sy, boundary MSE (sum / W) * wy (RMSE its square root), MAD (sum / W) * sy.  The totals are the
 * same integer sums as without a spacing (a dataset-level mean is scaled by its reader). */
OCTM_API int octm_derive_metrics_spacing(const uint64_t* counts, const int64_t* thick_absdiff, const int64_t* bnd_sq,
                        const int64_t* bnd_abs, const uint32_t* n_pts, const double* max_sq,
                        const double* p95_sq, const double* sum_dist, const uint32_t* contour_flags,
                        int64_t n_items, int H, int W, int num_classes, const double* spacing /* HOST [2] */,
                        double* class_metrics, double* boundary_metrics, double* totals, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OCTM_H_ */
