/* libofc -- C-ABI of the B200 (sm_100a) flow -> grid -> k-means -> cosine hot path.
 *
 * The reference (menmitsu/opticalFlowClustering, k-means-color-clustering/) has
 * no FFI of its own: its hot path is Python calling cv2 / scikit-learn.  Each
 * entry point below replaces one of those library calls (cited per function);
 * the Python package opticalflowclustering_b200 binds them with ctypes and
 * re-exports the reference's own function/class names on top.
 *
 * Conventions
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer
 *     owned by the caller (the Python side allocates with torch);
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all
 *     work is stream-ordered, no call synchronises the device;
 *   - return 0 on success, a negative OFC_ERR_* otherwise; ofc_last_error()
 *     gives the message (thread-local).
 */
#ifndef OFC_H_
#define OFC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFC_OK 0
#define OFC_ERR_INVALID (-1)
#define OFC_ERR_UNSUPPORTED (-2)
#define OFC_ERR_CUDA (-3)
#define OFC_ERR_WORKSPACE (-4)

int ofc_version(void);
const char* ofc_last_error(void);

/* ---- optional per-kernel timing (benchmark / profiling aid) ----------------
 * Between begin and end every kernel launch is bracketed by cudaEvents on its
 * launch stream; end() synchronises on them and returns, per kernel kind, the
 * summed device time (ms) and the launch count.  Kinds: 0 bgr2gray, 1 prefilter,
 * 2 polyexp, 3 minmax_init, 4 flow_encode, 5 grid_cells, 6 flow_minmax,
 * 7 draw_grid, 8 kmeans, 9 cosine, 10 flow_upsample, 12+l flow_iter at pyramid level l (0 = full
 * resolution).  n_kinds must be >= 20.  The record list is mutex-protected (launches from several host
 * threads are all recorded); begin/end themselves are meant to be called from one thread. */
int ofc_profile_begin(void);
int ofc_profile_end(float* ms_by_kind, int* launches_by_kind, int n_kinds);

/* ---- Farneback dense optical flow --------------------------------------
 * Replaces cv.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels,
 * winsize, iterations, poly_n, poly_sigma, flags)
 *   reference: computeOpticalFlowModule.py:20-22, computeOpticalFlow.py:99-101.
 * A plan fixes the frame size and parameters (pyramid geometry, filter taps,
 * workspace layout) for up to `max_frames` frames per call.  winsize 4..65 (cv2's quirk kept: the window is
 * 2 (winsize / 2) + 1 wide, the box sums are scaled by 1 / winsize^2), poly_n 5 or 7.  flags: 0 (box window,
 * the reference's literal), OFC_FLOW_GAUSSIAN (cv2.OPTFLOW_FARNEBACK_GAUSSIAN: Gaussian
 * window of winsize | 1 taps, any odd winsize <= 65) and/or OFC_FLOW_USE_INITIAL_FLOW
 * (cv2.OPTFLOW_USE_INITIAL_FLOW, through ofc_farneback_pair_init); anything else ->
 * OFC_ERR_UNSUPPORTED.
 * Threading: a plan (its side stream, events and the workspace handed to its calls) must be used by ONE
 * stream / host thread at a time; different plans are independent.  The shared-memory opt-in of every
 * kernel is recorded per device, so one process may drive several GPUs. */
#define OFC_FLOW_USE_INITIAL_FLOW 4
#define OFC_FLOW_GAUSSIAN 256
typedef struct ofc_flow_plan ofc_flow_plan;

int ofc_flow_plan_create(ofc_flow_plan** plan, int width, int height, int max_frames,
                         double pyr_scale, int levels, int winsize, int iterations,
                         int poly_n, double poly_sigma, int flags);
void ofc_flow_plan_destroy(ofc_flow_plan* plan);
size_t ofc_flow_plan_workspace_bytes(const ofc_flow_plan* plan);
/* keep != 0: also write the pre-filtered image I of the full-resolution level to the workspace
 * (buffer kind 0 below); by default it is fused into the polynomial expansion and never stored. */
int ofc_flow_plan_keep_intermediates(ofc_flow_plan* plan, int keep);
int ofc_flow_plan_num_levels(const ofc_flow_plan* plan);
/* level 0 = coarsest ... num_levels-1 = full resolution */
int ofc_flow_plan_level_size(const ofc_flow_plan* plan, int level, int* w, int* h);
/* byte offset inside the workspace of a level's buffer (for parity tests of
 * the intermediates): kind 0 = I f32[h][w], 1 = RA f32x4[h][w], 2 = RB f32[h][w],
 * 3 / 4 = flow ping/pong f32x2[h][w]; *frame_stride_bytes = distance between
 * consecutive frames (or pairs). */
int ofc_flow_plan_buffer(const ofc_flow_plan* plan, int level, int kind,
                         size_t* offset_bytes, size_t* frame_stride_bytes);

/* n_frames consecutive gray frames u8[n_frames][H][W] -> n_frames-1 flow fields
 * f32[n_frames-1][H][W][2]; pair t is (frame t, frame t+1) and the pre-filter
 * and polynomial expansion of each frame are computed once (streaming reuse).
 * minmax (nullable) receives per pair the IEEE bits of min and max |flow|
 * (u32[n_frames-1][2]) for ofc_flow_to_bgr. */
int ofc_farneback_sequence(const ofc_flow_plan* plan, const uint8_t* gray, int n_frames,
                           float* flow, uint32_t* minmax,
                           void* workspace, size_t workspace_bytes, void* stream);
/* one independent pair, the literal cv2 call */
int ofc_farneback_pair(const ofc_flow_plan* plan, const uint8_t* prev, const uint8_t* next,
                       float* flow, uint32_t* minmax,
                       void* workspace, size_t workspace_bytes, void* stream);

/* the cv2 call with flags & OPTFLOW_USE_INITIAL_FLOW: init_flow f32[H][W][2] seeds the coarsest
 * pyramid level (cv::resize INTER_AREA, times the level's scale); plan created with that flag */
int ofc_farneback_pair_init(const ofc_flow_plan* plan, const uint8_t* prev, const uint8_t* next,
                            const float* init_flow, float* flow, uint32_t* minmax,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Streaming form of ofc_farneback_pair for the reference's per-frame loop (ComputeOpticalFLow keeps prev_gray and is
 * called once per decoded frame, computeOpticalFlowModule.py:18-36): the plan keeps the previous frame's pre-filtered
 * image and polynomial expansion in its workspace (two frame slots used alternately), so every call expands ONE
 * frame instead of two.  begin(first frame) primes slot 0; next(frame) returns the flow previous -> frame.  Same bits as
 * ofc_farneback_pair(previous, frame).  The plan needs max_frames >= 2; the same workspace must be passed every call. */
int ofc_farneback_stream_begin(ofc_flow_plan* plan, const uint8_t* first_gray, void* workspace, size_t workspace_bytes,
                               void* stream);
int ofc_farneback_stream_next(ofc_flow_plan* plan, const uint8_t* gray, float* flow, uint32_t* minmax, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- 8-bit colour ---------------------------------------------------------
 * cv.cvtColor(frame, COLOR_BGR2GRAY)        computeOpticalFlowModule.py:16,19 */
int ofc_bgr2gray(const uint8_t* bgr, uint8_t* gray, int64_t n_pixels, void* stream);
/* cv2.cvtColor(x, COLOR_BGR2HSV) on n 8-bit pixels (H 0..179): KmeanGrids.py:92,336,
 * color_kmeans.py:121 (applied there to cell means / cluster centres). */
int ofc_bgr2hsv(const uint8_t* bgr, uint8_t* hsv, int64_t n_pixels, void* stream);
/* min / max of |flow| per frame (IEEE bits), for flows that did not come from
 * ofc_farneback_*; first step of cv.normalize(..., NORM_MINMAX)  :31 */
int ofc_flow_minmax(const float* flow, int n_frames, int64_t n_pixels, uint32_t* minmax, void* stream);
/* cv.cartToPolar + hue byte + cv.normalize + cv.cvtColor(HSV2BGR)  :25-33.
 * mag_sum (nullable, f64[n_frames]) receives the sum of |flow| per frame for
 * the "Average Magnitude" series of computeOpticalFlow.py:114-117,146-149.
 * The row width matters: cv2's HSV2BGR truncates in its 32-pixel SIMD body and
 * rounds in the scalar tail (last width % 32 pixels of each row). */
int ofc_flow_to_bgr(const float* flow, int n_frames, int height, int width, const uint32_t* minmax,
                    uint8_t* bgr, double* mag_sum, void* stream);
/* Same, additionally writing the reference's `mask` image (H, 255, V) that ComputeOpticalFLow keeps as an
 * attribute (computeOpticalFlowModule.py:14-15, 28-31): hsv u8 [n_frames][H][W][3]. */
int ofc_flow_to_hsv(const float* flow, int n_frames, int height, int width, const uint32_t* minmax,
                    uint8_t* bgr, uint8_t* hsv, void* stream);
/* ofc_flow_to_bgr + ofc_grid_cells in one kernel (one CTA per grid cell and frame): the visualisation is written
 * once and never read back; the per-cell outputs are those of ofc_grid_cells (any of them may be NULL).
 * Replaces computeOpticalFlowModule.py:25-33 followed by overlayGridAndComputeAvgColor (KmeanGrids.py:52-113)
 * and the k = 1 colour cluster (:269-339) for every frame of the batch. */
int ofc_flow_to_bgr_grid(const float* flow, int n_frames, int height, int width, const uint32_t* minmax, uint8_t* bgr,
                         double* mag_sum, int rows, int cols, int draw_lines, int threshold, uint8_t* avg_bgr,
                         uint8_t* avg_hue, uint8_t* km_centre, uint8_t* km_hue, void* stream);

/* ---- grid-cell aggregation ------------------------------------------------
 * overlayGridAndComputeAvgColor (KmeanGrids.py:52-113,
 * drawGridsAndOutputCSV.py:47-135) and, for n_clusters = 1, the per-cell
 * preprocess_image + KMeans(1) + rint + BGR2HSV of KmeanGrids.py:269-339 /
 * color_kmeans.py:35-135.  cells = rows*cols in the reference's row-major
 * order; any output pointer may be NULL.
 *   draw_lines  reproduce the state of the white 1-px rectangles the reference
 *               draws between the mean and the k-means stage (SURVEY.md Q3)
 *   threshold   preprocess_image's "channel < 30 -> 0" (0 disables)         */
int ofc_grid_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols,
                   int draw_lines, int threshold,
                   uint8_t* avg_bgr /* [n][cells][3] */, uint8_t* avg_hue /* [n][cells] */,
                   uint8_t* km_centre /* [n][cells][4] */, uint8_t* km_hue /* [n][cells] */,
                   uint32_t* km_sums /* [n][cells][4] */, void* stream);
/* cv2.rectangle(frame,(x1,y1),(x2,y2),(255,255,255),1) for every cell  KmeanGrids.py:108 */
int ofc_draw_grid(uint8_t* bgr, int n_frames, int height, int width, int rows, int cols, void* stream);

/* ---- k-means (Lloyd) --------------------------------------------------------
 * Replaces sklearn.cluster.KMeans(n_clusters=k).fit(X) / .predict(X) as called at
 *   reference: KmeanGrids.py:299-304, color_kmeans.py:65-78
 * (scikit-learn 1.9.0 dense Lloyd, SURVEY.md A.5).  The host loop (stopping rule,
 * optional cross-GPU all-reduce of `sums`/`counts` between ofc_kmeans_sums and
 * ofc_kmeans_centres) lives in opticalflowclustering_b200/kmeans.py.
 * All calls are batched over `batch` independent problems of equal shape
 * (X is [batch][n][d], row-major); the reference runs one fit per grid cell.
 * dtype: OFC_U8 (worked in float64 like sklearn), OFC_F32 (float32), OFC_F64.
 * `active` (nullable, u8 [batch]) selects the problems a call touches: problems
 * that already met the stopping rule are frozen while the rest keep iterating. */
#define OFC_U8 0
#define OFC_F32 1
#define OFC_F64 2
/* OR-ed into the dtype of ofc_kmeans_assign / _sums / _step / _relocate (and accepted by
 * ofc_kmeans_step_supported): every problem of the batch reads the same X [n][d] -- several
 * starts of one fit (KMeans n_init) without a copy of the rows per start.  Everything else
 * (centres, labels, sums, ...) stays per problem.  A problem's results are the bits it gets
 * when run alone (batch = 1).  Such a batch needs at most batch * ofc_kmeans_workspace_bytes(1, n, d, k)
 * bytes of workspace.  ofc_kmeans_far_points / _far_payload (row-sharded fits) return
 * OFC_ERR_UNSUPPORTED for it. */
#define OFC_KMEANS_SHARED_ROWS 0x100

size_t ofc_kmeans_workspace_bytes(int batch, int64_t n, int d, int k);
/* the (small) prefix of that workspace ofc_kmeans_assign and ofc_kmeans_centres need on their own */
size_t ofc_kmeans_assign_workspace_bytes(int batch, int64_t n, int d, int k);

/* E-step: labels[i] = first strict minimum over j of ||c_j||^2 - 2 (x_i - mean).c_j
 * (_k_means_lloyd.pyx:160-213).  mean [batch][d] (nullable) is subtracted from every
 * row on the fly (KMeans.fit centres X, _kmeans.py:1487-1493; predict does not).
 * prev_labels/n_changed (nullable): n_changed[b] = #{i: labels[i] != prev_labels[i]}.
 * inertia (nullable, [batch]) = sum of squared distances to the
 * chosen centres; min_dist (nullable, [batch][n]) the per-point values. */
int ofc_kmeans_assign(const void* X, int dtype, int batch, int64_t n, int d, int k,
                      const double* mean, const double* centres /* [batch][k][d] */,
                      int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed,
                      double* inertia, double* min_dist, const uint8_t* active,
                      void* workspace, size_t workspace_bytes, void* stream);

/* M-step sums: sums[b][j][:] = sum over members of (x - mean) (or its square when
 * `square`), counts[b][j] = members; labels NULL = one cluster holding everything
 * (column statistics for KMeans' tolerance, _kmeans.py:285-293).  Deterministic:
 * private accumulators folded in a fixed order, no floating-point atomics. */
int ofc_kmeans_sums(const void* X, int dtype, int batch, int64_t n, int d, int k,
                    const double* mean, const int32_t* labels, int square,
                    double* sums /* [batch][k][d] */, int64_t* counts /* [batch][k] */, const uint8_t* active,
                    void* workspace, size_t workspace_bytes, void* stream);

/* E-step and M-step sums of one Lloyd iteration in ONE pass over X, for the reference's own shape: uint8 rows
 * (pixels, hues) with d <= 32 whose [k][d] integer accumulators fit shared memory (ofc_kmeans_step_supported).
 * Same labels / n_changed as ofc_kmeans_assign and the same (exact integer) raw sums / counts as ofc_kmeans_sums
 * with mean = NULL; `mean` only centres the rows for the distance, as in ofc_kmeans_assign. */
int ofc_kmeans_step_supported(int dtype, int d, int k);
int ofc_kmeans_step(const void* X, int dtype, int batch, int64_t n, int d, int k,
                    const double* mean, const double* centres, int32_t* labels, const int32_t* prev_labels,
                    uint64_t* n_changed, double* sums /* [batch][k][d] */, int64_t* counts /* [batch][k] */,
                    const uint8_t* active, void* workspace, size_t workspace_bytes, void* stream);

/* centres[b][j] = sums/counts (use_reciprocal: sums * (1/count) as sklearn's _average_centers)
 * minus mean_sub (nullable); empty clusters copy the heaviest cluster; shift_tot[b] =
 * sum_j ||new_j - old_j||^2 (_k_means_common.pyx:274-311).  centres: old in, new out. */
int ofc_kmeans_centres(int batch, int d, int k, const double* sums, const int64_t* counts,
                       const double* mean_sub, int use_reciprocal, double* centres, double* shift_tot,
                       const uint8_t* active, void* workspace, size_t workspace_bytes, void* stream);
/* ofc_kmeans_centres + sklearn's stopping rule (_kmeans.py:705-758) on the device, so the Lloyd loop needs no
 * device->host read per iteration: a problem stops when n_changed == 0 (labels repeated) or shift <= tol[b];
 * it then clears active[b], sets just_done[b] (and, for batch > 1, its labels are copied from labels_cur into
 * labels_other so both ping-pong buffers hold them).  n_iter[b] = iteration + 1 for every problem still running;
 * *n_active += number of problems that continue (the host polls it asynchronously).  round_f32: store the
 * centres rounded to float32 (float32 data).  NULL tol / n_changed / active / just_done / n_iter / n_active /
 * labels_* skip the corresponding part.  it_counter (may be NULL): the iteration number is read from the device
 * (and incremented afterwards) instead of `iteration`, and the running count goes to n_active[*it_counter] -- so one
 * iteration can be captured in a CUDA graph and replayed. */
int ofc_kmeans_update(int batch, int64_t n, int d, int k, const double* sums, const int64_t* counts, const double* mean_sub,
                      int use_reciprocal, int round_f32, double* centres, double* shift_tot, const uint64_t* n_changed,
                      const double* tol, int iteration, uint8_t* active, uint8_t* just_done, int32_t* n_iter,
                      int32_t* n_active, const int32_t* labels_cur, int32_t* labels_other, int32_t* it_counter,
                      void* workspace, size_t workspace_bytes, void* stream);

/* MiniBatchKMeans centre update, the arithmetic behind the reference's color-quantization/quant.py:18-20
 * (clt = MiniBatchKMeans(n_clusters); clt.fit_predict(image)) -> scikit-learn 1.9.0 _minibatch_update_dense
 * (sklearn/cluster/_k_means_minibatch.pyx:60-110): for one mini-batch Xb [batch_rows][d] with labels from
 * ofc_kmeans_assign,  c_new = (c_old * weight_sum + members in batch order) / (weight_sum + n_members), weight_sums
 * updated in place; clusters without a member keep their centre.  float32 data is worked in float32. */
int ofc_minibatch_update(const void* Xb, int dtype, int batch_rows, int d, int k, const int32_t* labels,
                         const double* centres_old, double* centres_new, double* weight_sums, void* stream);

/* The same with sample weights, as MiniBatchKMeans.partial_fit(X, sample_weight=w) steps: per cluster,
 * wsum = the members' weights in batch order; if wsum > 0, c_new = (c_old * weight_sum + x w of the members in batch
 * order) / (weight_sum + wsum) and weight_sum += wsum, else the cluster keeps its centre and weight sum.  weights
 * [batch_rows] are float64 holding values of the working type (float32 values for float32 rows).  Every product and
 * sum is rounded on its own, as sklearn's loop; the result is that left fold's bits for every dtype and batch size.
 * Both calls take any batch_rows >= 1 (a whole 1080p frame is one batch): one CTA per cluster streams the batch in
 * order, on exact integer prefix sums where every increment is an integer, on the sequential fold elsewhere.
 * centres_old and centres_new must not overlap. */
int ofc_minibatch_update_weighted(const void* Xb, int dtype, int batch_rows, int d, int k, const int32_t* labels,
                                  const double* weights, const double* centres_old, double* centres_new,
                                  double* weight_sums, void* stream);

/* Empty-cluster relocation on the sums/counts (_k_means_common.pyx:167-211): every empty
 * cluster, in index order, takes the point farthest from the (old) centre of its label.
 * Distances use (x - mean) against centres_old; raw_sums says whether `sums` holds sums of
 * the raw rows (uint8 path) or of the centred rows.  Returns immediately on the device for
 * problems without an empty cluster, so it can be launched every iteration; call it
 * between ofc_kmeans_sums and ofc_kmeans_centres.  scratch (f64 [batch][n], may be NULL): with it the row
 * distances are computed once by the whole grid and the picks read them (same result; without it one CTA per
 * problem re-reads X once per empty cluster, which is only tolerable for small problems). */
int ofc_kmeans_relocate(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                        const int32_t* labels, const double* centres_old, double* sums, int64_t* counts,
                        int raw_sums, const uint8_t* active, double* scratch, void* stream);

/* ---- weighted fits: KMeans.fit(X, sample_weight=w) ----
 * The weighted twins of ofc_kmeans_assign / _sums / _update / _relocate.  weights f64 [batch][n] (>= 0, not all 0;
 * the caller validates them), or ONE [n] vector for every problem under OFC_KMEANS_SHARED_ROWS, like X.  Where the
 * unweighted calls have int64 member counts these take float64 weight sums `weight_sums [batch][k]`.  Labels do not
 * depend on the weights.  Every weighted form folds in the unweighted order, so weights of all ones give exactly the
 * unweighted bits.  Real-valued weights are summed deterministically (fixed order, no floating-point atomics).  uint8
 * rows with integer-valued weights keep exact sums: every x w and every partial sum stays below 2^53.
 *
 * ofc_kmeans_assign_weighted: ofc_kmeans_assign with inertia = sum_i w_i ||x_i - c_label||^2
 *   (_inertia_dense, _k_means_common.pyx:94-124); min_dist stays unweighted. */
int ofc_kmeans_assign_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                               const double* centres, const double* weights, int32_t* labels, const int32_t* prev_labels,
                               uint64_t* n_changed, double* inertia, double* min_dist, const uint8_t* active, void* workspace,
                               size_t workspace_bytes, void* stream);
/* M-step: sums[b][j][:] = sum over members of (x - mean) w, weight_sums[b][j] = sum of their weights
 * (_k_means_lloyd.pyx:216-218).  Same workspace as ofc_kmeans_sums. */
int ofc_kmeans_sums_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                             const int32_t* labels, const double* weights, double* sums, double* weight_sums,
                             const uint8_t* active, void* workspace, size_t workspace_bytes, void* stream);
/* ofc_kmeans_update on weight sums (_average_centers, _k_means_common.pyx:264-286): centres = sums / weight where
 * weight > 0, otherwise the centre of the heaviest cluster by weight (the first on ties).  Stopping rule unchanged. */
int ofc_kmeans_update_weighted(int batch, int64_t n, int d, int k, const double* sums, const double* weight_sums,
                               const double* mean_sub, int use_reciprocal, int round_f32, double* centres, double* shift_tot,
                               const uint64_t* n_changed, const double* tol, int iteration, uint8_t* active, uint8_t* just_done,
                               int32_t* n_iter, int32_t* n_active, const int32_t* labels_cur, int32_t* labels_other,
                               int32_t* it_counter, void* workspace, size_t workspace_bytes, void* stream);
/* ofc_kmeans_relocate on weight sums (_relocate_empty_clusters_dense, _k_means_common.pyx:167-211): a cluster is
 * empty when its WEIGHT is 0 (members of weight 0 only count as empty); the farthest rows are chosen by unweighted
 * distance; the moved row carries x w and w.  scratch (f64 [batch][n]) is required. */
int ofc_kmeans_relocate_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                                 const int32_t* labels, const double* centres_old, const double* weights, double* sums,
                                 double* weight_sums, int raw_sums, const uint8_t* active, double* scratch, void* stream);

/* Row-sharded data (one shard per GPU): the search half of that relocation.  out_val / out_idx [batch][n_far] =
 * this shard's n_far farthest rows (squared distance to the old centre of their label; largest first, lowest
 * index on ties; idx -1 past the shard's size).  The host merges the ranks' lists and applies the moves to the
 * all-reduced sums (opticalflowclustering_b200/kmeans.py, _relocate_across_ranks).  scratch: as above. */
int ofc_kmeans_far_points(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                          const int32_t* labels, const double* centres_old, int n_far,
                          double* out_val, int64_t* out_idx, double* scratch, void* stream);

/* The same relocation for row-sharded data WITHOUT a host round trip: after the all-reduce of sums / counts every rank
 * calls ofc_kmeans_far_payload (payload f64 [batch][n_far][3 + d] = value, global row index, label, row -- all -1 when
 * no cluster is empty, in which case the row pass is skipped on the device), all-gathers the payloads into
 * all_payload [world][batch][n_far][3 + d] and calls ofc_kmeans_relocate_merge, which applies the same moves on every
 * rank: each empty cluster, in index order, takes the globally farthest remaining row (ties: lowest global index).
 * More than n_far clusters empty at once sets *overflow (sticky, may be NULL); the caller then falls back to
 * ofc_kmeans_far_points with a larger list. */
int ofc_kmeans_far_payload(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                           const int32_t* labels, const double* centres_old, const int64_t* counts, int raw_sums,
                           int n_far, int64_t row_offset, double* payload, double* scratch, const uint8_t* active,
                           void* stream);
int ofc_kmeans_relocate_merge(int batch, int d, int k, int world, int n_far, const double* all_payload, double* sums,
                              int64_t* counts, int32_t* overflow, const uint8_t* active, void* stream);

/* The exchange step of the row-sharded fit over NVLink peer memory, one kernel per rank and exchange instead of one
 * library collective per buffer (replaces, for ranks on one node, the all-reduce of sums / counts / label changes and the
 * all-gather of the far-point payloads above; what a multi-worker KMeans.fit of KmeanGrids.py:299-304 has to exchange
 * per Lloyd iteration).  Each rank owns one buffer: ofc_peer_alloc (cudaMalloc, zeroed; `handle64` = its 64-byte CUDA
 * IPC handle, to be sent to the other ranks by whatever transport the host has), ofc_peer_open maps a peer's buffer
 * into this process.  Layout: ofc_peer_header_bytes() of flags, then regions the caller lays out (offsets multiple of
 * 16).  `bufs` = DEVICE array of `world` pointers (own buffer at [rank]).
 * ofc_peer_exchange, enqueued by every rank on its own stream after the kernels that filled its region:
 *   mode 0: out_f64[i] = sum over ranks (in rank order: bit-identical on every rank) of the region's first n_f64 doubles,
 *           out_i64[i] = the same for the n_i64 int64 that follow;
 *   mode 1: out_f64[src][i] = rank src's n_f64 doubles (all-gather).
 * gate (device int64[gate_n], identical on all ranks, may be NULL): the exchange is skipped unless one entry is zero
 * ("some cluster is empty").  A region may be rewritten once ANOTHER exchange has completed after the one that read it
 * (alternate two regions).  A rank that waits longer than timeout_s (<= 0: 10 s) for a peer sets the error word that
 * ofc_peer_error reads back (after a stream synchronise) instead of hanging the device. */
size_t ofc_peer_header_bytes(void);
int ofc_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int ofc_peer_open(const unsigned char* handle64, void** ptr);
int ofc_peer_close(void* ptr);
int ofc_peer_free(void* ptr);
int ofc_peer_exchange(const void* bufs, int world, int rank, size_t region_offset, int mode, int64_t n_f64, int64_t n_i64,
                      double* out_f64, int64_t* out_i64, const int64_t* gate, int gate_n, double timeout_s, void* stream);
int ofc_peer_error(const void* own_buffer, int* err);

/* Whole Lloyd runs on the device, one CTA per problem: the reference's per-cell fits
 * (KMeans(n_clusters=k).fit on every grid cell of a frame, KmeanGrids.py:376-392) in ONE launch --
 * column statistics, seeding, all iterations, relocation, sklearn's stopping rule, closing E-step.
 * X u8 [batch][n][d], d <= 8, k <= 64, n <= 2^20.  init [batch][k][d] (float64) gives the same labels /
 * centres / n_iter as the stepwise calls above; init == NULL seeds with k-means++ (sklearn's procedure,
 * counter-based random stream from `seed`; workspace >= batch*n*8 bytes).  counts = members per cluster
 * of the final labels (the reference's bincount of predict(), KmeanGrids.py:304-307). */
int ofc_kmeans_cells(const uint8_t* X, int batch, int64_t n, int d, int k, const double* init, uint64_t seed,
                     int max_iter, double tol, int32_t* labels, double* centres, double* inertia,
                     int32_t* n_iter, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);

/* The reference's main loop over one frame's cells, fused: image_dict ROI + preprocess_image
 * (KmeanGrids.py:85,113,269-286: white row 0 / column 0 when draw_lines, channel < threshold -> 0, alpha) +
 * KMeans(n_clusters=k).fit per cell (k-means++ from `seed`, problem index (first_frame + frame) * cells + cell,
 * so results do not depend on how a clip is cut into calls) + largest cluster -> np.rint -> BGR2HSV hue
 * (:288-339, :376-392), one CTA per cell, the cell's pixels staged once in shared memory.  k <= 16.
 * Out (each may be NULL): dom_centre u8 [n_frames][cells][4], dom_hue u8 [n_frames][cells],
 * centres f64 [n_frames][cells][k][4], counts i64 [n_frames][cells][k], n_iter i32 [n_frames][cells].
 * Same numbers as ofc_grid_extract_cells + ofc_kmeans_cells(init = NULL, same seed) at first_frame = 0. */
size_t ofc_grid_kmeans_cells_workspace_bytes(int n_frames, int height, int width, int rows, int cols, int k);
int ofc_grid_kmeans_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols, int draw_lines,
                          int threshold, int swap_rb, int k, uint64_t seed, uint64_t first_frame, int max_iter, double tol,
                          uint8_t* dom_centre, uint8_t* dom_hue, double* centres, int64_t* counts, int32_t* n_iter,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- k-means, dense corner on the tensor cores --------------------------------
 * The same sklearn E-step / M-step (KmeanGrids.py:299-304, color_kmeans.py:65-78;
 * _k_means_lloyd.pyx:160-213) for ONE float32 problem whose distance step is a real GEMM
 * (d >= 32, d % 4 == 0, 2 <= k <= 8192; the 1M x D sweep of BASELINE configs[4]).
 * ofc_kmeans_tc_prepare: xc = float32(x - float32(mean)) (KMeans.fit centres float32 data in
 *   float32, _kmeans.py:1487-1493; mean nullable), stored split as Xh = its top 11 significant
 *   bits (exact in TF32) and Xl = xc - Xh (exact), and xnorm[i] = |xc_i|; once per fit.
 * ofc_kmeans_tc_assign: 3xTF32 tcgen05 distance GEMM (lo.hi + hi.lo + hi.hi; TMA-fed, accumulators
 *   in tensor memory) as a filter + float32 re-evaluation of every row whose two best distances
 *   are closer than the remaining error bound: labels are bit-identical to
 *   ofc_kmeans_assign(OFC_F32) on xc.  n_changed / inertia as there (nullable); n_rechecked
 *   (nullable, device u32) = rows re-evaluated.
 * ofc_kmeans_tc_sums: M-step over a label-sorted member list (stable counting sort, float64 sums
 *   in ascending row order per cluster; deterministic, no floating-point atomics).
 * All three share one workspace of ofc_kmeans_tc_workspace_bytes(n, d, k) bytes. */
size_t ofc_kmeans_tc_workspace_bytes(int64_t n, int d, int k);
int ofc_kmeans_tc_prepare(const float* X, const double* mean /* [d] */, int64_t n, int d,
                          float* Xh /* [n][d] */, float* Xl /* [n][d] */, float* xnorm /* [n] */, void* stream);
int ofc_kmeans_tc_assign(const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d, int k,
                         const double* centres /* [k][d] */, int32_t* labels, const int32_t* prev_labels,
                         uint64_t* n_changed, double* inertia, uint32_t* n_rechecked,
                         void* workspace, size_t workspace_bytes, void* stream);
int ofc_kmeans_tc_sums(const float* Xh, const float* Xl, int64_t n, int d, int k, const int32_t* labels,
                       double* sums /* [k][d] */, int64_t* counts /* [k] */,
                       void* workspace, size_t workspace_bytes, void* stream);
/* The same for uint8 rows (the reference's pixels / hues, which sklearn works in float64): the split rows hold
 * float32(x - mean) with the float64 column mean; the tensor-core filter's bound also covers that rounding, and
 * every near-tie is re-evaluated on the ORIGINAL bytes in the float64 arithmetic of ofc_kmeans_assign(OFC_U8):
 * labels bit-identical to it (and so to sklearn given the same centres).  ofc_kmeans_tc_sums_u8 sums the raw
 * bytes (exact integers, what ofc_kmeans_sums gives for OFC_U8 with mean = NULL). */
int ofc_kmeans_tc_prepare_u8(const uint8_t* X, const double* mean /* [d] */, int64_t n, int d,
                             float* Xh, float* Xl, float* xnorm, void* stream);
int ofc_kmeans_tc_assign_u8(const uint8_t* X, const double* mean, const float* Xh, const float* Xl, const float* xnorm,
                            int64_t n, int d, int k, const double* centres, int32_t* labels,
                            const int32_t* prev_labels, uint64_t* n_changed, uint32_t* n_rechecked,
                            void* workspace, size_t workspace_bytes, void* stream);
int ofc_kmeans_tc_sums_u8(const uint8_t* X, int64_t n, int d, int k, const int32_t* labels,
                          double* sums, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);
/* Weighted fits on the tensor cores (weights f64 [n], as for ofc_kmeans_sums_weighted); the E-step's labels do not
 * depend on the weights.  _assign_weighted: inertia = sum_i w_i ||x_i - c_label||^2 (_inertia_dense).  _sums_weighted /
 * _sums_u8_weighted: sums of x w and weight_sums[j] = sum of the members' weights (_k_means_lloyd.pyx:216-218), in the
 * member list's order; counts = members as before. */
int ofc_kmeans_tc_assign_weighted(const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d, int k,
                                  const double* centres, const double* weights, int32_t* labels, const int32_t* prev_labels,
                                  uint64_t* n_changed, double* inertia, uint32_t* n_rechecked,
                                  void* workspace, size_t workspace_bytes, void* stream);
int ofc_kmeans_tc_sums_weighted(const float* Xh, const float* Xl, int64_t n, int d, int k, const int32_t* labels,
                                const double* weights, double* sums, int64_t* counts, double* weight_sums,
                                void* workspace, size_t workspace_bytes, void* stream);
int ofc_kmeans_tc_sums_u8_weighted(const uint8_t* X, int64_t n, int d, int k, const int32_t* labels, const double* weights,
                                   double* sums, int64_t* counts, double* weight_sums, void* workspace, size_t workspace_bytes,
                                   void* stream);

/* ---- k-means transform: row-to-centre distances ----------------------------
 * Replaces KMeans.transform(X) / MiniBatchKMeans.transform(X) (and the transform half of fit_transform), which
 * scikit-learn 1.9.0 computes as euclidean_distances(X, cluster_centers_) (sklearn/cluster/_kmeans.py _transform,
 * sklearn/metrics/pairwise.py _euclidean_distances; float32 inputs are upcast chunk by chunk to float64 by
 * _euclidean_distances_upcast because the norm form cancels).  out[i][j] = sqrt(d2) with d2 one sequential float64 fma
 * chain over t = 0 .. d-1 of (double(X[i][t]) - centres[j][t])^2 -- the direct difference, on the un-centred rows,
 * correctly rounded square roots.  With out_f32 the output is float32: sqrtf(float(d2)), sklearn's float32 path after its
 * float64 chunk.  An element depends only on its row and centre (not on n, k or the kernel form).
 * dtype OFC_U8 / OFC_F32 / OFC_F64; centres f64 [k][d] (float32 values for a float32 fit); out f64 [n][k], or f32 [n][k]
 * when out_f32, which is valid with OFC_F32 rows only (OFC_ERR_INVALID otherwise).  n may exceed 2^31 / k. */
int ofc_kmeans_distances(const void* X, int dtype, int64_t n, int d, int k,
                         const double* centres /* [k][d] */, void* out /* [n][k] */, int out_f32, void* stream);

/* image_dict ROIs (KmeanGrids.py:85,113) + preprocess_image (:269-286) for every cell:
 * out u8 [n_frames][rows*cols][ (H/rows)*(W/cols) ][4] = (c0, c1, c2, alpha).  draw_lines:
 * white row 0 / column 0 as at the reference's k-means stage (SURVEY.md Q3); swap_rb:
 * read_image's BGR->RGB (color_kmeans.py:32-33). */
int ofc_grid_extract_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols,
                           int draw_lines, int threshold, int swap_rb, uint8_t* out, void* stream);

/* ---- cosine similarity ------------------------------------------------------
 * findCosineDifferentVectors.py:5-66: sims[i] = cos(a, b[i:i+n]) for i in 0..m-n
 * (0 when a norm is 0), *best = max, *best_idx = LAST i attaining it. */
int ofc_sliding_cosine(const double* a, int n, const double* b, int64_t m,
                       double* sims /* [m-n+1] */, double* best, int64_t* best_idx, void* stream);
/* out[i] = cos(X[i,:], q) for the n rows of X [n][d] (the 1M-row sweep; same formula). */
int ofc_row_cosine(const void* X, int dtype, int64_t n, int d, const double* q, double* out, void* stream);
/* computeVectorDistance.py:22-43 on two length-n columns: *cos = sklearn cosine_similarity of
 * the flattened vectors, quirk_row[j] = a[0]*b[j] / (|a[j]|*|b[j]|) (the script's printed
 * "Cosine similarity" row, :25,29), *l1 = sum |a-b|.  Any output may be NULL. */
int ofc_vector_distance(const double* a, const double* b, int64_t n, double* cos, double* quirk_row,
                        double* l1, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OFC_H_ */
