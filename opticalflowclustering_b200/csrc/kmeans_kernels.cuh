// Parameter blocks and launchers of kmeans_kernels.cu / cosine_kernels.cu (internal header).
#pragma once
#include "ofc_common.cuh"

namespace ofc {

enum { DT_U8 = 0, DT_F32 = 1, DT_F64 = 2 };

static inline size_t dtype_size(int dtype) { return dtype == DT_U8 ? 1 : (dtype == DT_F32 ? 4 : 8); }

struct KmAssignParams {
    const void* X;               // [batch][n][d], or one [n][d] for every problem (x_stride = 0)
    int64_t x_stride;            // elements between two problems' rows: n * d, or 0 (OFC_KMEANS_SHARED_ROWS)
    int dtype;
    int64_t n;
    int d, k;
    const double* mean;          // [batch][d] subtracted from every row, or null
    const double* centres;       // [batch][k][d]
    const double* c2;            // [batch][k] squared norms (generic path only)
    int32_t* labels;             // [batch][n] out
    const int32_t* prev_labels;  // [batch][n] or null
    unsigned long long* n_changed;   // [batch] (+= labels that differ from prev_labels) or null
    double* inertia_partial;     // [batch][gridDim.x] or null
    double* min_dist;            // [batch][n] squared distance to the chosen centre, or null
    const unsigned char* active; // [batch] problems to process (null = all)
    const double* weights = nullptr;   // [batch][n] sample weights (inertia = sum w_i d_i), or null (unweighted)
    int64_t w_stride = 0;        // n, or 0 when every problem reads one [n] vector (OFC_KMEANS_SHARED_ROWS)
};

struct KmSumsParams {
    const void* X;
    int64_t x_stride;            // as in KmAssignParams
    int dtype;
    int64_t n;
    int d, k;
    const double* mean;          // [batch][d] or null
    const int32_t* labels;       // [batch][n] or null (everything in cluster 0)
    int square;                  // accumulate (x-mean)^2 instead of (x-mean)
    double* partial;             // [batch][splits][k][d]
    long long* cnt_partial;      // [batch][splits][k]
    int splits;
    int dt;                      // dims per lane group (power of two <= 32)
    int kt;                      // clusters per shared-memory pass
    const unsigned char* active; // [batch] or null
    const double* weights = nullptr;   // as in KmAssignParams: sums of x w and weight sums instead of member counts
    int64_t w_stride = 0;
    double* wcnt_partial = nullptr;    // [batch][splits][k] weight partials (weighted only; in place of cnt_partial)
};

int launch_kmeans_assign(KmAssignParams p, int batch, double* c2_ws, void* stream);
int launch_kmeans_sums(const KmSumsParams& p, int batch, double* sums, long long* counts, void* stream);
// p.weights set: weight_sums[b][j] = sum of the members' weights (float64) in place of the member counts
int launch_kmeans_sums_weighted(const KmSumsParams& p, int batch, double* sums, double* weight_sums, void* stream);
// fused E-step + M-step sums for uint8 rows whose [k][d] accumulators fit shared memory (one pass over X)
int kmeans_step_grid(int64_t n, int batch);
size_t kmeans_step_smem(int d, int k);
int launch_kmeans_step_u8(KmAssignParams p, int batch, double* partial, long long* cnt_partial, double* sums, long long* counts,
                          void* stream);
int launch_kmeans_centres(int batch, int d, int k, const double* sums, const long long* counts, const double* mean_sub,
                          int use_reciprocal, double* centres, double* shift_tot, double* shift_ws,
                          const unsigned char* active, void* stream);
int launch_kmeans_update(int batch, int d, int k, const double* sums, const long long* counts, const double* mean_sub,
                         int use_reciprocal, int round_f32, double* centres, double* shift_tot, double* shift_ws,
                         const unsigned long long* n_changed, const double* tol, int it, unsigned char* active,
                         unsigned char* just_done, int* n_iter, int* n_active, int64_t n, const int32_t* labels_cur,
                         int32_t* labels_other, int* it_counter, void* stream);
// the same driven by float64 cluster weights (empty = weight 0, the heaviest cluster by weight)
int launch_kmeans_update(int batch, int d, int k, const double* sums, const double* weight_sums, const double* mean_sub,
                         int use_reciprocal, int round_f32, double* centres, double* shift_tot, double* shift_ws,
                         const unsigned long long* n_changed, const double* tol, int it, unsigned char* active,
                         unsigned char* just_done, int* n_iter, int* n_active, int64_t n, const int32_t* labels_cur,
                         int32_t* labels_other, int* it_counter, void* stream);
// weights NULL: unit weights (the unweighted kernel)
int launch_minibatch_update(const void* Xb, int dtype, int bs, int d, int k, const int32_t* labels, const double* weights,
                            const double* centres_old, double* centres_new, double* weight_sums, void* stream);
int launch_kmeans_relocate(const void* X, int64_t x_stride, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                           const int32_t* labels, const double* centres_old, double* sums, long long* counts,
                           int raw_sums, const unsigned char* active, double* scratch, void* stream);
// weighted: a cluster is empty when its weight is 0; the moved row carries x w and w (weights [batch][n], w_stride n or 0);
// always the two-kernel form (scratch required)
int launch_kmeans_relocate_weighted(const void* X, int64_t x_stride, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                                    const int32_t* labels, const double* centres_old, const double* weights, int64_t w_stride,
                                    double* sums, double* weight_sums, int raw_sums, const unsigned char* active, double* scratch,
                                    void* stream);
int launch_kmeans_far_payload(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                              const double* centres_old, const long long* counts, int raw_sums, int n_far, long long row_offset,
                              double* payload, double* scratch, const unsigned char* active, void* stream);
int launch_kmeans_relocate_merge(int batch, int d, int k, int world, int n_far, const double* allpay, double* sums, long long* counts,
                                 int* overflow, const unsigned char* active, void* stream);
int launch_kmeans_far_points(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                             const double* centres_old, int n_far, double* out_val, long long* out_idx, double* scratch, void* stream);
int launch_inertia_reduce(const double* partial, int parts, int batch, double* inertia, const unsigned char* active,
                          void* stream);
int launch_kmeans_cells(const unsigned char* X, int batch, int64_t n, int d, int k, const double* init,
                        unsigned long long seed, int max_iter, double tol, int32_t* labels, double* centres,
                        double* inertia, int32_t* n_iter, long long* counts, double* scratch, void* stream);
// fast per-cell Lloyd runs for 4-channel uint8 rows, k <= 16 (cells_kmeans.cu)
struct KmCellsFastParams {
    const unsigned char* X;        // [batch][n][4] packed rows, or null when the cells are gathered from `bgr`
    const unsigned char* bgr;      // [n_frames][H][W][3] flow visualisation (cell gather + preprocess_image fused in)
    int64_t frame_stride;          // bytes between frames
    int W, H, cols, cells, x_step, y_step, draw_lines, threshold, swap_rb;
    int n, k;
    const double* init;            // [batch][k][4] or null (k-means++ from `seed`)
    unsigned long long seed, problem_offset;
    int max_iter;
    double tol;
    int32_t* labels;               // [batch][n]      or null
    double* centres;               // [batch][k][4]   or null
    double* inertia;               // [batch]         or null
    int32_t* n_iter;               // [batch]         or null
    long long* counts;             // [batch][k]      or null
    unsigned char* dom_centre;     // [batch][4] np.rint of the largest cluster's centre, or null
    unsigned char* dom_hue;        // [batch]    BGR2HSV hue of its first three channels, or null
    unsigned* closest_ws;          // [batch][n] k-means++ scratch when it does not fit shared memory
    int closest_in_smem;           // set by the launcher
};
bool kmeans_cells_fast_supported(int64_t n, int d, int k);
size_t kmeans_cells_fast_workspace(int batch, int64_t n, int k, bool seeding);
int launch_kmeans_cells_fast(KmCellsFastParams p, int batch, void* stream);
// fused uint8 step for 4-channel rows, k <= 8 (cells_kmeans.cu): float32-filtered E-step + packed register M-step
bool kmeans_step_u8d4_usable(const KmAssignParams& p, int batch);
int launch_kmeans_step_u8d4(const KmAssignParams& p, int batch, int grid, double* partial, long long* cnt_partial, void* stream);
int kmeans_assign_grid(int64_t n);
// row-to-centre distances (kmeans_distances.cu); out_f32 only with float32 rows (the caller checks)
int launch_kmeans_distances(const void* X, int dtype, int64_t n, int d, int k, const double* centres, void* out, int out_f32,
                            void* stream);
int kmeans_sums_splits(int64_t n, int batch);

int launch_sliding_cosine(const double* a, int n, const double* b, int64_t m, double* sims, double* best,
                          long long* best_idx, void* stream);
int launch_row_cosine(const void* X, int dtype, int64_t n, int d, const double* q, double* out, void* stream);
int launch_vector_distance(const double* a, const double* b, int64_t n, double* cos_out, double* quirk_row,
                           double* l1, void* stream);
int launch_extract_cells(const unsigned char* bgr, int n_frames, int H, int W, int rows, int cols, int draw_lines,
                         int threshold, int swap_rb, unsigned char* out, void* stream);

}  // namespace ofc
