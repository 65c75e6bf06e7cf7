// Elkan's k-means step kernels (ofc_kmeans_elkan_* in ofc.h): scikit-learn 1.9.0's dense Elkan iteration
// (sklearn/cluster/_k_means_elkan.pyx) with the triangle-inequality bounds kept on the device.
//
// Arithmetic: every distance is _euclidean_dense_dense (_k_means_common.pyx:16-43) in the working type W (float for
// float32 rows, double for uint8 and float64 rows): the features in groups of four, each group summed as
// ((d0^2 + d1^2) + d2^2) + d3^2 and then added to the running total, the remainder added one feature at a time, every
// product and sum rounded on its own (explicit _rn intrinsics, so nvcc cannot contract them into fma), the square root
// correctly rounded in W.  A row is centred as sklearn's working copy holds it: x - mean rounded in W (uint8 rows:
// double(x) - mean).  So a label, an upper bound and every lower bound are the bits sklearn's loops produce from the
// same centres and centre half-distances.
//
// Launch forms, chosen from (d, k, W) alone -- one thread per row in all of them:
//   * the centres (as W), the half-distances chd [k][k] and dnc [k] in shared memory when they fit 48 KB, else read
//     from global memory (L1/L2 resident: k^2 + k d values);
//   * the centred row in registers for d <= 4 and d <= 16, else re-read from global memory per distance.
// A warp per row (lanes splitting the features) would change the summation order, and lanes splitting the centres
// would have to replay the sequential label / upper-bound updates, so neither is used.
#include <math.h>

#include "ofc_common.cuh"
#include "kmeans_kernels.cuh"

namespace ofc {

__device__ __forceinline__ double el_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float el_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double el_sub(double a, double b) { return __dadd_rn(a, -b); }
__device__ __forceinline__ float el_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double el_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float el_mul(float a, float b) { return __fmul_rn(a, b); }
#ifndef OFC_EMULATE
__device__ __forceinline__ double el_sqrt(double a) { return __dsqrt_rn(a); }
#else
static inline double el_sqrt(double a) { return sqrt(a); }
#endif
__device__ __forceinline__ float el_sqrt(float a) { return __fsqrt_rn(a); }

constexpr int EL_THREADS = 256;
constexpr size_t EL_SMEM_MAX = 48 * 1024;

// _euclidean_dense_dense of a(t) and b(t), t < d (squared when `squared`)
template <class W, class A, class B>
__device__ __forceinline__ W el_dist(const A& a, const B& b, int d, bool squared) {
    W r = (W)0;
    int t = 0;
    for (; t + 4 <= d; t += 4) {
        const W d0 = el_sub(a(t), b(t)), d1 = el_sub(a(t + 1), b(t + 1)), d2 = el_sub(a(t + 2), b(t + 2)),
                d3 = el_sub(a(t + 3), b(t + 3));
        r = el_add(r, el_add(el_add(el_add(el_mul(d0, d0), el_mul(d1, d1)), el_mul(d2, d2)), el_mul(d3, d3)));
    }
    for (; t < d; ++t) {
        const W df = el_sub(a(t), b(t));
        r = el_add(r, el_mul(df, df));
    }
    return squared ? r : el_sqrt(r);
}

// the same with a[] in registers (d <= DR): every index a compile-time constant, the same operations in the same order
template <class W, int DR, class B>
__device__ __forceinline__ W el_dist_reg(const W (&a)[DR], const B& b, int d, bool squared) {
    W r = (W)0;
    const int g4 = d & ~3;
#pragma unroll
    for (int t = 0; t < DR; t += 4) {
        if (t + 4 <= d) {
            const W d0 = el_sub(a[t], b(t)), d1 = el_sub(a[t + 1], b(t + 1)), d2 = el_sub(a[t + 2], b(t + 2)),
                    d3 = el_sub(a[t + 3], b(t + 3));
            r = el_add(r, el_add(el_add(el_add(el_mul(d0, d0), el_mul(d1, d1)), el_mul(d2, d2)), el_mul(d3, d3)));
        }
    }
#pragma unroll
    for (int t = 0; t < DR; ++t) {
        if (t >= g4 && t < d) {
            const W df = el_sub(a[t], b(t));
            r = el_add(r, el_mul(df, df));
        }
    }
    return squared ? r : el_sqrt(r);
}

// the centre geometry one problem's CTA reads: staged in shared memory (SM) or straight from global memory
template <class W, bool SM>
struct ElkanGeo {
    const double* gc;           // [k][d] centres (global)
    const W* gh;                // [k][k] half-distances (global)
    const W* gn;                // [k] distance to the next centre (global), or null
    W* s;                       // shared: centres [k][d] as W, then chd [k][k], then dnc [k]
    int d, k;
    __device__ __forceinline__ W c(int j, int t) const { return SM ? s[j * d + t] : (W)gc[(int64_t)j * d + t]; }
    __device__ __forceinline__ W h(int a, int b) const { return SM ? s[k * d + a * k + b] : gh[(int64_t)a * k + b]; }
    __device__ __forceinline__ W dn(int j) const { return SM ? s[k * d + k * k + j] : gn[j]; }
    __device__ void stage() {
        if (!SM) return;
        for (int e = threadIdx.x; e < k * d; e += blockDim.x) s[e] = (W)gc[e];
        for (int e = threadIdx.x; e < k * k; e += blockDim.x) s[k * d + e] = gh[e];
        if (gn)
            for (int e = threadIdx.x; e < k; e += blockDim.x) s[k * d + k * k + e] = gn[e];
        __syncthreads();
    }
};

// centre j of a geometry as an accessor t -> W
template <class G>
struct ElkanCentre {
    const G& g;
    int j;
    __device__ __forceinline__ auto operator()(int t) const { return g.c(j, t); }
};

// a [k][d] float64 array's row j as W
template <class W>
struct ElkanRowOf {
    const double* p;
    __device__ __forceinline__ W operator()(int t) const { return (W)p[t]; }
};

template <class W>
static size_t elkan_smem_bytes(int d, int k) { return ((size_t)k * d + (size_t)k * k + k) * sizeof(W); }

// one row, centred in W: in registers (DR > 0, d <= DR) or re-read from global memory (DR = 0)
template <class T, class W, int DR>
struct ElkanRow {
    W x[DR > 0 ? DR : 4];
    const T* g;
    const double* mean;
    int d;
    __device__ __forceinline__ void load(const T* row, const double* m, int d_) {
        g = row; mean = m; d = d_;
        if (DR > 0) {
#pragma unroll
            for (int t = 0; t < (DR > 0 ? DR : 4); ++t) x[t] = t < d ? centred(t) : (W)0;
        }
    }
    __device__ __forceinline__ W centred(int t) const {
        return mean ? el_sub((W)g[t], (W)mean[t]) : (W)g[t];
    }
    __device__ __forceinline__ W operator()(int t) const { return centred(t); }
    template <class B>
    __device__ __forceinline__ W dist(const B& b, bool squared) const {
        if constexpr (DR > 0) return el_dist_reg<W, DR>(x, b, d, squared);
        else return el_dist<W>(*this, b, d, squared);
    }
};

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ bool el_runs(const unsigned char* active, const unsigned char* also, int b) {
    return (!active || active[b]) || (also && also[b]);
}

// ---- init_bounds_dense (_k_means_elkan.pyx:24-97) ------------------------------------------------------------------
template <class T, class W, int DR, bool SM>
__global__ void __launch_bounds__(EL_THREADS, 1) kmeans_elkan_init_kernel(const T* __restrict__ Xall, int64_t x_stride, int64_t n,
                                                                     int d, int k, const double* __restrict__ mean_all,
                                                                     const double* __restrict__ centres_all,
                                                                     const W* __restrict__ chd_all, int32_t* __restrict__ labels_all,
                                                                     W* __restrict__ upper_all, W* __restrict__ lower_all,
                                                                     const unsigned char* __restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    OFC_DYN_SMEM(W, smem);
    ElkanGeo<W, SM> geo{centres_all + (int64_t)b * k * d, chd_all + (int64_t)b * k * k, nullptr, smem, d, k};
    geo.stage();
    const T* X = Xall + b * x_stride;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    for (int64_t i = (int64_t)blockIdx.x * EL_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * EL_THREADS) {
        ElkanRow<T, W, DR> x;
        x.load(X + i * d, mean, d);
        W* lo = lower_all + ((int64_t)b * n + i) * k;
        int best = 0;
        W m = x.dist(ElkanCentre<decltype(geo)>{geo, 0}, false);
        lo[0] = m;
        for (int j = 1; j < k; ++j) {
            if (m > geo.h(best, j)) {
                const W dj = x.dist(ElkanCentre<decltype(geo)>{geo, j}, false);
                lo[j] = dj;
                if (dj < m) { m = dj; best = j; }
            } else {
                lo[j] = (W)0;                                   // never computed: sklearn's np.zeros
            }
        }
        labels_all[(int64_t)b * n + i] = best;
        upper_all[(int64_t)b * n + i] = m;
    }
}

// ---- the label half of _update_chunk_dense (_k_means_elkan.pyx:352-427) ------------------------------------------------
template <class T, class W, int DR, bool SM>
__global__ void __launch_bounds__(EL_THREADS, 1) kmeans_elkan_step_kernel(const T* __restrict__ Xall, int64_t x_stride, int64_t n,
                                                                     int d, int k, const double* __restrict__ mean_all,
                                                                     const double* __restrict__ centres_all,
                                                                     const W* __restrict__ chd_all, const W* __restrict__ dnc_all,
                                                                     const int32_t* labels_in_all, int32_t* labels_all,
                                                                     const int32_t* __restrict__ prev_all, W* __restrict__ upper_all,
                                                                     W* __restrict__ lower_all, unsigned long long* n_changed,
                                                                     unsigned long long* n_dist, const unsigned char* __restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    OFC_DYN_SMEM(W, smem);
    ElkanGeo<W, SM> geo{centres_all + (int64_t)b * k * d, chd_all + (int64_t)b * k * k, dnc_all + (int64_t)b * k, smem, d, k};
    geo.stage();
    const T* X = Xall + b * x_stride;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    unsigned long long changed = 0, evaluated = 0;
    for (int64_t i = (int64_t)blockIdx.x * EL_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * EL_THREADS) {
        const int64_t r = (int64_t)b * n + i;
        int label = labels_in_all[r];
        W ub = upper_all[r];
        if (!(geo.dn(label) >= ub)) {                           // dnc first: a settled row reads one label and one bound
            ElkanRow<T, W, DR> x;
            x.load(X + i * d, mean, d);
            W* lo = lower_all + r * k;
            bool tight = false;
            for (int j = 0; j < k; ++j) {
                if (j != label && ub > lo[j] && ub > geo.h(label, j)) {
                    if (!tight) {
                        ub = x.dist(ElkanCentre<decltype(geo)>{geo, label}, false);
                        lo[label] = ub;
                        tight = true;
                        ++evaluated;
                    }
                    if (ub > lo[j] || ub > geo.h(label, j)) {
                        const W dj = x.dist(ElkanCentre<decltype(geo)>{geo, j}, false);
                        lo[j] = dj;
                        ++evaluated;
                        if (dj < ub) { label = j; ub = dj; }
                    }
                }
            }
            upper_all[r] = ub;
        }
        labels_all[r] = label;
        changed += prev_all ? (label != prev_all[r] ? 1ull : 0ull) : 1ull;     // no previous labels: sklearn's -1 start
    }
    changed = warp_sum_u64(changed);
    evaluated = warp_sum_u64(evaluated);
    if ((threadIdx.x & 31) == 0) {
        if (n_changed && changed) atomicAdd(n_changed + b, changed);
        if (n_dist && evaluated) atomicAdd(n_dist + b, evaluated);
    }
}

__global__ void kmeans_elkan_zero_kernel(int batch, unsigned long long* n_changed, const unsigned char* active) {
    for (int b = threadIdx.x; b < batch; b += blockDim.x)
        if (!active || active[b]) n_changed[b] = 0ull;
}

// ---- _center_shift (_k_means_common.pyx:298-311) and the bound update of elkan_iter_chunked_dense (:336-343) ----------
template <class W>
__global__ void __launch_bounds__(EL_THREADS) kmeans_elkan_shift_kernel(int d, int k, const double* __restrict__ old_all,
                                                                       const double* __restrict__ new_all, W* __restrict__ shift_all,
                                                                       const unsigned char* active, const unsigned char* also) {
    const int b = blockIdx.x;
    if (!el_runs(active, also, b)) return;
    const double* o = old_all + (int64_t)b * k * d;
    const double* c = new_all + (int64_t)b * k * d;
    for (int j = threadIdx.x; j < k; j += EL_THREADS)
        shift_all[(int64_t)b * k + j] = el_dist<W>(ElkanRowOf<W>{c + (int64_t)j * d}, ElkanRowOf<W>{o + (int64_t)j * d}, d, false);
}

template <class W>
__global__ void __launch_bounds__(EL_THREADS) kmeans_elkan_bounds_kernel(int64_t n, int k, const W* __restrict__ shift_all,
                                                                        const int32_t* __restrict__ labels_all, W* __restrict__ upper_all,
                                                                        W* __restrict__ lower_all, const unsigned char* active,
                                                                        const unsigned char* also) {
    const int b = blockIdx.y;
    if (!el_runs(active, also, b)) return;
    OFC_DYN_SMEM(W, s_shift);
    for (int j = threadIdx.x; j < k; j += EL_THREADS) s_shift[j] = shift_all[(int64_t)b * k + j];
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * EL_THREADS;
    for (int64_t i = (int64_t)blockIdx.x * EL_THREADS + threadIdx.x; i < n; i += stride) {
        const int64_t r = (int64_t)b * n + i;
        upper_all[r] = el_add(upper_all[r], s_shift[labels_all[r]]);
    }
    // lower -= shift, clamped at 0: one pass over the [n][k] bounds, the column index carried incrementally
    W* lo = lower_all + (int64_t)b * n * k;
    const int64_t total = n * k;
    int64_t e = (int64_t)blockIdx.x * EL_THREADS + threadIdx.x;
    if (e >= total) return;
    int j = (int)(e % k);
    const int step = (int)(stride % k);
    for (; e < total; e += stride) {
        W v = el_sub(lo[e], s_shift[j]);
        if (v < (W)0) v = (W)0;
        lo[e] = v;
        j += step;
        if (j >= k) j -= k;
    }
}

// ---- centre half-distances: halve ofc_kmeans_distances' output in W, dnc = np.partition(chd, 1, axis=0)[1] -----------
__global__ void kmeans_elkan_to_f32_kernel(int64_t count, const double* __restrict__ src, float* __restrict__ dst) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
        dst[e] = (float)src[e];
}

template <class W>
__global__ void __launch_bounds__(EL_THREADS) kmeans_elkan_halve_kernel(int k, W* __restrict__ chd_all, W* __restrict__ dnc_all) {
    const int b = blockIdx.x;
    // chd is exactly symmetric (the distance kernel squares x - c), so column j's second smallest is row j's
    for (int j = threadIdx.x; j < k; j += EL_THREADS) {
        W* row = chd_all + ((int64_t)b * k + j) * k;
        W m1 = (W)INFINITY, m2 = (W)INFINITY;
        for (int i = 0; i < k; ++i) {
            const W v = el_mul(row[i], (W)0.5);
            row[i] = v;
            if (v < m1) { m2 = m1; m1 = v; }
            else if (v < m2) m2 = v;
        }
        dnc_all[(int64_t)b * k + j] = m2;
    }
}

// ---- _inertia_dense (_k_means_common.pyx:105-135) of given labels ---------------------------------------------------------
template <class T, class W>
__global__ void __launch_bounds__(EL_THREADS) kmeans_elkan_inertia_kernel(const T* __restrict__ Xall, int64_t x_stride, int64_t n,
                                                                         int d, int k, const double* __restrict__ mean_all,
                                                                         const double* __restrict__ centres_all,
                                                                         const int32_t* __restrict__ labels_all,
                                                                         const double* __restrict__ weights, int64_t w_stride,
                                                                         double* __restrict__ partial, const unsigned char* active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const T* X = Xall + b * x_stride;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    const double* C = centres_all + (int64_t)b * k * d;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * EL_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * EL_THREADS) {
        ElkanRow<T, W, 0> x;
        x.load(X + i * d, mean, d);
        const int l = labels_all[(int64_t)b * n + i];
        W sq = x.dist(ElkanRowOf<W>{C + (int64_t)l * d}, true);
        if (weights) sq = el_mul(sq, (W)weights[b * w_stride + i]);
        acc += (double)sq;
    }
    __shared__ double red[EL_THREADS];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = EL_THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[(int64_t)b * gridDim.x + blockIdx.x] = red[0];
}

// ---- launchers ------------------------------------------------------------------------------------------------------------
static unsigned elkan_row_blocks(int64_t n) {
    int64_t blocks = (n + EL_THREADS - 1) / EL_THREADS;
    if (blocks > 148 * 8) blocks = 148 * 8;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

// the launch form of the init and step kernels, from (dtype, d, k) alone
static int kmeans_elkan_form(int dtype, int d, int k) {
    const size_t bytes = dtype == DT_F32 ? elkan_smem_bytes<float>(d, k) : elkan_smem_bytes<double>(d, k);
    const int smem = bytes <= EL_SMEM_MAX ? 1 : 0;
    const int regs = d <= 4 ? 2 : (d <= 16 ? 1 : 0);
    return smem * 4 + regs;                  // bit 2: geometry in shared memory; bits 0-1: row in registers (2: d <= 4, 1: d <= 16)
}

template <class T, class W>
static int launch_elkan_typed(const ElkanArgs& a, void* stream) {
    const int form = kmeans_elkan_form(a.dtype, a.d, a.k);
    const bool sm = (form & 4) != 0;
    const size_t smem = sm ? elkan_smem_bytes<W>(a.d, a.k) : 0;
    const dim3 grid(elkan_row_blocks(a.n), (unsigned)a.batch);
    const T* X = (const T*)a.X;
    W* upper = (W*)a.upper;
    W* lower = (W*)a.lower;
    const W* chd = (const W*)a.chd;
    const W* dnc = (const W*)a.dnc;
#define OFC_EL(DR, SMF)                                                                                                       \
    do {                                                                                                                      \
        if (a.init)                                                                                                           \
            OFC_LAUNCH((kmeans_elkan_init_kernel<T, W, DR, SMF>), grid, dim3(EL_THREADS), smem, stream, X, a.x_stride, a.n,   \
                       a.d, a.k, a.mean, a.centres, chd, a.labels, upper, lower, a.active);                                   \
        else                                                                                                                  \
            OFC_LAUNCH((kmeans_elkan_step_kernel<T, W, DR, SMF>), grid, dim3(EL_THREADS), smem, stream, X, a.x_stride, a.n,   \
                       a.d, a.k, a.mean, a.centres, chd, dnc, a.labels_in, a.labels, a.prev_labels, upper, lower,             \
                       a.n_changed, a.n_dist, a.active);                                                                      \
    } while (0)
    if (sm) {
        if ((form & 3) == 2) OFC_EL(4, true);
        else if ((form & 3) == 1) OFC_EL(16, true);
        else OFC_EL(0, true);
    } else {
        if ((form & 3) == 2) OFC_EL(4, false);
        else if ((form & 3) == 1) OFC_EL(16, false);
        else OFC_EL(0, false);
    }
#undef OFC_EL
    OFC_CHECK_LAUNCH(a.init ? "kmeans_elkan_init" : "kmeans_elkan_step");
    return OFC_OK;
}

int launch_kmeans_elkan(const ElkanArgs& a, void* stream) {
    if (a.batch <= 0 || a.n <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    if (!a.init && a.n_changed) {
        OFC_LAUNCH(kmeans_elkan_zero_kernel, dim3(1), dim3(128), 0, stream, a.batch, a.n_changed, a.active);
        OFC_CHECK_LAUNCH("kmeans_elkan_zero");
    }
    if (a.dtype == DT_U8) return launch_elkan_typed<unsigned char, double>(a, stream);
    if (a.dtype == DT_F32) return launch_elkan_typed<float, float>(a, stream);
    return launch_elkan_typed<double, double>(a, stream);
}

template <class W>
static int launch_bounds_typed(int batch, int64_t n, int d, int k, const double* centres_old, const double* centres,
                               const int32_t* labels, W* upper, W* lower, const unsigned char* active, const unsigned char* just_done,
                               W* shift, void* stream) {
    OFC_LAUNCH(kmeans_elkan_shift_kernel<W>, dim3(batch), dim3(EL_THREADS), 0, stream, d, k, centres_old, centres, shift, active,
               just_done);
    OFC_CHECK_LAUNCH("kmeans_elkan_shift");
    int64_t blocks = (n * k + EL_THREADS - 1) / EL_THREADS;
    if (blocks > 148 * 16) blocks = 148 * 16;
    const size_t smem = (size_t)k * sizeof(W);
    OFC_SMEM_OPTIN(kmeans_elkan_bounds_kernel<W>, smem);
    OFC_LAUNCH(kmeans_elkan_bounds_kernel<W>, dim3((unsigned)blocks, batch), dim3(EL_THREADS), smem, stream, n, k, shift, labels,
               upper, lower, active, just_done);
    OFC_CHECK_LAUNCH("kmeans_elkan_bounds");
    return OFC_OK;
}

int launch_kmeans_elkan_bounds(int dtype, int batch, int64_t n, int d, int k, const double* centres_old, const double* centres,
                               const int32_t* labels, void* upper, void* lower, const unsigned char* active,
                               const unsigned char* just_done, void* shift_ws, void* stream) {
    if (batch <= 0 || n <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    if (dtype == DT_F32)
        return launch_bounds_typed<float>(batch, n, d, k, centres_old, centres, labels, (float*)upper, (float*)lower, active, just_done,
                                          (float*)shift_ws, stream);
    return launch_bounds_typed<double>(batch, n, d, k, centres_old, centres, labels, (double*)upper, (double*)lower, active, just_done,
                                       (double*)shift_ws, stream);
}

int launch_kmeans_elkan_centres(int dtype, int batch, int d, int k, const double* centres, void* chd, void* dnc, float* f32_ws,
                                void* stream) {
    if (batch <= 0) return OFC_OK;
    const bool f32 = dtype == DT_F32;
    const size_t wsz = f32 ? 4 : 8;
    if (f32) {
        ProfScope prof(PK_KMEANS, stream);
        const int64_t count = (int64_t)batch * k * d;
        OFC_LAUNCH(kmeans_elkan_to_f32_kernel, dim3((unsigned)((count + 255) / 256 < 1024 ? (count + 255) / 256 : 1024)), dim3(256), 0,
                   stream, count, centres, f32_ws);
        OFC_CHECK_LAUNCH("kmeans_elkan_to_f32");
    }
    // the centres against themselves through ofc_kmeans_distances (direct difference, float32 output after a float32 fit)
    for (int b = 0; b < batch; ++b) {
        const void* cb = f32 ? (const void*)(f32_ws + (int64_t)b * k * d) : (const void*)(centres + (int64_t)b * k * d);
        const int rc = launch_kmeans_distances(cb, f32 ? DT_F32 : DT_F64, k, d, k, centres + (int64_t)b * k * d,
                                               (char*)chd + (size_t)b * k * k * wsz, f32 ? 1 : 0, stream);
        if (rc != OFC_OK) return rc;
    }
    ProfScope prof(PK_KMEANS, stream);
    if (f32) OFC_LAUNCH(kmeans_elkan_halve_kernel<float>, dim3(batch), dim3(EL_THREADS), 0, stream, k, (float*)chd, (float*)dnc);
    else OFC_LAUNCH(kmeans_elkan_halve_kernel<double>, dim3(batch), dim3(EL_THREADS), 0, stream, k, (double*)chd, (double*)dnc);
    OFC_CHECK_LAUNCH("kmeans_elkan_halve");
    return OFC_OK;
}

int launch_kmeans_elkan_inertia(const void* X, int64_t x_stride, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                                const double* centres, const int32_t* labels, const double* weights, int64_t w_stride, double* partial,
                                int parts, double* inertia, const unsigned char* active, void* stream) {
    if (batch <= 0 || n <= 0) return OFC_OK;
    {
        ProfScope prof(PK_KMEANS, stream);
        const dim3 grid((unsigned)parts, (unsigned)batch);
#define OFC_EI(T, W) OFC_LAUNCH((kmeans_elkan_inertia_kernel<T, W>), grid, dim3(EL_THREADS), 0, stream, (const T*)X, x_stride, n, d, k, \
                                mean, centres, labels, weights, w_stride, partial, active)
        if (dtype == DT_U8) OFC_EI(unsigned char, double);
        else if (dtype == DT_F32) OFC_EI(float, float);
        else OFC_EI(double, double);
#undef OFC_EI
        OFC_CHECK_LAUNCH("kmeans_elkan_inertia");
    }
    return launch_inertia_reduce(partial, parts, batch, inertia, active, stream);
}

}  // namespace ofc
