// Row-to-centre Euclidean distances for KMeans.transform / MiniBatchKMeans.transform (ofc_kmeans_distances in ofc.h).
//
// out[i][j] = sqrt(d2) with d2 = one sequential float64 fma chain over t = 0 .. d-1 of (double(x_it) - c_jt)^2; float32
// output is sqrtf(float(d2)), which is what scikit-learn's float32 path does after its float64 chunk.  An element
// therefore depends on its own row and centre only -- not on n, k, the launch geometry or which of the two forms below
// computed it:
//   * small form (d <= 16, k <= 64: the reference's pixels): one row per thread, the row in registers, the centres in
//     shared memory; a warp stages its [32 x 16] output tile in shared memory so the global stores are coalesced.  These
//     shapes are bound by writing the output (n k 8 bytes against n d read).
//   * dense form (everything else): a 64-row x 128-centre tile per CTA, 4 x 8 accumulators per thread, the feature
//     slices streamed through shared memory (centres by cp.async, rows through registers where they become float64),
//     double-buffered.  FP64-pipe bound: two instructions (sub, fma) per row, centre and feature.
// Feature padding in the last slice is zero on both sides, and fma(0, 0, acc) == acc, so the chain is unchanged.
#include <math.h>

#include "ofc_common.cuh"
#include "kmeans_kernels.cuh"

namespace ofc {

#ifndef OFC_EMULATE
__device__ __forceinline__ void dist_cp_async8(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void dist_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void dist_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
#else
// host-side debug emulation: copies are immediate
static inline void dist_cp_async8(void* dst, const void* src) { memcpy(dst, src, 8); }
static inline void dist_cp_async_commit() {}
static inline void dist_cp_async_wait_all() {}
#endif

template <class OUT> __device__ __forceinline__ OUT dist_from_sq(double d2);
template <> __device__ __forceinline__ double dist_from_sq<double>(double d2) { return sqrt(d2); }
template <> __device__ __forceinline__ float dist_from_sq<float>(double d2) { return sqrtf((float)d2); }

// ---- small form -------------------------------------------------------------------------------------------------
constexpr int DS_THREADS = 128;
constexpr int DS_KC = 16;                     // centres per staged chunk
constexpr int DS_MAX_D = 16, DS_MAX_K = 64;      // past d = 16 the row no longer fits the registers well

template <class T, class OUT, int DMAX>
__global__ void __launch_bounds__(DS_THREADS) kmeans_distances_small_kernel(const T* __restrict__ X, int64_t n, int d, int k,
                                                                           const double* __restrict__ centres,
                                                                           OUT* __restrict__ out) {
    // dynamic shared memory: the warps' output tiles, then the centres (sized to k d, so more CTAs fit an SM)
    OFC_DYN_SMEM(double, smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double (*stage)[DS_KC + 1] = reinterpret_cast<double (*)[DS_KC + 1]>(smem + warp * 32 * (DS_KC + 1));
    double* s_c = smem + DS_THREADS * (DS_KC + 1);
    for (int e = threadIdx.x; e < k * d; e += DS_THREADS) s_c[e] = centres[e];
    __syncthreads();
    const int64_t n_tiles = (n + DS_THREADS - 1) / DS_THREADS;
    double x[DMAX];
    int64_t tile = blockIdx.x;
    {
        const int64_t row = tile * DS_THREADS + threadIdx.x;
#pragma unroll
        for (int t = 0; t < DMAX; ++t) x[t] = (row < n && t < d) ? (double)X[row * d + t] : 0.0;
    }
    for (; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * DS_THREADS + warp * 32;       // this warp's first row
        // the next tile's row is loaded while this one is computed and stored
        T xn[DMAX];                                                 // in its own type: fewer registers
        const int64_t nrow = (tile + gridDim.x) * DS_THREADS + threadIdx.x;
#pragma unroll
        for (int t = 0; t < DMAX; ++t) xn[t] = (nrow < n && t < d) ? X[nrow * d + t] : T(0);
        for (int c0 = 0; c0 < k; c0 += DS_KC) {
            const int kc = min(DS_KC, k - c0);
            for (int j = 0; j < kc; ++j) {
                const double* c = s_c + (c0 + j) * d;
                double d2 = 0.0;
#pragma unroll
                for (int t = 0; t < DMAX; ++t) {
                    if (t < d) {
                        const double df = x[t] - c[t];
                        d2 = fma(df, df, d2);
                    }
                }
                stage[lane][j] = d2;
            }
            __syncwarp();
            // the warp's 32 rows x kc centres: element e is row e / kc, centre c0 + e % kc
            const int rows_here = n - row0 < 32 ? (int)(n - row0) : 32;
            for (int e = lane; e < 32 * kc; e += 32) {
                const int r = e / kc, j = e - r * kc;
                if (r < rows_here) out[(row0 + r) * k + c0 + j] = dist_from_sq<OUT>(stage[r][j]);
            }
            __syncwarp();
        }
#pragma unroll
        for (int t = 0; t < DMAX; ++t) x[t] = (double)xn[t];
    }
}

// ---- dense form -------------------------------------------------------------------------------------------------
constexpr int DD_BM = 64, DD_BN = 128, DD_BK = 16, DD_THREADS = 256;
constexpr int DD_XS = DD_BM + 2, DD_CS = DD_BN + 2;           // padded strides (doubles), 16-byte aligned rows
constexpr size_t DD_SMEM = (size_t)2 * DD_BK * (DD_XS + DD_CS) * sizeof(double);

template <class T>
__device__ __forceinline__ void dense_load_x(const T* __restrict__ X, int64_t n, int d, int64_t row0, int t0, double (&xr)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = threadIdx.x + DD_THREADS * i;
        const int r = e / DD_BK, t = e % DD_BK;
        const int64_t row = row0 + r;
        xr[i] = (row < n && t0 + t < d) ? (double)X[row * d + t0 + t] : 0.0;
    }
}

__device__ __forceinline__ void dense_store_x(double* sx, const double (&xr)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = threadIdx.x + DD_THREADS * i;
        sx[(e % DD_BK) * DD_XS + e / DD_BK] = xr[i];
    }
}

__device__ __forceinline__ void dense_load_c(const double* __restrict__ centres, int d, int k, int c0, int t0, double* sc) {
#pragma unroll
    for (int i = 0; i < DD_BK * DD_BN / DD_THREADS; ++i) {
        const int e = threadIdx.x + DD_THREADS * i;
        const int j = e / DD_BK, t = e % DD_BK;
        double* dst = sc + t * DD_CS + j;
        if (c0 + j < k && t0 + t < d) dist_cp_async8(dst, centres + (int64_t)(c0 + j) * d + t0 + t);
        else *dst = 0.0;
    }
}

template <class T, class OUT>
__global__ void __launch_bounds__(DD_THREADS, 2) kmeans_distances_dense_kernel(const T* __restrict__ X, int64_t n, int d, int k,
                                                                           const double* __restrict__ centres,
                                                                           OUT* __restrict__ out) {
    OFC_DYN_SMEM(double, smem);
    double* const sx = smem;                          // [2][DD_BK][DD_XS]
    double* const sc = smem + 2 * DD_BK * DD_XS;      // [2][DD_BK][DD_CS]
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int64_t row0 = (int64_t)blockIdx.x * DD_BM;
    const int c0 = blockIdx.y * DD_BN;
    double acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0;
    const int n_slices = (d + DD_BK - 1) / DD_BK;
    double xr[4];
    dense_load_x(X, n, d, row0, 0, xr);
    dense_load_c(centres, d, k, c0, 0, sc);
    dist_cp_async_commit();
    dense_store_x(sx, xr);
    dist_cp_async_wait_all();
    __syncthreads();
    for (int s = 0; s < n_slices; ++s) {
        const int cur = s & 1;
        const bool more = s + 1 < n_slices;
        if (more) {                               // the next slice is in flight while this one is computed
            dense_load_c(centres, d, k, c0, (s + 1) * DD_BK, sc + (cur ^ 1) * DD_BK * DD_CS);
            dist_cp_async_commit();
            dense_load_x(X, n, d, row0, (s + 1) * DD_BK, xr);
        }
        const double* xs = sx + cur * DD_BK * DD_XS + ty * 4;
        const double* cs = sc + cur * DD_BK * DD_CS + tx;
#pragma unroll 4
        for (int t = 0; t < DD_BK; ++t) {
            double xv[4], cv[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) xv[i] = xs[t * DD_XS + i];
#pragma unroll
            for (int j = 0; j < 8; ++j) cv[j] = cs[t * DD_CS + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const double df = xv[i] - cv[j];
                    acc[i][j] = fma(df, df, acc[i][j]);
                }
        }
        if (more) dense_store_x(sx + (cur ^ 1) * DD_BK * DD_XS, xr);
        dist_cp_async_wait_all();
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t row = row0 + ty * 4 + i;
        if (row >= n) continue;
        OUT* o = out + row * k;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int col = c0 + tx + 16 * j;
            if (col < k) o[col] = dist_from_sq<OUT>(acc[i][j]);
        }
    }
}

static bool kmeans_distances_small_form(int d, int k) { return d <= DS_MAX_D && k <= DS_MAX_K; }

template <class T, class OUT>
static int launch_distances_typed(const T* X, int64_t n, int d, int k, const double* centres, OUT* out, void* stream) {
    if (kmeans_distances_small_form(d, k)) {
        int64_t blocks = (n + DS_THREADS - 1) / DS_THREADS;
        if (blocks > 148 * 10) blocks = 148 * 10;
        const size_t smem = (size_t)(DS_THREADS * (DS_KC + 1) + k * d) * sizeof(double);
#define OFC_DS(DM) OFC_LAUNCH((kmeans_distances_small_kernel<T, OUT, DM>), dim3((unsigned)blocks), dim3(DS_THREADS), smem, stream, \
                              X, n, d, k, centres, out)
        if (d <= 4) OFC_DS(4);
        else if (d <= 8) OFC_DS(8);
        else OFC_DS(16);
#undef OFC_DS
        OFC_CHECK_LAUNCH("kmeans_distances_small");
        return OFC_OK;
    }
    const int64_t row_tiles = (n + DD_BM - 1) / DD_BM;
    const int col_tiles = (k + DD_BN - 1) / DD_BN;
    if (row_tiles > 0x7fffffff || col_tiles > 65535) {
        set_error("ofc_kmeans_distances: too many tiles (n=%lld, k=%d)", (long long)n, k);
        return OFC_ERR_UNSUPPORTED;
    }
    OFC_SMEM_OPTIN((kmeans_distances_dense_kernel<T, OUT>), DD_SMEM);
    OFC_LAUNCH((kmeans_distances_dense_kernel<T, OUT>), dim3((unsigned)row_tiles, (unsigned)col_tiles), dim3(DD_THREADS), DD_SMEM,
               stream, X, n, d, k, centres, out);
    OFC_CHECK_LAUNCH("kmeans_distances_dense");
    return OFC_OK;
}

int launch_kmeans_distances(const void* X, int dtype, int64_t n, int d, int k, const double* centres, void* out, int out_f32,
                            void* stream) {
    ProfScope prof(PK_KMEANS, stream);
    if (out_f32) return launch_distances_typed((const float*)X, n, d, k, centres, (float*)out, stream);
    if (dtype == DT_U8) return launch_distances_typed((const unsigned char*)X, n, d, k, centres, (double*)out, stream);
    if (dtype == DT_F32) return launch_distances_typed((const float*)X, n, d, k, centres, (double*)out, stream);
    return launch_distances_typed((const double*)X, n, d, k, centres, (double*)out, stream);
}

}  // namespace ofc
