// Lloyd k-means for sm_100a: E-step (assign) and M-step (deterministic partial sums).
//
// Replaces the arithmetic behind the reference's
//   clt = KMeans(n_clusters = k); clt.fit(X); clt.predict(X)
// (reference k-means-color-clustering/KmeanGrids.py:299-304, color_kmeans.py:65-78),
// i.e. scikit-learn 1.9.0's dense Lloyd iteration (SURVEY.md Appendix A.5):
//   E-step  label = first strict minimum over j of  ||c_j||^2 - 2 x.c_j   (ties -> lowest j)
//   M-step  c_j = sum of the members / count; empty clusters take the farthest points.
//
// uint8 input (the reference's pixels and hues) is promoted to float64 exactly as
// sklearn does; float32 input is worked in float32.  The M-step never uses
// floating-point atomics: every lane group owns a private accumulator in shared
// memory, the copies are folded in a fixed order, and so are the per-CTA partials.
// For uint8 data the sums are integers held exactly in float64, so any reduction
// order (including the cross-GPU all-reduce) gives the same bits.
//
// All kernels take a batch dimension (independent problems of equal shape): the
// reference runs one fit per grid cell per frame (350 per frame).
#include <stdlib.h>
#include <type_traits>
#include "ofc_common.cuh"
#include "kmeans_kernels.cuh"

namespace ofc {

template <typename W> __device__ __forceinline__ W fma_w(W a, W b, W c);
template <> __device__ __forceinline__ double fma_w<double>(double a, double b, double c) { return fma(a, b, c); }
template <> __device__ __forceinline__ float fma_w<float>(float a, float b, float c) { return fmaf(a, b, c); }

// ||c||^2 of one centre in the working type: float64 in numpy's einsum order (norm_sq_numpy_f64), float32 as a
// sequential fma chain
__device__ __forceinline__ double centre_norm_sq(const double* c, int d) { return norm_sq_numpy_f64(c, d); }
__device__ __forceinline__ float centre_norm_sq(const float* c, int d) {
    float s = 0.f;
    for (int t = 0; t < d; ++t) s = fmaf(c[t], c[t], s);
    return s;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum in a fixed order (xor tree inside a warp, warps 0..7 in sequence)
__device__ __forceinline__ double block_sum_256(double v, double* s_red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < 8; ++w) t += s_red[w];
    __syncthreads();
    return t;      // valid in thread 0
}

// ---------------------------------------------------------------------------
// E-step, one thread per point: the row lives in registers (d <= DP), the
// centres and their squared norms in shared memory.
// ---------------------------------------------------------------------------
// WT: p.weights is set and the inertia is sum_i w_i ||x_i - c||^2 (sklearn's _inertia_dense); labels and min_dist do
// not depend on the weights.  Every weighted form below keeps the unweighted fold order, so unit weights give its bits.
template <typename T, typename W, int DP, bool WT>
__global__ void __launch_bounds__(256) kmeans_assign_small_kernel(KmAssignParams p) {
    OFC_DYN_SMEM(unsigned char, raw);
    W* sc = reinterpret_cast<W*>(raw);               // [k][d]
    W* sc2 = sc + (size_t)p.k * p.d;                  // [k]
    W* smean = sc2 + p.k;                             // [d]
    __shared__ double s_red[8];
    const int b = blockIdx.y, tid = threadIdx.x, d = p.d, k = p.k;
    if (p.active && !p.active[b]) return;
    const double* cen = p.centres + (int64_t)b * k * d;
    for (int i = tid; i < k * d; i += 256) sc[i] = (W)cen[i];
    for (int i = tid; i < d; i += 256) smean[i] = p.mean ? (W)p.mean[(int64_t)b * d + i] : (W)0;
    __syncthreads();
    for (int j = tid; j < k; j += 256) sc2[j] = centre_norm_sq(sc + j * d, d);
    __syncthreads();

    const T* X = reinterpret_cast<const T*>(p.X) + (int64_t)b * p.x_stride;
    int32_t* labels = p.labels + (int64_t)b * p.n;
    const int32_t* prev = p.prev_labels ? p.prev_labels + (int64_t)b * p.n : nullptr;
    const double* wt = WT ? p.weights + (int64_t)b * p.w_stride : nullptr;
    double inert = 0.0;
    unsigned changed = 0;
    for (int64_t base = (int64_t)blockIdx.x * 256; base < p.n; base += (int64_t)gridDim.x * 256) {
        const int64_t i = base + tid;
        if (i < p.n) {
            W x[DP];
            const T* row = X + i * d;
            if (sizeof(T) == 1 && DP == 4 && d == 4) {
                const uchar4 q = *reinterpret_cast<const uchar4*>(row);
                x[0] = (W)q.x - smean[0]; x[1] = (W)q.y - smean[1];
                x[2] = (W)q.z - smean[2]; x[3] = (W)q.w - smean[3];
#pragma unroll
                for (int t = 4; t < DP; ++t) x[t] = (W)0;
            } else {
#pragma unroll
                for (int t = 0; t < DP; ++t) x[t] = t < d ? (W)row[t] - smean[t] : (W)0;
            }
            W best = (W)0;
            int label = 0;
            for (int j = 0; j < k; ++j) {
                const W* c = sc + j * d;
                W dot = (W)0;
#pragma unroll
                for (int t = 0; t < DP; ++t)
                    if (t < d) dot = fma_w<W>(x[t], c[t], dot);
                const W dist = fma_w<W>((W)-2, dot, sc2[j]);
                if (j == 0 || dist < best) { best = dist; label = j; }
            }
            labels[i] = label;
            if (prev && prev[i] != label) ++changed;
            if (p.inertia_partial || p.min_dist) {
                const W* c = sc + label * d;
                W sq = (W)0;
#pragma unroll
                for (int t = 0; t < DP; ++t)
                    if (t < d) { W df = x[t] - c[t]; sq = fma_w<W>(df, df, sq); }
                inert += WT ? (double)sq * wt[i] : (double)sq;
                if (p.min_dist) p.min_dist[(int64_t)b * p.n + i] = (double)sq;
            }
        }
    }
    if (p.inertia_partial) {
        double t = block_sum_256(inert, s_red);
        if (tid == 0) p.inertia_partial[(int64_t)b * gridDim.x + blockIdx.x] = t;
    }
    if (p.n_changed && prev) {
        // integer counts: any order gives the same total
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
        if ((tid & 31) == 0 && changed) atomicAdd(p.n_changed + b, (unsigned long long)changed);
    }
}

// ---------------------------------------------------------------------------
// E-step, generic shape (large d, or k*d beyond shared memory): one warp per
// point, lanes stride over the features, centres read through L1/L2.
// ---------------------------------------------------------------------------
template <typename T, typename W, bool WT>
__global__ void __launch_bounds__(256) kmeans_assign_generic_kernel(KmAssignParams p) {
    __shared__ double s_red[8];
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, d = p.d, k = p.k;
    if (p.active && !p.active[b]) return;
    const double* cen = p.centres + (int64_t)b * k * d;
    const double* c2 = p.c2 + (int64_t)b * k;
    const double* mean = p.mean ? p.mean + (int64_t)b * d : nullptr;
    const T* X = reinterpret_cast<const T*>(p.X) + (int64_t)b * p.x_stride;
    int32_t* labels = p.labels + (int64_t)b * p.n;
    const int32_t* prev = p.prev_labels ? p.prev_labels + (int64_t)b * p.n : nullptr;
    const double* wt = WT ? p.weights + (int64_t)b * p.w_stride : nullptr;
    double inert = 0.0;
    unsigned changed = 0;
    for (int64_t i = (int64_t)blockIdx.x * 8 + warp; i < p.n; i += (int64_t)gridDim.x * 8) {
        const T* row = X + i * d;
        W best = (W)0;
        int label = 0;
        for (int j = 0; j < k; ++j) {
            const double* c = cen + (int64_t)j * d;
            W part = (W)0;
            for (int t = lane; t < d; t += 32) {
                W xv = (W)row[t] - (mean ? (W)mean[t] : (W)0);
                part = fma_w<W>(xv, (W)c[t], part);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            const W dist = fma_w<W>((W)-2, part, (W)c2[j]);
            if (j == 0 || dist < best) { best = dist; label = j; }
        }
        if (lane == 0) {
            labels[i] = label;
            if (prev && prev[i] != label) ++changed;
        }
        if (p.inertia_partial || p.min_dist) {
            const double* c = cen + (int64_t)label * d;
            W sq = (W)0;
            for (int t = lane; t < d; t += 32) {
                W df = ((W)row[t] - (mean ? (W)mean[t] : (W)0)) - (W)c[t];
                sq = fma_w<W>(df, df, sq);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
            if (lane == 0) {
                inert += WT ? (double)sq * wt[i] : (double)sq;
                if (p.min_dist) p.min_dist[(int64_t)b * p.n + i] = (double)sq;
            }
        }
    }
    if (p.inertia_partial) {
        double t = block_sum_256(inert, s_red);
        if (tid == 0) p.inertia_partial[(int64_t)b * gridDim.x + blockIdx.x] = t;
    }
    if (p.n_changed && prev && lane == 0 && changed) atomicAdd(p.n_changed + b, (unsigned long long)changed);
}

// ---------------------------------------------------------------------------
// E-step, medium shape (32 < d <= 32*NT, centres fit shared memory): one warp per point like the generic
// kernel and in exactly its arithmetic order (lanes stride over the features, fma chain, xor-tree reduction),
// but the centred row is loaded ONCE into registers and the centres (in the working precision) and their
// norms live in shared memory -- X is read once per iteration and nothing else leaves the SM.
// ---------------------------------------------------------------------------
template <typename T, typename W, int NT, bool WT>
__global__ void __launch_bounds__(256) kmeans_assign_medium_kernel(KmAssignParams p) {
    OFC_DYN_SMEM(unsigned char, raw);
    W* sc = reinterpret_cast<W*>(raw);                        // [k][d]
    W* sc2 = sc + (size_t)p.k * p.d;                           // [k]
    __shared__ double s_red[8];
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, d = p.d, k = p.k;
    if (p.active && !p.active[b]) return;
    const double* cen = p.centres + (int64_t)b * k * d;
    const double* c2 = p.c2 + (int64_t)b * k;
    for (int i = tid; i < k * d; i += 256) sc[i] = (W)cen[i];
    for (int i = tid; i < k; i += 256) sc2[i] = (W)c2[i];
    __syncthreads();
    const double* mean = p.mean ? p.mean + (int64_t)b * d : nullptr;
    W m[NT];
#pragma unroll
    for (int u = 0; u < NT; ++u) { const int t = lane + 32 * u; m[u] = (mean && t < d) ? (W)mean[t] : (W)0; }
    const T* X = reinterpret_cast<const T*>(p.X) + (int64_t)b * p.x_stride;
    int32_t* labels = p.labels + (int64_t)b * p.n;
    const int32_t* prev = p.prev_labels ? p.prev_labels + (int64_t)b * p.n : nullptr;
    const double* wt = WT ? p.weights + (int64_t)b * p.w_stride : nullptr;
    double inert = 0.0;
    unsigned changed = 0;
    for (int64_t i = (int64_t)blockIdx.x * 8 + warp; i < p.n; i += (int64_t)gridDim.x * 8) {
        const T* row = X + i * d;
        W x[NT];
#pragma unroll
        for (int u = 0; u < NT; ++u) { const int t = lane + 32 * u; x[u] = t < d ? (W)row[t] - m[u] : (W)0; }
        W best = (W)0;
        int label = 0;
        for (int j = 0; j < k; ++j) {
            const W* c = sc + (size_t)j * d;
            W part = (W)0;
#pragma unroll
            for (int u = 0; u < NT; ++u) { const int t = lane + 32 * u; if (t < d) part = fma_w<W>(x[u], c[t], part); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            const W dist = fma_w<W>((W)-2, part, sc2[j]);
            if (j == 0 || dist < best) { best = dist; label = j; }
        }
        if (lane == 0) {
            labels[i] = label;
            if (prev && prev[i] != label) ++changed;
        }
        if (p.inertia_partial || p.min_dist) {
            const W* c = sc + (size_t)label * d;
            W sq = (W)0;
#pragma unroll
            for (int u = 0; u < NT; ++u) { const int t = lane + 32 * u; if (t < d) { const W df = x[u] - c[t]; sq = fma_w<W>(df, df, sq); } }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
            if (lane == 0) {
                inert += WT ? (double)sq * wt[i] : (double)sq;
                if (p.min_dist) p.min_dist[(int64_t)b * p.n + i] = (double)sq;
            }
        }
    }
    if (p.inertia_partial) {
        double t = block_sum_256(inert, s_red);
        if (tid == 0) p.inertia_partial[(int64_t)b * gridDim.x + blockIdx.x] = t;
    }
    if (p.n_changed && prev && lane == 0 && changed) atomicAdd(p.n_changed + b, (unsigned long long)changed);
}

__global__ void kmeans_c2_kernel(const double* centres, double* c2, int d, int k, int as_float) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (j >= k) return;
    const double* c = centres + ((int64_t)b * k + j) * d;
    if (as_float) {
        float s = 0.f;
        for (int t = 0; t < d; ++t) s = fmaf((float)c[t], (float)c[t], s);
        c2[(int64_t)b * k + j] = (double)s;
    } else {
        c2[(int64_t)b * k + j] = norm_sq_numpy_f64(c, d);
    }
}

// inertia[b] = sum of the per-CTA partials in CTA order
__global__ void inertia_reduce_kernel(const double* partial, int parts, double* inertia, const unsigned char* active) {
    const int b = blockIdx.x;
    if (active && !active[b]) return;
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < parts; ++i) s += partial[(int64_t)b * parts + i];
        inertia[b] = s;
    }
}

// ---------------------------------------------------------------------------
// M-step partial sums.  grid = (splits, feature tiles, batch); a warp is cut
// into G = 32/dt lane groups, group g of warp w owns accumulator copy (w, g) of
// [kt][dt] doubles and walks its own subsequence of the split's points, so no
// two lanes ever touch the same word.  Copies are folded in index order.
// WT (weighted, _k_means_lloyd.pyx:216-218): every member adds (x - mean) w and
// its weight w to a float64 weight accumulator in place of the integer count.
// ---------------------------------------------------------------------------
template <typename T, bool WT>
__global__ void __launch_bounds__(256) kmeans_sums_kernel(KmSumsParams p) {
    using Cnt = typename std::conditional<WT, double, int>::type;
    using CntSum = typename std::conditional<WT, double, long long>::type;
    OFC_DYN_SMEM(double, acc);                         // [8*G][kt][dt]
    const int dt = p.dt, G = 32 / dt, kt = p.kt, d = p.d, k = p.k;
    Cnt* cnt = reinterpret_cast<Cnt*>(acc + (size_t)8 * G * kt * dt);   // [8*G][kt]
    const int split = blockIdx.x, dtile = blockIdx.y, b = blockIdx.z;
    if (p.active && !p.active[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane / dt, t = lane - g * dt, dim = dtile * dt + t;
    const bool dim_ok = dim < d;
    const int64_t chunk = (p.n + p.splits - 1) / p.splits;
    const int64_t lo = (int64_t)split * chunk, hi = lo + chunk < p.n ? lo + chunk : p.n;
    const int copy = warp * G + g;
    double* my = acc + (size_t)copy * kt * dt + t;
    Cnt* mycnt = cnt + copy * kt;
    const double m = (p.mean && dim_ok) ? p.mean[(int64_t)b * d + dim] : 0.0;
    const T* X = reinterpret_cast<const T*>(p.X) + (int64_t)b * p.x_stride;
    const int32_t* labels = p.labels ? p.labels + (int64_t)b * p.n : nullptr;
    const double* wt = WT ? p.weights + (int64_t)b * p.w_stride : nullptr;

    for (int k0 = 0; k0 < k; k0 += kt) {
        const int kk = k - k0 < kt ? k - k0 : kt;
        for (int j = 0; j < kk; ++j) {
            my[j * dt] = 0.0;
            if (t == 0) mycnt[j] = 0;
        }
        __syncwarp();
        for (int64_t i = lo + copy; i < hi; i += 8 * G) {
            const int j = (labels ? labels[i] : 0) - k0;
            if ((unsigned)j < (unsigned)kk) {
                if (dim_ok) {
                    double v = (double)X[i * d + dim] - m;
                    if (p.square) v *= v;
                    if (WT) v *= wt[i];
                    my[j * dt] += v;
                }
                if (t == 0) {
                    if constexpr (WT) mycnt[j] += wt[i];
                    else mycnt[j] += 1;
                }
            }
        }
        __syncthreads();
        for (int e = tid; e < kk * dt; e += 256) {
            const int j = e / dt, tt = e - j * dt;
            double s = 0.0;
            for (int c = 0; c < 8 * G; ++c) s += acc[((size_t)c * kt + j) * dt + tt];
            if (dtile * dt + tt < d)
                p.partial[(((int64_t)b * p.splits + split) * k + k0 + j) * d + dtile * dt + tt] = s;
        }
        if (dtile == 0) {
            for (int j = tid; j < kk; j += 256) {
                CntSum c = 0;
                for (int q = 0; q < 8 * G; ++q) c += cnt[q * kt + j];
                if (WT) p.wcnt_partial[((int64_t)b * p.splits + split) * k + k0 + j] = (double)c;
                else p.cnt_partial[((int64_t)b * p.splits + split) * k + k0 + j] = (long long)c;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// One Lloyd iteration in ONE pass for the reference's own shape -- uint8 rows with a handful of
// features and clusters (pixels: d = 4, hues per frame: d <= 32): E-step exactly as
// kmeans_assign_small_kernel, and in the same pass every thread adds its row to a thread-private
// integer accumulator [k][d] (+ member count) in shared memory, laid out [slot][thread] so no two
// threads ever share a word or a bank.  The sums are exact integers, so the CTA reduction and the
// fold over CTAs give the same bits as kmeans_sums_kernel in any order; X is read once per
// iteration instead of twice and no floating-point atomic exists anywhere.
// ---------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(256) kmeans_step_u8_kernel(KmAssignParams p, double* __restrict__ partial,
                                                             long long* __restrict__ cnt_partial) {
    OFC_DYN_SMEM(unsigned char, raw);
    const int b = blockIdx.y, tid = threadIdx.x, d = p.d, k = p.k;
    if (p.active && !p.active[b]) return;
    double* sc = reinterpret_cast<double*>(raw);              // [k][d]
    double* sc2 = sc + (size_t)k * d;                          // [k]
    double* smean = sc2 + k;                                   // [d]
    unsigned* acc = reinterpret_cast<unsigned*>(smean + d);    // [k*d + k][256]
    const int slots = k * d + k;
    const double* cen = p.centres + (int64_t)b * k * d;
    for (int i = tid; i < k * d; i += 256) sc[i] = cen[i];
    for (int i = tid; i < d; i += 256) smean[i] = p.mean ? p.mean[(int64_t)b * d + i] : 0.0;
    for (int s = 0; s < slots; ++s) acc[s * 256 + tid] = 0u;
    __syncthreads();
    for (int j = tid; j < k; j += 256) sc2[j] = norm_sq_numpy_f64(sc + j * d, d);
    __syncthreads();
    const unsigned char* X = reinterpret_cast<const unsigned char*>(p.X) + (int64_t)b * p.x_stride;
    int32_t* labels = p.labels + (int64_t)b * p.n;
    const int32_t* prev = p.prev_labels ? p.prev_labels + (int64_t)b * p.n : nullptr;
    unsigned changed = 0;
    for (int64_t base = (int64_t)blockIdx.x * 256; base < p.n; base += (int64_t)gridDim.x * 256) {
        const int64_t i = base + tid;
        if (i < p.n) {
            unsigned xr[DP];
            double x[DP];
            const unsigned char* row = X + i * d;
            if (DP == 4 && d == 4) {
                const uchar4 q = *reinterpret_cast<const uchar4*>(row);
                xr[0] = q.x; xr[1] = q.y; xr[2] = q.z; xr[3] = q.w;
            } else {
#pragma unroll
                for (int t = 0; t < DP; ++t) xr[t] = t < d ? row[t] : 0u;
            }
#pragma unroll
            for (int t = 0; t < DP; ++t) x[t] = t < d ? (double)xr[t] - smean[t] : 0.0;
            double best = 0.0;
            int label = 0;
            for (int j = 0; j < k; ++j) {
                const double* c = sc + j * d;
                double dot = 0.0;
#pragma unroll
                for (int t = 0; t < DP; ++t)
                    if (t < d) dot = fma(x[t], c[t], dot);
                const double dist = fma(-2.0, dot, sc2[j]);
                if (j == 0 || dist < best) { best = dist; label = j; }
            }
            labels[i] = label;
            if (prev && prev[i] != label) ++changed;
            unsigned* a = acc + (size_t)label * d * 256 + tid;
#pragma unroll
            for (int t = 0; t < DP; ++t)
                if (t < d) a[t * 256] += xr[t];
            acc[(size_t)(k * d + label) * 256 + tid] += 1u;
        }
    }
    __syncthreads();
    // CTA totals: warp w folds slots w, w + 8, ... (integers: any order gives the same bits)
    const int lane = tid & 31, warp = tid >> 5;
    for (int s = warp; s < slots; s += 8) {
        unsigned long long v = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) v += acc[s * 256 + q * 32 + lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) {
            if (s < k * d) partial[((int64_t)b * gridDim.x + blockIdx.x) * k * d + s] = (double)v;
            else cnt_partial[((int64_t)b * gridDim.x + blockIdx.x) * k + (s - k * d)] = (long long)v;
        }
    }
    if (p.n_changed && prev) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
        if (lane == 0 && changed) atomicAdd(p.n_changed + b, (unsigned long long)changed);
    }
}

// sums[b][j][t] = sum over splits (in split order) of the partials; counts (or weight sums) likewise
template <typename C>
__global__ void kmeans_fold_kernel(const double* partial, const C* cnt_partial, int splits, int k, int d,
                                   double* sums, C* counts, const unsigned char* active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t kd = (int64_t)k * d;
    if (e < kd) {
        double s = 0.0;
        for (int sp = 0; sp < splits; ++sp) s += partial[((int64_t)b * splits + sp) * kd + e];
        sums[(int64_t)b * kd + e] = s;
    }
    if (e < k && counts) {
        C c = 0;
        for (int sp = 0; sp < splits; ++sp) c += cnt_partial[((int64_t)b * splits + sp) * k + e];
        counts[(int64_t)b * k + e] = c;
    }
}

// ---------------------------------------------------------------------------
// centres from (all-reduced) sums and counts; an empty cluster copies the heaviest
// cluster's row as sklearn's in-place _average_centers (_k_means_common.pyx:274-295)
// finds it: not yet divided -- the heaviest cluster's centred SUM -- when the empty
// cluster's index is the lower one, its new centre otherwise (raw sums are centred
// as S - W mean); shift_tot = sum_j ||new-old||^2 taken as (sqrt(.))^2 like
// sklearn's center_shift (:298-311, _kmeans.py:733).  One CTA per problem.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kmeans_centres_kernel(int d, int k, const double* sums, const long long* counts,
                                                             const double* mean_sub, int use_reciprocal,
                                                             double* centres, double* shift_tot, double* shift_ws,
                                                             const unsigned char* active) {
    const int b = blockIdx.x, tid = threadIdx.x;
    if (active && !active[b]) return;
    const double* S = sums + (int64_t)b * k * d;
    const long long* Cn = counts + (int64_t)b * k;
    double* C = centres + (int64_t)b * k * d;
    double* sh = shift_ws + (int64_t)b * k;
    __shared__ int s_heavy;
    if (tid == 0) {
        int best = 0;
        for (int j = 1; j < k; ++j) if (Cn[j] > Cn[best]) best = j;
        s_heavy = best;
    }
    __syncthreads();
    const int heavy = s_heavy;
    for (int j = tid; j < k; j += 256) {
        const int src = Cn[j] > 0 ? j : heavy;
        const double w = (double)Cn[src];
        const double alpha = 1.0 / w;
        double ss = 0.0;
        if (src != j && j < heavy) {                     // the heaviest cluster's centred sum
            for (int t = 0; t < d; ++t) {
                double v = S[(int64_t)src * d + t];
                if (mean_sub) v = fma(-w, mean_sub[(int64_t)b * d + t], v);
                const double df = v - C[(int64_t)j * d + t];
                ss = fma(df, df, ss);
                C[(int64_t)j * d + t] = v;
            }
        } else {
            for (int t = 0; t < d; ++t) {
                double v = S[(int64_t)src * d + t];
                v = use_reciprocal ? v * alpha : v / w;
                if (mean_sub) v -= mean_sub[(int64_t)b * d + t];
                const double df = v - C[(int64_t)j * d + t];
                ss = fma(df, df, ss);
                C[(int64_t)j * d + t] = v;
            }
        }
        const double s = sqrt(ss);
        sh[j] = s * s;
    }
    __syncthreads();
    if (tid == 0 && shift_tot) {
        double tot = 0.0;
        for (int j = 0; j < k; ++j) tot += sh[j];
        shift_tot[b] = tot;
    }
}

// ---------------------------------------------------------------------------
// End of one Lloyd iteration, entirely on the device: new centres (kmeans_centres_kernel's arithmetic),
// optional float32 rounding of the stored centres, and sklearn's stopping rule (_kmeans.py:705-758) --
// a problem stops when its labels repeated (n_changed == 0, "strict") or when the squared centre shift is
// <= tol.  Stopped problems clear their `active` byte (every kernel skips them from then on) and raise
// `just_done` (their labels are copied into both label buffers by kmeans_freeze_labels_kernel); the number
// of problems still running is accumulated in *n_active, which the host reads asynchronously, a few
// iterations behind, to know when to stop enqueuing.  One CTA per problem.  CW = double: `counts` are the float64
// weight sums of a weighted fit (_average_centers: empty = weight 0, np.argmax of the weights).
// ---------------------------------------------------------------------------
template <typename CW>
__global__ void __launch_bounds__(256) kmeans_update_kernel(int d, int k, const double* sums, const CW* counts,
                                                            const double* mean_sub, int use_reciprocal, int round_f32,
                                                            double* centres, double* shift_tot, double* shift_ws,
                                                            const unsigned long long* n_changed, const double* tol, int it_arg,
                                                            unsigned char* active, unsigned char* just_done, int* n_iter,
                                                            int* n_active_base, const int* it_counter) {
    const int b = blockIdx.x, tid = threadIdx.x;
    // it_counter: the iteration number lives on the device (the loop body is replayed from a CUDA graph, so it cannot be a
    // launch argument); the "still running" count then goes to slot [it] of n_active_base
    const int it = it_counter ? *it_counter : it_arg;
    int* n_active = n_active_base ? n_active_base + (it_counter ? it : 0) : nullptr;
    if (just_done && tid == 0) just_done[b] = 0;
    if (active && !active[b]) return;
    const double* S = sums + (int64_t)b * k * d;
    const CW* Cn = counts + (int64_t)b * k;
    double* C = centres + (int64_t)b * k * d;
    double* sh = shift_ws + (int64_t)b * k;
    __shared__ int s_heavy;
    if (tid == 0) {
        int best = 0;
        for (int j = 1; j < k; ++j) if (Cn[j] > Cn[best]) best = j;
        s_heavy = best;
    }
    __syncthreads();
    const int heavy = s_heavy;
    for (int j = tid; j < k; j += 256) {
        const int src = Cn[j] > 0 ? j : heavy;
        const double w = (double)Cn[src];
        const double alpha = 1.0 / w;
        double ss = 0.0;
        if (src != j && j < heavy) {                     // the heaviest cluster's centred sum (kmeans_centres_kernel)
            for (int t = 0; t < d; ++t) {
                double v = S[(int64_t)src * d + t];
                if (mean_sub) v = fma(-w, mean_sub[(int64_t)b * d + t], v);
                const double df = v - C[(int64_t)j * d + t];
                ss = fma(df, df, ss);
                C[(int64_t)j * d + t] = round_f32 ? (double)(float)v : v;
            }
        } else {
            for (int t = 0; t < d; ++t) {
                double v = S[(int64_t)src * d + t];
                v = use_reciprocal ? v * alpha : v / w;
                if (mean_sub) v -= mean_sub[(int64_t)b * d + t];
                const double df = v - C[(int64_t)j * d + t];
                ss = fma(df, df, ss);
                C[(int64_t)j * d + t] = round_f32 ? (double)(float)v : v;
            }
        }
        const double s = sqrt(ss);
        sh[j] = s * s;
    }
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        for (int j = 0; j < k; ++j) tot += sh[j];
        if (shift_tot) shift_tot[b] = tot;
        if (n_iter) n_iter[b] = it + 1;
        bool stop = false;
        if (n_changed && n_changed[b] == 0ull) stop = true;                 // labels repeated: strict convergence
        else if (tol && tot <= tol[b]) stop = true;
        if (stop) {
            if (active) active[b] = 0;
            if (just_done) just_done[b] = 1;
        } else if (n_active) {
            atomicAdd(n_active, 1);
        }
    }
}

// ---------------------------------------------------------------------------
// MiniBatchKMeans centre update (reference color-quantization/quant.py:18-20 -> scikit-learn 1.9.0
// sklearn/cluster/_k_means_minibatch.pyx:60-110, update_center_dense): per cluster, in the mini-batch's sample
// order,  c_new = (c_old * weight_sum + sum of the members) / (weight_sum + n_members);  clusters without a member keep
// their centre.  One thread per (cluster, feature) walks the batch sequentially -- the reference's accumulation
// order, so the float result is the same; float32 data is worked in float32 like sklearn (W = float).
// ---------------------------------------------------------------------------
template <typename T, typename W>
__global__ void __launch_bounds__(256) minibatch_update_kernel(const T* __restrict__ Xb, int bs, int d, int k,
                                                               const int32_t* __restrict__ labels, const double* __restrict__ centres_old,
                                                               double* __restrict__ centres_new, double* __restrict__ weight_sums) {
    OFC_DYN_SMEM(int, s_lab);                            // [bs]
    __shared__ int s_any;
    for (int i = threadIdx.x; i < bs; i += 256) s_lab[i] = labels[i];
    __syncthreads();
    for (int e0 = 0; e0 < k * d; e0 += 256) {
        const int e = e0 + threadIdx.x;
        int cnt = 0, j = 0;
        if (e < k * d) {
            j = e / d;
            const int t = e - j * d;
            for (int i = 0; i < bs; ++i) cnt += s_lab[i] == j ? 1 : 0;
            const W c_old = (W)centres_old[e];
            W out = c_old;
            if (cnt > 0) {
                const W ws = (W)weight_sums[j];
                W acc = c_old * ws;
                for (int i = 0; i < bs; ++i)
                    if (s_lab[i] == j) acc += (W)Xb[(int64_t)i * d + t];
                const W ws_new = ws + (W)cnt;
                const W alpha = (W)1 / ws_new;
                out = acc * alpha;
            }
            centres_new[e] = (double)out;
        }
        __syncthreads();                                  // every feature of a cluster has read its old weight
        if (e < k * d && e - j * d == 0 && cnt > 0) weight_sums[j] = (double)((W)weight_sums[j] + (W)cnt);
        if (threadIdx.x == 0) s_any = 0;
        __syncthreads();
    }
}

__global__ void kmeans_counter_inc_kernel(int* counter) { *counter += 1; }

// problems that stopped in this iteration keep the labels they stopped with in BOTH ping-pong buffers
__global__ void __launch_bounds__(256) kmeans_freeze_labels_kernel(int64_t n, const unsigned char* just_done, const int32_t* cur,
                                                                   int32_t* other) {
    const int b = blockIdx.y;
    if (!just_done[b]) return;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        other[(int64_t)b * n + i] = cur[(int64_t)b * n + i];
}

// The empty clusters of a problem (count or weight sum 0) as a bit mask of (k + 31) / 32 words in shared memory, taken
// by the CTA of NT threads before the first relocation move.  sklearn lists them once (_k_means_common.pyx:176): a
// cluster that a move empties (its only member, or its only member of positive weight, was moved) stays empty for
// this iteration, whatever its index.
template <int NT, typename C>
__device__ __forceinline__ void snapshot_empty(const C* counts, int k, unsigned* mask) {
    for (int w = threadIdx.x; w < (k + 31) >> 5; w += NT) {
        unsigned m = 0u;
        for (int j = w * 32; j < min(k, w * 32 + 32); ++j) m |= (counts[j] == 0 ? 1u : 0u) << (j & 31);
        mask[w] = m;
    }
    __syncthreads();
}

__device__ __forceinline__ bool in_mask(const unsigned* mask, int e) { return (mask[e >> 5] >> (e & 31)) & 1u; }

static inline size_t empty_mask_bytes(int k) { return (size_t)((k + 31) / 32) * sizeof(unsigned); }

// ---------------------------------------------------------------------------
// empty-cluster relocation (_k_means_common.pyx:167-211): the clusters empty
// before the first move, in index order, each take the farthest remaining point
// (squared distance to the OLD centre of its label); labels are left untouched.
// One CTA of 1024 threads per problem; it returns at once when no cluster is
// empty, so the host launches it unconditionally (no device->host round trip).
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(1024) kmeans_relocate_kernel(const T* Xall, int64_t x_stride, int64_t n, int d, int k, const double* mean_all,
                                                                const int32_t* labels_all, const double* centres_all,
                                                                double* sums_all, long long* counts_all,
                                                                int raw_sums, const unsigned char* active) {
    OFC_DYN_SMEM(long long, s_taken);                  // [k] indices already given away, then the empty-cluster mask
    unsigned* s_empty = reinterpret_cast<unsigned*>(s_taken + k);
    const int b = blockIdx.x, tid = threadIdx.x;
    if (active && !active[b]) return;
    long long* counts = counts_all + (int64_t)b * k;
    __shared__ int s_any;
    if (tid == 0) {
        int any = 0;
        for (int j = 0; j < k; ++j) any |= counts[j] == 0;
        s_any = any;
    }
    __syncthreads();
    if (!s_any) return;
    snapshot_empty<1024>(counts, k, s_empty);
    const T* X = Xall + (int64_t)b * x_stride;
    const int32_t* labels = labels_all + (int64_t)b * n;
    const double* cen = centres_all + (int64_t)b * k * d;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    double* sums = sums_all + (int64_t)b * k * d;
    __shared__ double s_val[32];
    __shared__ long long s_idx[32];
    __shared__ long long s_pick;
    int n_taken = 0;
    for (int e = 0; e < k; ++e) {
        if (!in_mask(s_empty, e)) continue;
        double bv = -1.0;
        long long bi = -1;
        for (int64_t i = tid; i < n; i += 1024) {
            bool taken = false;
            for (int q = 0; q < n_taken; ++q) taken |= s_taken[q] == i;
            if (taken) continue;
            const double* c = cen + (int64_t)labels[i] * d;
            double v = 0.0;
            for (int t = 0; t < d; ++t) {
                const double df = ((double)X[i * d + t] - (mean ? mean[t] : 0.0)) - c[t];
                v = fma(df, df, v);
            }
            if (v > bv) { bv = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
        __syncthreads();
        if (tid == 0) {
            double v = -1.0;
            long long idx = -1;
            for (int w = 0; w < 32; ++w)
                if (s_idx[w] >= 0 && (idx < 0 || s_val[w] > v || (s_val[w] == v && s_idx[w] < idx))) { v = s_val[w]; idx = s_idx[w]; }
            if (n_taken == 0 && !(v > 0.0)) idx = -1;               // np.max(distances) == 0: nothing to do
            s_pick = idx;
            if (idx >= 0) s_taken[n_taken] = idx;
        }
        __syncthreads();
        const long long fi = s_pick;
        if (fi < 0) return;
        ++n_taken;
        const int old = labels[fi];
        for (int t = tid; t < d; t += 1024) {
            const double x = (double)X[fi * d + t] - ((mean && !raw_sums) ? mean[t] : 0.0);
            sums[(int64_t)old * d + t] -= x;
            sums[(int64_t)e * d + t] = x;
        }
        if (tid == 0) {
            counts[e] = 1;
            counts[old] -= 1;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// The same relocation in two kernels for large problems: (1) every row's squared distance to the old centre of its
// label, written to a scratch array by the whole grid (the arithmetic of kmeans_relocate_kernel: sequential fma over
// the features) -- skipped at once when no cluster is empty, unless `force`; (2) one CTA per problem picks, per empty
// cluster in index order, the farthest remaining row from the scratch (ties: lowest index), marks it taken and moves
// it in the sums.  kmeans_relocate_kernel re-reads all of X once per empty cluster through ONE CTA: 369 ms per
// launch on 1 M x 128 float32 rows with a handful of empty clusters (ncu r02e) against ~1 ms this way.
// C = double: a weighted fit (_relocate_empty_clusters_dense): `counts` are the clusters' weight sums, a cluster is
// empty when its weight is 0, the distances stay unweighted and the moved row carries x w and w.
// ---------------------------------------------------------------------------
template <typename T, typename C>
__global__ void __launch_bounds__(256) kmeans_rowdist_kernel(const T* Xall, int64_t x_stride, int64_t n, int d, int k, const double* mean_all,
                                                             const int32_t* labels_all, const double* centres_all,
                                                             const C* counts_all, double* scratch_all, int force,
                                                             const unsigned char* active) {
    const int b = blockIdx.y, tid = threadIdx.x;
    if (active && !active[b]) return;
    __shared__ int s_any;
    if (!force) {
        if (tid == 0) s_any = 0;
        __syncthreads();
        const C* counts = counts_all + (int64_t)b * k;
        int any = 0;
        for (int j = tid; j < k; j += 256) any |= counts[j] == 0;
        if (any) s_any = 1;
        __syncthreads();
        if (!s_any) return;
    }
    const T* X = Xall + (int64_t)b * x_stride;
    const int32_t* labels = labels_all + (int64_t)b * n;
    const double* cen = centres_all + (int64_t)b * k * d;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    double* scratch = scratch_all + (int64_t)b * n;
    for (int64_t i = (int64_t)blockIdx.x * 256 + tid; i < n; i += (int64_t)gridDim.x * 256) {
        const double* c = cen + (int64_t)labels[i] * d;
        const T* row = X + i * d;
        double v = 0.0;
        for (int t = 0; t < d; ++t) {
            const double df = ((double)row[t] - (mean ? mean[t] : 0.0)) - c[t];
            v = fma(df, df, v);
        }
        scratch[i] = v;
    }
}

// block-wide arg-max over scratch[0..n): largest value, lowest index among equals; -1 when nothing is left
__device__ __forceinline__ void block_argmax_1024(const double* scratch, int64_t n, double* s_val, long long* s_idx, double& out_v,
                                                  long long& out_i) {
    const int tid = threadIdx.x;
    double bv = -1.0;
    long long bi = -1;
    for (int64_t i = tid; i < n; i += 1024) {
        const double v = scratch[i];
        if (v > bv) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
    __syncthreads();
    double v = -1.0;
    long long idx = -1;
    for (int w = 0; w < 32; ++w)
        if (s_idx[w] >= 0 && (idx < 0 || s_val[w] > v || (s_val[w] == v && s_idx[w] < idx))) { v = s_val[w]; idx = s_idx[w]; }
    __syncthreads();
    out_v = v;
    out_i = idx;
}

template <typename T, typename C>
__global__ void __launch_bounds__(1024) kmeans_relocate_apply_kernel(const T* Xall, int64_t x_stride, int64_t n, int d, int k, const double* mean_all,
                                                                      const int32_t* labels_all, double* scratch_all, double* sums_all,
                                                                      C* counts_all, int raw_sums, const unsigned char* active,
                                                                      const double* weights_all, int64_t w_stride) {
    constexpr bool WT = std::is_same<C, double>::value;
    OFC_DYN_SMEM(unsigned, s_empty);                   // [(k + 31) / 32] the empty-cluster mask
    const int b = blockIdx.x, tid = threadIdx.x;
    if (active && !active[b]) return;
    C* counts = counts_all + (int64_t)b * k;
    __shared__ int s_any;
    __shared__ double s_val[32];
    __shared__ long long s_idx[32];
    if (tid == 0) s_any = 0;
    __syncthreads();
    {
        int any = 0;
        for (int j = tid; j < k; j += 1024) any |= counts[j] == 0;
        if (any) s_any = 1;
    }
    __syncthreads();
    if (!s_any) return;
    snapshot_empty<1024>(counts, k, s_empty);
    const T* X = Xall + (int64_t)b * x_stride;
    const int32_t* labels = labels_all + (int64_t)b * n;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    double* sums = sums_all + (int64_t)b * k * d;
    double* scratch = scratch_all + (int64_t)b * n;
    int n_taken = 0;
    for (int e = 0; e < k; ++e) {
        if (!in_mask(s_empty, e)) continue;
        double v;
        long long fi;
        block_argmax_1024(scratch, n, s_val, s_idx, v, fi);
        if (n_taken == 0 && !(v > 0.0)) return;        // np.max(distances) == 0: nothing to do
        if (fi < 0) return;
        ++n_taken;
        const int old = labels[fi];
        const double wf = WT ? weights_all[(int64_t)b * w_stride + fi] : 1.0;
        for (int t = tid; t < d; t += 1024) {
            double x = (double)X[fi * d + t] - ((mean && !raw_sums) ? mean[t] : 0.0);
            if (WT) x *= wf;
            sums[(int64_t)old * d + t] -= x;
            sums[(int64_t)e * d + t] = x;
        }
        if (tid == 0) {
            if constexpr (WT) {
                counts[e] = wf;
                counts[old] -= wf;
            } else {
                counts[e] = 1;
                counts[old] -= 1;
            }
            scratch[fi] = -1.0;                        // taken
        }
        __syncthreads();
        __threadfence_block();
    }
}

// the listing form for row-sharded data: the n_far farthest rows of this shard from the scratch distances
__global__ void __launch_bounds__(1024) kmeans_far_list_kernel(int64_t n, double* scratch_all, int n_far, double* out_val,
                                                               long long* out_idx) {
    const int b = blockIdx.x, tid = threadIdx.x;
    __shared__ double s_val[32];
    __shared__ long long s_idx[32];
    double* scratch = scratch_all + (int64_t)b * n;
    for (int e = 0; e < n_far; ++e) {
        double v;
        long long idx;
        block_argmax_1024(scratch, n, s_val, s_idx, v, idx);
        if (tid == 0) {
            out_val[(int64_t)b * n_far + e] = v;
            out_idx[(int64_t)b * n_far + e] = idx;
            if (idx >= 0) scratch[idx] = -1.0;
        }
        __syncthreads();
        __threadfence_block();
    }
}

// ---------------------------------------------------------------------------
// Empty-cluster relocation for ROW-SHARDED data without a host round trip (SURVEY.md section 8e).  Per iteration,
// after the all-reduce of sums / counts, every rank launches
//   kmeans_rowdist_kernel        row distances of its shard (returns at once when no cluster is empty),
//   kmeans_far_payload_kernel    its n_far farthest rows as [value, global row index, label, row...] records
//                                (value -1 = no candidate; all -1 when no cluster is empty),
//   [all-gather of the records],
//   kmeans_relocate_merge_kernel every rank applies the same moves to the all-reduced sums: each empty cluster, in index
//                                order, takes the globally farthest remaining row (ties: lowest global index).
// Same result as kmeans_relocate_kernel on the whole set.  More empty clusters than n_far at once raise *overflow
// (sticky); the host, which polls it a few iterations late, then redoes the fit with the host-merged path.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(1024) kmeans_far_payload_kernel(const T* Xall, int64_t n, int d, int k, const double* mean_all,
                                                                   const int32_t* labels_all, const long long* counts_all,
                                                                   double* scratch_all, int raw_sums, int n_far, long long row_offset,
                                                                   double* payload_all, const unsigned char* active) {
    const int b = blockIdx.x, tid = threadIdx.x;
    const int rec = 3 + d;
    double* payload = payload_all + (int64_t)b * n_far * rec;
    __shared__ int s_any;
    __shared__ double s_val[32];
    __shared__ long long s_idx[32];
    if (tid == 0) s_any = 0;
    __syncthreads();
    if (!(active && !active[b])) {
        const long long* counts = counts_all + (int64_t)b * k;
        int any = 0;
        for (int j = tid; j < k; j += 1024) any += counts[j] == 0 ? 1 : 0;
        if (any) atomicAdd(&s_any, any);
    }
    __syncthreads();
    // only as many candidates as there are empty clusters can ever be used (every rank sees the same all-reduced counts)
    const int wanted = min(s_any, n_far);
    for (int e = wanted + tid; e < n_far; e += 1024) { payload[(int64_t)e * rec] = -1.0; payload[(int64_t)e * rec + 1] = -1.0; }
    if (!s_any || n <= 0) {
        for (int e = tid; e < wanted; e += 1024) { payload[(int64_t)e * rec] = -1.0; payload[(int64_t)e * rec + 1] = -1.0; }
        return;
    }
    const T* X = Xall + (int64_t)b * n * d;
    const int32_t* labels = labels_all + (int64_t)b * n;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    double* scratch = scratch_all + (int64_t)b * n;
    for (int e = 0; e < wanted; ++e) {
        double v;
        long long idx;
        block_argmax_1024(scratch, n, s_val, s_idx, v, idx);
        double* r = payload + (int64_t)e * rec;
        if (idx < 0) {
            if (tid == 0) { r[0] = -1.0; r[1] = -1.0; }
        } else {
            if (tid == 0) {
                r[0] = v; r[1] = (double)(idx + row_offset); r[2] = (double)labels[idx];
                scratch[idx] = -1.0;
            }
            for (int t = tid; t < d; t += 1024) r[3 + t] = (double)X[idx * d + t] - ((mean && !raw_sums) ? mean[t] : 0.0);
        }
        __syncthreads();
        __threadfence_block();
    }
}

// allpay [world][batch][n_far][3 + d]; one CTA per problem
__global__ void __launch_bounds__(256) kmeans_relocate_merge_kernel(int batch, int d, int k, int world, int n_far, const double* allpay,
                                                                    double* sums_all, long long* counts_all, int* overflow,
                                                                    const unsigned char* active) {
    const int b = blockIdx.x, tid = threadIdx.x;
    if (active && !active[b]) return;
    const int rec = 3 + d, ncand = world * n_far;
    long long* counts = counts_all + (int64_t)b * k;
    double* sums = sums_all + (int64_t)b * k * d;
    OFC_DYN_SMEM(unsigned char, s_used);                  // [ncand], then the empty-cluster mask (4-byte aligned)
    unsigned* s_mask = reinterpret_cast<unsigned*>(s_used + ((ncand + 3) & ~3));
    __shared__ int s_pick, s_empty, s_state;
    if (tid == 0) {
        int ne = 0;
        for (int j = 0; j < k; ++j) ne += counts[j] == 0;
        s_state = ne == 0 ? 0 : (ne > n_far ? 2 : 1);
        if (ne > n_far && overflow) atomicExch(overflow, 1);
    }
    for (int c = tid; c < ncand; c += 256) s_used[c] = 0;
    __syncthreads();
    if (s_state != 1) return;
    snapshot_empty<256>(counts, k, s_mask);
    auto cand = [&](int c) -> const double* {
        const int r = c / n_far, e = c - r * n_far;
        return allpay + (((int64_t)r * batch + b) * n_far + e) * rec;
    };
    int e_next = 0;
    for (int round = 0;; ++round) {
        if (tid == 0) {
            int e = e_next;
            while (e < k && !in_mask(s_mask, e)) ++e;
            s_empty = e;
            int best = -1;
            if (e < k) {
                for (int c = 0; c < ncand; ++c) {
                    if (s_used[c]) continue;
                    const double* r = cand(c);
                    if (r[1] < 0.0) continue;
                    if (best < 0) { best = c; continue; }
                    const double* q = cand(best);
                    if (r[0] > q[0] || (r[0] == q[0] && r[1] < q[1])) best = c;
                }
                if (best >= 0 && round == 0 && !(cand(best)[0] > 0.0)) best = -1;      // np.max(distances) == 0: nothing to do
            }
            s_pick = best;
            if (best >= 0) s_used[best] = 1;
        }
        __syncthreads();
        const int e = s_empty, best = s_pick;
        if (e >= k || best < 0) return;
        const double* r = cand(best);
        const int old = (int)r[2];
        for (int t = tid; t < d; t += 256) {
            sums[(int64_t)old * d + t] -= r[3 + t];
            sums[(int64_t)e * d + t] = r[3 + t];
        }
        __syncthreads();
        if (tid == 0) { counts[e] = 1; counts[old] -= 1; }
        e_next = e + 1;
        __syncthreads();
    }
}

// The search half of the relocation for row-sharded data (SURVEY.md section 8e): this rank's n_far farthest rows
// (squared distance to the old centre of their label, same arithmetic and tie rule as kmeans_relocate_kernel:
// largest first, lowest index on ties).  The host merges the ranks' lists and applies the moves to the
// all-reduced sums.  One CTA of 1024 threads per problem.
template <typename T>
__global__ void __launch_bounds__(1024) kmeans_far_points_kernel(const T* Xall, int64_t n, int d, int k, const double* mean_all,
                                                                  const int32_t* labels_all, const double* centres_all, int n_far,
                                                                  double* out_val, long long* out_idx) {
    OFC_DYN_SMEM(long long, s_taken);                  // [n_far]
    const int b = blockIdx.x, tid = threadIdx.x;
    const T* X = Xall + (int64_t)b * n * d;
    const int32_t* labels = labels_all + (int64_t)b * n;
    const double* cen = centres_all + (int64_t)b * k * d;
    const double* mean = mean_all ? mean_all + (int64_t)b * d : nullptr;
    __shared__ double s_val[32];
    __shared__ long long s_idx[32];
    for (int e = 0; e < n_far; ++e) {
        double bv = -1.0;
        long long bi = -1;
        for (int64_t i = tid; i < n; i += 1024) {
            bool taken = false;
            for (int q = 0; q < e; ++q) taken |= s_taken[q] == i;
            if (taken) continue;
            const double* c = cen + (int64_t)labels[i] * d;
            double v = 0.0;
            for (int t = 0; t < d; ++t) {
                const double df = ((double)X[i * d + t] - (mean ? mean[t] : 0.0)) - c[t];
                v = fma(df, df, v);
            }
            if (v > bv) { bv = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
        __syncthreads();
        if (tid == 0) {
            double v = -1.0;
            long long idx = -1;
            for (int w = 0; w < 32; ++w)
                if (s_idx[w] >= 0 && (idx < 0 || s_val[w] > v || (s_val[w] == v && s_idx[w] < idx))) { v = s_val[w]; idx = s_idx[w]; }
            s_taken[e] = idx;
            out_val[(int64_t)b * n_far + e] = v;
            out_idx[(int64_t)b * n_far + e] = idx;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// Whole Lloyd runs on the device: one CTA per problem, for the reference's per-cell fits
// (350 small uint8 problems per frame, KmeanGrids.py:376-392).  Column statistics, optional
// k-means++ seeding, every E-step / M-step, empty-cluster relocation, the stopping rule of
// sklearn's _kmeans_single_lloyd and the final E-step + inertia all happen inside the kernel,
// so a frame's fits cost one launch and no host round trip.  Same arithmetic as the stepwise
// kernels above (same fma chains, exact integer sums), hence the same labels / centres / n_iter
// as kmeans.lloyd() for the same initial centres.
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

struct KmCellsParams {
    const unsigned char* X;      // [batch][n][d]
    int n, d, k;
    const double* init;          // [batch][k][d] or null (k-means++)
    unsigned long long seed;
    int max_iter;
    double tol;
    int32_t* labels;             // [batch][n]
    double* centres;             // [batch][k][d]
    double* inertia;             // [batch]
    int32_t* n_iter;             // [batch]
    long long* counts;           // [batch][k] members of the final labels
    double* scratch;             // [batch][n] (k-means++ only)
};

template <int DP>
__global__ void __launch_bounds__(256) kmeans_cells_kernel(KmCellsParams p) {
    OFC_DYN_SMEM(double, sm);
    const int n = p.n, d = p.d, k = p.k, b = blockIdx.x, tid = threadIdx.x;
    double* cc = sm;                              // [k][d] centred centres
    double* c2 = cc + k * d;                      // [k]
    double* cnew = c2 + k;                        // [k][d]
    double* shift = cnew + k * d;                 // [k]
    double* mean = shift + k;                     // [d]
    double* s_red = mean + d;                     // [8]
    unsigned* s_sum = reinterpret_cast<unsigned*>(s_red + 8);   // [k][d]
    int* s_cnt = reinterpret_cast<int*>(s_sum + k * d);         // [k]
    __shared__ unsigned long long s_stat[16];     // sum x, sum x^2 per dim (d <= 8)
    __shared__ double s_tol, s_val[8];
    __shared__ long long s_idx[8], s_pick;
    __shared__ int s_heavy, s_stop, s_changed;            // one word per decision: no reuse between barriers
    __shared__ unsigned long long s_empty;                // the clusters empty before the first relocation move (k <= 64)
    const unsigned char* X = p.X + (int64_t)b * n * d;
    int32_t* labels = p.labels + (int64_t)b * n;

    auto load_x = [&](int i, double (&x)[DP]) {
        const unsigned char* row = X + (int64_t)i * d;
        if (DP == 4 && d == 4) {
            const uchar4 q = *reinterpret_cast<const uchar4*>(row);
            x[0] = (double)q.x; x[1] = (double)q.y; x[2] = (double)q.z; x[3] = (double)q.w;
        } else {
#pragma unroll
            for (int t = 0; t < DP; ++t) x[t] = t < d ? (double)row[t] : 0.0;
        }
    };
    auto block_sum = [&](double v) -> double {       // fixed order; result in every thread
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0) s_red[tid >> 5] = v;
        __syncthreads();
        double tsum = 0.0;
        for (int w = 0; w < 8; ++w) tsum += s_red[w];
        __syncthreads();
        return tsum;
    };

    // ---- column statistics: mean, tolerance ------------------------------------------------
    if (tid < 16) s_stat[tid] = 0ull;
    __syncthreads();
    {
        unsigned long long sx[DP], sxx[DP];
#pragma unroll
        for (int t = 0; t < DP; ++t) { sx[t] = 0ull; sxx[t] = 0ull; }
        for (int i = tid; i < n; i += 256) {
            double x[DP];
            load_x(i, x);
#pragma unroll
            for (int t = 0; t < DP; ++t) {
                const unsigned long long v = (unsigned long long)x[t];
                sx[t] += v; sxx[t] += v * v;
            }
        }
#pragma unroll
        for (int t = 0; t < DP; ++t) {
            if (t < d) {
                atomicAdd(&s_stat[t], sx[t]);
                atomicAdd(&s_stat[8 + t], sxx[t]);
            }
        }
    }
    __syncthreads();
    if (tid == 0) {
        double vs = 0.0;
        for (int t = 0; t < d; ++t) {
            mean[t] = (double)s_stat[t] / (double)n;
            const unsigned long long num = (unsigned long long)n * s_stat[8 + t] - s_stat[t] * s_stat[t];   // exact for n <= 2^20
            vs += (double)num / ((double)n * (double)n);
        }
        s_tol = vs / (double)d * p.tol;
    }
    __syncthreads();

    // ---- initial centres ----------------------------------------------------------------------
    if (p.init) {
        for (int e = tid; e < k * d; e += 256) cc[e] = p.init[(int64_t)b * k * d + e] - mean[e % d];
    } else {
        // k-means++ (sklearn/_kmeans.py:181-268): first centre uniform, then 2+int(log k) candidates per step
        // drawn in proportion to the squared distance to the closest chosen centre, keeping the candidate with
        // the lowest potential.  Distances are exact (integers); the random stream is a counter-based hash of
        // (seed, problem, draw), not numpy's -- the reference leaves random_state unset (SURVEY.md Q9).
        double* closest = p.scratch + (int64_t)b * n;
        const int trials = 2 + (int)log((double)k);
        unsigned long long ctr = splitmix64(p.seed ^ (0xD1B54A32D192ED03ull * (unsigned long long)(b + 1)));
        auto uniform = [&]() -> double { ctr = splitmix64(ctr); return (double)(ctr >> 11) * (1.0 / 9007199254740992.0); };
        auto dist_to = [&](int i, int c) -> double {
            const unsigned char* a = X + (int64_t)i * d;
            const unsigned char* q = X + (int64_t)c * d;
            double s = 0.0;
            for (int t = 0; t < d; ++t) { const double df = (double)a[t] - (double)q[t]; s += df * df; }
            return s;
        };
        int first = (int)(uniform() * (double)n);
        if (first >= n) first = n - 1;
        for (int t = tid; t < d; t += 256) cc[t] = (double)X[(int64_t)first * d + t] - mean[t];
        double part = 0.0;
        for (int i = tid; i < n; i += 256) { const double v = dist_to(i, first); closest[i] = v; part += v; }
        double pot = block_sum(part);
        const int chunk = (n + 255) / 256;               // contiguous ranges for the cumulative sum
        for (int c = 1; c < k; ++c) {
            double best_pot = 0.0;
            int best = -1;
            for (int tr = 0; tr < trials; ++tr) {
                const double r = uniform() * pot;          // same value in every thread
                // searchsorted(cumsum(closest), r): thread-range sums, then the owner scans its range
                const int lo = tid * chunk, hi = min(n, lo + chunk);
                double loc = 0.0;
                for (int i = lo; i < hi; ++i) loc += closest[i];
                // running sum over the 256 range sums by one thread (k is small, n moderate)
                __shared__ double s_part[256];
                s_part[tid] = loc;
                __syncthreads();
                if (tid == 0) {
                    double run = 0.0;
                    long long cand = n - 1;
                    for (int q = 0; q < 256; ++q) {
                        const double nxt = run + s_part[q];
                        if (r < nxt || q == 255) {
                            const int l2 = q * chunk, h2 = min(n, l2 + chunk);
                            double acc = run;
                            cand = h2 > l2 ? h2 - 1 : n - 1;
                            for (int i = l2; i < h2; ++i) { acc += closest[i]; if (r < acc) { cand = i; break; } }
                            break;
                        }
                        run = nxt;
                    }
                    if (cand > n - 1) cand = n - 1;
                    s_pick = cand;
                }
                __syncthreads();
                const int cand = (int)s_pick;
                double pp = 0.0;
                for (int i = tid; i < n; i += 256) pp += fmin(closest[i], dist_to(i, cand));
                const double cp = block_sum(pp);
                if (best < 0 || cp < best_pot) { best_pot = cp; best = cand; }
            }
            for (int i = tid; i < n; i += 256) closest[i] = fmin(closest[i], dist_to(i, best));
            for (int t = tid; t < d; t += 256) cc[c * d + t] = (double)X[(int64_t)best * d + t] - mean[t];
            pot = best_pot;
            __syncthreads();
        }
    }
    __syncthreads();

    // ---- Lloyd iterations --------------------------------------------------------------------------
    auto e_step_label = [&](const double (&x)[DP]) -> int {
        double xc[DP];
#pragma unroll
        for (int t = 0; t < DP; ++t) xc[t] = t < d ? x[t] - mean[t] : 0.0;
        double bestd = 0.0;
        int label = 0;
        for (int j = 0; j < k; ++j) {
            const double* c = cc + j * d;
            double dot = 0.0;
#pragma unroll
            for (int t = 0; t < DP; ++t)
                if (t < d) dot = fma(xc[t], c[t], dot);
            const double dist = fma(-2.0, dot, c2[j]);
            if (j == 0 || dist < bestd) { bestd = dist; label = j; }
        }
        return label;
    };
    bool strict = false;
    int iters = 0;
    for (int it = 0; it < p.max_iter; ++it) {
        for (int j = tid; j < k; j += 256) {
            c2[j] = norm_sq_numpy_f64(cc + j * d, d);
            s_cnt[j] = 0;
        }
        for (int e = tid; e < k * d; e += 256) s_sum[e] = 0u;
        if (tid == 0) s_changed = 0;
        __syncthreads();
        int changed = 0;
        for (int i = tid; i < n; i += 256) {
            double x[DP];
            load_x(i, x);
            const int label = e_step_label(x);
            if (it == 0 || labels[i] != label) ++changed;
            labels[i] = label;
#pragma unroll
            for (int t = 0; t < DP; ++t)
                if (t < d) atomicAdd(&s_sum[label * d + t], (unsigned)x[t]);
            atomicAdd(&s_cnt[label], 1);
        }
        if (changed) atomicAdd(&s_changed, changed);
        __syncthreads();
        // the clusters empty now, in index order, take the farthest points (distance to the old centre of their label)
        if (tid == 0) {
            unsigned long long empty = 0ull;
            for (int j = 0; j < k; ++j) empty |= (unsigned long long)(s_cnt[j] == 0) << j;
            s_empty = empty;
        }
        __syncthreads();
        if (s_empty) {
            long long* taken = reinterpret_cast<long long*>(cnew);     // scratch until the centre update
            int n_taken = 0;
            for (int e = 0; e < k; ++e) {
                if (!((s_empty >> e) & 1ull)) continue;
                double bv = -1.0;
                long long bi = -1;
                for (int i = tid; i < n; i += 256) {
                    bool tk = false;
                    for (int q = 0; q < n_taken; ++q) tk |= taken[q] == i;
                    if (tk) continue;
                    double x[DP];
                    load_x(i, x);
                    const double* c = cc + labels[i] * d;
                    double v = 0.0;
                    for (int t = 0; t < d; ++t) { const double df = (x[t] - mean[t]) - c[t]; v = fma(df, df, v); }
                    if (v > bv) { bv = v; bi = i; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
                }
                if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
                __syncthreads();
                if (tid == 0) {
                    double v = -1.0;
                    long long idx = -1;
                    for (int w = 0; w < 8; ++w)
                        if (s_idx[w] >= 0 && (idx < 0 || s_val[w] > v || (s_val[w] == v && s_idx[w] < idx))) { v = s_val[w]; idx = s_idx[w]; }
                    if (n_taken == 0 && !(v > 0.0)) idx = -1;
                    s_pick = idx;
                    if (idx >= 0) {
                        taken[n_taken] = idx;
                        const int old = labels[idx];
                        for (int t = 0; t < d; ++t) {
                            const unsigned xv = X[idx * d + t];
                            s_sum[old * d + t] -= xv;
                            s_sum[e * d + t] = xv;
                        }
                        s_cnt[e] = 1;
                        s_cnt[old] -= 1;
                    }
                }
                __syncthreads();
                if (s_pick < 0) break;
                ++n_taken;
            }
            __syncthreads();
        }
        // centres, shift
        if (tid == 0) {
            int heavy = 0;
            for (int j = 1; j < k; ++j) if (s_cnt[j] > s_cnt[heavy]) heavy = j;
            s_heavy = heavy;
        }
        __syncthreads();
        for (int j = tid; j < k; j += 256) {
            const int srcj = s_cnt[j] > 0 ? j : s_heavy;
            const bool as_sum = srcj != j && j < srcj;         // the heaviest cluster's centred sum (kmeans_centres_kernel)
            const double wgt = (double)s_cnt[srcj];
            double ss = 0.0;
            for (int t = 0; t < d; ++t) {
                const double sv = (double)s_sum[srcj * d + t];
                const double v = as_sum ? fma(-wgt, mean[t], sv) : sv / wgt - mean[t];
                const double df = v - cc[j * d + t];
                ss = fma(df, df, ss);
                cnew[j * d + t] = v;
            }
            const double sr = sqrt(ss);
            shift[j] = sr * sr;
        }
        __syncthreads();
        for (int e = tid; e < k * d; e += 256) cc[e] = cnew[e];
        if (tid == 0) {
            double tot = 0.0;
            for (int j = 0; j < k; ++j) tot += shift[j];
            int stop = 0;
            if (s_changed == 0) stop = 2;                 // labels repeated: strict convergence
            else if (tot <= s_tol) stop = 1;
            s_stop = stop;
        }
        __syncthreads();
        iters = it + 1;
        if (s_stop) { strict = s_stop == 2; break; }
    }
    (void)strict;   // the closing E-step below is idempotent for a strict stop (kmeans.lloyd does the same)

    // ---- closing E-step on the final centres, inertia, member counts ------------------------------
    for (int j = tid; j < k; j += 256) {
        c2[j] = norm_sq_numpy_f64(cc + j * d, d);
        s_cnt[j] = 0;
    }
    __syncthreads();
    double inert = 0.0;
    for (int i = tid; i < n; i += 256) {
        double x[DP];
        load_x(i, x);
        const int label = e_step_label(x);
        labels[i] = label;
        atomicAdd(&s_cnt[label], 1);
        const double* c = cc + label * d;
        double sq = 0.0;
#pragma unroll
        for (int t = 0; t < DP; ++t)
            if (t < d) { const double df = (x[t] - mean[t]) - c[t]; sq = fma(df, df, sq); }
        inert += sq;
    }
    const double tot_inertia = block_sum(inert);
    __syncthreads();
    for (int e = tid; e < k * d; e += 256) p.centres[(int64_t)b * k * d + e] = cc[e] + mean[e % d];
    for (int j = tid; j < k; j += 256) p.counts[(int64_t)b * k + j] = s_cnt[j];
    if (tid == 0) {
        p.inertia[b] = tot_inertia;
        p.n_iter[b] = iters;
    }
}

int launch_kmeans_cells(const unsigned char* X, int batch, int64_t n, int d, int k, const double* init,
                        unsigned long long seed, int max_iter, double tol, int32_t* labels, double* centres,
                        double* inertia, int32_t* n_iter, long long* counts, double* scratch, void* stream) {
    if (batch <= 0) return OFC_OK;
    KmCellsParams p;
    p.X = X; p.n = (int)n; p.d = d; p.k = k; p.init = init; p.seed = seed; p.max_iter = max_iter; p.tol = tol;
    p.labels = labels; p.centres = centres; p.inertia = inertia; p.n_iter = n_iter; p.counts = counts; p.scratch = scratch;
    const size_t smem = (size_t)(2 * k * d + 2 * k + d + 8) * sizeof(double) + (size_t)k * d * sizeof(unsigned) + (size_t)k * sizeof(int);
    ProfScope prof(PK_KMEANS, stream);
    if (d <= 4) {
        OFC_SMEM_OPTIN(kmeans_cells_kernel<4>, smem);
        OFC_LAUNCH(kmeans_cells_kernel<4>, dim3(batch), dim3(256), smem, stream, p);
    } else {
        OFC_SMEM_OPTIN(kmeans_cells_kernel<8>, smem);
        OFC_LAUNCH(kmeans_cells_kernel<8>, dim3(batch), dim3(256), smem, stream, p);
    }
    OFC_CHECK_LAUNCH("kmeans_cells");
    return OFC_OK;
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
int kmeans_assign_grid(int64_t n) {
    int64_t tiles = (n + 255) / 256;
    int64_t cap = 148 * 8;
    return (int)(tiles < 1 ? 1 : (tiles < cap ? tiles : cap));
}

int kmeans_sums_splits(int64_t n, int batch) {
    int64_t want = (n + 4095) / 4096;                  // >= 4096 points per split
    int64_t cap = (148 * 4 + batch - 1) / batch;
    if (cap < 1) cap = 1;
    if (want > cap) want = cap;
    return (int)(want < 1 ? 1 : want);
}

template <typename T, typename W, bool WT>
static int assign_small_dispatch(const KmAssignParams& p, dim3 grid, size_t smem, void* stream) {
#define OFC_KM_CASE(DPV)                                                                                     \
    {                                                                                                        \
        OFC_SMEM_OPTIN((kmeans_assign_small_kernel<T, W, DPV, WT>), smem);                                   \
        OFC_LAUNCH((kmeans_assign_small_kernel<T, W, DPV, WT>), grid, dim3(256), smem, stream, p);           \
    }
    if (p.d <= 4) OFC_KM_CASE(4)
    else if (p.d <= 8) OFC_KM_CASE(8)
    else if (p.d <= 16) OFC_KM_CASE(16)
    else OFC_KM_CASE(32)
#undef OFC_KM_CASE
    return OFC_OK;
}

template <bool WT>
static int launch_assign(KmAssignParams p, int batch, double* c2_ws, void* stream) {
    if (batch > 65535) { set_error("batch=%d exceeds 65535", batch); return OFC_ERR_UNSUPPORTED; }
    const size_t wsz = p.dtype == DT_F32 ? 4 : 8;
    const size_t smem = ((size_t)p.k * p.d + p.k + p.d) * wsz;
    ProfScope prof(PK_KMEANS, stream);
    if (p.d <= 32 && smem <= 200 * 1024) {
        dim3 grid(kmeans_assign_grid(p.n), batch);
        int rc;
        if (p.dtype == DT_U8) rc = assign_small_dispatch<unsigned char, double, WT>(p, grid, smem, stream);
        else if (p.dtype == DT_F32) rc = assign_small_dispatch<float, float, WT>(p, grid, smem, stream);
        else rc = assign_small_dispatch<double, double, WT>(p, grid, smem, stream);
        if (rc != OFC_OK) return rc;
        OFC_CHECK_LAUNCH("kmeans_assign_small");
        return OFC_OK;
    }
    if (!c2_ws) { set_error("k-means workspace missing"); return OFC_ERR_WORKSPACE; }
    OFC_LAUNCH(kmeans_c2_kernel, dim3(cdiv(p.k, 128), batch), dim3(128), 0, stream, p.centres, c2_ws, p.d, p.k,
               p.dtype == DT_F32 ? 1 : 0);
    OFC_CHECK_LAUNCH("kmeans_c2");
    p.c2 = c2_ws;
    int64_t g = (p.n + 7) / 8;
    if (g > 148 * 16) g = 148 * 16;
    dim3 grid((int)g, batch);
    // inertia partials are indexed by gridDim.x and sized with kmeans_assign_grid(n) by the caller:
    // (n+7)/8 >= (n+255)/256 and the cap above is larger, so clamping gives exactly that count
    const int parts = kmeans_assign_grid(p.n);
    if ((int)grid.x > parts) grid.x = parts;
    // centres fit shared memory and the row fits a warp's registers: same arithmetic, X read once
    // (test seam: OFC_KMEANS_MEDIUM=0 runs the generic kernel, the tests' reference)
    const size_t msmem = ((size_t)p.k * p.d + p.k) * wsz;
    if (!seam_off("OFC_KMEANS_MEDIUM") && p.d <= 512 && msmem <= 200 * 1024) {
#define OFC_KM_MED(TT, WW, NTV)                                                                                        \
    {                                                                                                                  \
        OFC_SMEM_OPTIN((kmeans_assign_medium_kernel<TT, WW, NTV, WT>), msmem);                                         \
        OFC_LAUNCH((kmeans_assign_medium_kernel<TT, WW, NTV, WT>), grid, dim3(256), msmem, stream, p);                 \
    }
#define OFC_KM_MED_NT(TT, WW)                                                                                          \
    {                                                                                                                  \
        if (p.d <= 64) OFC_KM_MED(TT, WW, 2)                                                                           \
        else if (p.d <= 96) OFC_KM_MED(TT, WW, 3)                                                                      \
        else if (p.d <= 128) OFC_KM_MED(TT, WW, 4)                                                                     \
        else if (p.d <= 192) OFC_KM_MED(TT, WW, 6)                                                                     \
        else if (p.d <= 256) OFC_KM_MED(TT, WW, 8)                                                                     \
        else if (p.d <= 384) OFC_KM_MED(TT, WW, 12)                                                                    \
        else OFC_KM_MED(TT, WW, 16)                                                                                    \
    }
        if (p.dtype == DT_U8) OFC_KM_MED_NT(unsigned char, double)
        else if (p.dtype == DT_F32) OFC_KM_MED_NT(float, float)
        else OFC_KM_MED_NT(double, double)
#undef OFC_KM_MED_NT
#undef OFC_KM_MED
        OFC_CHECK_LAUNCH("kmeans_assign_medium");
        return OFC_OK;
    }
    if (p.dtype == DT_U8) OFC_LAUNCH((kmeans_assign_generic_kernel<unsigned char, double, WT>), grid, dim3(256), 0, stream, p);
    else if (p.dtype == DT_F32) OFC_LAUNCH((kmeans_assign_generic_kernel<float, float, WT>), grid, dim3(256), 0, stream, p);
    else OFC_LAUNCH((kmeans_assign_generic_kernel<double, double, WT>), grid, dim3(256), 0, stream, p);
    OFC_CHECK_LAUNCH("kmeans_assign_generic");
    return OFC_OK;
}

// p.weights set: the weighted-inertia instantiations (the labels are the same)
int launch_kmeans_assign(KmAssignParams p, int batch, double* c2_ws, void* stream) {
    if (batch <= 0 || p.n <= 0) return OFC_OK;
    return p.weights ? launch_assign<true>(p, batch, c2_ws, stream) : launch_assign<false>(p, batch, c2_ws, stream);
}

// fold of the fused step's per-CTA partials: integers held exactly in float64, so a warp per element can
// add them in any order (lanes stride over the CTAs, xor tree) and still give the bits of the serial fold
__global__ void __launch_bounds__(256) kmeans_fold_exact_kernel(const double* __restrict__ partial, const long long* __restrict__ cnt_partial,
                                                                int splits, int k, int d, double* __restrict__ sums,
                                                                long long* __restrict__ counts, const unsigned char* active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int lane = threadIdx.x & 31;
    const int64_t e = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int64_t kd = (int64_t)k * d;
    if (e < kd) {
        double s = 0.0;
        for (int sp = lane; sp < splits; sp += 32) s += partial[((int64_t)b * splits + sp) * kd + e];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sums[(int64_t)b * kd + e] = s;
    } else if (e < kd + k) {
        const int64_t j = e - kd;
        long long c = 0;
        for (int sp = lane; sp < splits; sp += 32) c += cnt_partial[((int64_t)b * splits + sp) * k + j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) counts[(int64_t)b * k + j] = c;
    }
}

// grid of the fused uint8 step: every thread's 32-bit accumulators must hold 255 * its rows
int kmeans_step_grid(int64_t n, int batch) {
    int64_t tiles = (n + 4095) / 4096;                 // >= 4096 rows per CTA: the zero / fold overhead stays small
    int64_t cap = (148 * 4 + batch - 1) / batch;
    if (cap < 1) cap = 1;
    int64_t g = tiles < cap ? tiles : cap;
    const int64_t need = (n + (int64_t)256 * 8000000 - 1) / ((int64_t)256 * 8000000);   // <= 8M rows per thread
    if (g < need) g = need;
    return (int)(g < 1 ? 1 : g);
}

size_t kmeans_step_smem(int d, int k) { return ((size_t)k * d + k + d) * 8 + ((size_t)k * d + k) * 256 * 4; }

int launch_kmeans_step_u8(KmAssignParams p, int batch, double* partial, long long* cnt_partial, double* sums, long long* counts,
                          void* stream) {
    if (batch <= 0 || p.n <= 0) return OFC_OK;
    if (batch > 65535) { set_error("batch=%d exceeds 65535", batch); return OFC_ERR_UNSUPPORTED; }
    const size_t smem = kmeans_step_smem(p.d, p.k);
    if (p.d > 32 || smem > 200 * 1024) { set_error("fused k-means step: shape d=%d k=%d does not fit shared memory", p.d, p.k); return OFC_ERR_UNSUPPORTED; }
    const int grid = kmeans_step_grid(p.n, batch);
    ProfScope prof(PK_KMEANS, stream);
#define OFC_KM_STEP(DPV)                                                                                                \
    {                                                                                                                 \
        OFC_SMEM_OPTIN((kmeans_step_u8_kernel<DPV>), smem);                                                           \
        OFC_LAUNCH((kmeans_step_u8_kernel<DPV>), dim3(grid, batch), dim3(256), smem, stream, p, partial, cnt_partial); \
    }
    // Centres stay in shared memory at every d.  (Centres held in registers were measured slower at d = 4, k = 8: 1.15
    // against 0.75 ms per 64 M rows -- the 64 extra registers cost more occupancy than the broadcasts they save.)
    if (kmeans_step_u8d4_usable(p, batch)) {
        // the reference's pixel shape: float32-filtered E-step + packed register M-step, same bits (cells_kmeans.cu)
        int rc = launch_kmeans_step_u8d4(p, batch, grid, partial, cnt_partial, stream);
        if (rc != OFC_OK) return rc;
    } else if (p.d <= 4) OFC_KM_STEP(4)
    else if (p.d <= 8) OFC_KM_STEP(8)
    else if (p.d <= 16) OFC_KM_STEP(16)
    else OFC_KM_STEP(32)
#undef OFC_KM_STEP
    OFC_CHECK_LAUNCH("kmeans_step_u8");
    const int64_t kd = (int64_t)p.k * p.d;
    OFC_LAUNCH(kmeans_fold_exact_kernel, dim3((unsigned)((kd + p.k + 7) / 8), batch), dim3(256), 0, stream, partial, cnt_partial, grid,
               p.k, p.d, sums, counts, p.active);
    OFC_CHECK_LAUNCH("kmeans_fold_exact");
    return OFC_OK;
}

int launch_inertia_reduce(const double* partial, int parts, int batch, double* inertia, const unsigned char* active,
                          void* stream) {
    OFC_LAUNCH(inertia_reduce_kernel, dim3(batch), dim3(32), 0, stream, partial, parts, inertia, active);
    OFC_CHECK_LAUNCH("inertia_reduce");
    return OFC_OK;
}

// C = long long: member counts; C = double: weight sums (p.weights set)
template <typename C>
static int launch_sums(const KmSumsParams& p, int batch, double* sums, C* counts, void* stream) {
    constexpr bool WT = std::is_same<C, double>::value;
    if (batch <= 0) return OFC_OK;
    if (batch > 65535) { set_error("batch=%d exceeds 65535", batch); return OFC_ERR_UNSUPPORTED; }
    const int G = 32 / p.dt;
    const size_t smem = (size_t)8 * G * p.kt * p.dt * sizeof(double) + (size_t)8 * G * p.kt * (WT ? sizeof(double) : sizeof(int));
    dim3 grid(p.splits, cdiv(p.d, p.dt), batch);
    ProfScope prof(PK_KMEANS, stream);
#define OFC_KM_SUMS(TT)                                                                                      \
    {                                                                                                        \
        OFC_SMEM_OPTIN((kmeans_sums_kernel<TT, WT>), smem);                                                  \
        OFC_LAUNCH((kmeans_sums_kernel<TT, WT>), grid, dim3(256), smem, stream, p);                          \
    }
    if (p.dtype == DT_U8) OFC_KM_SUMS(unsigned char)
    else if (p.dtype == DT_F32) OFC_KM_SUMS(float)
    else OFC_KM_SUMS(double)
#undef OFC_KM_SUMS
    OFC_CHECK_LAUNCH("kmeans_sums");
    const int64_t kd = (int64_t)p.k * p.d;
    const C* cnt_partial;
    if constexpr (WT) cnt_partial = p.wcnt_partial;
    else cnt_partial = p.cnt_partial;
    OFC_LAUNCH(kmeans_fold_kernel<C>, dim3((unsigned)((kd + 255) / 256), batch), dim3(256), 0, stream, p.partial,
               cnt_partial, p.splits, p.k, p.d, sums, counts, p.active);
    OFC_CHECK_LAUNCH("kmeans_fold");
    return OFC_OK;
}

int launch_kmeans_sums(const KmSumsParams& p, int batch, double* sums, long long* counts, void* stream) {
    return launch_sums<long long>(p, batch, sums, counts, stream);
}

int launch_kmeans_sums_weighted(const KmSumsParams& p, int batch, double* sums, double* weight_sums, void* stream) {
    return launch_sums<double>(p, batch, sums, weight_sums, stream);
}

int launch_kmeans_centres(int batch, int d, int k, const double* sums, const long long* counts, const double* mean_sub,
                          int use_reciprocal, double* centres, double* shift_tot, double* shift_ws,
                          const unsigned char* active, void* stream) {
    if (batch <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    OFC_LAUNCH(kmeans_centres_kernel, dim3(batch), dim3(256), 0, stream, d, k, sums, counts, mean_sub, use_reciprocal,
               centres, shift_tot, shift_ws, active);
    OFC_CHECK_LAUNCH("kmeans_centres");
    return OFC_OK;
}

template <typename C>
static int launch_update(int batch, int d, int k, const double* sums, const C* counts, const double* mean_sub,
                         int use_reciprocal, int round_f32, double* centres, double* shift_tot, double* shift_ws,
                         const unsigned long long* n_changed, const double* tol, int it, unsigned char* active,
                         unsigned char* just_done, int* n_iter, int* n_active, int64_t n, const int32_t* labels_cur,
                         int32_t* labels_other, int* it_counter, void* stream) {
    if (batch <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    OFC_LAUNCH(kmeans_update_kernel<C>, dim3(batch), dim3(256), 0, stream, d, k, sums, counts, mean_sub, use_reciprocal, round_f32,
               centres, shift_tot, shift_ws, n_changed, tol, it, active, just_done, n_iter, n_active, it_counter);
    OFC_CHECK_LAUNCH("kmeans_update");
    if (it_counter) {
        OFC_LAUNCH(kmeans_counter_inc_kernel, dim3(1), dim3(1), 0, stream, it_counter);
        OFC_CHECK_LAUNCH("kmeans_counter_inc");
    }
    if (batch > 1 && just_done && labels_cur && labels_other && n > 0) {
        int64_t bx = (n + 255) / 256;
        if (bx > 64) bx = 64;
        OFC_LAUNCH(kmeans_freeze_labels_kernel, dim3((unsigned)bx, batch), dim3(256), 0, stream, n, just_done, labels_cur, labels_other);
        OFC_CHECK_LAUNCH("kmeans_freeze_labels");
    }
    return OFC_OK;
}

int launch_kmeans_update(int batch, int d, int k, const double* sums, const long long* counts, const double* mean_sub,
                         int use_reciprocal, int round_f32, double* centres, double* shift_tot, double* shift_ws,
                         const unsigned long long* n_changed, const double* tol, int it, unsigned char* active,
                         unsigned char* just_done, int* n_iter, int* n_active, int64_t n, const int32_t* labels_cur,
                         int32_t* labels_other, int* it_counter, void* stream) {
    return launch_update(batch, d, k, sums, counts, mean_sub, use_reciprocal, round_f32, centres, shift_tot, shift_ws, n_changed, tol,
                         it, active, just_done, n_iter, n_active, n, labels_cur, labels_other, it_counter, stream);
}

int launch_kmeans_update(int batch, int d, int k, const double* sums, const double* weight_sums, const double* mean_sub,
                         int use_reciprocal, int round_f32, double* centres, double* shift_tot, double* shift_ws,
                         const unsigned long long* n_changed, const double* tol, int it, unsigned char* active,
                         unsigned char* just_done, int* n_iter, int* n_active, int64_t n, const int32_t* labels_cur,
                         int32_t* labels_other, int* it_counter, void* stream) {
    return launch_update(batch, d, k, sums, weight_sums, mean_sub, use_reciprocal, round_f32, centres, shift_tot, shift_ws, n_changed,
                         tol, it, active, just_done, n_iter, n_active, n, labels_cur, labels_other, it_counter, stream);
}

int launch_minibatch_update(const void* Xb, int dtype, int bs, int d, int k, const int32_t* labels, const double* centres_old,
                            double* centres_new, double* weight_sums, void* stream) {
    const size_t smem = (size_t)bs * sizeof(int);
    if (smem > 200 * 1024) { set_error("mini-batch of %d rows is too large (<= 51200)", bs); return OFC_ERR_UNSUPPORTED; }
    ProfScope prof(PK_KMEANS, stream);
#define OFC_MB(TT, WW)                                                                                               \
    {                                                                                                                \
        OFC_SMEM_OPTIN((minibatch_update_kernel<TT, WW>), smem);                                                     \
        OFC_LAUNCH((minibatch_update_kernel<TT, WW>), dim3(1), dim3(256), smem, stream, (const TT*)Xb, bs, d, k, labels, \
                   centres_old, centres_new, weight_sums);                                                           \
    }
    if (dtype == DT_U8) OFC_MB(unsigned char, double)
    else if (dtype == DT_F32) OFC_MB(float, float)
    else OFC_MB(double, double)
#undef OFC_MB
    OFC_CHECK_LAUNCH("minibatch_update");
    return OFC_OK;
}

static int rowdist_grid(int64_t n, int batch) {
    int64_t g = (n + 255) / 256;
    int64_t cap = (148 * 8 + batch - 1) / batch;
    if (cap < 1) cap = 1;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

template <typename T, typename C>
static int launch_rowdist(const void* X, int64_t x_stride, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                          const double* centres_old, const C* counts, double* scratch, int force,
                          const unsigned char* active, void* stream) {
    OFC_LAUNCH((kmeans_rowdist_kernel<T, C>), dim3(rowdist_grid(n, batch), batch), dim3(256), 0, stream, (const T*)X, x_stride, n, d, k, mean, labels,
               centres_old, counts, scratch, force, active);
    OFC_CHECK_LAUNCH("kmeans_rowdist");
    return OFC_OK;
}

int launch_kmeans_relocate(const void* X, int64_t x_stride, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                           const int32_t* labels, const double* centres_old, double* sums, long long* counts,
                           int raw_sums, const unsigned char* active, double* scratch, void* stream) {
    if (batch <= 0) return OFC_OK;
    if (batch > 65535) { set_error("batch=%d exceeds 65535", batch); return OFC_ERR_UNSUPPORTED; }
    ProfScope prof(PK_KMEANS, stream);
    if (scratch) {
        // two kernels: distances by the whole grid, then the pick loop (see kmeans_rowdist_kernel)
        int rc;
        if (dtype == DT_U8) rc = launch_rowdist<unsigned char>(X, x_stride, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        else if (dtype == DT_F32) rc = launch_rowdist<float>(X, x_stride, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        else rc = launch_rowdist<double>(X, x_stride, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        if (rc != OFC_OK) return rc;
        const size_t smem = empty_mask_bytes(k);
        if (dtype == DT_U8)
            OFC_LAUNCH((kmeans_relocate_apply_kernel<unsigned char, long long>), dim3(batch), dim3(1024), smem, stream, (const unsigned char*)X,
                       x_stride, n, d, k, mean, labels, scratch, sums, counts, raw_sums, active, nullptr, 0);
        else if (dtype == DT_F32)
            OFC_LAUNCH((kmeans_relocate_apply_kernel<float, long long>), dim3(batch), dim3(1024), smem, stream, (const float*)X, x_stride, n, d, k,
                       mean, labels, scratch, sums, counts, raw_sums, active, nullptr, 0);
        else
            OFC_LAUNCH((kmeans_relocate_apply_kernel<double, long long>), dim3(batch), dim3(1024), smem, stream, (const double*)X, x_stride, n, d,
                       k, mean, labels, scratch, sums, counts, raw_sums, active, nullptr, 0);
        OFC_CHECK_LAUNCH("kmeans_relocate_apply");
        return OFC_OK;
    }
    // the list of rows already given away (k words) and the empty-cluster mask in shared memory: opt in past 48 KB
    if (k > 25600) { set_error("k=%d too large for the relocation kernel (k <= 25600)", k); return OFC_ERR_UNSUPPORTED; }
    const size_t smem = (size_t)k * sizeof(long long) + empty_mask_bytes(k);
    OFC_SMEM_OPTIN(kmeans_relocate_kernel<unsigned char>, smem);
    OFC_SMEM_OPTIN(kmeans_relocate_kernel<float>, smem);
    OFC_SMEM_OPTIN(kmeans_relocate_kernel<double>, smem);
    if (dtype == DT_U8)
        OFC_LAUNCH(kmeans_relocate_kernel<unsigned char>, dim3(batch), dim3(1024), smem, stream, (const unsigned char*)X, x_stride, n, d, k,
                   mean, labels, centres_old, sums, counts, raw_sums, active);
    else if (dtype == DT_F32)
        OFC_LAUNCH(kmeans_relocate_kernel<float>, dim3(batch), dim3(1024), smem, stream, (const float*)X, x_stride, n, d, k, mean, labels,
                   centres_old, sums, counts, raw_sums, active);
    else
        OFC_LAUNCH(kmeans_relocate_kernel<double>, dim3(batch), dim3(1024), smem, stream, (const double*)X, x_stride, n, d, k, mean, labels,
                   centres_old, sums, counts, raw_sums, active);
    OFC_CHECK_LAUNCH("kmeans_relocate");
    return OFC_OK;
}

template <typename T>
static int relocate_weighted(const void* X, int64_t x_stride, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                             const double* centres_old, const double* weights, int64_t w_stride, double* sums, double* weight_sums,
                             int raw_sums, const unsigned char* active, double* scratch, void* stream) {
    int rc = launch_rowdist<T, double>(X, x_stride, batch, n, d, k, mean, labels, centres_old, weight_sums, scratch, 0, active, stream);
    if (rc != OFC_OK) return rc;
    OFC_LAUNCH((kmeans_relocate_apply_kernel<T, double>), dim3(batch), dim3(1024), empty_mask_bytes(k), stream, (const T*)X, x_stride, n, d,
               k, mean, labels, scratch, sums, weight_sums, raw_sums, active, weights, w_stride);
    OFC_CHECK_LAUNCH("kmeans_relocate_apply");
    return OFC_OK;
}

int launch_kmeans_relocate_weighted(const void* X, int64_t x_stride, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                                    const int32_t* labels, const double* centres_old, const double* weights, int64_t w_stride,
                                    double* sums, double* weight_sums, int raw_sums, const unsigned char* active, double* scratch,
                                    void* stream) {
    if (batch <= 0) return OFC_OK;
    if (batch > 65535) { set_error("batch=%d exceeds 65535", batch); return OFC_ERR_UNSUPPORTED; }
    ProfScope prof(PK_KMEANS, stream);
    if (dtype == DT_U8)
        return relocate_weighted<unsigned char>(X, x_stride, batch, n, d, k, mean, labels, centres_old, weights, w_stride, sums, weight_sums,
                                                raw_sums, active, scratch, stream);
    if (dtype == DT_F32)
        return relocate_weighted<float>(X, x_stride, batch, n, d, k, mean, labels, centres_old, weights, w_stride, sums, weight_sums,
                                        raw_sums, active, scratch, stream);
    return relocate_weighted<double>(X, x_stride, batch, n, d, k, mean, labels, centres_old, weights, w_stride, sums, weight_sums,
                                     raw_sums, active, scratch, stream);
}

int launch_kmeans_far_payload(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                              const double* centres_old, const long long* counts, int raw_sums, int n_far, long long row_offset,
                              double* payload, double* scratch, const unsigned char* active, void* stream) {
    if (batch <= 0 || n_far <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    int rc = OFC_OK;
    if (n > 0) {
        if (dtype == DT_U8) rc = launch_rowdist<unsigned char>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        else if (dtype == DT_F32) rc = launch_rowdist<float>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        else rc = launch_rowdist<double>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, counts, scratch, 0, active, stream);
        if (rc != OFC_OK) return rc;
    }
    if (dtype == DT_U8)
        OFC_LAUNCH(kmeans_far_payload_kernel<unsigned char>, dim3(batch), dim3(1024), 0, stream, (const unsigned char*)X, n, d, k, mean, labels,
                   counts, scratch, raw_sums, n_far, row_offset, payload, active);
    else if (dtype == DT_F32)
        OFC_LAUNCH(kmeans_far_payload_kernel<float>, dim3(batch), dim3(1024), 0, stream, (const float*)X, n, d, k, mean, labels, counts,
                   scratch, raw_sums, n_far, row_offset, payload, active);
    else
        OFC_LAUNCH(kmeans_far_payload_kernel<double>, dim3(batch), dim3(1024), 0, stream, (const double*)X, n, d, k, mean, labels, counts,
                   scratch, raw_sums, n_far, row_offset, payload, active);
    OFC_CHECK_LAUNCH("kmeans_far_payload");
    return OFC_OK;
}

int launch_kmeans_relocate_merge(int batch, int d, int k, int world, int n_far, const double* allpay, double* sums, long long* counts,
                                 int* overflow, const unsigned char* active, void* stream) {
    if (batch <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    const size_t smem = (((size_t)world * n_far + 3) & ~(size_t)3) + empty_mask_bytes(k);
    OFC_SMEM_OPTIN(kmeans_relocate_merge_kernel, smem);
    OFC_LAUNCH(kmeans_relocate_merge_kernel, dim3(batch), dim3(256), smem, stream, batch, d, k, world, n_far, allpay, sums, counts, overflow,
               active);
    OFC_CHECK_LAUNCH("kmeans_relocate_merge");
    return OFC_OK;
}

int launch_kmeans_far_points(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                             const double* centres_old, int n_far, double* out_val, long long* out_idx, double* scratch, void* stream) {
    if (batch <= 0 || n_far <= 0) return OFC_OK;
    ProfScope prof(PK_KMEANS, stream);
    if (scratch) {
        int rc;
        if (dtype == DT_U8) rc = launch_rowdist<unsigned char>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, (const long long*)nullptr, scratch, 1, nullptr, stream);
        else if (dtype == DT_F32) rc = launch_rowdist<float>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, (const long long*)nullptr, scratch, 1, nullptr, stream);
        else rc = launch_rowdist<double>(X, (int64_t)n * d, batch, n, d, k, mean, labels, centres_old, (const long long*)nullptr, scratch, 1, nullptr, stream);
        if (rc != OFC_OK) return rc;
        OFC_LAUNCH(kmeans_far_list_kernel, dim3(batch), dim3(1024), 0, stream, n, scratch, n_far, out_val, out_idx);
        OFC_CHECK_LAUNCH("kmeans_far_list");
        return OFC_OK;
    }
    const size_t smem = (size_t)n_far * sizeof(long long);
    if (smem > 40 * 1024) { set_error("n_far=%d too large", n_far); return OFC_ERR_UNSUPPORTED; }
    if (dtype == DT_U8)
        OFC_LAUNCH(kmeans_far_points_kernel<unsigned char>, dim3(batch), dim3(1024), smem, stream, (const unsigned char*)X, n, d, k, mean,
                   labels, centres_old, n_far, out_val, out_idx);
    else if (dtype == DT_F32)
        OFC_LAUNCH(kmeans_far_points_kernel<float>, dim3(batch), dim3(1024), smem, stream, (const float*)X, n, d, k, mean, labels,
                   centres_old, n_far, out_val, out_idx);
    else
        OFC_LAUNCH(kmeans_far_points_kernel<double>, dim3(batch), dim3(1024), smem, stream, (const double*)X, n, d, k, mean, labels,
                   centres_old, n_far, out_val, out_idx);
    OFC_CHECK_LAUNCH("kmeans_far_points");
    return OFC_OK;
}

}  // namespace ofc
