// Per-cell k-means of the reference's main loop, whole Lloyd runs on the device -- fast form for the
// reference's own shape (4-channel uint8 pixels, k <= 16):
//
//   for every frame folder, for every cell:  preprocess_image(roi); KMeans(n_clusters=k).fit(...);
//   predict; bincount; largest cluster's centre -> np.rint -> BGR2HSV hue
//   (reference k-means-color-clustering/KmeanGrids.py:376-392, :269-286, :288-339)
//
// One CTA per cell.  Same results, bit for bit, as kmeans_cells_kernel (kmeans_kernels.cu) and hence as
// the stepwise float64 kernels / scikit-learn's float64 Lloyd given the same initial centres; what changes
// is where the time goes:
//   * the cell's pixels are staged ONCE in shared memory as packed (c0,c1,c2,alpha) words -- optionally
//     gathered straight from the flow visualisation (white grid lines, < 30 -> 0 threshold and alpha applied
//     on the way in), so the [frames][cells][n][4] copy of ofc_grid_extract_cells never exists;
//   * E-step: a float32 evaluation of ||c||^2 - 2 x.c on the un-centred bytes is only a FILTER.  Its error
//     against the float64 reference chain is below E = 0.25 for any uint8 row and any centres inside the
//     data range (derivation at e_step()); a row whose best and second-best filtered distances are more than
//     1.0 (= 4 E) apart has a unique float64 minimum at the same index.  Every other row (exact ties
//     included) is re-evaluated with the float64 fma chain of the reference kernels, so labels are identical;
//   * M-step: cluster sums are exact integers and are updated INCREMENTALLY from the rows whose label
//     changed (shared-memory integer atomics); after the first couple of iterations that is a few rows;
//   * k-means++ seeding works on exact integer distances (dp4a), all candidates of a step are scored in one
//     pass, and the weighted pick is a parallel prefix scan instead of one thread's running sum.  The picks
//     are those of kmeans_cells_kernel for the same seed (integer sums are order-independent).
#include <math.h>
#include <stdlib.h>

#include "ofc_common.cuh"
#include "color_math.cuh"
#include "kmeans_kernels.cuh"

namespace ofc {

namespace {

__device__ __forceinline__ unsigned long long cells_splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// squared Euclidean distance of two packed 4-byte rows (exact, <= 260 100)
__device__ __forceinline__ unsigned dist4(unsigned a, unsigned b) {
#ifndef OFC_EMULATE
    const unsigned v = __vabsdiffu4(a, b);
    return __dp4a(v, v, 0u);
#else
    unsigned s = 0;
    for (int t = 0; t < 4; ++t) {
        const int df = (int)((a >> (8 * t)) & 255u) - (int)((b >> (8 * t)) & 255u);
        s += (unsigned)(df * df);
    }
    return s;
#endif
}

// byte t of w as a float, without an integer->float conversion: 0x4B0000bb is 2^23 + bb
template <int T> __device__ __forceinline__ float byte_as_float(unsigned w) {
#ifndef OFC_EMULATE
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540 + T)) - 8388608.f;
#else
    return (float)((w >> (8 * T)) & 255u);
#endif
}

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
    return __shfl_xor_sync(0xffffffffu, v, m);
}

__device__ __forceinline__ unsigned warp_sum_u32(unsigned v) {
#ifndef OFC_EMULATE
    return __reduce_add_sync(0xffffffffu, v);
#else
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
#endif
}

// two bytes of a packed row as 16-bit fields of one word: (byte A) | (byte B) << 16
template <int SEL> __device__ __forceinline__ unsigned spread2(unsigned w) {
#ifndef OFC_EMULATE
    return __byte_perm(w, 0u, SEL);
#else
    const unsigned a = (w >> (8 * (SEL & 7))) & 255u, b = (w >> (8 * ((SEL >> 8) & 7))) & 255u;
    return a | (b << 16);
#endif
}

}  // namespace

// KP = 8 steps two rows per thread with the plain label chain, so it fits 80 registers = 3 CTAs per SM (64 registers
// at 4 CTAs spill 316 bytes).  Measured on 1080p visualisation cells, k = 8 (r02f / r02g): 0.241 ms per frame, against
// 0.264 with four rows per step and 0.285 with the index packed into the mantissa (one more ALU-pipe op per distance).
template <int KP>
__global__ void __launch_bounds__(256, KP <= 8 ? 3 : 2) kmeans_cells_fast_kernel(KmCellsFastParams p) {
    constexpr int RU = KP == 8 ? 2 : 4;                   // rows per thread step of the E-step
    constexpr bool PACK = KP != 8;                        // E-step arg-min index packed into the distances' low bits
    constexpr int D = 4;
    OFC_DYN_SMEM(unsigned char, smraw);
    const int n = p.n, k = p.k, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b = blockIdx.x;
    // ---- shared memory carve-up (doubles first: 8-byte alignment) --------------------------------------
    double* cc = reinterpret_cast<double*>(smraw);      // [KP][4] centred centres (float64: the reference values)
    double* c2 = cc + KP * D;                             // [KP]
    double* cnew = c2 + KP;                               // [KP][4]
    double* shift = cnew + KP * D;                        // [KP]
    double* mean = shift + KP;                            // [4]
    double* s_red = mean + D;                             // [8]
    unsigned long long* s_u64 = reinterpret_cast<unsigned long long*>(s_red + 8);   // [8 warps][8] scratch
    float* s_cf = reinterpret_cast<float*>(s_u64 + 64);   // [KP][5] un-centred float32 centres + squared norm
    unsigned* s_sum = reinterpret_cast<unsigned*>(s_cf + KP * 5);    // [KP][4] exact channel sums of the current labels
    int* s_cnt = reinterpret_cast<int*>(s_sum + KP * D);             // [KP]
    int* s_moves = s_cnt + KP;                                        // [KP][3] relocation moves of this iteration
    unsigned* xs = reinterpret_cast<unsigned*>(s_moves + KP * 3);     // [n] packed rows
    unsigned* closest = xs + n;                                       // [n] (seeding, when it fits) -- may be global
    unsigned char* lab = reinterpret_cast<unsigned char*>(p.closest_in_smem ? closest + n : xs + n);   // [n]
    __shared__ unsigned long long s_stat[8];
    __shared__ double s_tol;
    __shared__ double s_val[8];
    __shared__ int s_idx[8];
    __shared__ int s_pick, s_stop, s_changed, s_nmoves, s_exact;
    __shared__ int s_cand[8];
    if (!p.closest_in_smem) closest = p.closest_ws + b * n;

    // ---- stage the cell --------------------------------------------------------------------------------
    if (p.bgr) {
        // image_dict ROI + preprocess_image (KmeanGrids.py:85,113,269-286): white row 0 / column 0 (the state of
        // the frame at the reference's k-means stage, SURVEY.md Q3), channel < threshold -> 0,
        // alpha = 255 * (BGR2GRAY(thresholded) > 0)
        const int frame = (int)(b / p.cells), cell = (int)(b - (int64_t)frame * p.cells);
        const int cy = cell / p.cols, cx = cell - cy * p.cols;
        const int x1 = cx * p.x_step, y1 = cy * p.y_step;
        const unsigned char* img = p.bgr + (int64_t)frame * p.frame_stride;
        for (int i = tid; i < n; i += 256) {
            const int ly = i / p.x_step, lx = i - ly * p.x_step;
            const unsigned char* px = img + ((int64_t)(y1 + ly) * p.W + (x1 + lx)) * 3;
            unsigned c0 = px[0], c1 = px[1], c2v = px[2];
            if (p.draw_lines && (ly == 0 || lx == 0)) c0 = c1 = c2v = 255u;
            if (p.swap_rb) { const unsigned t = c0; c0 = c2v; c2v = t; }
            if (p.threshold) {
                c0 = c0 < (unsigned)p.threshold ? 0u : c0;
                c1 = c1 < (unsigned)p.threshold ? 0u : c1;
                c2v = c2v < (unsigned)p.threshold ? 0u : c2v;
            }
            const unsigned gray = (3735u * c0 + 19235u * c1 + 9798u * c2v + 16384u) >> 15;
            xs[i] = c0 | (c1 << 8) | (c2v << 16) | (gray > 0 ? 0xFF000000u : 0u);
        }
    } else {
        const unsigned* X = reinterpret_cast<const unsigned*>(p.X) + b * n;
        for (int i = tid; i < n; i += 256) xs[i] = X[i];
    }
    for (int i = tid; i < n; i += 256) lab[i] = 255;
    if (tid < 8) s_stat[tid] = 0ull;
    __syncthreads();

    // ---- column statistics: mean, tolerance (exact integers) -------------------------------------------
    {
        unsigned sx[D] = {0, 0, 0, 0}, sxx[D] = {0, 0, 0, 0};      // <= 4096 rows per thread: fits 32 bits
        for (int i = tid; i < n; i += 256) {
            const unsigned w = xs[i];
#pragma unroll
            for (int t = 0; t < D; ++t) {
                const unsigned v = (w >> (8 * t)) & 255u;
                sx[t] += v; sxx[t] += v * v;
            }
        }
#pragma unroll
        for (int t = 0; t < D; ++t) {
            unsigned long long a = sx[t], q = sxx[t];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { a += shfl_xor_u64(a, o); q += shfl_xor_u64(q, o); }
            if (lane == 0) { atomicAdd(&s_stat[t], a); atomicAdd(&s_stat[4 + t], q); }
        }
    }
    __syncthreads();
    if (tid == 0) {
        double vs = 0.0;
        for (int t = 0; t < D; ++t) {
            mean[t] = (double)s_stat[t] / (double)n;
            const unsigned long long num = (unsigned long long)n * s_stat[4 + t] - s_stat[t] * s_stat[t];
            vs += (double)num / ((double)n * (double)n);
        }
        s_tol = vs / (double)D * p.tol;
        s_exact = 0;
    }
    __syncthreads();

    // ---- initial centres -------------------------------------------------------------------------------
    if (p.init) {
        for (int e = tid; e < k * D; e += 256) cc[e] = p.init[b * k * D + e] - mean[e & 3];
    } else {
        // k-means++ (sklearn/cluster/_kmeans.py:181-268): first centre uniform; then 2 + int(log k) candidates per
        // step drawn in proportion to the squared distance to the closest chosen centre, keeping the candidate with
        // the lowest potential (first one on ties).  Counter-based random stream of (seed, problem): the reference
        // leaves random_state unset (SURVEY.md Q9).
        const int trials = 2 + (int)log((double)k);                 // <= 4 for k <= 16
        unsigned long long ctr = cells_splitmix64(p.seed ^ (0xD1B54A32D192ED03ull * (unsigned long long)(p.problem_offset + b + 1)));
        auto uniform = [&]() -> double { ctr = cells_splitmix64(ctr); return (double)(ctr >> 11) * (1.0 / 9007199254740992.0); };
        int chunk = (n + 255) / 256;
        chunk |= 1;                                                  // odd stride: conflict-free contiguous ranges
        const int lo = min(n, tid * chunk), hi = min(n, lo + chunk);
        int first = (int)(uniform() * (double)n);
        if (first >= n) first = n - 1;
        unsigned chosen = xs[first];
        if (tid < D) cc[tid] = (double)((chosen >> (8 * tid)) & 255u) - mean[tid];
        for (int c = 1; c < k; ++c) {
            // pass B of the previous step: fold the newly chosen centre into `closest`, range sums on the way
            unsigned long long loc = 0ull;
            for (int i = lo; i < hi; ++i) {
                const unsigned dnew = dist4(xs[i], chosen);
                const unsigned v = c == 1 ? dnew : min(closest[i], dnew);
                closest[i] = v;
                loc += v;
            }
            // inclusive prefix sums of the 256 range sums
            unsigned long long incl = loc;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            if (lane == 31) s_u64[warp] = incl;
            __syncthreads();
            unsigned long long before = 0ull, pot_u = 0ull;
            for (int w = 0; w < 8; ++w) { const unsigned long long v = s_u64[w]; if (w < warp) before += v; pot_u += v; }
            incl += before;
            const unsigned long long excl = incl - loc;
            const double pot = (double)pot_u;
            // the weighted picks: first row whose running sum exceeds r (the last row when none does)
            for (int tr = 0; tr < trials; ++tr) {
                const double r = uniform() * pot;                    // same value in every thread
                const bool below = r < (double)incl;
                const bool owner = below && !(r < (double)excl);
                if (owner) {
                    unsigned long long acc = excl;
                    int cand = hi - 1;
                    for (int i = lo; i < hi; ++i) { acc += closest[i]; if (r < (double)acc) { cand = i; break; } }
                    s_cand[tr] = cand;
                }
                if (tid == 255 && !(r < (double)pot_u)) s_cand[tr] = n - 1;
            }
            __syncthreads();
            // pass A: potential of every candidate
            unsigned candx[4];
            unsigned long long pp[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
            for (int tr = 0; tr < 4; ++tr) candx[tr] = xs[s_cand[tr < trials ? tr : 0]];
            for (int i = lo; i < hi; ++i) {
                const unsigned x = xs[i], cl = closest[i];
#pragma unroll
                for (int tr = 0; tr < 4; ++tr) pp[tr] += min(cl, dist4(x, candx[tr]));
            }
#pragma unroll
            for (int tr = 0; tr < 4; ++tr) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) pp[tr] += shfl_xor_u64(pp[tr], o);
                if (lane == 0) s_u64[8 + warp * 4 + tr] = pp[tr];
            }
            __syncthreads();
            int best = 0;
            unsigned long long best_pot = 0ull;
            for (int tr = 0; tr < trials; ++tr) {
                unsigned long long tot = 0ull;
                for (int w = 0; w < 8; ++w) tot += s_u64[8 + w * 4 + tr];
                if (tr == 0 || tot < best_pot) { best_pot = tot; best = tr; }
            }
            chosen = candx[best];
            if (tid < D) cc[c * D + tid] = (double)((chosen >> (8 * tid)) & 255u) - mean[tid];
            __syncthreads();                                         // s_cand / s_u64 are rewritten by the next step
        }
    }
    __syncthreads();

    // ---- Lloyd iterations ------------------------------------------------------------------------------
    // float64 label of one row: the fma chain of kmeans_cells_kernel / kmeans_assign_small_kernel
    auto exact_label = [&](unsigned w) -> int {
        double xc[D];
#pragma unroll
        for (int t = 0; t < D; ++t) xc[t] = (double)((w >> (8 * t)) & 255u) - mean[t];
        double bestd = 0.0;
        int label = 0;
        for (int j = 0; j < k; ++j) {
            const double* c = cc + j * D;
            double dot = 0.0;
#pragma unroll
            for (int t = 0; t < D; ++t) dot = fma(xc[t], c[t], dot);
            const double dist = fma(-2.0, dot, c2[j]);
            if (j == 0 || dist < bestd) { bestd = dist; label = j; }
        }
        return label;
    };
    // Filtered E-step over this thread's rows.  With u = 2^-24, x in [0,255]^4 and un-centred centres c' = c + mean
    // inside [0,255]^4 (means of data rows):  rounding c' to float32 moves x.c' by <= 4*255*255 u; the four-fma dot
    // product adds <= 4 u * 260100; rounding ||c'||^2 adds <= 260100 u; the closing fma adds <= 780300 u; with the
    // factor 2 on the dot product the total is < 3.7e6 u = 0.22 < E = 0.25.  ||x - c'||^2 and the centred float64
    // chain differ by a per-row constant (||x||^2 - ||x - mean||^2 terms cancel between clusters), and the float64
    // chain's own rounding (< 1e-9) is far inside the margin, so a filtered gap > MARGIN (below) fixes the arg-min.
    // RU rows per thread step and no serial best/second chain: the distances of a row are independent, the
    // minimum is a tree, the label the lowest index that attains it, and "near tie" = more than one distance within
    // 1.0 of the minimum -- so a thread always has RU rows' worth of independent arithmetic in flight.
    auto e_step = [&](auto&& on_label) {
        float fx[KP], fy[KP], fz[KP], fw[KP], fq[KP];
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            fx[j] = s_cf[j * 5 + 0]; fy[j] = s_cf[j * 5 + 1]; fz[j] = s_cf[j * 5 + 2]; fw[j] = s_cf[j * 5 + 3]; fq[j] = s_cf[j * 5 + 4];
        }
        // filtered values carry: the float32 evaluation error E < 0.25, the rounding of the shifted norm (< 0.07) and the
        // index bits (< KP ulp of values below 2^21 = KP / 8); twice their sum, rounded up, separates "unique minimum"
        constexpr float MARGIN = !PACK ? 1.5f : (KP <= 4 ? 2.f : (KP <= 8 ? 3.f : 5.f));
        for (int i0 = tid; i0 < n; i0 += 256 * RU) {
            unsigned w[RU];
            int label[RU];
            bool near[RU];
#pragma unroll
            for (int r = 0; r < RU; ++r) w[r] = xs[min(i0 + 256 * r, n - 1)];
#pragma unroll
            for (int r = 0; r < RU; ++r) {
                const float x0 = byte_as_float<0>(w[r]), x1 = byte_as_float<1>(w[r]), x2 = byte_as_float<2>(w[r]), x3 = byte_as_float<3>(w[r]);
                float dj[KP];
#pragma unroll
                for (int j = 0; j < KP; ++j) {
                    float dot = x0 * fx[j];
                    dot = fmaf(x1, fy[j], dot);
                    dot = fmaf(x2, fz[j], dot);
                    dot = fmaf(x3, fw[j], dot);
                    // the cluster index rides in the low mantissa bits (distances are positive, see prepare_centres): the
                    // minimum of the packed values is the arg-min, lowest index first among equal distances
                    const float dv = fmaf(-2.f, dot, fq[j]);
                    dj[j] = PACK ? __uint_as_float((__float_as_uint(dv) & ~(unsigned)(KP - 1)) | (unsigned)j) : dv;
                }
                float m[KP];
#pragma unroll
                for (int j = 0; j < KP; ++j) m[j] = dj[j];
#pragma unroll
                for (int st = KP / 2; st > 0; st >>= 1)
#pragma unroll
                    for (int j = 0; j < st; ++j) m[j] = fminf(m[j], m[j + st]);
                const float best = m[0], lim = best + MARGIN;
                int lb = PACK ? (int)(__float_as_uint(best) & (unsigned)(KP - 1)) : KP - 1;
                int cnt = 0;
#pragma unroll
                for (int j = KP - 1; j >= 0; --j) {
                    if (!PACK) lb = dj[j] == best ? j : lb;
                    cnt += dj[j] <= lim ? 1 : 0;
                }
                label[r] = lb;
                near[r] = cnt > 1;
            }
#pragma unroll
            for (int r = 0; r < RU; ++r) {
                const int i = i0 + 256 * r;
                if (i < n) {
                    if (near[r]) label[r] = exact_label(w[r]);
                    on_label(i, w[r], label[r]);
                }
            }
        }
    };
    // Centres outside the data range (an empty cluster holding the heaviest cluster's centred sum, or such initial
    // centres).  One farther than 2^19 (squared) from [0,255]^4 is farther from every row than any centre inside
    // [-1,256]^4 can be (4 * 256^2 = 2^18): it never wins, so the filter leaves it out like a padding cluster (the float64
    // chain of the near-ties still sees it).  That needs one centre inside the range, which every centre computed by an
    // update has -- the heaviest cluster's mean -- but initial centres need not.  Any other centre outside [-1,256]^4
    // voids the filter's bound: from then on every row takes the float64 chain -- the same rows per thread, in the same
    // order.  s_exact is set in prepare_centres and sticky (no reset between barriers); the unit of slack keeps means
    // that round a few ulp past 0 or 255 on the filter, and with |c'_t| <= 256 the bound above still stays below E.  The
    // test is uniform and outside the row loop, so the filtered loop is unchanged.
    auto lloyd_e_step = [&](auto&& on_label) {
        if (s_exact) {
            for (int i = tid; i < n; i += 256) { const unsigned w = xs[i]; on_label(i, w, exact_label(w)); }
        } else {
            e_step(on_label);
        }
    };
    // c2 (float64), float32 filter copies; padding clusters can never win.  `updated`: the centres come from an update
    auto prepare_centres = [&](bool updated) {
        for (int j = tid; j < KP; j += 256) {
            if (j < k) {
                double squ = 0.0, out = 0.0;
                bool inside = true;
                const double sq = norm_sq_numpy_f64(cc + j * D, D);
                for (int t = 0; t < D; ++t) {
                    const double u = cc[j * D + t] + mean[t];
                    squ += u * u;
                    s_cf[j * 5 + t] = (float)u;
                    inside = inside && u >= -1.0 && u <= 256.0;
                    const double o = fmax(fmax(-u, u - 255.0), 0.0);
                    out += o * o;
                }
                c2[j] = sq;
                if (updated && out > 524288.0) {
                    for (int t = 0; t < D; ++t) s_cf[j * 5 + t] = 0.f;
                    s_cf[j * 5 + 4] = 3.0e38f;
                    continue;
                }
                if (!inside) s_exact = 1;
                // + 2^18: ||c'||^2 - 2 x.c' >= -||x||^2 >= -260100, so every filtered distance is a positive float below 2^21
                s_cf[j * 5 + 4] = (float)(squ + 262144.0);
            } else {
                for (int t = 0; t < D; ++t) s_cf[j * 5 + t] = 0.f;
                s_cf[j * 5 + 4] = 3.0e38f;
            }
        }
    };

    for (int e = tid; e < KP * D; e += 256) s_sum[e] = 0u;
    for (int j = tid; j < KP; j += 256) s_cnt[j] = 0;
    int iters = 0;
    bool strict = false;
    for (int it = 0; it < p.max_iter; ++it) {
        prepare_centres(it > 0);
        if (tid == 0) { s_changed = 0; s_nmoves = 0; }
        // M-step of this iteration: the first E-step labels every row, so its sums are built from scratch in registers
        // (16-bit fields, warp reductions -- no contended atomics); every later iteration updates them from the rows
        // whose label moved.  Both are exact integer arithmetic, so the choice cannot change a bit.  Measured on
        // 350 x 5852 random rows (r02c): k = 3 / 8 / 16 -> 0.47 / 1.11 / 1.67 ms, against 0.53 / 1.49 / 2.32 ms
        // rebuilding every iteration.
        const bool full = it == 0;
        if (full) {
            for (int e = tid; e < KP * D; e += 256) s_sum[e] = 0u;
            for (int j = tid; j < KP; j += 256) s_cnt[j] = 0;
        }
        __syncthreads();
        int changed = 0;
        if (full) {
            lloyd_e_step([&](int i, unsigned, int label) {
                if (lab[i] != label) { ++changed; lab[i] = (unsigned char)label; }
            });
            unsigned a0[KP], a1[KP], ac[KP];
#pragma unroll
            for (int j = 0; j < KP; ++j) { a0[j] = 0u; a1[j] = 0u; ac[j] = 0u; }
            for (int i = tid; i < n; i += 256) {               // this thread's own rows: it wrote their labels itself
                const unsigned w = xs[i];
                const int l = lab[i];
                const unsigned p0 = spread2<0x4140>(w), p1 = spread2<0x4342>(w);
#pragma unroll
                for (int j = 0; j < KP; ++j) {
                    const bool mine = l == j;
                    a0[j] += mine ? p0 : 0u;
                    a1[j] += mine ? p1 : 0u;
                    ac[j] += mine ? 1u : 0u;
                }
            }
#pragma unroll
            for (int j = 0; j < KP; ++j) {
                if (j < k) {                                   // uniform
                    const unsigned s0 = warp_sum_u32(a0[j] & 0xFFFFu), s1 = warp_sum_u32(a0[j] >> 16);
                    const unsigned s2 = warp_sum_u32(a1[j] & 0xFFFFu), s3 = warp_sum_u32(a1[j] >> 16);
                    const unsigned sc = warp_sum_u32(ac[j]);
                    if (lane == 0 && sc) {
                        atomicAdd(&s_sum[j * D + 0], s0); atomicAdd(&s_sum[j * D + 1], s1);
                        atomicAdd(&s_sum[j * D + 2], s2); atomicAdd(&s_sum[j * D + 3], s3);
                        atomicAdd(&s_cnt[j], (int)sc);
                    }
                }
            }
        } else {
            lloyd_e_step([&](int i, unsigned w, int label) {
                const int old = lab[i];
                if (old != label) {
                    ++changed;
                    lab[i] = (unsigned char)label;
#pragma unroll
                    for (int t = 0; t < D; ++t) {
                        const unsigned v = (w >> (8 * t)) & 255u;
                        if (v) {
                            atomicAdd(&s_sum[label * D + t], v);
                            atomicAdd(&s_sum[old * D + t], 0u - v);
                        }
                    }
                    atomicAdd(&s_cnt[label], 1);
                    atomicAdd(&s_cnt[old], -1);
                }
            });
        }
        if (changed) atomicAdd(&s_changed, changed);
        __syncthreads();
        // empty clusters take the farthest points (squared distance to the old centre of their label); the labels
        // stay as they are (_k_means_common.pyx:167-211), so the moves are undone on the running sums below.
        // The member counts are final behind the barrier above: every thread takes the set of empty clusters from them
        // itself (no flag, no barrier), once -- a cluster that a move empties stays empty in this iteration
        unsigned empty = 0u;
        for (int j = 0; j < k; ++j) empty |= (s_cnt[j] == 0 ? 1u : 0u) << j;
        if (empty) {
            for (int e = 0; e < k; ++e) {
                if (!((empty >> e) & 1u)) continue;
                const int n_taken = s_nmoves;
                double bv = -1.0;
                int bi = -1;
                for (int i = tid; i < n; i += 256) {
                    bool tk = false;
                    for (int q = 0; q < n_taken; ++q) tk |= s_moves[q * 3] == i;
                    if (tk) continue;
                    const unsigned w = xs[i];
                    const double* c = cc + lab[i] * D;
                    double v = 0.0;
#pragma unroll
                    for (int t = 0; t < D; ++t) { const double df = ((double)((w >> (8 * t)) & 255u) - mean[t]) - c[t]; v = fma(df, df, v); }
                    if (v > bv) { bv = v; bi = i; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
                }
                if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
                __syncthreads();
                if (tid == 0) {
                    double v = -1.0;
                    int idx = -1;
                    for (int w = 0; w < 8; ++w)
                        if (s_idx[w] >= 0 && (idx < 0 || s_val[w] > v || (s_val[w] == v && s_idx[w] < idx))) { v = s_val[w]; idx = s_idx[w]; }
                    if (n_taken == 0 && !(v > 0.0)) idx = -1;          // np.max(distances) == 0: nothing to do
                    s_pick = idx;
                    if (idx >= 0) {
                        const int old = lab[idx];
                        const unsigned w = xs[idx];
                        s_moves[n_taken * 3] = idx; s_moves[n_taken * 3 + 1] = old; s_moves[n_taken * 3 + 2] = e;
                        s_nmoves = n_taken + 1;
                        for (int t = 0; t < D; ++t) {
                            const unsigned xv = (w >> (8 * t)) & 255u;
                            s_sum[old * D + t] -= xv;
                            s_sum[e * D + t] = xv;
                        }
                        s_cnt[e] = 1;
                        s_cnt[old] -= 1;
                    }
                }
                __syncthreads();
                if (s_pick < 0) break;
            }
            __syncthreads();
        }
        // centres, shift, stopping rule: all of it by warp 0 (k <= 16 <= 32 lanes) between two __syncwarp, while the
        // other warps go straight to the barrier at the end of the iteration -- three CTA-wide barriers per iteration
        // instead of six (ncu r03q: barrier waits were 28 % of the stall samples at ~10 pixels per thread)
        if (warp == 0) {
            int heavy = 0;
            for (int j = 1; j < k; ++j) if (s_cnt[j] > s_cnt[heavy]) heavy = j;
            for (int j = lane; j < k; j += 32) {
                const int srcj = s_cnt[j] > 0 ? j : heavy;
                const bool as_sum = srcj != j && j < srcj;     // the heaviest cluster's centred sum (kmeans_cells_kernel)
                const double wgt = (double)s_cnt[srcj];
                double ss = 0.0;
                for (int t = 0; t < D; ++t) {
                    const double sv = (double)s_sum[srcj * D + t];
                    const double v = as_sum ? fma(-wgt, mean[t], sv) : sv / wgt - mean[t];
                    const double df = v - cc[j * D + t];
                    ss = fma(df, df, ss);
                    cnew[j * D + t] = v;
                }
                const double sr = sqrt(ss);
                shift[j] = sr * sr;
            }
            __syncwarp();
            for (int e = lane; e < k * D; e += 32) cc[e] = cnew[e];
        }
        if (tid == 0) {
            double tot = 0.0;
            for (int j = 0; j < k; ++j) tot += shift[j];
            int stop = 0;
            if (s_changed == 0) stop = 2;                 // labels repeated: strict convergence
            else if (tot <= s_tol) stop = 1;
            s_stop = stop;
            // the running sums go back to "sums of the current labels" (the relocated rows keep their label)
            for (int q = s_nmoves - 1; q >= 0; --q) {
                const int idx = s_moves[q * 3], old = s_moves[q * 3 + 1], e = s_moves[q * 3 + 2];
                const unsigned w = xs[idx];
                for (int t = 0; t < D; ++t) {
                    const unsigned xv = (w >> (8 * t)) & 255u;
                    s_sum[old * D + t] += xv;
                    s_sum[e * D + t] = 0u;
                }
                s_cnt[e] = 0;
                s_cnt[old] += 1;
            }
        }
        __syncthreads();
        iters = it + 1;
        if (s_stop) { strict = s_stop == 2; break; }
    }

    // ---- closing E-step on the final centres: labels, member counts, inertia -----------------------------
    // After a strict stop the labels are already those of the final centres and s_cnt their member counts
    // (_kmeans.py:745-755 skips the extra E-step too), so the pass only runs when its by-products are wanted.
    int32_t* labels_out = p.labels ? p.labels + b * n : nullptr;
    double inert = 0.0;
    const bool want_inertia = p.inertia != nullptr;
    const bool closing = !strict || want_inertia || labels_out != nullptr;
    if (closing) {
        prepare_centres(iters > 0);
        for (int j = tid; j < KP; j += 256) s_cnt[j] = 0;
    }
    __syncthreads();
    if (closing) lloyd_e_step([&](int i, unsigned w, int label) {
        lab[i] = (unsigned char)label;
        if (labels_out) labels_out[i] = label;
        atomicAdd(&s_cnt[label], 1);
        if (want_inertia) {
            const double* c = cc + label * D;
            double sq = 0.0;
#pragma unroll
            for (int t = 0; t < D; ++t) { const double df = ((double)((w >> (8 * t)) & 255u) - mean[t]) - c[t]; sq = fma(df, df, sq); }
            inert += sq;
        }
    });
    if (want_inertia) {                                    // fixed order: xor tree inside a warp, warps 0..7 in sequence
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) inert += __shfl_xor_sync(0xffffffffu, inert, o);
        if (lane == 0) s_red[warp] = inert;
    }
    __syncthreads();
    if (p.centres)
        for (int e = tid; e < k * D; e += 256) p.centres[b * k * D + e] = cc[e] + mean[e & 3];
    if (p.counts)
        for (int j = tid; j < k; j += 256) p.counts[b * k + j] = s_cnt[j];
    if (tid == 0) {
        if (want_inertia) {
            double tot = 0.0;
            for (int w = 0; w < 8; ++w) tot += s_red[w];
            p.inertia[b] = tot;
        }
        if (p.n_iter) p.n_iter[b] = iters;
        if (p.dom_centre || p.dom_hue) {
            // largest cluster (first one on equal shares: the reference's stable sort, KmeanGrids.py:317), np.rint,
            // the cast to uint8 of its first three channels, BGR2HSV hue (:326-336)
            int top = 0;
            for (int j = 1; j < k; ++j) if (s_cnt[j] > s_cnt[top]) top = j;
            int c[D];
            for (int t = 0; t < D; ++t) {
                const double v = rint(cc[top * D + t] + mean[t]);
                c[t] = v < 0.0 ? 0 : (v > 255.0 ? 255 : (int)v);
            }
            if (p.dom_centre)
                for (int t = 0; t < D; ++t) p.dom_centre[b * D + t] = (unsigned char)c[t];
            if (p.dom_hue) p.dom_hue[b] = (unsigned char)hue_of_bgr(c[0], c[1], c[2]);
        }
    }
}

// ---------------------------------------------------------------------------
// One stepwise Lloyd iteration (E-step + exact integer M-step sums) for the reference's pixel shape -- uint8 rows
// with 4 channels, k <= 8 -- as ONE pass: kmeans_step_u8_kernel's results (labels, n_changed, per-CTA integer
// partial sums, bit for bit) with the float32-filtered E-step of the per-cell kernel above and the M-step in packed
// 16-bit register fields (flushed through warp reductions every 256 rows of a thread).  Four rows per thread step
// (one 16-byte load, one 16-byte label store).  The centres of the stepwise API are arbitrary (any initial centres),
// so the filter margin is computed from them:  |filtered - exact| <= 2^-24 (3060 ||c'||_1 + 2 ||c'||^2) per cluster
// (derivation at e_step() above, with |x_t| <= 255); rows whose two best filtered distances are closer than 8x the
// largest such bound are re-evaluated with the float64 chain.
// ---------------------------------------------------------------------------
template <int KP>
__global__ void __launch_bounds__(256, 2) kmeans_step_u8d4_kernel(KmAssignParams p, double* __restrict__ partial,
                                                                  long long* __restrict__ cnt_partial) {
    constexpr int D = 4;
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, k = p.k;
    if (p.active && !p.active[b]) return;
    __shared__ double s_c[KP * D], s_c2[KP], s_mean[D];
    __shared__ float s_cf[KP * 5], s_bound[KP];
    __shared__ unsigned s_acc[KP * 5];
    const double* cen = p.centres + (int64_t)b * k * D;
    for (int i = tid; i < KP * D; i += 256) s_c[i] = i < k * D ? cen[i] : 0.0;
    if (tid < D) s_mean[tid] = p.mean ? p.mean[(int64_t)b * D + tid] : 0.0;
    for (int i = tid; i < KP * 5; i += 256) s_acc[i] = 0u;
    __syncthreads();
    if (tid < KP) {
        const int j = tid;
        if (j < k) {
            s_c2[j] = norm_sq_numpy_f64(s_c + j * D, D);
            double l1 = 0.0, l2 = 0.0;
            for (int t = 0; t < D; ++t) {
                const double u = s_c[j * D + t] + s_mean[t];
                l1 += fabs(u); l2 += u * u;
                s_cf[j * 5 + t] = (float)u;
            }
            s_cf[j * 5 + 4] = (float)l2;
            s_bound[j] = (float)((3060.0 * l1 + 2.0 * l2) * (1.0 / 16777216.0));
        } else {
            s_c2[j] = 0.0;
            for (int t = 0; t < D; ++t) s_cf[j * 5 + t] = 0.f;
            s_cf[j * 5 + 4] = 3.0e38f;
            s_bound[j] = 0.f;
        }
    }
    __syncthreads();
    float margin = 0.f;
#pragma unroll
    for (int j = 0; j < KP; ++j) margin = fmaxf(margin, s_bound[j]);
    margin = 8.f * margin + 1e-6f;
    float fx[KP], fy[KP], fz[KP], fw[KP], fq[KP];
#pragma unroll
    for (int j = 0; j < KP; ++j) {
        fx[j] = s_cf[j * 5 + 0]; fy[j] = s_cf[j * 5 + 1]; fz[j] = s_cf[j * 5 + 2]; fw[j] = s_cf[j * 5 + 3]; fq[j] = s_cf[j * 5 + 4];
    }
    auto exact_label = [&](unsigned w) -> int {            // kmeans_step_u8_kernel's float64 chain
        double xc[D];
#pragma unroll
        for (int t = 0; t < D; ++t) xc[t] = (double)((w >> (8 * t)) & 255u) - s_mean[t];
        double bestd = 0.0;
        int label = 0;
        for (int j = 0; j < k; ++j) {
            double dot = 0.0;
#pragma unroll
            for (int t = 0; t < D; ++t) dot = fma(xc[t], s_c[j * D + t], dot);
            const double dist = fma(-2.0, dot, s_c2[j]);
            if (j == 0 || dist < bestd) { bestd = dist; label = j; }
        }
        return label;
    };
    auto filter_label = [&](unsigned w, bool& near) -> int {
        const float x0 = byte_as_float<0>(w), x1 = byte_as_float<1>(w), x2 = byte_as_float<2>(w), x3 = byte_as_float<3>(w);
        float dj[KP], m[KP];
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            float dot = x0 * fx[j];
            dot = fmaf(x1, fy[j], dot);
            dot = fmaf(x2, fz[j], dot);
            dot = fmaf(x3, fw[j], dot);
            dj[j] = fmaf(-2.f, dot, fq[j]);
            m[j] = dj[j];
        }
#pragma unroll
        for (int st = KP / 2; st > 0; st >>= 1)
#pragma unroll
            for (int j = 0; j < st; ++j) m[j] = fminf(m[j], m[j + st]);
        const float best = m[0], lim = best + margin;
        int lb = KP - 1, cnt = 0;
#pragma unroll
        for (int j = KP - 1; j >= 0; --j) {
            lb = dj[j] == best ? j : lb;
            cnt += dj[j] <= lim ? 1 : 0;
        }
        near = cnt > 1;
        return lb;
    };

    const int64_t n = p.n, n4 = n >> 2;
    const uint4* X4 = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(p.X) + (int64_t)b * p.x_stride);
    int4* L4 = reinterpret_cast<int4*>(p.labels + (int64_t)b * n);
    const int4* P4 = p.prev_labels ? reinterpret_cast<const int4*>(p.prev_labels + (int64_t)b * n) : nullptr;
    unsigned a0[KP], a1[KP], ac[KP];
#pragma unroll
    for (int j = 0; j < KP; ++j) { a0[j] = 0u; a1[j] = 0u; ac[j] = 0u; }
    auto flush = [&]() {                                   // warp-collective: every thread of the CTA calls it together
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            if (j < k) {
                const unsigned s0 = warp_sum_u32(a0[j] & 0xFFFFu), s1 = warp_sum_u32(a0[j] >> 16);
                const unsigned s2 = warp_sum_u32(a1[j] & 0xFFFFu), s3 = warp_sum_u32(a1[j] >> 16);
                const unsigned sc = warp_sum_u32(ac[j]);
                if (lane == 0 && sc) {
                    atomicAdd(&s_acc[j * 5 + 0], s0); atomicAdd(&s_acc[j * 5 + 1], s1);
                    atomicAdd(&s_acc[j * 5 + 2], s2); atomicAdd(&s_acc[j * 5 + 3], s3);
                    atomicAdd(&s_acc[j * 5 + 4], sc);
                }
            }
            a0[j] = 0u; a1[j] = 0u; ac[j] = 0u;
        }
    };
    unsigned changed = 0;
    int since_flush = 0;
    for (int64_t base = (int64_t)blockIdx.x * 256; base < n4; base += (int64_t)gridDim.x * 256) {
        const int64_t g = base + tid;
        if (g < n4) {
            const uint4 q = X4[g];
            const unsigned w[4] = {q.x, q.y, q.z, q.w};
            int lab[4];
            bool near[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) lab[r] = filter_label(w[r], near[r]);
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (near[r]) lab[r] = exact_label(w[r]);
            L4[g] = make_int4(lab[0], lab[1], lab[2], lab[3]);
            if (P4) {
                const int4 pl = P4[g];
                changed += (pl.x != lab[0]) + (pl.y != lab[1]) + (pl.z != lab[2]) + (pl.w != lab[3]);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const unsigned p0 = spread2<0x4140>(w[r]), p1 = spread2<0x4342>(w[r]);
#pragma unroll
                for (int j = 0; j < KP; ++j) {
                    const bool mine = lab[r] == j;
                    a0[j] += mine ? p0 : 0u;
                    a1[j] += mine ? p1 : 0u;
                    ac[j] += mine ? 1u : 0u;
                }
            }
        }
        since_flush += 4;
        if (since_flush >= 256) { flush(); since_flush = 0; }
    }
    flush();
    // the n % 4 last rows: scalar, exact chain
    if (blockIdx.x == 0 && tid < (int)(n & 3)) {
        const int64_t i = (n4 << 2) + tid;
        const unsigned w = reinterpret_cast<const unsigned*>(reinterpret_cast<const unsigned char*>(p.X) + (int64_t)b * p.x_stride)[i];
        const int label = exact_label(w);
        p.labels[(int64_t)b * n + i] = label;
        if (p.prev_labels && p.prev_labels[(int64_t)b * n + i] != label) ++changed;
        for (int t = 0; t < D; ++t) atomicAdd(&s_acc[label * 5 + t], (w >> (8 * t)) & 255u);
        atomicAdd(&s_acc[label * 5 + 4], 1u);
    }
    __syncthreads();
    for (int e = tid; e < k * D; e += 256)
        partial[((int64_t)b * gridDim.x + blockIdx.x) * k * D + e] = (double)s_acc[(e >> 2) * 5 + (e & 3)];
    for (int j = tid; j < k; j += 256) cnt_partial[((int64_t)b * gridDim.x + blockIdx.x) * k + j] = (long long)s_acc[j * 5 + 4];
    if (p.n_changed && p.prev_labels) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
        if (lane == 0 && changed) atomicAdd(p.n_changed + b, (unsigned long long)changed);
    }
}

bool kmeans_step_u8d4_usable(const KmAssignParams& p, int batch) {
    if (p.dtype != DT_U8 || p.d != 4 || p.k < 1 || p.k > 8) return false;
    if (((uintptr_t)p.X & 15) || ((uintptr_t)p.labels & 15) || (p.prev_labels && ((uintptr_t)p.prev_labels & 15))) return false;
    return batch <= 1 || (p.n & 3) == 0;                           // else the next problem's rows would be misaligned
}

int launch_kmeans_step_u8d4(const KmAssignParams& p, int batch, int grid, double* partial, long long* cnt_partial, void* stream) {
    if (p.k <= 4) {
        OFC_LAUNCH(kmeans_step_u8d4_kernel<4>, dim3(grid, batch), dim3(256), 0, stream, p, partial, cnt_partial);
    } else {
        OFC_LAUNCH(kmeans_step_u8d4_kernel<8>, dim3(grid, batch), dim3(256), 0, stream, p, partial, cnt_partial);
    }
    OFC_CHECK_LAUNCH("kmeans_step_u8d4");
    return OFC_OK;
}

// shared memory of one CTA; *closest_in_smem says whether the k-means++ scratch fits as well
static size_t cells_fast_smem(int n, int kp, bool want_closest, int* closest_in_smem) {
    const size_t fixed = (size_t)(2 * kp * 4 + 2 * kp + 4 + 8) * 8 + 64 * 8 + (size_t)kp * 5 * 4 + (size_t)kp * 4 * 4 + (size_t)kp * 4 +
                         (size_t)kp * 3 * 4;
    const size_t rows = (size_t)n * 4 + ((size_t)n + 15) / 16 * 16;
    size_t with = fixed + rows + (size_t)n * 4;
    if (want_closest && with <= 100 * 1024) { *closest_in_smem = 1; return with; }
    *closest_in_smem = 0;
    return fixed + rows;
}

bool kmeans_cells_fast_supported(int64_t n, int d, int k) {
    int dummy;
    return d == 4 && k >= 1 && k <= 16 && n >= 1 && n <= (1 << 20) && cells_fast_smem((int)n, 16, false, &dummy) <= 200 * 1024;
}

size_t kmeans_cells_fast_workspace(int batch, int64_t n, int k, bool seeding) {
    int in_smem = 0;
    const int kp = k <= 4 ? 4 : (k <= 8 ? 8 : 16);
    cells_fast_smem((int)n, kp, seeding, &in_smem);
    return (seeding && !in_smem) ? (size_t)batch * n * 4 : 0;
}

int launch_kmeans_cells_fast(KmCellsFastParams p, int batch, void* stream) {
    if (batch <= 0) return OFC_OK;
    const int kp = p.k <= 4 ? 4 : (p.k <= 8 ? 8 : 16);
    int in_smem = 0;
    const size_t smem = cells_fast_smem(p.n, kp, p.init == nullptr, &in_smem);
    p.closest_in_smem = in_smem;
    if (p.init == nullptr && !in_smem && p.closest_ws == nullptr) {
        set_error("k-means++ seeding of %d-row cells needs %zu bytes of workspace", p.n, (size_t)batch * p.n * 4);
        return OFC_ERR_WORKSPACE;
    }
    ProfScope prof(PK_KMEANS, stream);
#define OFC_CELLS_FAST(KPV)                                                                     \
    {                                                                                           \
        OFC_SMEM_OPTIN((kmeans_cells_fast_kernel<KPV>), smem);                                  \
        OFC_LAUNCH((kmeans_cells_fast_kernel<KPV>), dim3(batch), dim3(256), smem, stream, p);   \
    }
    if (kp == 4) OFC_CELLS_FAST(4)
    else if (kp == 8) OFC_CELLS_FAST(8)
    else OFC_CELLS_FAST(16)
#undef OFC_CELLS_FAST
    OFC_CHECK_LAUNCH("kmeans_cells_fast");
    return OFC_OK;
}

}  // namespace ofc
