// Common definitions for the sm_100a kernels of libofc.
//
// Two build modes:
//   * nvcc -gencode arch=compute_100a,code=sm_100a  -> the product (libofc.so)
//   * g++ -DOFC_EMULATE -include tests/emu/cuda_emu.h -> a host-side *debug
//     emulation* of the same kernel sources (fibers standing in for CUDA
//     threads).  It exists only so kernel indexing can be debugged in a
//     container without a GPU; it is built and loaded by tests/ only and is
//     never reachable from the Python package (see tests/emu/README.md).
#pragma once

#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>

#ifndef OFC_EMULATE
#include <cuda_runtime.h>
#define OFC_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
#define OFC_DYN_SMEM(type, name) extern __shared__ __align__(16) unsigned char name##_raw_[]; \
    type* name = reinterpret_cast<type*>(name##_raw_)
#else
#define OFC_LAUNCH(kernel, grid, block, smem, stream, ...) \
    ofc_emu::launch((grid), (block), (smem), [=]() { kernel(__VA_ARGS__); })
#define OFC_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(ofc_emu::dyn_smem())
#endif

#define OFC_OK 0
#define OFC_ERR_INVALID (-1)
#define OFC_ERR_UNSUPPORTED (-2)
#define OFC_ERR_CUDA (-3)
#define OFC_ERR_WORKSPACE (-4)

namespace ofc {

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

#define OFC_CUDA(call)                                              \
    do {                                                            \
        int ofc_rc_ = ::ofc::check_cuda((call), #call);             \
        if (ofc_rc_ != OFC_OK) return ofc_rc_;                      \
    } while (0)

#define OFC_CHECK_LAUNCH(name) OFC_CUDA(cudaGetLastError())

// Opt a kernel in to more than 48 KB of dynamic shared memory.  The attribute is per device, so the
// "already done" cache is keyed by (current device, kernel) and guarded by a mutex: one process may
// drive several GPUs and several host threads may launch (ofc_api.cu).
int smem_optin(const void* kernel, size_t bytes);
#define OFC_SMEM_OPTIN(kernel, bytes)                                                   \
    do {                                                                                \
        if ((size_t)(bytes) > 48 * 1024) {                                              \
            int ofc_rc_ = ::ofc::smem_optin(reinterpret_cast<const void*>(kernel), (size_t)(bytes)); \
            if (ofc_rc_ != OFC_OK) return ofc_rc_;                                      \
        }                                                                               \
    } while (0)

#define OFC_REQUIRE(cond, ...)                                      \
    do {                                                            \
        if (!(cond)) {                                              \
            ::ofc::set_error(__VA_ARGS__);                          \
            return OFC_ERR_INVALID;                                 \
        }                                                           \
    } while (0)

// Optional per-kernel timing (ofc_profile_begin / ofc_profile_end in ofc.h): when
// enabled every launcher brackets its kernel with two cudaEvents on the launch
// stream.  Off by default; costs nothing then.
enum ProfKind {
    PK_GRAY = 0, PK_PREFILTER, PK_POLYEXP, PK_MINMAX_INIT, PK_ENCODE, PK_GRID, PK_FLOW_MINMAX, PK_DRAW,
    PK_KMEANS, PK_COSINE, PK_UPSAMPLE, PK_RESERVED1,
    PK_ITER_L0 = 12,             // flow_iter at full resolution; +1 per coarser level (up to 8)
    PK_COUNT = 20
};
struct ProfScope {
    int kind; void* stream; bool on; int index;
    ProfScope(int kind, void* stream);
    ~ProfScope();
};
extern int g_prof_level;         // pyramid level (0 = finest) of the flow_iter launch being issued

// Test seam (DESIGN §5a.5): true when the environment variable `name` is set to 0, which selects the form a fast
// kernel replaced and gives the same bits.  Read on every call, so one process can run and compare both forms.
static inline bool seam_off(const char* name) {
    const char* e = getenv(name);
    return e && atoi(e) == 0;
}

static inline double host_dmul(double a, double b) { volatile double r = a * b; return r; }
static inline double host_dadd(double a, double b) { volatile double r = a + b; return r; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__host__ __device__ __forceinline__ int clampi(int v, int lo, int hi) {
    return v < lo ? lo : (v > hi ? hi : v);
}

// BORDER_REFLECT_101 for |overshoot| < n (single reflection is enough on this
// path: the Gaussian radius is always smaller than the image).
__host__ __device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    const int p = 2 * (n - 1);
    i %= p;
    if (i < 0) i += p;
    return i >= n ? p - i : i;
}

// same map for -n < i < 2n-1 without the modulo (n >= 2)
__host__ __device__ __forceinline__ int reflect101_near(int i, int n) {
    return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i);
}

// Squared norm of a float64 centre in the summation order of numpy's einsum("ij,ij->i"), which is what scikit-learn's
// row_norms(centers, squared=True) evaluates (sklearn/utils/extmath.py; numpy einsum_sumprod, 128-bit lanes on x86-64:
// two interleaved partial sums, four vectors per unrolled step accumulated from the last to the first, products and
// sums rounded separately -- no fma).  Verified bit for bit against numpy 2.3 for d = 1 .. 100.  It matters on integer
// lattice data (uint8 rows with few features), where rows sit EXACTLY on bisectors and the last bit of ||c||^2 decides
// the label: with a sequential fma chain 31 of 20 000 labels of the d = 2 sklearn golden flip.
__host__ __device__ __forceinline__ double norm_sq_numpy_f64(const double* c, int d) {
#ifdef __CUDA_ARCH__
#define OFC_DMUL(a, b) __dmul_rn((a), (b))
#define OFC_DADD(a, b) __dadd_rn((a), (b))
#else
#define OFC_DMUL(a, b) ::ofc::host_dmul((a), (b))
#define OFC_DADD(a, b) ::ofc::host_dadd((a), (b))
#endif
    double v0 = 0.0, v1 = 0.0;
    int i = 0;
    for (; d - i >= 8; i += 8) {
        v0 = OFC_DADD(OFC_DMUL(c[i], c[i]), OFC_DADD(OFC_DMUL(c[i + 2], c[i + 2]), OFC_DADD(OFC_DMUL(c[i + 4], c[i + 4]),
                                                                                         OFC_DADD(OFC_DMUL(c[i + 6], c[i + 6]), v0))));
        v1 = OFC_DADD(OFC_DMUL(c[i + 1], c[i + 1]), OFC_DADD(OFC_DMUL(c[i + 3], c[i + 3]), OFC_DADD(OFC_DMUL(c[i + 5], c[i + 5]),
                                                                                                 OFC_DADD(OFC_DMUL(c[i + 7], c[i + 7]), v1))));
    }
    for (; i < d; i += 2) {
        v0 = OFC_DADD(OFC_DMUL(c[i], c[i]), v0);
        if (i + 1 < d) v1 = OFC_DADD(OFC_DMUL(c[i + 1], c[i + 1]), v1);
    }
    return OFC_DADD(v0, v1);
#undef OFC_DMUL
#undef OFC_DADD
}

// byte T of a word as a float without an integer->float conversion: 0x4B0000bb is 2^23 + bb
template <int T> __device__ __forceinline__ float byte_to_float(unsigned w) {
#ifndef OFC_EMULATE
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540 + T)) - 8388608.f;
#else
    return (float)((w >> (8 * T)) & 255u);
#endif
}

}  // namespace ofc
