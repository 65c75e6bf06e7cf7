// k-means for the dense corner (float32 rows, d >= 32, k >= 16): the E-step's distance matrix
// is a real GEMM there (2 n k d flop against n d bytes, SURVEY.md section 8d), so it runs on the
// 5th-generation tensor cores; the M-step walks a label-sorted (CSR) member list.
//
// Replaces, for that shape, the arithmetic behind the reference's
//   clt = KMeans(n_clusters = k); clt.fit(X); clt.predict(X)
// (reference k-means-color-clustering/KmeanGrids.py:299-304, color_kmeans.py:65-78): scikit-learn's
// Lloyd E-step  label = first strict minimum over j of ||c_j||^2 - 2 x.c_j  (_k_means_lloyd.pyx:196-213).
//
// E-step (kmeans_assign_tc_kernel), one persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer: 128 x 32 float tiles of the rows (A hi, A lo) and BN x 32 tiles of the centres
//               (B hi, B lo) into a shared-memory ring (128-byte swizzle, mbarrier complete_tx);
//   warp 1      one elected thread issues tcgen05.mma.kind::tf32 (M = 128, N = BN, K = 8) with the
//               128 x BN float32 accumulator in tensor memory; two accumulators (2 x BN <= 512 columns)
//               so the epilogue of one tile overlaps the MMAs of the next;
//   warps 2..9  epilogue: tcgen05.ld of the accumulator (one row per thread, two warp sets splitting the
//               columns, next chunk in flight while one is scanned), dist = c2 - 2 acc, running minimum plus
//               a short history of the near-minimum distances per row.
// TF32 keeps 10 mantissa bits, so every operand is split once into hi = its top 11 significant bits
// and lo = the exact remainder (x = hi + lo, both float32), and x.c is formed as lo.hi + hi.lo + hi.hi
// -- three MMAs per step ("3xTF32"), the hi parts exact in TF32 whatever the hardware does with the low
// bits.  What is left (the lo.lo term, the TF32 image of the lo parts, float32 accumulation) is bounded
// by (2^-19 + d 2^-23) |x| |c| per dot product, and the tensor-core distances only FILTER: a row whose
// two best distances are further apart than that bound keeps its arg-min; every other row is appended
// to a list and re-evaluated by kmeans_assign_fix_kernel in exactly the float32 arithmetic of
// kmeans_assign_generic_kernel (the two or three centres inside the bound; all k when there are more).  Labels are therefore bit-identical to the CUDA-core float32 path.
//
// GPU only (no host-side emulation: tests/emu skips tc_*.cu).
#include <cuda.h>
#include <stdlib.h>
#include "ofc_common.cuh"
#include "../../include/ofc.h"

namespace ofc {
namespace {

constexpr int BM = 128;          // rows per tile (= TMEM lanes)
constexpr int BK = 32;           // floats per shared-memory row: 128 bytes = one swizzle atom
constexpr int TC_THREADS = 320;      // TMA warp, MMA warp, 2 x 4 epilogue warps

struct TcParams {
    int64_t n;
    int d, k;
    const float* c2;             // [k] squared norms of the float32 centres
    const float* xnorm;          // [n] row norms
    const float* cmax;           // [1] largest centre norm
    float tol_scale;             // bound on |TF32 distance difference error| / (|x| cmax)
    float tol_c2;                // ... plus this times cmax^2 (rounding of the squared norms; uint8 path only)
    int32_t* labels;
    int4* amb;                   // [n] (row, best, second, third | candidates << 16) of rows to re-evaluate
    unsigned* amb_count;
    unsigned* error_flag;
    int stages;                  // ring depth (centre-resident form: row stages only)
    unsigned tile_bytes;         // shared memory taken by the operand tiles (ring [+ resident centres])
};

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol bug must not hang the GPU -- after ~4 s the kernel flags the error and traps.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity, unsigned* error_flag) {
    unsigned ok = 0;
    long long t0 = 0;
    for (unsigned spin = 0;; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) return;
        if ((spin & 1023u) == 1023u) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 8000000000ll) {
                if (error_flag) atomicExch(error_flag, 1u + bar);
                __trap();
            }
        }
    }
}
__device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                 "l"(map), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void umma_tf32(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// issue only: the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld32_issue(unsigned taddr, unsigned (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, rows of 128 bytes, 128-byte swizzle (what TMA writes with SWIZZLE_128B):
// 8-row groups 1024 bytes apart (SBO), LBO unused, descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t make_desc_sw128(unsigned addr) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

template <int BN> struct TcCfg {
    static constexpr unsigned A_BYTES = BM * BK * 4, B_BYTES = BN * BK * 4, STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int STAGES = BN == 256 ? 2 : (BN == 128 ? 3 : 4);
};

// BRES (k <= BN and few K-steps): the centre tiles (hi and lo, every K-step) are loaded ONCE and stay resident in
// shared memory; the ring then only carries the rows, a third of the bytes per row block -- the small-d corner is
// bound by the latency of refilling the ring, not by the tensor cores.
constexpr int MAX_STAGES = 8;

template <int BN, bool BRES>
__global__ void __launch_bounds__(TC_THREADS, 1)
kmeans_assign_tc_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                        const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl, TcParams p) {
    constexpr unsigned A_BYTES = TcCfg<BN>::A_BYTES, B_BYTES = TcCfg<BN>::B_BYTES;
    constexpr unsigned STAGE_BYTES = BRES ? 2 * A_BYTES : TcCfg<BN>::STAGE_BYTES;
    const int STAGES = p.stages;
    // instruction descriptor: D = f32, A = B = tf32, both K-major, N = BN, M = 128
    constexpr unsigned IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(BN >> 3) << 17) | ((unsigned)(BM >> 4) << 24);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.tile_bytes);
    // bars: full[MAX_STAGES], empty[MAX_STAGES], tfull[2], tempty[2], bfull
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * MAX_STAGES + 5);
    const unsigned bar0 = smem_addr(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (MAX_STAGES + s); };
    auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * MAX_STAGES + a); };
    auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * MAX_STAGES + 2 + a); };
    const unsigned bfull_bar = bar0 + 8u * (2 * MAX_STAGES + 4);
    unsigned char* bres = smem + (size_t)STAGES * STAGE_BYTES;          // resident centre tiles (BRES)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_mtiles = (int)((p.n + BM - 1) / BM);
    const int n_ntiles = (p.k + BN - 1) / BN;
    const int n_ktiles = (p.d + BK - 1) / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
        mbar_init(bfull_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            if (BRES) {
                mbar_expect_tx(bfull_bar, (unsigned)n_ktiles * 2u * B_BYTES);
                for (int kt = 0; kt < n_ktiles; ++kt) {
                    const unsigned b_dst = smem_addr(bres + (size_t)kt * 2 * B_BYTES);
                    tma_load_2d(b_dst, &tmBh, bfull_bar, kt * BK, 0);
                    tma_load_2d(b_dst + B_BYTES, &tmBl, bfull_bar, kt * BK, 0);
                }
            }
            unsigned it = 0;
            for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x)
                for (int nt = 0; nt < n_ntiles; ++nt)
                    for (int kt = 0; kt < n_ktiles; ++kt, ++it) {
                        const int s = it % STAGES;
                        const unsigned ph = (it / STAGES) & 1u;
                        mbar_wait(empty_bar(s), ph ^ 1u, p.error_flag);
                        mbar_expect_tx(full_bar(s), STAGE_BYTES);
                        const unsigned a_dst = smem_addr(smem + (size_t)s * STAGE_BYTES);
                        tma_load_2d(a_dst, &tmAh, full_bar(s), kt * BK, mt * BM);
                        tma_load_2d(a_dst + A_BYTES, &tmAl, full_bar(s), kt * BK, mt * BM);
                        if (!BRES) {
                            tma_load_2d(a_dst + 2 * A_BYTES, &tmBh, full_bar(s), kt * BK, nt * BN);
                            tma_load_2d(a_dst + 2 * A_BYTES + B_BYTES, &tmBl, full_bar(s), kt * BK, nt * BN);
                        }
                    }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            unsigned it = 0, unit = 0;
            if (BRES) { mbar_wait(bfull_bar, 0u, p.error_flag); tc_fence_after(); }
            for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x)
                for (int nt = 0; nt < n_ntiles; ++nt, ++unit) {
                    const unsigned acc = unit & 1u, aph = (unit >> 1) & 1u;
                    mbar_wait(tempty_bar(acc), aph ^ 1u, p.error_flag);
                    tc_fence_after();
                    const unsigned tmem_d = tmem_base + acc * BN;
                    for (int kt = 0; kt < n_ktiles; ++kt, ++it) {
                        const int s = it % STAGES;
                        const unsigned ph = (it / STAGES) & 1u;
                        mbar_wait(full_bar(s), ph, p.error_flag);
                        tc_fence_after();
                        const unsigned a_addr = smem_addr(smem + (size_t)s * STAGE_BYTES);
                        const uint64_t ah = make_desc_sw128(a_addr), al = make_desc_sw128(a_addr + A_BYTES);
                        const unsigned b_addr = BRES ? smem_addr(bres + (size_t)kt * 2 * B_BYTES) : a_addr + 2 * A_BYTES;
                        const uint64_t bh = make_desc_sw128(b_addr), bl = make_desc_sw128(b_addr + B_BYTES);
#pragma unroll
                        for (int k4 = 0; k4 < BK / 8; ++k4) {    // 8 floats = 32 bytes per MMA: +2 in 16-byte units
                            umma_tf32(tmem_d, al + 2u * k4, bh + 2u * k4, IDESC, (kt | k4) != 0);
                            umma_tf32(tmem_d, ah + 2u * k4, bl + 2u * k4, IDESC, 1u);
                            umma_tf32(tmem_d, ah + 2u * k4, bh + 2u * k4, IDESC, 1u);
                        }
                        umma_commit(empty_bar(s));               // frees the stage once these MMAs have read it
                    }
                    umma_commit(tfull_bar(acc));
                }
        }
    } else {
        // Epilogue: warps 2..5 take the even 32-column chunks of every accumulator, warps 6..9 the odd ones (a warp
        // may only read the TMEM lane quarter warp % 4, so the two sets cover the same 128 rows); each thread keeps a
        // running minimum (first strict minimum in centre order) plus a four-deep history of every distance that
        // came within the row's error bound of its running minimum: whatever ends within the bound of the FINAL
        // minimum is in a history unless it was pushed out while still eligible (`lost`).  The odd set hands its
        // state over through shared memory at the end of the row block and the even set decides.
        const int q = warp & 3;                                   // TMEM lane quarter this warp may read
        const int half = warp >= 6 ? 1 : 0;
        const float cmax = __ldg(p.cmax);
        float* xch = reinterpret_cast<float*>(tmem_slot + 4);     // [128][12] hand-over
        unsigned unit = 0;
        for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x) {
            const int64_t row = (int64_t)mt * BM + q * 32 + lane;
            const float tol = p.tol_scale * __ldg(p.xnorm + (row < p.n ? row : p.n - 1)) * cmax + p.tol_c2 * cmax * cmax;
            float m1 = __int_as_float(0x7f800000), thr = m1;
            int a1 = 0x7fffffff;
            float h0 = m1, h1 = m1, h2 = m1, h3 = m1;
            int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
            bool lost = false;
            for (int nt = 0; nt < n_ntiles; ++nt, ++unit) {
                const unsigned acc = unit & 1u, aph = (unit >> 1) & 1u;
                mbar_wait(tfull_bar(acc), aph, p.error_flag);
                tc_fence_after();
                const unsigned trow = tmem_base + acc * BN + ((unsigned)(q * 32) << 16);
                // two register buffers, statically named: the next chunk of this warp is in flight while one is scanned
                unsigned bufA[32], bufB[32];
                constexpr int NCH = BN / 32;
                auto scan = [&](const unsigned (&buf)[32], int j0) {
                    const float4* c2v = reinterpret_cast<const float4*>(p.c2 + j0);   // padded with +inf past k
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4) {
                        const float4 cc = __ldg(c2v + g4);
                        const float cj[4] = {cc.x, cc.y, cc.z, cc.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float dist = fmaf(-2.f, __uint_as_float(buf[g4 * 4 + e]), cj[e]);
                            if (dist <= thr) {
                                const int j = j0 + g4 * 4 + e;
                                const float out = h3;
                                h3 = h2; i3 = i2; h2 = h1; i2 = i1; h1 = h0; i1 = i0; h0 = dist; i0 = j;
                                if (dist < m1) { m1 = dist; a1 = j; thr = dist + tol; }
                                lost = lost || out <= thr;
                            }
                        }
                    }
                };
                const int jt = nt * BN;
                int c = half;
                if (c < NCH && jt + c * 32 < p.k) tmem_ld32_issue(trow + c * 32, bufA);
                tmem_ld_wait();
#pragma unroll 1
                while (c < NCH && jt + c * 32 < p.k) {
                    if (c + 2 < NCH && jt + (c + 2) * 32 < p.k) tmem_ld32_issue(trow + (c + 2) * 32, bufB);
                    scan(bufA, jt + c * 32);
                    tmem_ld_wait();
                    c += 2;
                    if (!(c < NCH && jt + c * 32 < p.k)) break;
                    if (c + 2 < NCH && jt + (c + 2) * 32 < p.k) tmem_ld32_issue(trow + (c + 2) * 32, bufA);
                    scan(bufB, jt + c * 32);
                    tmem_ld_wait();
                    c += 2;
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(acc));
            }
            // hand-over of the odd set's state; named barrier 1 over the 256 epilogue threads
            float* slot = xch + (q * 32 + lane) * 12;
            if (half) {
                slot[0] = m1; slot[1] = __int_as_float(a1); slot[2] = lost ? 1.f : 0.f;
                slot[3] = h0; slot[4] = __int_as_float(i0); slot[5] = h1; slot[6] = __int_as_float(i1);
                slot[7] = h2; slot[8] = __int_as_float(i2); slot[9] = h3; slot[10] = __int_as_float(i3);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (!half && row < p.n) {
                const float om1 = slot[0];
                const int oa1 = __float_as_int(slot[1]);
                const float oh[4] = {slot[3], slot[5], slot[7], slot[9]};
                const int oi[4] = {__float_as_int(slot[4]), __float_as_int(slot[6]), __float_as_int(slot[8]), __float_as_int(slot[10])};
                lost = lost || slot[2] != 0.f;
                // first strict minimum over both halves: the lower centre index wins a tie
                if (om1 < m1 || (om1 == m1 && oa1 < a1)) { m1 = om1; a1 = oa1; }
                thr = m1 + tol;
                p.labels[row] = a1;
                // the other centres inside the bound of the final minimum
                int cand[8], nc = 0;
                if (i0 != a1 && h0 <= thr) cand[nc++] = i0;
                if (i1 != a1 && h1 <= thr) cand[nc++] = i1;
                if (i2 != a1 && h2 <= thr) cand[nc++] = i2;
                if (i3 != a1 && h3 <= thr) cand[nc++] = i3;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (oi[u] != a1 && oh[u] <= thr) cand[nc++] = oi[u];
                if (nc > 0 || lost || !(m1 < __int_as_float(0x7f800000))) {
                    // 2 or 3 candidates are listed; otherwise (0) all k centres are re-evaluated
                    const int ncand = (lost || nc > 2 || nc == 0) ? 0 : nc + 1;
                    const unsigned pos = atomicAdd(p.amb_count, 1u);
                    p.amb[pos] = make_int4((int)row, a1, nc > 0 ? cand[0] : 0, (nc > 1 ? cand[1] : 0) | (ncand << 16));
                }
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");      // the slots are free for the next row block
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}

// one float32 distance in the arithmetic of kmeans_assign_generic_kernel<float, float>: lanes stride over
// the features, xor-tree reduction, dist = fma(-2, dot, c2)
__device__ __forceinline__ float exact_dist(const float* __restrict__ x, const float* __restrict__ c, float c2, int d, int lane) {
    float part = 0.f;
    for (int t = lane; t < d; t += 32) part = fmaf(x[t], c[t], part);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    return fmaf(-2.f, part, c2);
}

// rows the tensor-core filter could not decide: one warp per row; the row (hi + lo, exactly the centred
// float32 row) is staged once in the warp's slice of shared memory when it fits
__global__ void __launch_bounds__(256) kmeans_assign_fix_kernel(const float* __restrict__ Xh, const float* __restrict__ Xl, int d, int k,
                                                                const float* __restrict__ C, const float* __restrict__ c2,
                                                                const int4* __restrict__ amb, const unsigned* __restrict__ amb_count,
                                                                int32_t* __restrict__ labels, float* __restrict__ row_ws, int use_smem) {
    OFC_DYN_SMEM(float, s_rows);                     // [8][d] when use_smem
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned n_amb = *amb_count;
    float* x = use_smem ? s_rows + (size_t)warp * d : row_ws + ((size_t)blockIdx.x * 8 + warp) * d;
    for (unsigned e = blockIdx.x * 8 + warp; e < n_amb; e += gridDim.x * 8) {
        const int4 a = amb[e];
        const float* rh = Xh + (int64_t)a.x * d;
        const float* rl = Xl + (int64_t)a.x * d;
        __syncwarp();
        for (int t = lane; t < d; t += 32) x[t] = rh[t] + rl[t];
        __syncwarp();
        int label;
        const int ncand = a.w >> 16;
        if (ncand) {
            // first strict minimum in ascending centre order over the listed candidates
            int c0 = a.y, c1 = a.z, c2i = ncand == 3 ? (a.w & 0xffff) : 0x7fffffff, t;
            if (c1 < c0) { t = c0; c0 = c1; c1 = t; }
            if (c2i < c1) { t = c1; c1 = c2i; c2i = t; }
            if (c1 < c0) { t = c0; c0 = c1; c1 = t; }
            float best = exact_dist(x, C + (int64_t)c0 * d, c2[c0], d, lane);
            label = c0;
            const float d1 = exact_dist(x, C + (int64_t)c1 * d, c2[c1], d, lane);
            if (d1 < best) { best = d1; label = c1; }
            if (ncand == 3) {
                const float d2 = exact_dist(x, C + (int64_t)c2i * d, c2[c2i], d, lane);
                if (d2 < best) { best = d2; label = c2i; }
            }
        } else {
            float best = 0.f;
            label = 0;
            for (int j = 0; j < k; ++j) {
                const float dist = exact_dist(x, C + (int64_t)j * d, c2[j], d, lane);
                if (j == 0 || dist < best) { best = dist; label = j; }
            }
        }
        if (lane == 0) labels[a.x] = label;
    }
}

// hi = the top 11 significant bits (exact in TF32), lo = the exact remainder
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    lo = v - hi;
}

// uint8 rows (worked in float64 by sklearn and by ofc_kmeans_assign(OFC_U8)): the same re-evaluation in the
// float64 arithmetic of kmeans_assign_generic_kernel<unsigned char, double> on the ORIGINAL bytes
__device__ __forceinline__ double exact_dist64(const double* __restrict__ x, const double* __restrict__ c, double c2, int d, int lane) {
    double part = 0.0;
    for (int t = lane; t < d; t += 32) part = fma(x[t], c[t], part);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    return fma(-2.0, part, c2);
}

__global__ void __launch_bounds__(256) kmeans_assign_fix_u8_kernel(const unsigned char* __restrict__ X, const double* __restrict__ mean, int d,
                                                                   int k, const double* __restrict__ C, const double* __restrict__ c2,
                                                                   const int4* __restrict__ amb, const unsigned* __restrict__ amb_count,
                                                                   int32_t* __restrict__ labels, double* __restrict__ row_ws, int use_smem) {
    OFC_DYN_SMEM(double, s_rows);                    // [8][d] when use_smem
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned n_amb = *amb_count;
    double* x = use_smem ? s_rows + (size_t)warp * d : row_ws + ((size_t)blockIdx.x * 8 + warp) * d;
    for (unsigned e = blockIdx.x * 8 + warp; e < n_amb; e += gridDim.x * 8) {
        const int4 a = amb[e];
        const unsigned char* row = X + (int64_t)a.x * d;
        __syncwarp();
        for (int t = lane; t < d; t += 32) x[t] = (double)row[t] - (mean ? mean[t] : 0.0);
        __syncwarp();
        int label;
        const int ncand = a.w >> 16;
        if (ncand) {
            int c0 = a.y, c1 = a.z, c2i = ncand == 3 ? (a.w & 0xffff) : 0x7fffffff, t;
            if (c1 < c0) { t = c0; c0 = c1; c1 = t; }
            if (c2i < c1) { t = c1; c1 = c2i; c2i = t; }
            if (c1 < c0) { t = c0; c0 = c1; c1 = t; }
            double best = exact_dist64(x, C + (int64_t)c0 * d, c2[c0], d, lane);
            label = c0;
            const double d1 = exact_dist64(x, C + (int64_t)c1 * d, c2[c1], d, lane);
            if (d1 < best) { best = d1; label = c1; }
            if (ncand == 3) {
                const double d2 = exact_dist64(x, C + (int64_t)c2i * d, c2[c2i], d, lane);
                if (d2 < best) { best = d2; label = c2i; }
            }
        } else {
            double best = 0.0;
            label = 0;
            for (int j = 0; j < k; ++j) {
                const double dist = exact_dist64(x, C + (int64_t)j * d, c2[j], d, lane);
                if (j == 0 || dist < best) { best = dist; label = j; }
            }
        }
        if (lane == 0) labels[a.x] = label;
    }
}

// c2 in float64 in the order of kmeans_c2_kernel (numpy's einsum order, norm_sq_numpy_f64) for the re-evaluation, and its float32
// image (padded with +inf) for the tensor-core epilogue
__global__ void centres_c2_f64_kernel(const double* __restrict__ c, double* __restrict__ c2d, float* __restrict__ c2f, int d, int k,
                                      int k_pad) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) {
        if (j < k_pad) c2f[j] = __int_as_float(0x7f800000);
        return;
    }
    const double* r = c + (int64_t)j * d;
    const double s = norm_sq_numpy_f64(r, d);
    c2d[j] = s;
    c2f[j] = (float)s;
}

// uint8 rows: xc = float32(x - mean) with the float64 column mean (KMeans.fit works uint8 data in float64)
__global__ void __launch_bounds__(256) prepare_rows_u8_kernel(const unsigned char* __restrict__ X, const double* __restrict__ mean, int64_t n,
                                                              int d, float* __restrict__ Xh, float* __restrict__ Xl,
                                                              float* __restrict__ xnorm) {
    const int lane = threadIdx.x & 31;
    for (int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); i < n; i += (int64_t)gridDim.x * 8) {
        const unsigned char* row = X + i * d;
        float s = 0.f;
        for (int t = lane; t < d; t += 32) {
            const float v = (float)((double)row[t] - (mean ? mean[t] : 0.0));
            split_tf32(v, Xh[i * d + t], Xl[i * d + t]);
            s = fmaf(v, v, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) xnorm[i] = sqrtf(s);
    }
}

// centres f64 -> f32 copy and its hi / lo split (the B operands)
__global__ void centres_to_f32_kernel(const double* __restrict__ c, float* __restrict__ out, float* __restrict__ hi, float* __restrict__ lo,
                                      int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = (float)c[i];
        out[i] = v;
        split_tf32(v, hi[i], lo[i]);
    }
}
// c2[j] in the order of kmeans_c2_kernel(as_float): sequential fma chain over the features
__global__ void centres_c2_kernel(const float* __restrict__ c, float* __restrict__ c2, int d, int k, int k_pad) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) {
        if (j < k_pad) c2[j] = __int_as_float(0x7f800000);       // past the last centre: never the minimum
        return;
    }
    const float* r = c + (int64_t)j * d;
    float s = 0.f;
    for (int t = 0; t < d; ++t) s = fmaf(r[t], r[t], s);
    c2[j] = s;
}
__global__ void __launch_bounds__(1024) centres_cmax_kernel(const float* __restrict__ c2, int k, float* __restrict__ cmax,
                                                             unsigned* __restrict__ amb_count) {
    __shared__ float s[32];
    float m = 0.f;
    for (int j = threadIdx.x; j < k; j += 1024) m = fmaxf(m, c2[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) m = fmaxf(m, s[w]);
        *cmax = sqrtf(m);
        *amb_count = 0u;
    }
}

// xc = float32(x - float32 mean) (KMeans.fit centres float32 data in float32, _kmeans.py:1487-1493), stored as
// its hi / lo split, and the row norms the tensor-core filter's error bound needs; one warp per row
__global__ void __launch_bounds__(256) prepare_rows_kernel(const float* __restrict__ X, const double* __restrict__ mean, int64_t n,
                                                           int d, float* __restrict__ Xh, float* __restrict__ Xl, float* __restrict__ xnorm) {
    const int lane = threadIdx.x & 31;
    for (int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); i < n; i += (int64_t)gridDim.x * 8) {
        const float* row = X + i * d;
        float s = 0.f;
        for (int t = lane; t < d; t += 32) {
            const float v = row[t] - (mean ? (float)mean[t] : 0.f);
            split_tf32(v, Xh[i * d + t], Xl[i * d + t]);
            s = fmaf(v, v, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) xnorm[i] = sqrtf(s);
    }
}

__global__ void __launch_bounds__(256) labels_changed_kernel(const int32_t* __restrict__ a, const int32_t* __restrict__ b, int64_t n,
                                                             unsigned long long* __restrict__ n_changed) {
    unsigned c = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) c += a[i] != b[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(n_changed, (unsigned long long)c);     // integers: order-free
}

// inertia partials: sum over the rows of a CTA of ||x - c_label||^2 (float32 per row like the assign kernels,
// float64 across rows), one warp per row, fixed order inside the CTA; folded in CTA order afterwards.
// WT: each row's term times its weight (unit weights give the unweighted bits)
template <bool WT>
__global__ void __launch_bounds__(256) inertia_rows_kernel(const float* __restrict__ Xh, const float* __restrict__ Xl, int64_t n, int d,
                                                           const float* __restrict__ C, const int32_t* __restrict__ labels,
                                                           const double* __restrict__ weights, double* __restrict__ partial) {
    __shared__ double s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * 8 + warp; i < n; i += (int64_t)gridDim.x * 8) {
        const float* rh = Xh + i * d;
        const float* rl = Xl + i * d;
        const float* c = C + (int64_t)labels[i] * d;
        float sq = 0.f;
        for (int t = lane; t < d; t += 32) { const float df = (rh[t] + rl[t]) - c[t]; sq = fmaf(df, df, sq); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        acc += WT ? (double)sq * weights[i] : (double)sq;
    }
    if (lane == 0) s_w[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_w[w];
        partial[blockIdx.x] = t;
    }
}
__global__ void fold_partials_kernel(const double* __restrict__ partial, int parts, double* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < parts; ++i) s += partial[i];
        *out = s;
    }
}

// ---------------------------------------------------------------------------
// M-step over a label-sorted member list (deterministic, no floating-point atomics).
//   1  csr_hist:    one warp per chunk of 1024 consecutive rows counts its labels (shared-memory table)
//   2  csr_scan:    per cluster, running start of every chunk's members; clusters laid end to end;
//                   every cluster's list is cut into segments of SEG members
//   3  csr_scatter: the same walk as (1) writes the row indices -- ascending inside every cluster
//   4  seg_sums:    grid (segment, 128-feature tile): float64 sums of the segment's rows, in list order
//   5  seg_fold:    sums[j][t] = the cluster's segment partials in order; counts[j]
// Weighted (WT, _k_means_lloyd.pyx:216-218): every row adds x w, and one more column (t == d) sums the weights, folded
// into weight_sums[j]; same list order, so unit weights give the unweighted bits.
// ---------------------------------------------------------------------------
constexpr int CHUNK = 1024;
constexpr int SEG = 512;

template <bool SCATTER>
__global__ void __launch_bounds__(256) csr_walk_kernel(const int32_t* __restrict__ labels, int64_t n, int k, unsigned* __restrict__ table,
                                                       int32_t* __restrict__ order) {
    extern __shared__ unsigned s_cnt[];              // [8][k]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t chunk = (int64_t)blockIdx.x * 8 + warp;
    const int64_t lo = chunk * CHUNK;
    unsigned* cnt = s_cnt + (size_t)warp * k;
    unsigned* tab = table + chunk * k;
    if (lo < n) {
        for (int j = lane; j < k; j += 32) cnt[j] = SCATTER ? tab[j] : 0u;
    }
    __syncwarp();
    if (lo >= n) return;
    const int64_t hi = lo + CHUNK < n ? lo + CHUNK : n;
    for (int64_t base = lo; base < hi; base += 32) {
        const int64_t i = base + lane;
        const bool ok = i < hi;
        const int l = ok ? labels[i] : -1 - lane;                        // distinct dummies for idle lanes
        const unsigned peers = __match_any_sync(0xffffffffu, l);
        const int leader = __ffs(peers) - 1;
        unsigned start = 0;
        if (ok && lane == leader) { start = cnt[l]; cnt[l] = start + __popc(peers); }
        start = __shfl_sync(0xffffffffu, start, leader);
        if (SCATTER && ok) order[start + __popc(peers & ((1u << lane) - 1u))] = (int32_t)i;
        __syncwarp();
    }
    if (!SCATTER)
        for (int j = lane; j < k; j += 32) tab[j] = cnt[j];
}

// table[chunk][j] (counts) -> absolute start of chunk's members of cluster j in `order`; counts[j];
// seg_info[s] = (cluster, begin, end) for every segment; seg_first[j] = first segment of cluster j.
// One CTA: G = 1024 / k thread groups split the chunk range (G = 1 for k >= 1024).
__global__ void __launch_bounds__(1024) csr_scan_kernel(unsigned* __restrict__ table, int64_t n_chunks, int k, long long* __restrict__ counts,
                                                        int* __restrict__ seg_first, int4* __restrict__ seg_info, int* __restrict__ n_segs) {
    extern __shared__ unsigned s_scan[];             // [G][k] group totals, [k] cluster offsets, [k] first segments
    const int G = k >= 1024 ? 1 : 1024 / k;
    unsigned* s_tot = s_scan;
    unsigned* s_off = s_scan + (size_t)G * k;
    unsigned* s_seg = s_off + k;
    const int64_t per = (n_chunks + G - 1) / G;
    for (int e = threadIdx.x; e < G * k; e += 1024) {
        const int g = e / k, j = e - g * k;
        const int64_t c0 = g * per, c1 = c0 + per < n_chunks ? c0 + per : n_chunks;
        unsigned run = 0;
        for (int64_t c = c0; c < c1; ++c) run += table[c * k + j];
        s_tot[e] = run;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += 1024) {
        unsigned run = 0;
        for (int g = 0; g < G; ++g) { const unsigned v = s_tot[g * k + j]; s_tot[g * k + j] = run; run += v; }
        counts[j] = run;
        s_off[j] = run;                              // cluster size for now
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned off = 0, segs = 0;
        for (int j = 0; j < k; ++j) {
            const unsigned c = s_off[j];
            s_off[j] = off; off += c;
            s_seg[j] = segs; seg_first[j] = (int)segs; segs += (c + SEG - 1) / SEG;
        }
        seg_first[k] = (int)segs;
        *n_segs = (int)segs;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < G * k; e += 1024) {
        const int g = e / k, j = e - g * k;
        const int64_t c0 = g * per, c1 = c0 + per < n_chunks ? c0 + per : n_chunks;
        unsigned run = s_off[j] + s_tot[e];
        for (int64_t c = c0; c < c1; ++c) { const unsigned v = table[c * k + j]; table[c * k + j] = run; run += v; }
    }
    for (int j = threadIdx.x; j < k; j += 1024) {
        const unsigned off = s_off[j], c = (unsigned)counts[j];
        const unsigned ns = (c + SEG - 1) / SEG;
        for (unsigned s = 0; s < ns; ++s) {
            const unsigned b = off + s * SEG, e = (s + 1) * SEG < c ? off + (s + 1) * SEG : off + c;
            seg_info[s_seg[j] + s] = make_int4(j, (int)b, (int)e, 0);
        }
    }
}

// uint8 rows: sums of the raw bytes (exact integers in float64, what ofc_kmeans_sums gives for OFC_U8); weighted: float64
// sums of x w in list order (exact for integer weights while the sums stay below 2^53)
template <bool WT>
__global__ void __launch_bounds__(128) seg_sums_u8_kernel(const unsigned char* __restrict__ X, int d, const int32_t* __restrict__ order,
                                                          const int4* __restrict__ seg_info, const int* __restrict__ n_segs,
                                                          const double* __restrict__ weights, double* __restrict__ partial) {
    const int t = blockIdx.y * 128 + threadIdx.x;
    for (int s = blockIdx.x; s < *n_segs; s += gridDim.x) {
        const int4 si = seg_info[s];
        if constexpr (WT) {
            if (t <= d) {
                double acc = 0.0;
                for (int m = si.y; m < si.z; ++m) {
                    const int64_t r = order[m];
                    acc += t == d ? weights[r] : (double)X[r * d + t] * weights[r];
                }
                partial[(int64_t)s * (d + 1) + t] = acc;
            }
        } else if (t < d) {
            unsigned long long acc = 0;
            int m = si.y;
            for (; m + 4 <= si.z; m += 4) {
                const unsigned v0 = X[(int64_t)order[m] * d + t], v1 = X[(int64_t)order[m + 1] * d + t];
                const unsigned v2 = X[(int64_t)order[m + 2] * d + t], v3 = X[(int64_t)order[m + 3] * d + t];
                acc += v0 + v1 + v2 + v3;
            }
            for (; m < si.z; ++m) acc += X[(int64_t)order[m] * d + t];
            partial[(int64_t)s * d + t] = (double)acc;
        }
    }
}

template <bool WT>
__global__ void __launch_bounds__(128) seg_sums_kernel(const float* __restrict__ Xh, const float* __restrict__ Xl, int d,
                                                       const int32_t* __restrict__ order,
                                                       const int4* __restrict__ seg_info, const int* __restrict__ n_segs,
                                                       const double* __restrict__ weights, double* __restrict__ partial) {
    const int t = blockIdx.y * 128 + threadIdx.x;
    const int dp = WT ? d + 1 : d;                   // partial columns: the features (+ the weight)
    // one member's term: x (h + l exactly), x w, or (column d) w
    auto term = [&](int64_t r) -> double {
        if (WT && t == d) return weights[r];
        const int64_t o = r * d + t;
        const double x = (double)(Xh[o] + Xl[o]);
        return WT ? x * weights[r] : x;
    };
    for (int s = blockIdx.x; s < *n_segs; s += gridDim.x) {
        const int4 si = seg_info[s];
        double acc = 0.0;
        if (t < dp) {
            int m = si.y;
            for (; m + 4 <= si.z; m += 4) {
                const double a0 = term(order[m]), a1 = term(order[m + 1]), a2 = term(order[m + 2]), a3 = term(order[m + 3]);
                acc += a0; acc += a1; acc += a2; acc += a3;
            }
            for (; m < si.z; ++m) acc += term(order[m]);
            partial[(int64_t)s * dp + t] = acc;
        }
    }
}

template <bool WT>
__global__ void __launch_bounds__(128) seg_fold_kernel(const double* __restrict__ partial, int d, const int* __restrict__ seg_first,
                                                       double* __restrict__ sums, double* __restrict__ weight_sums) {
    const int j = blockIdx.x, t = blockIdx.y * 128 + threadIdx.x;
    const int dp = WT ? d + 1 : d;
    if (t >= dp) return;
    double s = 0.0;
    for (int g = seg_first[j]; g < seg_first[j + 1]; ++g) s += partial[(int64_t)g * dp + t];
    if (WT && t == d) weight_sums[j] = s;
    else sums[(int64_t)j * d + t] = s;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_rows_map(CUtensorMap* map, const float* base, int64_t rows, int d, int box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !sym) {
            set_error("cuTensorMapEncodeTiled is not available from the driver");
            return OFC_ERR_CUDA;
        }
        fn = (EncodeTiledFn)sym;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)d * 4};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return OFC_ERR_CUDA; }
    return OFC_OK;
}

int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaDeviceProp prop;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return 148;
        n = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    }
    return n;
}

struct TcLayout {
    size_t off_c32, off_ch, off_cl, off_c2, off_c2d, off_cmax, off_count, off_err, off_amb, off_part, off_table, off_order, off_segfirst, off_seginfo,
        off_nsegs, off_segpart, off_fixrows, total;
    int64_t n_chunks, max_segs;
    int parts;
};
TcLayout tc_layout(int64_t n, int d, int k) {
    TcLayout w;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    w.n_chunks = (n + CHUNK - 1) / CHUNK;
    w.max_segs = n / SEG + k + 1;
    w.parts = 148 * 8;
    w.off_c32 = take((size_t)k * d * 4);
    w.off_ch = take((size_t)k * d * 4);
    w.off_cl = take((size_t)k * d * 4);
    w.off_c2 = take((size_t)(k + 512) * 4);
    w.off_c2d = take((size_t)k * 8);
    w.off_cmax = take(4);
    w.off_count = take(4);
    w.off_err = take(4);
    w.off_amb = take((size_t)n * 16);
    w.off_part = take((size_t)w.parts * 8);
    w.off_table = take((size_t)(w.n_chunks + 8) * k * 4);
    w.off_order = take((size_t)n * 4);
    w.off_segfirst = take((size_t)(k + 1) * 4);
    w.off_seginfo = take((size_t)w.max_segs * 16);
    w.off_nsegs = take(4);
    w.off_segpart = take((size_t)w.max_segs * (d + 1) * 8);     // + 1: the weight column of a weighted M-step
    w.off_fixrows = take((size_t)148 * 4 * 8 * d * 8);
    w.total = off;
    return w;
}

template <int BN, bool BRES>
int launch_tc_form(const CUtensorMap& tmAh, const CUtensorMap& tmAl, const CUtensorMap& tmBh, const CUtensorMap& tmBl, const TcParams& p,
                   void* stream) {
    const size_t smem = (size_t)p.tile_bytes + 1024 + 256 + 128 * 12 * 4;
    OFC_SMEM_OPTIN((kmeans_assign_tc_kernel<BN, BRES>), smem);
    const int64_t mtiles = (p.n + BM - 1) / BM;
    const int grid = (int)(mtiles < sm_count() ? mtiles : sm_count());
    kmeans_assign_tc_kernel<BN, BRES><<<grid, TC_THREADS, smem, (cudaStream_t)stream>>>(tmAh, tmAl, tmBh, tmBl, p);
    OFC_CHECK_LAUNCH("kmeans_assign_tc");
    return OFC_OK;
}

template <int BN>
int launch_tc(const CUtensorMap& tmAh, const CUtensorMap& tmAl, const CUtensorMap& tmBh, const CUtensorMap& tmBl, TcParams p,
              void* stream) {
    // centre-resident form when one centre tile covers all k and the resident tiles leave room for >= 2 row stages
    const int n_ktiles = (p.d + BK - 1) / BK;
    const size_t bres_bytes = (size_t)n_ktiles * 2 * TcCfg<BN>::B_BYTES;
    const size_t budget = 200 * 1024;
    if (p.k <= BN && bres_bytes + 2 * (2 * TcCfg<BN>::A_BYTES) <= budget) {
        int st = (int)((budget - bres_bytes) / (2 * TcCfg<BN>::A_BYTES));
        if (st > MAX_STAGES) st = MAX_STAGES;
        p.stages = st;
        p.tile_bytes = (unsigned)((size_t)st * 2 * TcCfg<BN>::A_BYTES + bres_bytes);
        return launch_tc_form<BN, true>(tmAh, tmAl, tmBh, tmBl, p, stream);
    }
    p.stages = TcCfg<BN>::STAGES;
    p.tile_bytes = (unsigned)((size_t)TcCfg<BN>::STAGES * TcCfg<BN>::STAGE_BYTES);
    return launch_tc_form<BN, false>(tmAh, tmAl, tmBh, tmBl, p, stream);
}

int tc_shape_ok(int64_t n, int d, int k) {
    if (n < 1 || n > 0x7fffffffll) { set_error("tensor-core k-means: n=%lld outside [1, 2^31)", (long long)n); return OFC_ERR_UNSUPPORTED; }
    if (d < 32 || (d & 3)) { set_error("tensor-core k-means needs d >= 32 and d %% 4 == 0 (d=%d)", d); return OFC_ERR_UNSUPPORTED; }
    if (k < 2 || k > 8192) { set_error("tensor-core k-means needs 2 <= k <= 8192 (k=%d)", k); return OFC_ERR_UNSUPPORTED; }
    return OFC_OK;
}

}  // namespace
}  // namespace ofc

using namespace ofc;

extern "C" {

size_t ofc_kmeans_tc_workspace_bytes(int64_t n, int d, int k) {
    if (n <= 0 || d <= 0 || k <= 0) return 0;
    return tc_layout(n, d, k).total;
}

int ofc_kmeans_tc_prepare(const float* X, const double* mean, int64_t n, int d, float* Xh, float* Xl, float* xnorm, void* stream) {
    OFC_REQUIRE(X && Xh && Xl && xnorm && n >= 1 && d >= 1, "bad arguments");
    int64_t g = (n + 7) / 8;
    if (g > 148 * 16) g = 148 * 16;
    ProfScope prof(PK_KMEANS, stream);
    prepare_rows_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(X, mean, n, d, Xh, Xl, xnorm);
    OFC_CHECK_LAUNCH("prepare_rows");
    return OFC_OK;
}

// X8 != null: the rows are uint8 (worked in float64): float64 squared norms, float64 re-evaluation on the bytes
static int tc_assign_impl(const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d, int k, const double* centres,
                          int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed, double* inertia, uint32_t* n_rechecked,
                          void* workspace, size_t workspace_bytes, void* stream, const uint8_t* X8, const double* mean8,
                          const double* weights) {
    int rc = tc_shape_ok(n, d, k);
    if (rc != OFC_OK) return rc;
    OFC_REQUIRE(Xh && Xl && xnorm && centres && labels, "null buffer");
    OFC_REQUIRE(((uintptr_t)Xh & 15) == 0 && ((uintptr_t)Xl & 15) == 0, "rows must be 16-byte aligned");
    const TcLayout w = tc_layout(n, d, k);
    if (!workspace || workspace_bytes < w.total) { set_error("tensor-core k-means workspace too small: %zu < %zu", workspace_bytes, w.total); return OFC_ERR_WORKSPACE; }
    OFC_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    float* c32 = (float*)(ws + w.off_c32);
    float* ch = (float*)(ws + w.off_ch);
    float* cl = (float*)(ws + w.off_cl);
    float* c2 = (float*)(ws + w.off_c2);
    float* cmax = (float*)(ws + w.off_cmax);
    unsigned* count = (unsigned*)(ws + w.off_count);
    unsigned* err = (unsigned*)(ws + w.off_err);
    ProfScope prof(PK_KMEANS, stream);
    const int64_t kd = (int64_t)k * d;
    centres_to_f32_kernel<<<(int)((kd + 255) / 256 < 1184 ? (kd + 255) / 256 : 1184), 256, 0, st>>>(centres, c32, ch, cl, kd);
    OFC_CHECK_LAUNCH("centres_to_f32");
    double* c2d = (double*)(ws + w.off_c2d);
    if (X8) centres_c2_f64_kernel<<<cdiv(k + 256, 128), 128, 0, st>>>(centres, c2d, c2, d, k, k + 256);
    else centres_c2_kernel<<<cdiv(k + 256, 128), 128, 0, st>>>(c32, c2, d, k, k + 256);
    OFC_CHECK_LAUNCH("centres_c2");
    centres_cmax_kernel<<<1, 1024, 0, st>>>(c2, k, cmax, count);
    OFC_CHECK_LAUNCH("centres_cmax");
    OFC_CUDA(cudaMemsetAsync(err, 0, 4, st));

    const int BN = k <= 64 ? 64 : (k <= 128 ? 128 : 256);
    CUtensorMap tmAh, tmAl, tmBh, tmBl;
    rc = encode_rows_map(&tmAh, Xh, n, d, BM);
    if (rc == OFC_OK) rc = encode_rows_map(&tmAl, Xl, n, d, BM);
    if (rc == OFC_OK) rc = encode_rows_map(&tmBh, ch, k, d, BN);
    if (rc == OFC_OK) rc = encode_rows_map(&tmBl, cl, k, d, BN);
    if (rc != OFC_OK) return rc;
    TcParams p;
    p.n = n; p.d = d; p.k = k; p.c2 = c2; p.xnorm = xnorm; p.cmax = cmax;
    // per distance: 2 |x| |c| (2^-19 split remainder + d 2^-23 accumulation); two distances; x1.5 margin
    p.tol_scale = 1.5f * 4.f * (1.f / 524288.f + (float)d * (1.f / 8388608.f));
    p.tol_c2 = 0.f;
    if (X8) {
        // against the float64 distance of the bytes: also the float32 rounding of the centred row and of the centres
        // (2 x 2^-24 |x| |c| per dot product) and of the squared norms / the final fma (2^-24 (c2 + |dist|) each)
        p.tol_scale = 1.5f * 4.f * (1.f / 524288.f + 1.f / 4194304.f + (float)d * (1.f / 8388608.f));
        p.tol_c2 = 1.5f * 4.f * (1.f / 8388608.f);
    }
    p.labels = labels; p.amb = (int4*)(ws + w.off_amb); p.amb_count = count; p.error_flag = err;
    if (BN == 64) rc = launch_tc<64>(tmAh, tmAl, tmBh, tmBl, p, stream);
    else if (BN == 128) rc = launch_tc<128>(tmAh, tmAl, tmBh, tmBl, p, stream);
    else rc = launch_tc<256>(tmAh, tmAl, tmBh, tmBl, p, stream);
    if (rc != OFC_OK) return rc;
    const int fix_ctas = sm_count() < 148 ? sm_count() * 4 : 148 * 4;
    if (X8) {
        const size_t fix_smem = (size_t)8 * d * 8;
        const int use_smem = fix_smem <= 200 * 1024;
        if (use_smem) OFC_SMEM_OPTIN(kmeans_assign_fix_u8_kernel, fix_smem);
        kmeans_assign_fix_u8_kernel<<<fix_ctas, 256, use_smem ? fix_smem : 0, st>>>(X8, mean8, d, k, centres, c2d, (const int4*)(ws + w.off_amb),
                                                                                    count, labels, (double*)(ws + w.off_fixrows), use_smem);
    } else {
        const size_t fix_smem = (size_t)8 * d * 4;
        const int use_smem = fix_smem <= 200 * 1024;
        if (use_smem) OFC_SMEM_OPTIN(kmeans_assign_fix_kernel, fix_smem);
        kmeans_assign_fix_kernel<<<fix_ctas, 256, use_smem ? fix_smem : 0, st>>>(Xh, Xl, d, k, c32, c2, (const int4*)(ws + w.off_amb),
                                                                                 count, labels, (float*)(ws + w.off_fixrows), use_smem);
    }
    OFC_CHECK_LAUNCH("kmeans_assign_fix");
    if (n_rechecked) OFC_CUDA(cudaMemcpyAsync(n_rechecked, count, 4, cudaMemcpyDeviceToDevice, st));
    if (n_changed) {
        OFC_CUDA(cudaMemsetAsync(n_changed, 0, 8, st));
        if (prev_labels) {
            int64_t g = (n + 255) / 256;
            if (g > 148 * 8) g = 148 * 8;
            labels_changed_kernel<<<(int)g, 256, 0, st>>>(labels, prev_labels, n, (unsigned long long*)n_changed);
            OFC_CHECK_LAUNCH("labels_changed");
        }
    }
    if (inertia) {
        int64_t g = (n + 7) / 8;
        if (g > w.parts) g = w.parts;
        if (weights) inertia_rows_kernel<true><<<(int)g, 256, 0, st>>>(Xh, Xl, n, d, c32, labels, weights, (double*)(ws + w.off_part));
        else inertia_rows_kernel<false><<<(int)g, 256, 0, st>>>(Xh, Xl, n, d, c32, labels, nullptr, (double*)(ws + w.off_part));
        OFC_CHECK_LAUNCH("inertia_rows");
        fold_partials_kernel<<<1, 32, 0, st>>>((const double*)(ws + w.off_part), (int)g, inertia);
        OFC_CHECK_LAUNCH("fold_partials");
    }
    return OFC_OK;
}

int ofc_kmeans_tc_assign(const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d, int k, const double* centres, int32_t* labels,
                         const int32_t* prev_labels, uint64_t* n_changed, double* inertia, uint32_t* n_rechecked,
                         void* workspace, size_t workspace_bytes, void* stream) {
    return tc_assign_impl(Xh, Xl, xnorm, n, d, k, centres, labels, prev_labels, n_changed, inertia, n_rechecked, workspace,
                          workspace_bytes, stream, nullptr, nullptr, nullptr);
}

int ofc_kmeans_tc_assign_weighted(const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d, int k, const double* centres,
                                  const double* weights, int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed,
                                  double* inertia, uint32_t* n_rechecked, void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(weights != nullptr, "null weights");
    return tc_assign_impl(Xh, Xl, xnorm, n, d, k, centres, labels, prev_labels, n_changed, inertia, n_rechecked, workspace,
                          workspace_bytes, stream, nullptr, nullptr, weights);
}

int ofc_kmeans_tc_assign_u8(const uint8_t* X, const double* mean, const float* Xh, const float* Xl, const float* xnorm, int64_t n, int d,
                            int k, const double* centres, int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed,
                            uint32_t* n_rechecked, void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(X != nullptr, "null rows");
    return tc_assign_impl(Xh, Xl, xnorm, n, d, k, centres, labels, prev_labels, n_changed, nullptr, n_rechecked, workspace,
                          workspace_bytes, stream, X, mean, nullptr);
}

int ofc_kmeans_tc_prepare_u8(const uint8_t* X, const double* mean, int64_t n, int d, float* Xh, float* Xl, float* xnorm, void* stream) {
    OFC_REQUIRE(X && Xh && Xl && xnorm && n >= 1 && d >= 1, "bad arguments");
    int64_t g = (n + 7) / 8;
    if (g > 148 * 16) g = 148 * 16;
    ProfScope prof(PK_KMEANS, stream);
    prepare_rows_u8_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(X, mean, n, d, Xh, Xl, xnorm);
    OFC_CHECK_LAUNCH("prepare_rows_u8");
    return OFC_OK;
}

static int tc_sums_impl(const float* Xh, const float* Xl, const uint8_t* X8, int64_t n, int d, int k, const int32_t* labels, double* sums,
                        int64_t* counts, void* workspace, size_t workspace_bytes, void* stream, const double* weights = nullptr,
                        double* weight_sums = nullptr);

int ofc_kmeans_tc_sums(const float* Xh, const float* Xl, int64_t n, int d, int k, const int32_t* labels, double* sums, int64_t* counts,
                       void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(Xh && Xl, "null buffer");
    return tc_sums_impl(Xh, Xl, nullptr, n, d, k, labels, sums, counts, workspace, workspace_bytes, stream);
}

int ofc_kmeans_tc_sums_u8(const uint8_t* X, int64_t n, int d, int k, const int32_t* labels, double* sums, int64_t* counts,
                          void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(X != nullptr, "null buffer");
    return tc_sums_impl(nullptr, nullptr, X, n, d, k, labels, sums, counts, workspace, workspace_bytes, stream);
}

int ofc_kmeans_tc_sums_weighted(const float* Xh, const float* Xl, int64_t n, int d, int k, const int32_t* labels, const double* weights,
                                double* sums, int64_t* counts, double* weight_sums, void* workspace, size_t workspace_bytes,
                                void* stream) {
    OFC_REQUIRE(Xh && Xl && weights && weight_sums, "null buffer");
    return tc_sums_impl(Xh, Xl, nullptr, n, d, k, labels, sums, counts, workspace, workspace_bytes, stream, weights, weight_sums);
}

int ofc_kmeans_tc_sums_u8_weighted(const uint8_t* X, int64_t n, int d, int k, const int32_t* labels, const double* weights, double* sums,
                                   int64_t* counts, double* weight_sums, void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(X && weights && weight_sums, "null buffer");
    return tc_sums_impl(nullptr, nullptr, X, n, d, k, labels, sums, counts, workspace, workspace_bytes, stream, weights, weight_sums);
}

static int tc_sums_impl(const float* Xh, const float* Xl, const uint8_t* X8, int64_t n, int d, int k, const int32_t* labels, double* sums,
                        int64_t* counts, void* workspace, size_t workspace_bytes, void* stream, const double* weights,
                        double* weight_sums) {
    int rc = tc_shape_ok(n, d, k);
    if (rc != OFC_OK) return rc;
    OFC_REQUIRE(labels && sums && counts, "null buffer");
    const TcLayout w = tc_layout(n, d, k);
    if (!workspace || workspace_bytes < w.total) { set_error("tensor-core k-means workspace too small: %zu < %zu", workspace_bytes, w.total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* table = (unsigned*)(ws + w.off_table);
    int32_t* order = (int32_t*)(ws + w.off_order);
    int* seg_first = (int*)(ws + w.off_segfirst);
    int4* seg_info = (int4*)(ws + w.off_seginfo);
    int* n_segs = (int*)(ws + w.off_nsegs);
    double* partial = (double*)(ws + w.off_segpart);
    ProfScope prof(PK_KMEANS, stream);
    const int walk_ctas = (int)((w.n_chunks + 7) / 8);
    const size_t walk_smem = (size_t)8 * k * 4;
    OFC_SMEM_OPTIN(csr_walk_kernel<false>, walk_smem);
    OFC_SMEM_OPTIN(csr_walk_kernel<true>, walk_smem);
    csr_walk_kernel<false><<<walk_ctas, 256, walk_smem, st>>>(labels, n, k, table, nullptr);
    OFC_CHECK_LAUNCH("csr_hist");
    const size_t scan_smem = ((size_t)(k >= 1024 ? 1 : 1024 / k) * k + 2 * (size_t)k) * 4;
    OFC_SMEM_OPTIN(csr_scan_kernel, scan_smem);
    csr_scan_kernel<<<1, 1024, scan_smem, st>>>(table, w.n_chunks, k, (long long*)counts, seg_first, seg_info, n_segs);
    OFC_CHECK_LAUNCH("csr_scan");
    csr_walk_kernel<true><<<walk_ctas, 256, walk_smem, st>>>(labels, n, k, table, order);
    OFC_CHECK_LAUNCH("csr_scatter");
    const bool wt = weights != nullptr;
    const int dt = cdiv(wt ? d + 1 : d, 128);
    int64_t gx = w.max_segs;
    const int64_t cap = (int64_t)sm_count() * 32 / dt + 1;
    if (gx > cap) gx = cap;
    const dim3 sgrid((unsigned)gx, dt);
    if (X8 && wt) seg_sums_u8_kernel<true><<<sgrid, 128, 0, st>>>(X8, d, order, seg_info, n_segs, weights, partial);
    else if (X8) seg_sums_u8_kernel<false><<<sgrid, 128, 0, st>>>(X8, d, order, seg_info, n_segs, nullptr, partial);
    else if (wt) seg_sums_kernel<true><<<sgrid, 128, 0, st>>>(Xh, Xl, d, order, seg_info, n_segs, weights, partial);
    else seg_sums_kernel<false><<<sgrid, 128, 0, st>>>(Xh, Xl, d, order, seg_info, n_segs, nullptr, partial);
    OFC_CHECK_LAUNCH("seg_sums");
    if (wt) seg_fold_kernel<true><<<dim3(k, dt), 128, 0, st>>>(partial, d, seg_first, sums, weight_sums);
    else seg_fold_kernel<false><<<dim3(k, dt), 128, 0, st>>>(partial, d, seg_first, sums, nullptr);
    OFC_CHECK_LAUNCH("seg_fold");
    return OFC_OK;
}

}  // extern "C"
