// C-ABI entry points of libofc (declared in include/ofc.h) and the host-side
// Farneback driver: pyramid plan, workspace layout, per-level launch sequence.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/ofc.h"
#include "ofc_common.cuh"
#include "flow_kernels.cuh"
#include "grid_kernels.cuh"
#include "kmeans_kernels.cuh"
#include "viz_kernels.cuh"

namespace ofc {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return OFC_OK;
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return OFC_ERR_CUDA;
}

// per-(device, kernel) record of the dynamic shared memory already opted in to
int smem_optin(const void* kernel, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> done;
    int dev = 0;
    OFC_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = done[std::make_pair(dev, kernel)];
    if (bytes <= have) return OFC_OK;
#ifndef OFC_EMULATE
    OFC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
#endif
    have = bytes;
    return OFC_OK;
}

// ---- optional per-kernel event timing --------------------------------------
// The records are process-global and mutex-protected; a scope remembers its own record index, so launches
// from several host threads interleave without corrupting each other (their times then overlap, of course).
struct ProfRec { int kind; cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
int g_prof_level = 0;

ProfScope::ProfScope(int kind_, void* stream_) : kind(kind_), stream(stream_), on(g_prof_on), index(-1) {
    if (!on) return;
    ProfRec r;
    r.kind = kind;
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) { on = false; return; }
    cudaEventRecord(r.a, (cudaStream_t)stream);
    std::lock_guard<std::mutex> lock(g_prof_mu);
    index = (int)g_prof.size();
    g_prof.push_back(r);
}
ProfScope::~ProfScope() {
    if (!on) return;
    std::lock_guard<std::mutex> lock(g_prof_mu);
    if (index >= 0 && index < (int)g_prof.size()) cudaEventRecord(g_prof[index].b, (cudaStream_t)stream);
}

// cvRound: round half to even
static int cv_round(double v) { return (int)nearbyint(v); }

struct Level {
    int k;                 // pyramid index (0 = full resolution)
    int w, h;
    int ksz;
    double sigma;
    double sx, sy;         // cv::resize source/destination ratio
    int tx, ty, in_rows, in_pitch, taps_pad;
    size_t prefilter_smem;
    size_t off_I, off_RA, off_RB, off_flow[2];
    size_t taps_off;       // floats into the device tap table
};

}  // namespace ofc

struct ofc_flow_plan {
    int W, H, max_frames;
    double pyr_scale;
    int levels, winsize, iterations, poly_n;
    double poly_sigma;
    int flags;                       // OFC_FLOW_USE_INITIAL_FLOW | OFC_FLOW_GAUSSIAN
    ofc::GaussWindow gauss;          // window taps when OFC_FLOW_GAUSSIAN
    int keep_level0_I;               // also materialise I of the full-resolution level (fused away by default)
    // Side stream for the per-frame work (pre-filter + polynomial expansion), so that the large
    // full-resolution expansion overlaps the small, latency-bound iterations of the coarse levels.
    cudaStream_t side;
    cudaEvent_t ev_fork;
    std::vector<cudaEvent_t> ev_level;
    std::vector<ofc::Level> lv;      // coarsest first
    size_t workspace_bytes;
    float* d_taps;
    ofc::PolyParams poly;            // taps / inverse-Gram constants filled in
    // streaming use (ofc_farneback_stream_*): which of the two frame slots holds the previous frame's I / R
    int stream_slot;
    int stream_primed;
};

namespace ofc {

static void gaussian_taps(int ksize, double sigma, std::vector<float>& out) {
    out.resize(ksize);
    if (sigma <= 0 && ksize == 3) { out[0] = 0.25f; out[1] = 0.5f; out[2] = 0.25f; return; }
    if (sigma <= 0) sigma = ((ksize - 1) * 0.5 - 1) * 0.3 + 0.8;
    std::vector<double> g(ksize);
    double c = (ksize - 1) * 0.5, sum = 0;
    for (int i = 0; i < ksize; ++i) { double x = i - c; g[i] = exp(-(x * x) / (2.0 * sigma * sigma)); sum += g[i]; }
    for (int i = 0; i < ksize; ++i) out[i] = (float)(g[i] / sum);
}

// FarnebackPrepareGaussian: taps and the four inverse-Gram entries
static int prepare_poly(int n, double sigma, PolyParams& pp) {
    if (n > 7) { set_error("poly_n=%d unsupported", n); return OFC_ERR_UNSUPPORTED; }
    float g[15], xg[15], xxg[15];
    double s = 0;
    for (int x = -n; x <= n; ++x) { g[x + n] = (float)exp(-x * x / (2.0 * sigma * sigma)); s += g[x + n]; }
    s = 1.0 / s;
    for (int x = -n; x <= n; ++x) {
        g[x + n] = (float)(g[x + n] * s);
        xg[x + n] = (float)(x * g[x + n]);
        xxg[x + n] = (float)(x * x * g[x + n]);
    }
    double G[6][6];
    memset(G, 0, sizeof(G));
    for (int y = -n; y <= n; ++y)
        for (int x = -n; x <= n; ++x) {
            double w = (double)g[y + n] * g[x + n];
            G[0][0] += w;
            G[1][1] += w * x * x;
            G[3][3] += w * x * x * x * x;
            G[5][5] += w * x * x * y * y;
        }
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    // Gauss-Jordan inverse (6x6, symmetric positive definite)
    double A[6][12];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 12; ++j) A[i][j] = j < 6 ? G[i][j] : (j - 6 == i ? 1.0 : 0.0);
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        for (int r = c + 1; r < 6; ++r) if (fabs(A[r][c]) > fabs(A[piv][c])) piv = r;
        if (fabs(A[piv][c]) < 1e-300) { set_error("singular Gram matrix"); return OFC_ERR_INVALID; }
        if (piv != c) for (int j = 0; j < 12; ++j) { double t = A[c][j]; A[c][j] = A[piv][j]; A[piv][j] = t; }
        double d = 1.0 / A[c][c];
        for (int j = 0; j < 12; ++j) A[c][j] *= d;
        for (int r = 0; r < 6; ++r) if (r != c) {
            double f = A[r][c];
            if (f != 0) for (int j = 0; j < 12; ++j) A[r][j] -= f * A[c][j];
        }
    }
    for (int k = 0; k <= n; ++k) { pp.g[k] = g[n + k]; pp.xg[k] = xg[n + k]; pp.xxg[k] = xxg[n + k]; }
    pp.ig11 = (float)A[1][6 + 1];
    pp.ig03 = (float)A[0][6 + 3];
    pp.ig33 = (float)A[3][6 + 3];
    pp.ig55 = (float)A[5][6 + 5];
    return OFC_OK;
}

// stage1_frames / slot_first: the frames at `gray` are expanded into frame slots slot_first, slot_first + 1, ...;
// iterate: run the coarse-to-fine iterations for n_frames - 1 pairs whose "prev" frame sits in slot prev_slot and whose
// "next" frame is next_delta slots further (+1 for a batch; -1 / +1 alternating in streaming use).
static int run_farneback(const ofc_flow_plan* pl, const uint8_t* gray, int64_t gray_stride, int n_frames,
                         float* flow, uint32_t* minmax, void* workspace, size_t workspace_bytes, void* stream,
                         const float* init_flow = nullptr, int stage1_frames = -1, int slot_first = 0, bool iterate = true,
                         int prev_slot = 0, int next_delta = 1) {
    OFC_REQUIRE(pl != nullptr, "null plan");
    if ((pl->flags & OFC_FLOW_USE_INITIAL_FLOW) && !init_flow) {
        set_error("the plan was created with OPTFLOW_USE_INITIAL_FLOW: call ofc_farneback_pair_init with the initial flow");
        return OFC_ERR_INVALID;
    }
    if (!(pl->flags & OFC_FLOW_USE_INITIAL_FLOW)) init_flow = nullptr;
    OFC_REQUIRE(n_frames >= 2 && n_frames <= pl->max_frames, "n_frames=%d outside [2, %d]", n_frames, pl->max_frames);
    OFC_REQUIRE(gray && (flow || !iterate) && workspace, "null buffer");
    if (stage1_frames < 0) stage1_frames = n_frames;
    if (workspace_bytes < pl->workspace_bytes) {
        set_error("workspace too small: %zu < %zu", workspace_bytes, pl->workspace_bytes);
        return OFC_ERR_WORKSPACE;
    }
    OFC_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    char* ws = (char*)workspace;
    const int n_pairs = n_frames - 1;
    const int F = pl->max_frames;
    const int nl = (int)pl->lv.size();

    // stage 1: pre-filter + polynomial expansion of every frame at every level, coarsest first, on the
    // plan's side stream when it has one: level l's iterations (stage 2, caller's stream) wait only for
    // level l's event, so the big fine-level expansions run under the small coarse-level iterations.
    // (ofc_profile_begin turns the fork off: per-kernel event timing wants one stream.)
    const bool fork = pl->side != nullptr && !g_prof_on;
    void* const stream1 = fork ? (void*)pl->side : stream;
    if (fork) {
        OFC_CUDA(cudaEventRecord(pl->ev_fork, (cudaStream_t)stream));
        OFC_CUDA(cudaStreamWaitEvent(pl->side, pl->ev_fork, 0));
    }
    // an early error return must not leave the side stream running behind the caller's back: whatever
    // was enqueued there is joined into the caller's stream on every exit path
    struct SideJoin {
        cudaStream_t side, main; cudaEvent_t ev; bool armed;
        ~SideJoin() { if (armed && cudaEventRecord(ev, side) == cudaSuccess) cudaStreamWaitEvent(main, ev, 0); }
    } side_join{fork ? pl->side : nullptr, (cudaStream_t)stream, fork ? pl->ev_fork : cudaEvent_t(), fork};
    // the pre-filter of every level that is an exact power-of-two fraction of the frame: one launch
    std::vector<PrefilterParams> pfs(nl);
    std::vector<char> pf_done(nl, 0);
    for (int l = 0; l < nl; ++l) {
        const Level& L = pl->lv[l];
        PrefilterParams& pf = pfs[l];
        pf.gray = gray; pf.gray_stride = gray_stride;
        pf.out = (float*)(ws + L.off_I) + (int64_t)slot_first * L.w * L.h; pf.out_stride = (int64_t)L.w * L.h;
        pf.W = pl->W; pf.H = pl->H; pf.w = L.w; pf.h = L.h;
        pf.ksz = L.ksz; pf.sx = L.sx; pf.sy = L.sy;
        pf.taps = pl->d_taps + L.taps_off;
        pf.identity3 = (L.sigma <= 0 && L.ksz == 3 && L.w == pl->W && L.h == pl->H) ? 1 : 0;
        pf.tx = L.tx; pf.ty = L.ty; pf.in_rows = L.in_rows; pf.in_pitch = L.in_pitch; pf.taps_pad = L.taps_pad;
    }
    {
        int rc = stage1_frames > 0 ? launch_prefilter_pyramid(pfs.data(), nl, stage1_frames,
                                                             reinterpret_cast<bool*>(pf_done.data()), stream1)
                                   : OFC_OK;
        if (rc != OFC_OK) return rc;
    }
    for (int l = 0; l < nl; ++l) {
        const Level& L = pl->lv[l];
        const PrefilterParams& pf = pfs[l];
        int rc = OFC_OK;
        if (stage1_frames <= 0) {
            if (fork) OFC_CUDA(cudaEventRecord(pl->ev_level[l], pl->side));
            continue;
        }
        if (!pf.identity3 && !pf_done[l]) {
            rc = launch_prefilter(pf, stage1_frames, L.prefilter_smem, stream1);
            if (rc != OFC_OK) return rc;
        }
        PolyParams pp = pl->poly;
        pp.I = pf.out; pp.in_stride = pf.out_stride;
        pp.RA = (float4*)(ws + L.off_RA) + (int64_t)slot_first * L.w * L.h; pp.RB = (float*)(ws + L.off_RB) + (int64_t)slot_first * L.w * L.h;
        pp.out_stride = (int64_t)L.w * L.h; pp.w = L.w; pp.h = L.h;
        rc = launch_polyexp(pp, pl->poly_n, stage1_frames, pf.identity3 ? gray : nullptr, gray_stride,
                            (pl->keep_level0_I || pl->poly_n != 5) ? pf.out : nullptr, stream1);
        if (rc != OFC_OK) return rc;
        if (fork) OFC_CUDA(cudaEventRecord(pl->ev_level[l], pl->side));
    }
    if (!iterate) {
        // stage 1 only (priming a stream): join the side stream and leave
        if (fork) OFC_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, pl->ev_level[nl - 1], 0));
        side_join.armed = false;
        return OFC_OK;
    }
    if (minmax) {
        int rc = launch_minmax_init(minmax, n_pairs, stream);
        if (rc != OFC_OK) return rc;
    }
    // stage 2: coarse-to-fine iterations, all pairs of the batch per launch
    const float2* prev_flow = nullptr;
    int prev_w = 0, prev_h = 0;
    (void)F;
    for (int l = 0; l < nl; ++l) {
        const Level& L = pl->lv[l];
        const int64_t npx = (int64_t)L.w * L.h;
        if (fork) OFC_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, pl->ev_level[l], 0));
        for (int it = 0; it < pl->iterations; ++it) {
            IterParams ip;
            ip.RA = (const float4*)(ws + L.off_RA) + (int64_t)prev_slot * npx; ip.RB = (const float*)(ws + L.off_RB) + (int64_t)prev_slot * npx;
            ip.r_stride = npx; ip.r_next = (int64_t)next_delta * npx;
            ip.w = L.w; ip.h = L.h;
            ip.border[0] = 0.14f; ip.border[1] = 0.14f; ip.border[2] = 0.4472f; ip.border[3] = 0.4472f; ip.border[4] = 0.4472f;
            ip.blur_scale = 1.0 / ((double)pl->winsize * pl->winsize);
            {
                // float32 solve (solve2x2): the regulariser 1e-3 in units of the raw window sums, as two floats
                const double c = 1e-3 / (ip.blur_scale * ip.blur_scale);
                ip.solve_c_hi = (float)c;
                ip.solve_c_lo = (float)(c - (double)ip.solve_c_hi);
            }
            ip.upsample = 0; ip.wc = ip.hc = 0; ip.usx = ip.usy = 1.0; ip.flow_mul = 1.0;
            if (it == 0 && l == 0 && init_flow) {
                // cv2 flag 4: resize(flow0, INTER_AREA) * scale seeds the coarsest level (other ping-pong buffer)
                double scale = 1.0;
                for (int i = 0; i < L.k; ++i) scale *= pl->pyr_scale;
                float2* seed = (float2*)(ws + L.off_flow[1]);
                int rc = launch_flow_area_seed((const float2*)init_flow, (int64_t)pl->W * pl->H, pl->W, pl->H, seed, npx, L.w, L.h,
                                               (float)scale, n_pairs, stream);
                if (rc != OFC_OK) return rc;
                ip.flow_in = seed;
                ip.flow_in_stride = npx;
            } else if (it == 0) {
                ip.flow_in = prev_flow;
                ip.flow_in_stride = (int64_t)prev_w * prev_h;
                if (prev_flow) {
                    ip.upsample = 1; ip.wc = prev_w; ip.hc = prev_h;
                    ip.usx = 1.0 / ((double)L.w / prev_w);
                    ip.usy = 1.0 / ((double)L.h / prev_h);
                    ip.flow_mul = 1.0 / pl->pyr_scale;
                }
            } else {
                ip.flow_in = (const float2*)(ws + L.off_flow[(it - 1) & 1]);
                ip.flow_in_stride = npx;
            }
            const bool last = (l == nl - 1) && (it == pl->iterations - 1);
            ip.flow_out = last ? (float2*)flow : (float2*)(ws + L.off_flow[it & 1]);
            ip.flow_out_stride = npx;
            ip.minmax = last ? minmax : nullptr;
            g_prof_level = nl - 1 - l;
            int rc = launch_flow_iter(ip, pl->winsize, n_pairs, (float2*)(ws + L.off_flow[(it & 1) ^ 1]), stream,
                                      (pl->flags & OFC_FLOW_GAUSSIAN) ? &pl->gauss : nullptr);
            if (rc != OFC_OK) return rc;
        }
        prev_flow = (const float2*)(ws + L.off_flow[(pl->iterations - 1) & 1]);
        prev_w = L.w; prev_h = L.h;
    }
    side_join.armed = false;          // every level's event has been waited for above
    return OFC_OK;
}

}  // namespace ofc

using namespace ofc;

extern "C" {

int ofc_version(void) { return 100; }

int ofc_profile_begin(void) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_prof.clear();
    g_prof_on = true;
    return OFC_OK;
}

int ofc_profile_end(float* ms_by_kind, int* launches_by_kind, int n_kinds) {
    g_prof_on = false;
    std::lock_guard<std::mutex> lock(g_prof_mu);
    OFC_REQUIRE(ms_by_kind && launches_by_kind && n_kinds >= PK_COUNT, "need %d slots", (int)PK_COUNT);
    for (int i = 0; i < n_kinds; ++i) { ms_by_kind[i] = 0.f; launches_by_kind[i] = 0; }
    int rc = OFC_OK;
    for (auto& r : g_prof) {
        float ms = 0.f;
        if (rc == OFC_OK) rc = check_cuda(cudaEventSynchronize(r.b), "cudaEventSynchronize");
        if (rc == OFC_OK) rc = check_cuda(cudaEventElapsedTime(&ms, r.a, r.b), "cudaEventElapsedTime");
        if (rc == OFC_OK && r.kind >= 0 && r.kind < n_kinds) { ms_by_kind[r.kind] += ms; launches_by_kind[r.kind] += 1; }
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_prof.clear();
    return rc;
}

const char* ofc_last_error(void) { return g_error; }

int ofc_flow_plan_create(ofc_flow_plan** out, int width, int height, int max_frames,
                         double pyr_scale, int levels, int winsize, int iterations,
                         int poly_n, double poly_sigma, int flags) {
    OFC_REQUIRE(out != nullptr, "null plan pointer");
    *out = nullptr;
    if (flags & ~(OFC_FLOW_USE_INITIAL_FLOW | OFC_FLOW_GAUSSIAN)) {
        set_error("flags=%d unsupported: OPTFLOW_USE_INITIAL_FLOW (4) and OPTFLOW_FARNEBACK_GAUSSIAN (256) are the only flags", flags);
        return OFC_ERR_UNSUPPORTED;
    }
    OFC_REQUIRE(width >= 16 && height >= 16, "frame %dx%d too small", width, height);
    OFC_REQUIRE(max_frames >= 2, "max_frames must be >= 2");
    OFC_REQUIRE(pyr_scale > 0 && pyr_scale < 1, "pyr_scale must be in (0,1)");
    OFC_REQUIRE(levels >= 0 && iterations >= 1, "levels >= 0 and iterations >= 1 required");
    OFC_REQUIRE(winsize >= 4 && winsize <= 65, "winsize must be in [4, 65]");
    OFC_REQUIRE(poly_sigma > 0, "poly_sigma must be > 0");
    ofc_flow_plan* pl = new ofc_flow_plan();
    pl->W = width; pl->H = height; pl->max_frames = max_frames;
    pl->pyr_scale = pyr_scale; pl->levels = levels; pl->winsize = winsize;
    pl->iterations = iterations; pl->poly_n = poly_n; pl->poly_sigma = poly_sigma;
    pl->flags = flags;
    memset(&pl->gauss, 0, sizeof(pl->gauss));
    pl->d_taps = nullptr;
    pl->keep_level0_I = 0;
    pl->stream_slot = 0;
    pl->stream_primed = 0;
    pl->side = nullptr;
    pl->ev_fork = cudaEvent_t();
    memset(&pl->poly, 0, sizeof(pl->poly));
    int rc = prepare_poly(poly_n, poly_sigma, pl->poly);
    if (rc != OFC_OK) { delete pl; return rc; }
    if (poly_n != 5 && poly_n != 7) { set_error("poly_n=%d unsupported (5 or 7)", poly_n); delete pl; return OFC_ERR_UNSUPPORTED; }
    if (flags & OFC_FLOW_GAUSSIAN) {
        // FarnebackUpdateFlow_GaussianBlur: 2m+1 taps, sigma = m * 0.3, normalised in double, stored as float
        const int m = winsize / 2;
        if (m > 32) { set_error("winsize=%d unsupported with OPTFLOW_FARNEBACK_GAUSSIAN (<= 65)", winsize); delete pl; return OFC_ERR_UNSUPPORTED; }
        const double sigma = m * 0.3;
        double kk[33];
        double sum = 1.0;
        kk[0] = 1.0;
        for (int i = 1; i <= m; ++i) {
            const float t = (float)exp(-i * i / (2 * sigma * sigma));
            kk[i] = t;
            sum += (double)t * 2;
        }
        pl->gauss.r = m;
        pl->gauss.scale = 1.0;
        for (int i = 0; i <= m; ++i) pl->gauss.k[i] = (float)(kk[i] * (1.0 / sum));
    }
    // box window: radii 2..7, 10, 12 have unrolled kernels (launch_flow_iter), any other winsize in [4, 65] runs the
    // run-time-radius kernel
    // pyramid: levels+1 scales, cropped while the coarse side stays >= 32 (SURVEY.md A.1)
    int eff = 0;
    {
        double scale = 1.0;
        for (int k = 0; k < levels; ++k) {
            scale *= pyr_scale;
            if (width * scale < 32 || height * scale < 32) break;
            ++eff;
        }
    }
    std::vector<float> all_taps;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    for (int k = eff; k >= 0; --k) {
        Level L;
        L.k = k;
        double scale = 1.0;
        for (int i = 0; i < k; ++i) scale *= pyr_scale;
        L.sigma = (1.0 / scale - 1.0) * 0.5;
        int ksz = cv_round(L.sigma * 5) | 1;
        L.ksz = ksz < 3 ? 3 : ksz;
        L.w = cv_round(width * scale);
        L.h = cv_round(height * scale);
        L.sx = 1.0 / ((double)L.w / width);
        L.sy = 1.0 / ((double)L.h / height);
        if (L.ksz / 2 >= width || L.ksz / 2 >= height) {
            set_error("Gaussian radius %d exceeds the frame", L.ksz / 2);
            delete pl; return OFC_ERR_UNSUPPORTED;
        }
        std::vector<float> taps;
        gaussian_taps(L.ksz, L.sigma, taps);
        L.taps_off = all_taps.size();
        all_taps.insert(all_taps.end(), taps.begin(), taps.end());
        // prefilter tile: shrink until the staged window fits in shared memory
        L.tx = 32; L.ty = 8;
        for (;;) {
            int in_cols = (int)ceil((L.tx - 1) * L.sx) + L.ksz + 3;
            L.in_rows = (int)ceil((L.ty - 1) * L.sy) + L.ksz + 3;
            L.in_pitch = (in_cols + 3) / 4 * 4;
            L.taps_pad = (L.ksz + 3) / 4 * 4;
            L.prefilter_smem = (size_t)L.taps_pad * 4 + (size_t)L.in_rows * L.tx * 2 * 4 + (size_t)L.in_rows * L.in_pitch;
            if (L.prefilter_smem <= 200 * 1024) break;
            if (L.tx == 1 && L.ty == 1) { set_error("pyramid level %d needs too much shared memory", k); delete pl; return OFC_ERR_UNSUPPORTED; }
            if (L.tx >= 2 * L.ty && L.tx > 1) L.tx /= 2; else if (L.ty > 1) L.ty /= 2; else L.tx /= 2;
        }
        size_t npx = (size_t)L.w * L.h;
        L.off_I = take(npx * 4 * max_frames);
        L.off_RA = take(npx * 16 * max_frames);
        L.off_RB = take(npx * 4 * max_frames);
        L.off_flow[0] = take(npx * 8 * (max_frames - 1));
        L.off_flow[1] = take(npx * 8 * (max_frames - 1));
        pl->lv.push_back(L);
    }
    pl->workspace_bytes = off;
    void* d = nullptr;
    rc = check_cuda(cudaMalloc(&d, all_taps.size() * sizeof(float)), "cudaMalloc(taps)");
    if (rc != OFC_OK) { delete pl; return rc; }
    pl->d_taps = (float*)d;
    rc = check_cuda(cudaMemcpy(pl->d_taps, all_taps.data(), all_taps.size() * sizeof(float), cudaMemcpyHostToDevice), "cudaMemcpy(taps)");
    if (rc != OFC_OK) { cudaFree(d); delete pl; return rc; }
    // the side stream of stage 1 (run_farneback); without it everything runs on the caller's stream
    if (cudaStreamCreateWithFlags(&pl->side, cudaStreamNonBlocking) != cudaSuccess) pl->side = nullptr;
    if (pl->side) {
        bool ok = cudaEventCreateWithFlags(&pl->ev_fork, cudaEventDisableTiming) == cudaSuccess;
        pl->ev_level.resize(pl->lv.size());
        for (size_t i = 0; ok && i < pl->lv.size(); ++i)
            ok = cudaEventCreateWithFlags(&pl->ev_level[i], cudaEventDisableTiming) == cudaSuccess;
        if (!ok) { cudaStreamDestroy(pl->side); pl->side = nullptr; }
    }
    *out = pl;
    return OFC_OK;
}

void ofc_flow_plan_destroy(ofc_flow_plan* pl) {
    if (!pl) return;
    if (pl->d_taps) cudaFree(pl->d_taps);
    if (pl->side) {
        cudaStreamSynchronize(pl->side);
        cudaEventDestroy(pl->ev_fork);
        for (auto& e : pl->ev_level) cudaEventDestroy(e);
        cudaStreamDestroy(pl->side);
    }
    delete pl;
}

size_t ofc_flow_plan_workspace_bytes(const ofc_flow_plan* pl) { return pl ? pl->workspace_bytes : 0; }

int ofc_flow_plan_keep_intermediates(ofc_flow_plan* pl, int keep) {
    OFC_REQUIRE(pl != nullptr, "null plan");
    pl->keep_level0_I = keep ? 1 : 0;
    return OFC_OK;
}

int ofc_flow_plan_num_levels(const ofc_flow_plan* pl) { return pl ? (int)pl->lv.size() : 0; }

int ofc_flow_plan_level_size(const ofc_flow_plan* pl, int level, int* w, int* h) {
    OFC_REQUIRE(pl && level >= 0 && level < (int)pl->lv.size(), "bad level %d", level);
    if (w) *w = pl->lv[level].w;
    if (h) *h = pl->lv[level].h;
    return OFC_OK;
}

int ofc_flow_plan_buffer(const ofc_flow_plan* pl, int level, int kind, size_t* offset_bytes, size_t* frame_stride_bytes) {
    OFC_REQUIRE(pl && level >= 0 && level < (int)pl->lv.size(), "bad level %d", level);
    const Level& L = pl->lv[level];
    size_t npx = (size_t)L.w * L.h, o, s;
    switch (kind) {
        case 0: o = L.off_I; s = npx * 4; break;
        case 1: o = L.off_RA; s = npx * 16; break;
        case 2: o = L.off_RB; s = npx * 4; break;
        case 3: o = L.off_flow[0]; s = npx * 8; break;
        case 4: o = L.off_flow[1]; s = npx * 8; break;
        default: set_error("bad buffer kind %d", kind); return OFC_ERR_INVALID;
    }
    if (offset_bytes) *offset_bytes = o;
    if (frame_stride_bytes) *frame_stride_bytes = s;
    return OFC_OK;
}

int ofc_farneback_sequence(const ofc_flow_plan* plan, const uint8_t* gray, int n_frames, float* flow,
                           uint32_t* minmax, void* workspace, size_t workspace_bytes, void* stream) {
    if (!plan) { set_error("null plan"); return OFC_ERR_INVALID; }
    return run_farneback(plan, gray, (int64_t)plan->W * plan->H, n_frames, flow, minmax, workspace, workspace_bytes, stream);
}

int ofc_farneback_pair(const ofc_flow_plan* plan, const uint8_t* prev, const uint8_t* next, float* flow,
                       uint32_t* minmax, void* workspace, size_t workspace_bytes, void* stream) {
    if (!plan) { set_error("null plan"); return OFC_ERR_INVALID; }
    OFC_REQUIRE(prev && next, "null frame");
    return run_farneback(plan, prev, (int64_t)(next - prev), 2, flow, minmax, workspace, workspace_bytes, stream);
}

int ofc_farneback_pair_init(const ofc_flow_plan* plan, const uint8_t* prev, const uint8_t* next, const float* init_flow,
                            float* flow, uint32_t* minmax, void* workspace, size_t workspace_bytes, void* stream) {
    if (!plan) { set_error("null plan"); return OFC_ERR_INVALID; }
    OFC_REQUIRE(prev && next && init_flow, "null frame / initial flow");
    OFC_REQUIRE(plan->flags & OFC_FLOW_USE_INITIAL_FLOW, "the plan was created without OPTFLOW_USE_INITIAL_FLOW");
    OFC_REQUIRE(((uintptr_t)init_flow & 7) == 0, "initial flow must be 8-byte aligned");
    return run_farneback(plan, prev, (int64_t)(next - prev), 2, flow, minmax, workspace, workspace_bytes, stream, init_flow);
}

int ofc_farneback_stream_begin(ofc_flow_plan* plan, const uint8_t* first_gray, void* workspace, size_t workspace_bytes, void* stream) {
    if (!plan) { set_error("null plan"); return OFC_ERR_INVALID; }
    OFC_REQUIRE(first_gray != nullptr, "null frame");
    OFC_REQUIRE(!(plan->flags & OFC_FLOW_USE_INITIAL_FLOW), "streaming use does not take an initial flow");
    int rc = run_farneback(plan, first_gray, (int64_t)plan->W * plan->H, 2, nullptr, nullptr, workspace, workspace_bytes, stream, nullptr,
                           /*stage1_frames=*/1, /*slot_first=*/0, /*iterate=*/false);
    if (rc != OFC_OK) return rc;
    plan->stream_slot = 0;
    plan->stream_primed = 1;
    return OFC_OK;
}

int ofc_farneback_stream_next(ofc_flow_plan* plan, const uint8_t* gray, float* flow, uint32_t* minmax, void* workspace,
                              size_t workspace_bytes, void* stream) {
    if (!plan) { set_error("null plan"); return OFC_ERR_INVALID; }
    OFC_REQUIRE(gray && flow, "null buffer");
    OFC_REQUIRE(plan->stream_primed, "call ofc_farneback_stream_begin with the first frame");
    const int prev = plan->stream_slot, cur = prev ^ 1;
    int rc = run_farneback(plan, gray, (int64_t)plan->W * plan->H, 2, flow, minmax, workspace, workspace_bytes, stream, nullptr,
                           /*stage1_frames=*/1, /*slot_first=*/cur, /*iterate=*/true, /*prev_slot=*/prev, /*next_delta=*/cur - prev);
    if (rc != OFC_OK) return rc;
    plan->stream_slot = cur;
    return OFC_OK;
}

int ofc_bgr2gray(const uint8_t* bgr, uint8_t* gray, int64_t n_pixels, void* stream) {
    OFC_REQUIRE(n_pixels >= 0 && (n_pixels == 0 || (bgr && gray)), "bad arguments");
    OFC_REQUIRE(((uintptr_t)bgr & 3) == 0 && ((uintptr_t)gray & 3) == 0, "buffers must be 4-byte aligned");
    return launch_bgr2gray(bgr, gray, n_pixels, stream);
}

int ofc_bgr2hsv(const uint8_t* bgr, uint8_t* hsv, int64_t n_pixels, void* stream) {
    OFC_REQUIRE(n_pixels >= 0 && (n_pixels == 0 || (bgr && hsv)), "bad arguments");
    return launch_bgr2hsv(bgr, hsv, n_pixels, stream);
}

int ofc_flow_minmax(const float* flow, int n_frames, int64_t n_pixels, uint32_t* minmax, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && n_pixels >= 0, "bad sizes");
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(flow && minmax, "null buffer");
    int rc = launch_minmax_init(minmax, n_frames, stream);
    if (rc != OFC_OK) return rc;
    return launch_flow_minmax((const float2*)flow, n_pixels, n_frames, minmax, stream);
}

int ofc_flow_to_bgr(const float* flow, int n_frames, int height, int width, const uint32_t* minmax,
                    uint8_t* bgr, double* mag_sum, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height >= 0 && width >= 0, "bad sizes");
    const int64_t n_pixels = (int64_t)height * width;
    if (n_frames == 0 || n_pixels == 0) return OFC_OK;
    OFC_REQUIRE(flow && minmax && bgr, "null buffer");
    OFC_REQUIRE(((uintptr_t)flow & 15) == 0 && ((uintptr_t)bgr & 3) == 0, "flow must be 16-byte and bgr 4-byte aligned");
    if (mag_sum) OFC_CUDA(cudaMemsetAsync(mag_sum, 0, sizeof(double) * n_frames, (cudaStream_t)stream));
    VizParams p;
    p.flow = (const float2*)flow; p.n_px = n_pixels; p.width = width; p.minmax = minmax; p.bgr = bgr; p.mag_sum = mag_sum;
    p.hsv = nullptr;
    return launch_flow_encode(p, n_frames, stream);
}

int ofc_flow_to_hsv(const float* flow, int n_frames, int height, int width, const uint32_t* minmax, uint8_t* bgr, uint8_t* hsv,
                    void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height >= 0 && width >= 0, "bad sizes");
    const int64_t n_pixels = (int64_t)height * width;
    if (n_frames == 0 || n_pixels == 0) return OFC_OK;
    OFC_REQUIRE(flow && minmax && bgr && hsv, "null buffer");
    OFC_REQUIRE(((uintptr_t)flow & 15) == 0 && ((uintptr_t)bgr & 3) == 0 && ((uintptr_t)hsv & 3) == 0,
                "flow must be 16-byte, bgr / hsv 4-byte aligned");
    VizParams p;
    p.flow = (const float2*)flow; p.n_px = n_pixels; p.width = width; p.minmax = minmax; p.bgr = bgr; p.mag_sum = nullptr; p.hsv = hsv;
    return launch_flow_encode(p, n_frames, stream);
}

int ofc_flow_to_bgr_grid(const float* flow, int n_frames, int height, int width, const uint32_t* minmax, uint8_t* bgr,
                         double* mag_sum, int rows, int cols, int draw_lines, int threshold, uint8_t* avg_bgr, uint8_t* avg_hue,
                         uint8_t* km_centre, uint8_t* km_hue, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height > 0 && width > 0, "bad sizes");
    OFC_REQUIRE(rows > 0 && cols > 0 && rows <= height && cols <= width, "grid %dx%d does not fit %dx%d", rows, cols, height, width);
    OFC_REQUIRE(threshold >= 0 && threshold <= 255, "bad threshold");
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(flow && minmax && bgr, "null buffer");
    OFC_REQUIRE(((uintptr_t)flow & 7) == 0, "flow must be 8-byte aligned");
    if (mag_sum) OFC_CUDA(cudaMemsetAsync(mag_sum, 0, sizeof(double) * n_frames, (cudaStream_t)stream));
    VizParams p;
    p.flow = (const float2*)flow; p.n_px = (int64_t)height * width; p.width = width; p.minmax = minmax; p.bgr = bgr;
    p.mag_sum = mag_sum; p.hsv = nullptr;
    GridParams g;
    g.bgr = bgr; g.frame_stride = (int64_t)height * width * 3;
    g.W = width; g.H = height; g.rows = rows; g.cols = cols;
    g.x_step = width / cols; g.y_step = height / rows;
    OFC_REQUIRE((int64_t)g.x_step * g.y_step * 255 < (int64_t)1 << 32, "cell too large for 32-bit sums");
    g.draw_lines = draw_lines; g.threshold = threshold;
    g.avg_bgr = avg_bgr; g.avg_hue = avg_hue; g.km_centre = km_centre; g.km_hue = km_hue; g.km_sums = nullptr;
    return launch_flow_encode_grid(p, g, n_frames, stream);
}

int ofc_grid_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols,
                   int draw_lines, int threshold, uint8_t* avg_bgr, uint8_t* avg_hue,
                   uint8_t* km_centre, uint8_t* km_hue, uint32_t* km_sums, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height > 0 && width > 0, "bad sizes");
    OFC_REQUIRE(rows > 0 && cols > 0 && rows <= height && cols <= width, "grid %dx%d does not fit %dx%d", rows, cols, height, width);
    OFC_REQUIRE(threshold >= 0 && threshold <= 255, "bad threshold");
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(bgr != nullptr, "null frame buffer");
    GridParams p;
    p.bgr = bgr; p.frame_stride = (int64_t)height * width * 3;
    p.W = width; p.H = height; p.rows = rows; p.cols = cols;
    p.x_step = width / cols; p.y_step = height / rows;       // int(width / cols)
    OFC_REQUIRE((int64_t)p.x_step * p.y_step * 255 < (int64_t)1 << 32, "cell too large for 32-bit sums");
    p.draw_lines = draw_lines; p.threshold = threshold;
    p.avg_bgr = avg_bgr; p.avg_hue = avg_hue; p.km_centre = km_centre; p.km_hue = km_hue; p.km_sums = km_sums;
    return launch_grid_cells(p, n_frames, stream);
}

int ofc_draw_grid(uint8_t* bgr, int n_frames, int height, int width, int rows, int cols, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height > 0 && width > 0 && rows > 0 && cols > 0, "bad sizes");
    OFC_REQUIRE(rows <= height && cols <= width, "grid does not fit the frame");
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(bgr != nullptr, "null frame buffer");
    return launch_draw_grid(bgr, (int64_t)height * width * 3, width, height, rows, cols,
                            width / cols, height / rows, n_frames, stream);
}

// ---- k-means ---------------------------------------------------------------
namespace {
struct KmWorkspace {
    size_t off_c2, off_inertia, off_partial, off_cnt, off_shift, total;
    size_t assign_total;         // the prefix ofc_kmeans_assign / ofc_kmeans_centres need (no M-step partials)
    int parts, splits, dt, kt;
};
// shared: the problems read one X (OFC_KMEANS_SHARED_ROWS).  Their M-step then uses the split count of ONE problem, so
// the float sums of a problem are folded in the same order whatever the batch (uint8 sums are exact in any order);
// the layout stays within batch * km_layout(1, n, d, k).total, which is what the header promises the caller.
KmWorkspace km_layout(int batch, int64_t n, int d, int k, bool shared = false) {
    KmWorkspace w;
    w.parts = kmeans_assign_grid(n);
    w.splits = kmeans_sums_splits(n, shared ? 1 : batch);
    w.dt = 1;
    while (w.dt < 32 && w.dt < d) w.dt <<= 1;
    w.kt = k < 32 ? k : 32;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    w.off_c2 = take((size_t)batch * k * 8);
    w.off_inertia = take((size_t)batch * w.parts * 8);
    w.assign_total = off;
    // per-CTA partials of the M-step kernel (splits) or of the fused uint8 step (its own grid)
    const int step_grid = kmeans_step_grid(n, batch);
    const int parts = w.splits > step_grid ? w.splits : step_grid;
    w.off_partial = take((size_t)batch * parts * k * d * 8);
    w.off_cnt = take((size_t)batch * parts * k * 8);
    w.off_shift = take((size_t)batch * k * 8);
    w.total = off;
    return w;
}
}  // namespace

size_t ofc_kmeans_workspace_bytes(int batch, int64_t n, int d, int k) {
    if (batch <= 0 || n <= 0 || d <= 0 || k <= 0) return 0;
    return km_layout(batch, n, d, k).total;
}

size_t ofc_kmeans_assign_workspace_bytes(int batch, int64_t n, int d, int k) {
    if (batch <= 0 || n <= 0 || d <= 0 || k <= 0) return 0;
    return km_layout(batch, n, d, k).assign_total;
}

// splits the dtype argument of the stepwise calls into the element type and the OFC_KMEANS_SHARED_ROWS flag
static int km_check(const void* X, int& dtype, bool& shared, int batch, int64_t n, int d, int k) {
    shared = (dtype & OFC_KMEANS_SHARED_ROWS) != 0;
    dtype &= ~OFC_KMEANS_SHARED_ROWS;
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(batch >= 0 && n >= 0 && d >= 1 && k >= 1, "bad k-means shape batch=%d n=%lld d=%d k=%d", batch, (long long)n, d, k);
    OFC_REQUIRE(batch == 0 || n == 0 || X != nullptr, "null data");
    return OFC_OK;
}

int ofc_kmeans_assign(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                      const double* centres, int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed,
                      double* inertia, double* min_dist, const uint8_t* active, void* workspace, size_t workspace_bytes,
                      void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0 || n == 0) return OFC_OK;
    OFC_REQUIRE(centres && labels, "null centres / labels");
    KmWorkspace w = km_layout(batch, n, d, k, shared);
    if (!workspace || workspace_bytes < w.assign_total) { set_error("k-means workspace too small: %zu < %zu", workspace_bytes, w.assign_total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    KmAssignParams p;
    p.X = X; p.x_stride = shared ? 0 : n * d; p.dtype = dtype; p.n = n; p.d = d; p.k = k; p.mean = mean; p.centres = centres; p.c2 = nullptr;
    p.labels = labels; p.prev_labels = prev_labels; p.n_changed = (unsigned long long*)n_changed;
    p.inertia_partial = inertia ? (double*)(ws + w.off_inertia) : nullptr;
    p.min_dist = min_dist; p.active = active;
    if (n_changed) OFC_CUDA(cudaMemsetAsync(n_changed, 0, sizeof(uint64_t) * batch, (cudaStream_t)stream));
    rc = launch_kmeans_assign(p, batch, (double*)(ws + w.off_c2), stream);
    if (rc != OFC_OK) return rc;
    if (inertia) return launch_inertia_reduce((const double*)(ws + w.off_inertia), w.parts, batch, inertia, active, stream);
    return OFC_OK;
}

int ofc_kmeans_assign_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                               const double* centres, const double* weights, int32_t* labels, const int32_t* prev_labels,
                               uint64_t* n_changed, double* inertia, double* min_dist, const uint8_t* active, void* workspace,
                               size_t workspace_bytes, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0 || n == 0) return OFC_OK;
    OFC_REQUIRE(centres && labels && weights, "null centres / labels / weights");
    KmWorkspace w = km_layout(batch, n, d, k, shared);
    if (!workspace || workspace_bytes < w.assign_total) { set_error("k-means workspace too small: %zu < %zu", workspace_bytes, w.assign_total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    KmAssignParams p;
    p.X = X; p.x_stride = shared ? 0 : n * d; p.dtype = dtype; p.n = n; p.d = d; p.k = k; p.mean = mean; p.centres = centres; p.c2 = nullptr;
    p.labels = labels; p.prev_labels = prev_labels; p.n_changed = (unsigned long long*)n_changed;
    p.inertia_partial = inertia ? (double*)(ws + w.off_inertia) : nullptr;
    p.min_dist = min_dist; p.active = active;
    p.weights = weights; p.w_stride = shared ? 0 : n;
    if (n_changed) OFC_CUDA(cudaMemsetAsync(n_changed, 0, sizeof(uint64_t) * batch, (cudaStream_t)stream));
    rc = launch_kmeans_assign(p, batch, (double*)(ws + w.off_c2), stream);
    if (rc != OFC_OK) return rc;
    if (inertia) return launch_inertia_reduce((const double*)(ws + w.off_inertia), w.parts, batch, inertia, active, stream);
    return OFC_OK;
}

int ofc_kmeans_sums(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                    const int32_t* labels, int square, double* sums, int64_t* counts, const uint8_t* active,
                    void* workspace, size_t workspace_bytes, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(sums != nullptr, "null sums");
    OFC_REQUIRE(n > 0, "empty data");
    KmWorkspace w = km_layout(batch, n, d, k, shared);
    if (!workspace || workspace_bytes < w.total) { set_error("k-means workspace too small: %zu < %zu", workspace_bytes, w.total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    KmSumsParams p;
    p.X = X; p.x_stride = shared ? 0 : n * d; p.dtype = dtype; p.n = n; p.d = d; p.k = k; p.mean = mean; p.labels = labels; p.square = square;
    p.partial = (double*)(ws + w.off_partial); p.cnt_partial = (long long*)(ws + w.off_cnt);
    p.splits = w.splits; p.dt = w.dt; p.kt = w.kt; p.active = active;
    return launch_kmeans_sums(p, batch, sums, (long long*)counts, stream);
}

int ofc_kmeans_sums_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                             const int32_t* labels, const double* weights, double* sums, double* weight_sums,
                             const uint8_t* active, void* workspace, size_t workspace_bytes, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(sums && weight_sums && labels && weights, "null sums / weight_sums / labels / weights");
    OFC_REQUIRE(n > 0, "empty data");
    KmWorkspace w = km_layout(batch, n, d, k, shared);
    if (!workspace || workspace_bytes < w.total) { set_error("k-means workspace too small: %zu < %zu", workspace_bytes, w.total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    KmSumsParams p;
    p.X = X; p.x_stride = shared ? 0 : n * d; p.dtype = dtype; p.n = n; p.d = d; p.k = k; p.mean = mean; p.labels = labels; p.square = 0;
    p.partial = (double*)(ws + w.off_partial); p.cnt_partial = nullptr;
    p.splits = w.splits; p.dt = w.dt; p.kt = w.kt; p.active = active;
    // the weight partials take the place of the count partials (8 bytes each as well)
    p.weights = weights; p.w_stride = shared ? 0 : n; p.wcnt_partial = (double*)(ws + w.off_cnt);
    return launch_kmeans_sums_weighted(p, batch, sums, weight_sums, stream);
}

int ofc_kmeans_step_supported(int dtype, int d, int k) {
    return (dtype & ~OFC_KMEANS_SHARED_ROWS) == OFC_U8 && d >= 1 && d <= 32 && k >= 1 && kmeans_step_smem(d, k) <= 200 * 1024;
}

int ofc_kmeans_step(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const double* centres,
                    int32_t* labels, const int32_t* prev_labels, uint64_t* n_changed, double* sums, int64_t* counts,
                    const uint8_t* active, void* workspace, size_t workspace_bytes, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (!ofc_kmeans_step_supported(dtype, d, k)) {
        set_error("fused k-means step needs uint8 rows, d <= 32 and [k][d] accumulators that fit shared memory (dtype=%d d=%d k=%d)", dtype, d, k);
        return OFC_ERR_UNSUPPORTED;
    }
    if (batch == 0 || n == 0) return OFC_OK;
    OFC_REQUIRE(centres && labels && sums && counts, "null buffer");
    KmWorkspace w = km_layout(batch, n, d, k, shared);
    if (!workspace || workspace_bytes < w.total) { set_error("k-means workspace too small: %zu < %zu", workspace_bytes, w.total); return OFC_ERR_WORKSPACE; }
    char* ws = (char*)workspace;
    KmAssignParams p;
    p.X = X; p.x_stride = shared ? 0 : n * d; p.dtype = dtype; p.n = n; p.d = d; p.k = k; p.mean = mean; p.centres = centres; p.c2 = nullptr;
    p.labels = labels; p.prev_labels = prev_labels; p.n_changed = (unsigned long long*)n_changed;
    p.inertia_partial = nullptr; p.min_dist = nullptr; p.active = active;
    if (n_changed) OFC_CUDA(cudaMemsetAsync(n_changed, 0, sizeof(uint64_t) * batch, (cudaStream_t)stream));
    return launch_kmeans_step_u8(p, batch, (double*)(ws + w.off_partial), (long long*)(ws + w.off_cnt), sums, (long long*)counts, stream);
}

int ofc_kmeans_centres(int batch, int d, int k, const double* sums, const int64_t* counts, const double* mean_sub,
                       int use_reciprocal, double* centres, double* shift_tot, const uint8_t* active, void* workspace,
                       size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(batch >= 0 && d >= 1 && k >= 1, "bad shape");
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(sums && counts && centres, "null buffer");
    OFC_REQUIRE(workspace && workspace_bytes >= align_up((size_t)batch * k * 8, 256), "k-means workspace too small");
    // the shift scratch is the tail of the layout for any n; use the head of the workspace here
    return launch_kmeans_centres(batch, d, k, sums, (const long long*)counts, mean_sub, use_reciprocal, centres, shift_tot,
                                 (double*)workspace, active, stream);
}

int ofc_kmeans_update(int batch, int64_t n, int d, int k, const double* sums, const int64_t* counts, const double* mean_sub,
                      int use_reciprocal, int round_f32, double* centres, double* shift_tot, const uint64_t* n_changed,
                      const double* tol, int iteration, uint8_t* active, uint8_t* just_done, int32_t* n_iter, int32_t* n_active,
                      const int32_t* labels_cur, int32_t* labels_other, int32_t* it_counter, void* workspace, size_t workspace_bytes,
                      void* stream) {
    OFC_REQUIRE(batch >= 0 && d >= 1 && k >= 1 && n >= 0, "bad shape");
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(sums && counts && centres, "null buffer");
    OFC_REQUIRE(workspace && workspace_bytes >= align_up((size_t)batch * k * 8, 256), "k-means workspace too small");
    return launch_kmeans_update(batch, d, k, sums, (const long long*)counts, mean_sub, use_reciprocal, round_f32, centres, shift_tot,
                                (double*)workspace, (const unsigned long long*)n_changed, tol, iteration, active, just_done, n_iter,
                                n_active, n, labels_cur, labels_other, it_counter, stream);
}

int ofc_kmeans_update_weighted(int batch, int64_t n, int d, int k, const double* sums, const double* weight_sums,
                               const double* mean_sub, int use_reciprocal, int round_f32, double* centres, double* shift_tot,
                               const uint64_t* n_changed, const double* tol, int iteration, uint8_t* active, uint8_t* just_done,
                               int32_t* n_iter, int32_t* n_active, const int32_t* labels_cur, int32_t* labels_other,
                               int32_t* it_counter, void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(batch >= 0 && d >= 1 && k >= 1 && n >= 0, "bad shape");
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(sums && weight_sums && centres, "null buffer");
    OFC_REQUIRE(workspace && workspace_bytes >= align_up((size_t)batch * k * 8, 256), "k-means workspace too small");
    return launch_kmeans_update(batch, d, k, sums, weight_sums, mean_sub, use_reciprocal, round_f32, centres, shift_tot,
                                (double*)workspace, (const unsigned long long*)n_changed, tol, iteration, active, just_done, n_iter,
                                n_active, n, labels_cur, labels_other, it_counter, stream);
}

int ofc_minibatch_update(const void* Xb, int dtype, int batch_rows, int d, int k, const int32_t* labels, const double* centres_old,
                         double* centres_new, double* weight_sums, void* stream) {
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(batch_rows >= 1 && d >= 1 && k >= 1, "bad shape");
    OFC_REQUIRE(Xb && labels && centres_old && centres_new && weight_sums, "null buffer");
    return launch_minibatch_update(Xb, dtype, batch_rows, d, k, labels, nullptr, centres_old, centres_new, weight_sums, stream);
}

int ofc_minibatch_update_weighted(const void* Xb, int dtype, int batch_rows, int d, int k, const int32_t* labels,
                                  const double* weights, const double* centres_old, double* centres_new, double* weight_sums,
                                  void* stream) {
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(batch_rows >= 1 && d >= 1 && k >= 1, "bad shape");
    OFC_REQUIRE(Xb && labels && weights && centres_old && centres_new && weight_sums, "null buffer");
    return launch_minibatch_update(Xb, dtype, batch_rows, d, k, labels, weights, centres_old, centres_new, weight_sums, stream);
}

int ofc_kmeans_relocate(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                        const int32_t* labels, const double* centres_old, double* sums, int64_t* counts,
                        int raw_sums, const uint8_t* active, double* scratch, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0 || n == 0) return OFC_OK;
    OFC_REQUIRE(labels && centres_old && sums && counts, "null buffer");
    return launch_kmeans_relocate(X, shared ? 0 : n * d, dtype, batch, n, d, k, mean, labels, centres_old, sums, (long long*)counts, raw_sums, active, scratch,
                                  stream);
}

int ofc_kmeans_relocate_weighted(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean,
                                 const int32_t* labels, const double* centres_old, const double* weights, double* sums,
                                 double* weight_sums, int raw_sums, const uint8_t* active, double* scratch, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (batch == 0 || n == 0) return OFC_OK;
    OFC_REQUIRE(labels && centres_old && weights && sums && weight_sums && scratch, "null buffer");
    return launch_kmeans_relocate_weighted(X, shared ? 0 : n * d, dtype, batch, n, d, k, mean, labels, centres_old, weights, shared ? 0 : n,
                                           sums, weight_sums, raw_sums, active, scratch, stream);
}

int ofc_kmeans_far_points(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                          const double* centres_old, int n_far, double* out_val, int64_t* out_idx, double* scratch, void* stream) {
    bool shared;
    int rc = km_check(X, dtype, shared, batch, n, d, k);
    if (rc != OFC_OK) return rc;
    if (shared) { set_error("ofc_kmeans_far_points: row-sharded fits take one X per problem (no OFC_KMEANS_SHARED_ROWS)"); return OFC_ERR_UNSUPPORTED; }
    OFC_REQUIRE(n_far >= 1 && n_far <= k, "n_far=%d outside [1, k]", n_far);
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(n > 0 && labels && centres_old && out_val && out_idx, "null buffer / empty shard");
    return launch_kmeans_far_points(X, dtype, batch, n, d, k, mean, labels, centres_old, n_far, out_val, (long long*)out_idx, scratch,
                                    stream);
}

int ofc_kmeans_far_payload(const void* X, int dtype, int batch, int64_t n, int d, int k, const double* mean, const int32_t* labels,
                           const double* centres_old, const int64_t* counts, int raw_sums, int n_far, int64_t row_offset,
                           double* payload, double* scratch, const uint8_t* active, void* stream) {
    if (dtype & OFC_KMEANS_SHARED_ROWS) {
        set_error("ofc_kmeans_far_payload: row-sharded fits take one X per problem (no OFC_KMEANS_SHARED_ROWS)");
        return OFC_ERR_UNSUPPORTED;
    }
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(batch >= 0 && n >= 0 && d >= 1 && k >= 1, "bad shape");
    OFC_REQUIRE(n_far >= 1 && n_far <= k, "n_far=%d outside [1, k]", n_far);
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(counts && payload && (n == 0 || (X && labels && centres_old && scratch)), "null buffer");
    return launch_kmeans_far_payload(X, dtype, batch, n, d, k, mean, labels, centres_old, (const long long*)counts, raw_sums, n_far,
                                     (long long)row_offset, payload, scratch, active, stream);
}

int ofc_kmeans_relocate_merge(int batch, int d, int k, int world, int n_far, const double* all_payload, double* sums, int64_t* counts,
                              int32_t* overflow, const uint8_t* active, void* stream) {
    OFC_REQUIRE(batch >= 0 && d >= 1 && k >= 1 && world >= 1 && n_far >= 1, "bad shape");
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(all_payload && sums && counts, "null buffer");
    OFC_REQUIRE((size_t)world * n_far <= 200 * 1024, "too many candidates");
    return launch_kmeans_relocate_merge(batch, d, k, world, n_far, all_payload, sums, (long long*)counts, overflow, active, stream);
}

int ofc_kmeans_cells(const uint8_t* X, int batch, int64_t n, int d, int k, const double* init, uint64_t seed, int max_iter,
                     double tol, int32_t* labels, double* centres, double* inertia, int32_t* n_iter, int64_t* counts,
                     void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(batch >= 0 && n >= 1 && n <= (1 << 20) && d >= 1 && d <= 8 && k >= 1 && k <= 64 && max_iter >= 0,
                "unsupported shape for the per-cell kernel: n=%lld d=%d k=%d", (long long)n, d, k);
    OFC_REQUIRE(n >= k, "n_samples=%lld should be >= n_clusters=%d.", (long long)n, k);
    if (batch == 0) return OFC_OK;
    OFC_REQUIRE(X && labels && centres && inertia && n_iter && counts, "null buffer");
    if (!init && (!workspace || workspace_bytes < (size_t)batch * n * sizeof(double))) {
        set_error("k-means++ seeding needs %zu bytes of workspace", (size_t)batch * n * sizeof(double));
        return OFC_ERR_WORKSPACE;
    }
    // the reference's own shape (4 channels, small k) runs the shared-memory / filtered form (cells_kmeans.cu):
    // same labels, centres, n_iter, counts and inertia, bit for bit (test seam: OFC_CELLS_FAST=0 keeps the first kernel)
    if (!seam_off("OFC_CELLS_FAST") && kmeans_cells_fast_supported(n, d, k)) {
        KmCellsFastParams p;
        memset(&p, 0, sizeof(p));
        p.X = X; p.n = (int)n; p.k = k; p.init = init; p.seed = seed; p.problem_offset = 0; p.max_iter = max_iter; p.tol = tol;
        p.labels = labels; p.centres = centres; p.inertia = inertia; p.n_iter = n_iter; p.counts = (long long*)counts;
        p.closest_ws = (unsigned*)workspace;
        return launch_kmeans_cells_fast(p, batch, stream);
    }
    return launch_kmeans_cells(X, batch, n, d, k, init, seed, max_iter, tol, labels, centres, inertia, n_iter,
                               (long long*)counts, (double*)workspace, stream);
}

size_t ofc_grid_kmeans_cells_workspace_bytes(int n_frames, int height, int width, int rows, int cols, int k) {
    if (n_frames <= 0 || rows <= 0 || cols <= 0 || height < rows || width < cols) return 0;
    const int64_t n = (int64_t)(height / rows) * (width / cols);
    return kmeans_cells_fast_workspace(n_frames * rows * cols, n, k, true);
}

int ofc_grid_kmeans_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols, int draw_lines,
                          int threshold, int swap_rb, int k, uint64_t seed, uint64_t first_frame, int max_iter, double tol,
                          uint8_t* dom_centre, uint8_t* dom_hue, double* centres, int64_t* counts, int32_t* n_iter,
                          void* workspace, size_t workspace_bytes, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height > 0 && width > 0, "bad sizes");
    OFC_REQUIRE(rows > 0 && cols > 0 && rows <= height && cols <= width, "grid %dx%d does not fit %dx%d", rows, cols, height, width);
    OFC_REQUIRE(threshold >= 0 && threshold <= 255 && max_iter >= 0, "bad threshold / max_iter");
    const int64_t n = (int64_t)(height / rows) * (width / cols);
    OFC_REQUIRE(k >= 1 && n >= k, "n_samples=%lld should be >= n_clusters=%d.", (long long)n, k);
    if (!kmeans_cells_fast_supported(n, 4, k)) {
        set_error("per-cell k-means on the frame needs k <= 16 and cells of at most ~40 000 pixels (k=%d, %lld pixels): "
                  "gather the cells with ofc_grid_extract_cells and call ofc_kmeans_cells", k, (long long)n);
        return OFC_ERR_UNSUPPORTED;
    }
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(bgr && (dom_centre || dom_hue || centres), "null buffer");
    const size_t need = ofc_grid_kmeans_cells_workspace_bytes(n_frames, height, width, rows, cols, k);
    if (need && (!workspace || workspace_bytes < need)) {
        set_error("k-means++ seeding needs %zu bytes of workspace", need);
        return OFC_ERR_WORKSPACE;
    }
    KmCellsFastParams p;
    memset(&p, 0, sizeof(p));
    p.bgr = bgr; p.frame_stride = (int64_t)height * width * 3; p.W = width; p.H = height; p.cols = cols; p.cells = rows * cols;
    p.x_step = width / cols; p.y_step = height / rows; p.draw_lines = draw_lines; p.threshold = threshold; p.swap_rb = swap_rb;
    p.n = (int)n; p.k = k; p.init = nullptr; p.seed = seed; p.problem_offset = first_frame * (uint64_t)(rows * cols);
    p.max_iter = max_iter; p.tol = tol;
    p.centres = centres; p.counts = (long long*)counts; p.n_iter = n_iter; p.dom_centre = dom_centre; p.dom_hue = dom_hue;
    p.closest_ws = (unsigned*)workspace;
    return launch_kmeans_cells_fast(p, n_frames * rows * cols, stream);
}

int ofc_grid_extract_cells(const uint8_t* bgr, int n_frames, int height, int width, int rows, int cols,
                           int draw_lines, int threshold, int swap_rb, uint8_t* out, void* stream) {
    OFC_REQUIRE(n_frames >= 0 && height > 0 && width > 0, "bad sizes");
    OFC_REQUIRE(rows > 0 && cols > 0 && rows <= height && cols <= width, "grid %dx%d does not fit %dx%d", rows, cols, height, width);
    OFC_REQUIRE(threshold >= 0 && threshold <= 255, "bad threshold");
    if (n_frames == 0) return OFC_OK;
    OFC_REQUIRE(bgr && out, "null buffer");
    OFC_REQUIRE(((uintptr_t)out & 3) == 0, "out must be 4-byte aligned");
    return launch_extract_cells(bgr, n_frames, height, width, rows, cols, draw_lines, threshold, swap_rb, out, stream);
}

int ofc_kmeans_distances(const void* X, int dtype, int64_t n, int d, int k, const double* centres, void* out, int out_f32,
                         void* stream) {
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(!out_f32 || dtype == OFC_F32, "float32 output needs float32 rows (dtype %d)", dtype);
    OFC_REQUIRE(n >= 0 && d >= 1 && k >= 1, "bad shape n=%lld d=%d k=%d", (long long)n, d, k);
    if (n == 0) return OFC_OK;
    OFC_REQUIRE(X && centres && out, "null buffer");
    return launch_kmeans_distances(X, dtype, n, d, k, centres, out, out_f32 ? 1 : 0, stream);
}

// ---- cosine ----------------------------------------------------------------
int ofc_sliding_cosine(const double* a, int n, const double* b, int64_t m, double* sims, double* best,
                       int64_t* best_idx, void* stream) {
    OFC_REQUIRE(n >= 1 && m >= n, "need 1 <= n <= m (n=%d, m=%lld)", n, (long long)m);
    OFC_REQUIRE(a && b && sims && best && best_idx, "null buffer");
    OFC_REQUIRE((size_t)n * 8 <= 200 * 1024, "short vector too long for shared memory (n=%d)", n);
    return launch_sliding_cosine(a, n, b, m, sims, best, (long long*)best_idx, stream);
}

int ofc_row_cosine(const void* X, int dtype, int64_t n, int d, const double* q, double* out, void* stream) {
    OFC_REQUIRE(dtype == OFC_U8 || dtype == OFC_F32 || dtype == OFC_F64, "bad dtype %d", dtype);
    OFC_REQUIRE(n >= 0 && d >= 1, "bad shape");
    if (n == 0) return OFC_OK;
    OFC_REQUIRE(X && q && out, "null buffer");
    OFC_REQUIRE((size_t)d * 8 <= 200 * 1024, "query too long for shared memory (d=%d)", d);
    return launch_row_cosine(X, dtype, n, d, q, out, stream);
}

int ofc_vector_distance(const double* a, const double* b, int64_t n, double* cos_out, double* quirk_row, double* l1,
                        void* stream) {
    OFC_REQUIRE(n >= 1 && a && b, "bad arguments");
    return launch_vector_distance(a, b, n, cos_out, quirk_row, l1, stream);
}

}  // extern "C"
