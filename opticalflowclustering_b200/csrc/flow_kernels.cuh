// Kernel parameter blocks and launchers of flow_kernels.cu (internal header).
#pragma once
#include "ofc_common.cuh"

namespace ofc {

struct PrefilterParams {
    const unsigned char* gray;   // [n_frames][H][W]
    int64_t gray_stride;         // bytes between frames
    float* out;                  // [n_frames][h][w]
    int64_t out_stride;          // floats between frames
    int W, H, w, h;              // source / level size
    int ksz;                     // Gaussian taps (odd)
    double sx, sy;               // source/level ratio used by cv::resize
    const float* taps;           // device, ksz floats
    int tx, ty;                  // output tile
    int in_rows, in_pitch;       // staged source window (max over tiles)
    int taps_pad;
    int identity3;               // level is full resolution with the fixed [1/4,1/2,1/4] taps
};

struct PolyParams {
    const float* I;
    int64_t in_stride;
    float4* RA;
    float* RB;
    int64_t out_stride;          // pixels between frames
    int w, h;
    float g[8], xg[8], xxg[8];
    float ig11, ig03, ig33, ig55;
};

struct IterParams {
    const float4* RA;            // level's R for frame 0 of the batch
    const float* RB;
    int64_t r_stride;            // pixels between the "prev" frames of consecutive pairs
    int64_t r_next;              // pixels from a pair's "prev" frame to its "next" frame
    const float2* flow_in;       // null -> zero flow
    int64_t flow_in_stride;      // float2 between pairs
    int upsample;                // flow_in is the coarser level: bilinear resize * flow_mul
    int wc, hc;
    double usx, usy, flow_mul;
    float solve_c_hi, solve_c_lo; // 1e-3 / blur_scale^2 as two floats (solve2x2)
    float2* flow_out;
    int64_t flow_out_stride;
    int w, h;
    unsigned* minmax;            // [n_pairs][2] float bits (min, max) of |flow|, or null
    float border[5];
    double blur_scale;           // 1 / winsize^2
};

// OPTFLOW_FARNEBACK_GAUSSIAN window: k[0] centre tap, k[i] the tap at distance i (2r+1 taps)
struct GaussWindow {
    int r;
    float k[33];
    double scale;                // applied to the window sums before the solve (1 for the Gaussian window)
};

int launch_prefilter(const PrefilterParams& p, int n_frames, size_t smem, void* stream);
// all down-sampled levels whose size is an exact power-of-two fraction of the frame in ONE launch
// (prefilter_pyr_kernel); done[i] is set for the levels it covered, the others go through launch_prefilter
int launch_prefilter_pyramid(const PrefilterParams* levels, int n_levels, int n_frames, bool* done, void* stream);
// gray != null: full-resolution level with the fixed 3-tap pre-filter; I is produced from the 8-bit
// frame inside the expansion kernel (and written to I_out as a by-product)
int launch_polyexp(const PolyParams& p, int poly_n, int n_frames, const unsigned char* gray, int64_t gray_stride,
                   float* I_out, void* stream);
// scratch: a flow-sized buffer [n_pairs][h][w] the launch may overwrite (up-sampled input flow)
// gw != null: Gaussian window (cv2 flag 256) instead of the winsize x winsize box
int launch_flow_iter(const IterParams& p, int winsize, int n_pairs, float2* scratch, void* stream, const GaussWindow* gw = nullptr);
// cv::resize(INTER_AREA) of full-resolution flow fields to a coarser level, times mul (cv2 flag 4)
int launch_flow_area_seed(const float2* src, int64_t src_stride, int W, int H, float2* dst, int64_t dst_stride, int w, int h,
                          float mul, int n_pairs, void* stream);
int launch_minmax_init(unsigned* mm, int n_pairs, void* stream);

}  // namespace ofc
