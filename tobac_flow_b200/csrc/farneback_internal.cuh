// Internal launch interfaces shared by the Farneback translation units.
#pragma once
#include "tf_common.cuh"

namespace tf {

constexpr int kMaxBlurTaps = 96;
struct BlurTaps {
    int ksize;
    float w[kMaxBlurTaps];
};

// Levels of a frame at most 5424 px on its short side need up to 421 taps (one level at pyr_scale 32 / 5424);
// blurs wider than kMaxBlurTaps take the two-pass kernels with these taps.
constexpr int kMaxWideBlurTaps = 511;
struct WideBlurTaps {
    int ksize;
    float w[kMaxWideBlurTaps];
};

struct PolyConsts {
    int n;                      // poly_n: 5 or 7
    float g[8], xg[8], xxg[8];  // g[k], k = 0..n (symmetric / antisymmetric about 0)
    float ig11, ig03, ig33, ig55;
};
PolyConsts make_poly_consts(int n, double sigma);

// level image for 2*n_pairs images: out (2*n_pairs, h, w); tmp >= 2*n_pairs * rows*W floats
// two_pass: the separable path through `tmp` instead of the fused tile kernels (same bits; kept for parity tests)
// ksize > kMaxBlurTaps: the two-pass path with WideBlurTaps (two_pass is then implied)
int launch_pyramid_level(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, int h, int w, int ksize,
                         double sigma, float* tmp, float* out, cudaStream_t s, bool two_pass = false);

// dst (n_fields, h, w, 2) = resize(src (n_fields, sh, sw, 2)) * mul; src == nullptr -> zeros
int launch_flow_upsample(const float* src, float* dst, int n_fields, int sh, int sw, int h, int w, float mul,
                         cudaStream_t s);

// R: per image `img_stride` floats (a multiple of 4): a float4 plane (c0..c3) of h*w texels, then a float plane (c4)
inline long long r_img_stride(int h, int w) { return ((long long)5 * h * w + 3) / 4 * 4; }
int launch_polyexp(const float* I, float* R, long long img_stride, int n_img, int h, int w, const PolyConsts& pc,
                   cudaStream_t s);

// The flow up-sampling of a level fused into its first iteration (the default kernel only): instead of reading the level's
// initial flow, the kernel forms it from the previous (coarser) level's result with cv::resize's bilinear weights.
//   coarse (n_pairs, 2, sh, sw, 2); x0 / fx (w entries) and y0 / fy (h entries): first source index and weight of the
//   second one per destination column / row (launch_resize_tables); mul = 1 / pyr_scale
struct UpArgs {
    const float* coarse;
    const int* x0;
    const float* fx;
    const int* y0;
    const float* fy;
    int sh, sw;
    float mul;
};
int launch_resize_tables(int* x0, float* fx, int w, int sw, int* y0, float* fy, int h, int sh, cudaStream_t s);
bool fb_iteration_can_fuse_upsample();

// One Jacobi iteration (UpdateMatrices + 13x13 box + 2x2 solve) for n_pairs x 2 directions.
//   R          2*n_pairs images in the layout above: image 2p = prev, 2p+1 = next
//   flow_in    (n_pairs, 2, h, w, 2)   [pair][direction]
//   out_fwd/out_bwd + p*stride: where direction 0 / 1 results go (h, w, 2)
//   clamp > 0: clamp results to +-clamp
//   up != nullptr: flow_in is ignored, the initial flow is up-sampled from up->coarse inside the kernel
int launch_fb_iteration(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride, float* out_bwd,
                        long long bwd_stride, int n_pairs, int h, int w, int win, float clamp, bool full_res, cudaStream_t s,
                        const UpArgs* up = nullptr);

// The same Jacobi iteration for any window: box (win_size 3..63) or, with `gaussian`, OpenCV's Gaussian window
// (win_size 4..63).  Same buffers and addressing as launch_fb_iteration, no fused up-sampling.
int launch_fb_iteration_general(const float* R, long long img_stride, const float* flow_in, float* out_fwd,
                                long long fwd_stride, float* out_bwd, long long bwd_stride, int n_pairs, int h, int w,
                                int win, bool gaussian, float clamp, bool full_res, cudaStream_t s);

}  // namespace tf
