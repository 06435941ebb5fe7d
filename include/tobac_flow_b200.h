/*
 * tobac_flow_b200 — C ABI of the B200-native dense-flow hot path.
 *
 * This is the drop-in boundary: plain C, device pointers and sizes only (no torch types).  Each entry
 * point names the reference code it replaces (paths relative to the tobac-flow repository).  The
 * reference is Python on numpy + OpenCV, so a maintainer binds these with ctypes (INTEGRATION.md shows
 * the stub); `tobac_flow_b200/_lib.py` is that binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless marked "host";
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are asynchronous;
 *   - images are row-major (H, W); frame stacks (T, H, W); flow fields (H, W, 2) interleaved float32 with
 *     [...,0] = dx along W and [...,1] = dy along H   (tobac_flow/flow.py:408-416);
 *   - functions return 0 on success or a negative tf_status; tf_last_error() returns a thread-local
 *     human-readable message for the last failure.  Nothing throws, nothing falls back to the CPU.
 */
#ifndef TOBAC_FLOW_B200_H
#define TOBAC_FLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TF_ABI_VERSION 1

typedef enum tf_status {
    TF_OK = 0,
    TF_ERR_INVALID_ARGUMENT = -1,
    TF_ERR_WORKSPACE_TOO_SMALL = -2,
    TF_ERR_CUDA = -3,
    TF_ERR_UNSUPPORTED = -4
} tf_status;

/* element types of stencil operands/results */
typedef enum tf_dtype { TF_F32 = 0, TF_F64 = 1, TF_I32 = 2 } tf_dtype;

/* cv2.remap interpolation modes used by tobac_flow/convolve.py:46-54 */
typedef enum tf_interp { TF_NEAREST = 0, TF_LINEAR = 1, TF_CUBIC = 2, TF_LANCZOS4 = 3 } tf_interp;

/* per-step reducers (`func=`) the reference and its callers apply to the (n_taps, H, W) tap stack */
typedef enum tf_reducer {
    TF_RED_NONE = 0,           /* func=None: return the tap stack            convolve.py:332-345      */
    TF_RED_DIFF = 1,           /* Flow.diff reducer                          flow.py:182-186          */
    TF_RED_NANMEAN = 2,        /* lambda x: np.nanmean(x, 0)                 detection.py:53-55,187   */
    TF_RED_ANY = 3,            /* partial(np.any, axis=0)                    detection.py:313-320     */
    TF_RED_SOBEL = 4,          /* _sobel_func                                sobel.py:70-86           */
    TF_RED_SOBEL_UPHILL = 5,   /* _sobel_func_uphill                         sobel.py:32-48           */
    TF_RED_SOBEL_DOWNHILL = 6, /* _sobel_func_downhill                       sobel.py:51-67           */
    TF_RED_NANMAX = 7,         /* lambda x: np.nanmax(x, 0)   (commented-out variant, detection.py:57) */
    TF_RED_NANMIN = 8
} tf_reducer;

/* cv2.FarnebackOpticalFlow parameters; tf_fb_default_params() gives the factory defaults that
 * tobac_flow/utils/flow_utils.py:52-53 (cv2.optflow.createOptFlow_Farneback()) uses. */
typedef struct tf_fb_params {
    int num_levels;    /* 5   */
    double pyr_scale;  /* 0.5 (only 0.5 is supported) */
    int win_size;      /* 13  (odd, <= 25) */
    int num_iters;     /* 10  */
    int poly_n;        /* 5   (only 5 is supported) */
    double poly_sigma; /* 1.1 */
    float max_value;   /* clamp applied to the final flow (flow.py:60-61); <= 0 disables */
} tf_fb_params;

int tf_version(void);
const char* tf_last_error(void);
void tf_fb_default_params(tf_fb_params* p /* host */);

/* Number of pyramid levels OpenCV processes for an H x W image and, optionally, their sizes
 * (coarsest first; `hs`/`ws` host arrays of >= 8 ints, may be NULL). */
int tf_fb_level_plan(int H, int W, const tf_fb_params* p /* host */, int* hs /* host */, int* ws /* host */);

/* Host-side diagnostic: the polynomial-expansion constants of OpenCV's FarnebackPrepareGaussian for
 * (poly_n, poly_sigma): out[0..5] = g[0..5], out[6..11] = xg, out[12..17] = xxg, out[18..21] = ig11, ig03, ig33,
 * ig55.  `out` is a host array of 22 floats. */
int tf_fb_poly_constants(const tf_fb_params* p /* host */, float* out /* host */);

/* Stage-level entry points of the Farneback pipeline (parity tests against the oracle's per-stage restatement of
 * OpenCV's optflowgf.cpp; tf_farneback_pairs runs exactly these launches).
 *
 * tf_fb_pyramid_level: level image `level` (index into tf_fb_level_plan, coarsest first) of the quantised pair
 *   (q0, q1: (n_pairs, H, W) u8) = convertTo(CV_32F) -> GaussianBlur(ksize, sigma) -> resize(INTER_LINEAR), always
 *   from the full-resolution image.  out: (2 * n_pairs, h, w) fp32, image 2p = q0[p], 2p + 1 = q1[p].
 *   `workspace` as for tf_farneback_pairs.  flags bit 0: use the separable two-pass path through scratch instead of
 *   the fused tile kernels (both give the same bits).
 * tf_fb_polyexp: FarnebackPolyExp of `n_img` fp32 images I (n_img, h, w) -> R: per image `tf_fb_r_stride(h, w)`
 *   floats = a float4 plane (c0..c3 per pixel: OpenCV's r[0..3] order is c0 = d/dy, c1 = d/dx, c2 = yy, c3 = xx)
 *   followed by a float plane (c4 = xy). */
int tf_fb_pyramid_level(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, const tf_fb_params* p /* host */,
                        int level, float* out, void* workspace, size_t workspace_bytes, int flags, void* stream);
long long tf_fb_r_stride(int h, int w);
int tf_fb_polyexp(const float* I, int n_img, int h, int w, const tf_fb_params* p /* host */, float* R, void* stream);

/* Which fused-iteration kernel tf_farneback_pairs launches: 3 = the default (TMA-staged rows, tensor-memory ring, packed
 * fp32, two rows of gathers in flight, the flow up-sampling of a level fused into its first iteration), 4 = the same with
 * one row in flight, 5 = 3 with the up-sampling in its own kernel, 0 = the scalar LDG / shared-memory kernel,
 * 1 = the scalar kernel with its ring in tensor memory.  For A/B measurements and cross-check tests; the environment
 * variable TF_TMA sets the initial choice. */
int tf_fb_select_kernel(int which);

/* Bytes of scratch tf_farneback_pairs needs for `n_pairs` pairs of H x W frames. */
size_t tf_farneback_workspace_bytes(int n_pairs, int H, int W, const tf_fb_params* p /* host */);

/*
 * Per-pair normalisation + 8-bit quantisation.
 * Replaces linear_norm (tobac_flow/utils/normalisation_utils.py:59-72) followed by to_8bit(., 0, 1)
 * (:10-33) as called from calculate_flow (tobac_flow/flow.py:411-414): NaN-aware min/max over the
 * two-frame stack, scale to [0, 1], x255, non-finite -> 127 then patched from the other frame, truncate.
 * Pair p reads f0 + p*frame_stride and f1 + p*frame_stride (elements); writes q0/q1 + p*H*W.
 * `minmax_scratch`: 2*n_pairs floats.
 */
int tf_pair_normalise_u8(const float* f0, const float* f1, long long frame_stride, uint8_t* q0, uint8_t* q1,
                         int n_pairs, int H, int W, float* minmax_scratch, void* stream);

/* The same for float64 frames: numpy keeps the array dtype, so the reference then normalises in float64
 * (normalisation_utils.py:59-72, 10-33), which is not bit-identical to casting the frames to float32 first.
 * minmax_scratch: 2 * n_pairs doubles. */
int tf_pair_normalise_u8_f64(const double* f0, const double* f1, long long frame_stride, uint8_t* q0, uint8_t* q1,
                             int n_pairs, int H, int W, double* minmax_scratch, void* stream);

/*
 * Forward and backward Farneback flow for n_pairs quantised pairs.
 * Replaces of_model.calc(prev, next, None) and of_model.calc(next, prev, None)
 * (tobac_flow/flow.py:511,516; OpenCV FarnebackOpticalFlow::calc, flags = 0) including the clamp of
 * create_flow (flow.py:60-61).  Pair p: images q0/q1 + p*H*W; results fwd + p*fwd_stride and
 * bwd + p*bwd_stride (elements; calculate_flow stores them at forward_flow[i], backward_flow[i+1]).
 */
int tf_farneback_pairs(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                       long long bwd_stride, int n_pairs, int H, int W, const tf_fb_params* p /* host */,
                       void* workspace, size_t workspace_bytes, void* stream);

/* cv2.VariationalRefinement parameters; tf_vr_default_params() gives cv2.VariationalRefinement.create()'s defaults
 * (the module-level vr_model of tobac_flow/flow.py:359). */
typedef struct tf_vr_params {
    float alpha;                 /* 20   smoothness weight */
    float delta;                 /* 5    brightness-constancy weight */
    float gamma;                 /* 10   gradient-constancy weight */
    float omega;                 /* 1.6  SOR relaxation */
    int fixed_point_iterations;  /* 5 */
    int sor_iterations;          /* 5 */
    float zeta;                  /* 0.1 */
    float epsilon;               /* 0.001 */
} tf_vr_params;

void tf_vr_default_params(tf_vr_params* p /* host */);
size_t tf_vr_workspace_bytes(int n_pairs, int H, int W);

/*
 * Variational refinement of the forward and backward flow of n_pairs quantised pairs, in place.
 * Replaces vr_model.calc(prev, next, forward_flow) and vr_model.calc(next, prev, backward_flow)
 * (tobac_flow/flow.py:513-519, taken when vr_steps > 0; cv2.VariationalRefinement::calc).
 * Same pair addressing as tf_farneback_pairs.
 */
int tf_variational_refinement(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                              long long bwd_stride, int n_pairs, int H, int W, const tf_vr_params* p /* host */,
                              void* workspace, size_t workspace_bytes, void* stream);

/* cv2.DISOpticalFlow parameters (patch size 8, mean normalisation and spatial propagation on: the presets' values and
 * the only ones built).  tf_dis_default_params(p, preset) gives cv2.DISOpticalFlow_create(preset) for preset 0
 * (ULTRAFAST), 1 (FAST, the factory default) and 2 (MEDIUM), with max_value = 0. */
typedef struct tf_dis_params {
    int finest_scale;                       /* 2 / 2 / 1 (a frame too small for it lowers it, as calc() does) */
    int patch_stride;                       /* 4 / 4 / 3  (1..8) */
    int gradient_descent_iterations;        /* 12 / 16 / 25 */
    int variational_refinement_iterations;  /* 0 / 5 / 5  (fixed-point iterations of the per-scale refinement) */
    float vr_alpha, vr_delta, vr_gamma;     /* 20, 5, 10 */
    float vr_epsilon;                       /* 0.01 (the standalone refinement's default is 0.001) */
    float max_value;                        /* clamp of the final flow (create_flow's +-max_value); <= 0 disables */
} tf_dis_params;

void tf_dis_default_params(tf_dis_params* p /* host */, int preset);

/* HOST: the scales calc() runs for an H x W frame: *finest, *coarsest and, for finest <= s <= coarsest, the scale
 * image size hs[s] x ws[s] (host arrays of >= 16 ints; any pointer may be NULL).  Fails (TF_ERR_INVALID_ARGUMENT)
 * where OpenCV refuses the frame, and with TF_ERR_UNSUPPORTED where OpenCV would switch to patch size 12. */
int tf_dis_scale_plan(int H, int W, const tf_dis_params* p /* host */, int* finest, int* coarsest, int* hs /* host */,
                      int* ws /* host */);

/* Bytes of scratch tf_dis_pairs needs for `n_pairs` pairs of H x W frames (0 for a frame the plan refuses). */
size_t tf_dis_workspace_bytes(int n_pairs, int H, int W, const tf_dis_params* p /* host */);

/*
 * Forward and backward DIS flow of n_pairs quantised pairs: cv2.DISOpticalFlow.calc(q0, q1, None) and
 * .calc(q1, q0, None) with a fresh object per call, plus the +-max_value clamp.  Addressing as tf_farneback_pairs.
 */
int tf_dis_pairs(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd, long long bwd_stride,
                 int n_pairs, int H, int W, const tf_dis_params* p /* host */, void* workspace, size_t workspace_bytes,
                 void* stream);

/* Stage entry point: scale image `scale` of the DIS pyramid of each of the n_img u8 frames q (n_img, H, W) and its
 * spatialGradient: img (n_img, hs, ws) u8, gx / gy (n_img, hs, ws) int16.  workspace: tf_dis_workspace_bytes(n_img, ..) */
int tf_dis_scale_images(const uint8_t* q, int n_img, int H, int W, const tf_dis_params* p /* host */, int scale,
                        uint8_t* img, int16_t* gx, int16_t* gy, void* workspace, size_t workspace_bytes, void* stream);

/*
 * One smooth_flow_step (tobac_flow/flow.py:530-568) on n_pairs (fwd, bwd) fields in place semantics:
 * fwd' = nanmean(fwd, -warp(bwd by fwd)), bwd' = nanmean(bwd, -warp(fwd by bwd)), both from the old
 * fields; results go to fwd_out/bwd_out (must not alias the inputs).
 */
int tf_smooth_flow_step(const float* fwd, const float* bwd, float* fwd_out, float* bwd_out, long long stride,
                        int n_pairs, int H, int W, int interp, void* stream);

/*
 * Sequence end rules + clamp: forward[T-1] = -backward[T-1] (if mirror_last), backward[0] = -forward[0]
 * (if mirror_first)  (tobac_flow/flow.py:425-426), then clamp everything to +-max_value if max_value > 0
 * and `clamp_all` (flow.py:60-61).  fwd/bwd: (T, H, W, 2).
 */
int tf_flow_finalise(float* fwd, float* bwd, int T, int H, int W, float max_value, int clamp_all,
                     int mirror_first, int mirror_last, void* stream);

/*
 * Semi-Lagrangian 3x3x3 tap gather with a fused per-step reducer.
 * Replaces convolve.convolve / convolve_step / warp_flow / convolve_same_step
 * (tobac_flow/convolve.py:8-348), cv2.remap(BORDER_CONSTANT, fill) and the reducers listed in tf_reducer,
 * i.e. Flow.convolve / Flow.diff / Flow.sobel (tobac_flow/flow.py:105-234, tobac_flow/sobel.py).
 *
 *   cur0        frame t0 of the operand; frames contiguous, H*W elements apart, element type src_dtype
 *   n_frames    frames processed: t0 .. t0+n_frames-1
 *   has_prev    non-zero if frame t0-1 exists in memory at cur0 - H*W (else it is an all-`fill` frame,
 *               convolve.py:307-310);  has_next likewise for frame t0+n_frames (convolve.py:311-314)
 *   fflow0/bflow0   forward/backward flow of frame t0, (n_frames, H, W, 2) float32
 *   structure27 host array of 27 bytes, the 3x3x3 structuring element (non-zero = tap), order [t][y][x]
 *   stack_dtype the `dtype=` argument (type of the tap stack and of the result)
 *   out         reducer == TF_RED_NONE: (n_taps, n_frames, H, W) with tap stride `out_tap_stride` elements;
 *               otherwise (n_frames, H, W)
 *   fill        fill_value
 * With a reducer, outputs where the operand is NaN are set to `fill` (convolve.py:346-347).
 */
int tf_sl_convolve(const void* cur0, int n_frames, int has_prev, int has_next, const float* fflow0,
                   const float* bflow0, void* out, long long out_tap_stride, int H, int W, int src_dtype,
                   int stack_dtype, int interp, int reducer, const uint8_t* structure27 /* host */,
                   double fill, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * "Next" rows of the hot path (SURVEY.md section 8f, ranks 2 and 3): the per-frame filters of
 * detect_growth_markers and the semi-Lagrangian labelling, so the pipeline stays on the device between Flow operators.
 * Masks are uint8 (non-zero = True), one byte per pixel.
 * --------------------------------------------------------------------------------------------------------------- */

/* Bytes of scratch tf_flat_label / tf_binary_fill_holes need for a (T, H, W) stack. */
size_t tf_ccl_workspace_bytes(int T, int H, int W);

/*
 * flat_label (tobac_flow/utils/label_utils.py:143-180 -> scipy.ndimage.label with the time links of the structure
 * removed): 2-D connected components of every frame; numbering identical to scipy's (raster order of each component's
 * first pixel, continuing across frames).  connectivity 1 = cross, 2 = full 3x3 (the middle slab of `structure`).
 * labels: (T, H, W) int32 out; n_labels: device int32, may be NULL.
 */
int tf_flat_label(const uint8_t* mask, int32_t* labels, int T, int H, int W, int connectivity, int32_t* n_labels,
                  void* workspace, size_t workspace_bytes, void* stream);

/* scipy.ndimage.binary_fill_holes(mask, structure = 2-D cross per frame)  (tobac_flow/detection.py:72-87, 330-346). */
int tf_binary_fill_holes(const uint8_t* mask, uint8_t* out, int T, int H, int W, void* workspace, size_t workspace_bytes,
                         void* stream);

/*
 * scipy.ndimage.gaussian_filter(field, (0, sigma, sigma)) (detection.py:65, 149): correlate1d along y then x, 'reflect'
 * borders, fp64 accumulation in scipy's order, intermediate stored in the array dtype.  `weights` is the HOST array of
 * 2*radius+1 kernel weights exactly as scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius) returns them.
 * in/tmp/out: (T, H, W) of `dtype` (TF_F32 or TF_F64); tmp may not alias in or out.
 */
int tf_gaussian_filter_yx(const void* in, void* tmp, void* out, int dtype, int T, int H, int W,
                          const double* weights /* host */, int radius, void* stream);

/* The curvature test of get_curvature_filter (detection.py:66-70, 77, 85): second differences along x and y (zero on
 * the border), out = both < -threshold ("negative") or both > threshold (positive != 0). */
int tf_curvature_mask(const void* smoothed, uint8_t* out, int dtype, int T, int H, int W, double threshold, int positive,
                      void* stream);

/* scipy.ndimage.binary_opening(mask, structure = 2-D cross per frame)  (detection.py:75, 111, 234, 289). */
int tf_binary_opening_cross(const uint8_t* in, uint8_t* out, int T, int H, int W, void* stream);

/* scipy.ndimage.grey_opening(field, footprint = 2-D cross per frame)  (detection.py:105-107), 'reflect' borders and
 * scipy's NaN behaviour.  tmp: same shape/dtype, distinct from in and out. */
int tf_grey_opening_cross(const void* in, void* tmp, void* out, int dtype, int T, int H, int W, void* stream);

/* out[t] = (double)in[t] / dt[t]: Flow.diff(x) / get_time_diff_from_coord(x.t)[:, None, None]  (detection.py:99-101).
 * dt: device array of T doubles. */
int tf_scale_frames(const float* in, const double* dt, double* out, int T, int H, int W, void* stream);

/* out = a * mask (a's dtype; NaN * 0 stays NaN as in numpy)  (detection.py:105-108). */
int tf_mask_multiply(const void* a, const uint8_t* mask, void* out, int dtype, long long n, void* stream);

/* out = (a >= threshold)  (detection.py:111, 115). */
int tf_threshold_ge(const void* a, double threshold, uint8_t* out, int dtype, long long n, void* stream);

/* max(flat) into the device int32 *out_max (the `bins.size - 1` of label.py:139 for arbitrary input labels). */
int tf_label_max(const int32_t* flat, long long n, int32_t* out_max, void* stream);

/*
 * The overlap histogram of flow_label / flow_link_overlap (tobac_flow/label.py:139-163, 301-320;
 * find_overlapping_labels, utils/label_utils.py:352-376) for all labels at once.
 *   flat, back, fwd   n int32 each: the flat labels and the two outputs of
 *                     Flow.convolve(flat, method="nearest", structure = time taps only)  (label.py:133-137)
 *   sizes             out, n_labels+1 int32: np.bincount(flat)
 *   keys, counts      out, open-addressing table of `capacity` (a power of two) entries: key = dir<<62 | L<<31 | M with
 *                     dir 0 = forward, 1 = backward; empty slots keep key ~0
 *   flags             out, 2 int32: [0] table overflow (retry with a larger capacity), [1] a label outside 0..n_labels
 */
int tf_label_overlap_count(const int32_t* flat, const int32_t* back, const int32_t* fwd, long long n, int32_t* sizes,
                           int n_labels, unsigned long long* keys, int32_t* counts, long long capacity, int32_t* flags,
                           void* stream);

/* HOST function (all pointers host): the linking walk of label.py:139-163 over the table read back from
 * tf_label_overlap_count, in the reference's visiting order.  map[l] = final label of flat label l.  Returns the
 * number of linked objects, or a negative tf_status. */
int tf_label_link_groups(const unsigned long long* keys, const int32_t* counts, long long capacity, const int32_t* sizes,
                         int n_labels, double overlap, int absolute_overlap, int32_t* map);

/*
 * Per-label statistics for the marker filters of detect_growth_markers (tobac_flow/analysis.py:66-86:
 * filter_labels_by_length -> time extent from ndi.find_objects, filter_labels_by_mask -> labeled_comprehension(np.any)).
 * labels (T, hw) int32; mask_a / mask_b (T, hw) uint8 or NULL.  Outputs are device arrays of n_labels+1 int32:
 * tmin / tmax = first / last frame of each label (tmax = -1 when absent), any_a / any_b = 1 if the label touches the mask.
 */
int tf_label_stats(const int32_t* labels, const uint8_t* mask_a, const uint8_t* mask_b, int T, long long hw, int n_labels,
                   int32_t* tmin, int32_t* tmax, int32_t* any_a, int32_t* any_b, void* stream);

/* out[i] = map[flat[i]]  (label.py:165-170); map is a device array of n_labels+1 int32. */
int tf_relabel(const int32_t* flat, const int32_t* map, int32_t* out, long long n, int n_labels, void* stream);

/*
 * Launch accounting (used by bench.py; no reference counterpart).  Kernel classes:
 *   0 normalise, 1 pyramid, 2 polyexp, 3 flow upsample, 4 Farneback iteration (coarser levels),
 *   5 Farneback iteration at the full-resolution level, 6 semi-Lagrangian gather, 7 flow smoothing, 8 finalise,
 *   9 variational refinement, 10 labelling (flat_label, overlap graph, relabel), 11 detection filters.
 * Launch counts and algorithmic bytes are always accumulated; device time is measured with CUDA events recorded
 * on the launching stream while profiling is enabled.  tf_profile_read synchronises on the recorded events.
 */
int tf_profile_enable(int on);
int tf_profile_reset(void);
int tf_profile_read(int kernel_class, double* total_ms /* host */, double* total_bytes /* host */,
                    long long* launches /* host */);

/*
 * Semi-Lagrangian watershed flood: replaces tobac_flow._watershed.watershed_raveled (tobac_flow/_watershed.pyx:222-344) for
 * the plain watershed of its only call site (tobac_flow/watershed.py:147-160: compactness 0, no watershed lines).
 * ALL POINTERS ARE HOST POINTERS: the flood is a sequential priority queue ordered by (value, push age), as in the
 * reference.  `image`, `mask` (int8, 0 = excluded; the padded border must be 0) and `output` (int32 labels, in/out: non-zero
 * at the `n_markers` raveled `marker_locations`) have `n` elements; `structure[n_neighbors]` are the raveled neighbour
 * offsets; `forward_offset` / `backward_offset` (n elements) the raveled rounded flow displacement of every pixel, added to
 * the neighbours flagged in `forward_offset_locations` / `backward_offset_locations` (the t + 1 / t - 1 neighbours).
 */
int tf_watershed_flood_host(const float* image, const long long* marker_locations, long long n_markers,
                            const long long* structure, int n_neighbors, const int* forward_offset,
                            const int* backward_offset, const int* forward_offset_locations,
                            const int* backward_offset_locations, const signed char* mask, int* output, long long n);

#ifdef __cplusplus
}
#endif
#endif /* TOBAC_FLOW_B200_H */
