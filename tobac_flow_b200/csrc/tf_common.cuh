// Shared helpers for the tobac_flow_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tobac_flow_b200.h"

namespace tf {

void set_error(const char* fmt, ...);

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return TF_ERR_CUDA;
    }
    return TF_OK;
}

inline int cdiv(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// host-side cvRound (round half to even)
inline int cv_round(double v) { return (int)nearbyint(v); }

constexpr int kMaxLevels = 16;

struct LevelPlan {
    int n;                 // number of levels processed (coarsest first)
    int h[kMaxLevels], w[kMaxLevels], k[kMaxLevels], ksize[kMaxLevels];
    double sigma[kMaxLevels];
};

LevelPlan make_level_plan(int H, int W, const tf_fb_config& c);

// kernel classes for launch accounting (tf_profile_*)
enum KClass {
    KC_NORMALISE = 0, KC_PYRAMID, KC_POLYEXP, KC_UPSAMPLE, KC_FB_ITER, KC_FB_ITER_L0, KC_GATHER, KC_SMOOTH, KC_FINALISE,
    KC_VR, KC_LABEL, KC_MORPH, KC_COUNT
};

// RAII launch record: counts launches / algorithmic bytes, and times the enclosed launches with CUDA events on `s`
// when profiling is enabled.
class LaunchTimer {
public:
    LaunchTimer(int klass, double bytes, cudaStream_t s, int n_launches = 1);
    ~LaunchTimer();
    LaunchTimer(const LaunchTimer&) = delete;
    LaunchTimer& operator=(const LaunchTimer&) = delete;
private:
    int klass_;
    cudaStream_t s_;
    cudaEvent_t b_;
};

// streaming global loads/stores (data touched once per kernel: keep it out of L1)
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }

}  // namespace tf
