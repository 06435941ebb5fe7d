// Host orchestration of the batched coarse-to-fine Farneback schedule + small C-ABI entry points.
// Mirrors the control flow of OpenCV FarnebackOpticalFlowImpl::calc (fastPyramids = false, no initial flow) as the
// reference drives it from tobac_flow/flow.py:499-527, for a batch of pairs and both directions at once: the level images and polynomial
// expansions of a pair are shared by the forward and the backward flow (only the roles of R0/R1 swap).
#include <stdarg.h>
#include <string.h>

#include "farneback_internal.cuh"

namespace tf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

LevelPlan make_level_plan(int H, int W, const tf_fb_config& p) {
    LevelPlan lp{};
    const int min_size = 32;
    int k = 0;
    double scale = 1;
    for (; k < p.num_levels; ++k) {
        scale *= p.pyr_scale;
        if (W * scale < min_size || H * scale < min_size) break;
    }
    const int levels = k;
    lp.n = 0;
    for (k = levels; k >= 0 && lp.n < kMaxLevels; --k) {
        scale = 1;
        for (int i = 0; i < k; ++i) scale *= p.pyr_scale;
        const double sigma = (1. / scale - 1) * 0.5;
        int ksize = cv_round(sigma * 5) | 1;
        ksize = ksize > 3 ? ksize : 3;
        lp.k[lp.n] = k;
        lp.sigma[lp.n] = sigma;
        lp.ksize[lp.n] = ksize;
        lp.w[lp.n] = cv_round(W * scale);
        lp.h[lp.n] = cv_round(H * scale);
        ++lp.n;
    }
    return lp;
}

struct Workspace {
    float* tmp;    // blur pass A scratch   (2P, rows, W)
    float* I;      // level images          (2P, h, w)
    float* R;      // polynomial expansion  (2P, 5, h, w)
    float* flow[3];  // (P, 2, h, w, 2) ping / pong / previous level
    int* tab;        // resize tables of the fused flow up-sampling: x0 (W) | fx (W) | y0 (H) | fy (H)
    size_t total;
};

static Workspace carve(void* base, int n_pairs, int H, int W, const LevelPlan& lp) {
    // pass A scratch: max over levels of rows*W where rows = h (level 0) or 2h
    size_t tmp_px = 0;
    for (int i = 0; i < lp.n; ++i) {
        const size_t rows = (lp.h[i] == H) ? (size_t)lp.h[i] : (size_t)2 * lp.h[i];
        tmp_px = rows * W > tmp_px ? rows * W : tmp_px;
    }
    const size_t N = (size_t)H * W, P = (size_t)n_pairs;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 256);
        return o;
    };
    const size_t o_tmp = take(2 * P * tmp_px * 4), o_I = take(2 * P * N * 4), o_R = take(2 * P * (size_t)r_img_stride(H, W) * 4);
    const size_t o_f0 = take(P * 2 * N * 8), o_f1 = take(P * 2 * N * 8), o_f2 = take(P * 2 * N * 8);
    const size_t o_tab = take(2 * ((size_t)H + W) * 4);
    Workspace ws{};
    char* b = reinterpret_cast<char*>(base);
    ws.tmp = reinterpret_cast<float*>(b + o_tmp);
    ws.I = reinterpret_cast<float*>(b + o_I);
    ws.R = reinterpret_cast<float*>(b + o_R);
    ws.flow[0] = reinterpret_cast<float*>(b + o_f0);
    ws.flow[1] = reinterpret_cast<float*>(b + o_f1);
    ws.flow[2] = reinterpret_cast<float*>(b + o_f2);
    ws.tab = reinterpret_cast<int*>(b + o_tab);
    // tail pad: the staged (bulk-copy) rows of the iteration kernel are rounded up to 16-byte granules and may read a
    // few bytes past the last flow row
    ws.total = off + 256;
    return ws;
}

static int validate_params(const tf_fb_params* p) {
    if (!p) { set_error("farneback: params is NULL"); return TF_ERR_INVALID_ARGUMENT; }
    if (p->pyr_scale != 0.5) { set_error("farneback: only pyr_scale 0.5 is supported"); return TF_ERR_UNSUPPORTED; }
    if (p->poly_n != 5) { set_error("farneback: only poly_n 5 is supported"); return TF_ERR_UNSUPPORTED; }
    if (p->win_size != 13) { set_error("farneback: only win_size 13 is supported"); return TF_ERR_UNSUPPORTED; }
    if (p->num_levels < 0 || p->num_levels > 7 || p->num_iters < 1) {
        set_error("farneback: num_levels/num_iters out of range");
        return TF_ERR_INVALID_ARGUMENT;
    }
    return TF_OK;
}

static tf_fb_config to_config(const tf_fb_params& p) {
    tf_fb_config c{};
    c.num_levels = p.num_levels;
    c.pyr_scale = p.pyr_scale;
    c.win_size = p.win_size;
    c.num_iters = p.num_iters;
    c.poly_n = p.poly_n;
    c.poly_sigma = p.poly_sigma;
    c.max_value = p.max_value;
    c.flags = 0;
    return c;
}

// The range the GPU reproduces OpenCV over.  Gaussian windows of 2 and 3 (radius 1, sigma 0.3) and the box window of 1
// are excluded although OpenCV accepts them: their solve is so ill-conditioned that fp32 and OpenCV's arithmetic end
// up hundreds of pixels apart.
static int validate_config(const tf_fb_config* c) {
    if (!c) { set_error("farneback: config is NULL"); return TF_ERR_INVALID_ARGUMENT; }
    const bool gauss = c->flags == TF_FB_GAUSSIAN;
    const char* bad = nullptr;
    if (c->num_levels < 0 || c->num_levels > kMaxLevels - 1) bad = "num_levels must be in 0..15";
    else if (!(c->pyr_scale > 0 && c->pyr_scale < 1)) bad = "pyr_scale must be in (0, 1)";
    else if (c->num_iters < 1) bad = "num_iters must be >= 1";
    else if (c->poly_n != 5 && c->poly_n != 7) bad = "poly_n must be 5 or 7";
    else if (!(c->poly_sigma > 0)) bad = "poly_sigma must be > 0";
    else if (c->flags != 0 && !gauss) bad = "flags must be 0 or 256 (OPTFLOW_FARNEBACK_GAUSSIAN)";
    else if (c->win_size < (gauss ? 4 : 3) || c->win_size > 63)
        bad = gauss ? "win_size must be in 4..63 with the Gaussian window" : "win_size must be in 3..63";
    if (bad) { set_error("farneback: %s", bad); return TF_ERR_INVALID_ARGUMENT; }
    return TF_OK;
}

static int level_plan_impl(int H, int W, const tf_fb_config& c, int* hs, int* ws) {
    LevelPlan lp = make_level_plan(H, W, c);
    for (int i = 0; i < lp.n; ++i) {
        if (hs) hs[i] = lp.h[i];
        if (ws) ws[i] = lp.w[i];
    }
    return lp.n;
}

static int pyramid_level_impl(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, const tf_fb_config& c,
                              int level, float* out, void* workspace, size_t workspace_bytes, int flags, void* stream) {
    if (!q0 || !q1 || !out || !workspace || n_pairs < 0 || H <= 0 || W <= 0) {
        set_error("tf_fb_pyramid_level: invalid argument");
        return TF_ERR_INVALID_ARGUMENT;
    }
    const LevelPlan lp = make_level_plan(H, W, c);
    if (level < 0 || level >= lp.n) { set_error("tf_fb_pyramid_level: level %d out of range (%d levels)", level, lp.n); return TF_ERR_INVALID_ARGUMENT; }
    const Workspace ws = carve(workspace, n_pairs, H, W, lp);
    if (ws.total > workspace_bytes) {
        set_error("tf_fb_pyramid_level: workspace too small (%zu < %zu)", workspace_bytes, ws.total);
        return TF_ERR_WORKSPACE_TOO_SMALL;
    }
    return launch_pyramid_level(q0, q1, n_pairs, H, W, lp.h[level], lp.w[level], lp.ksize[level], lp.sigma[level], ws.tmp, out,
                                (cudaStream_t)stream, (flags & 1) != 0);
}

static int polyexp_impl(const float* I, int n_img, int h, int w, const tf_fb_config& c, float* R, void* stream) {
    if (!I || !R || n_img < 0 || h <= 0 || w <= 0) { set_error("tf_fb_polyexp: invalid argument"); return TF_ERR_INVALID_ARGUMENT; }
    const PolyConsts pc = make_poly_consts(c.poly_n, c.poly_sigma);
    return launch_polyexp(I, R, r_img_stride(h, w), n_img, h, w, pc, (cudaStream_t)stream);
}

static int farneback_pairs_impl(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                                long long bwd_stride, int n_pairs, int H, int W, const tf_fb_config& c, void* workspace,
                                size_t workspace_bytes, void* stream);

}  // namespace tf

using namespace tf;

extern "C" int tf_version(void) { return TF_ABI_VERSION; }
extern "C" const char* tf_last_error(void) { return g_err; }

extern "C" void tf_fb_default_params(tf_fb_params* p) {
    if (!p) return;
    p->num_levels = 5;
    p->pyr_scale = 0.5;
    p->win_size = 13;
    p->num_iters = 10;
    p->poly_n = 5;
    p->poly_sigma = 1.1;
    p->max_value = 20.f;
}

extern "C" int tf_fb_level_plan(int H, int W, const tf_fb_params* p, int* hs, int* ws) {
    if (validate_params(p) != TF_OK || H <= 0 || W <= 0) return TF_ERR_INVALID_ARGUMENT;
    return level_plan_impl(H, W, to_config(*p), hs, ws);
}

extern "C" int tf_fb_poly_constants(const tf_fb_params* p, float* out) {
    if (validate_params(p) != TF_OK || !out) return TF_ERR_INVALID_ARGUMENT;
    const PolyConsts pc = make_poly_consts(p->poly_n, p->poly_sigma);
    for (int i = 0; i < 6; ++i) { out[i] = pc.g[i]; out[6 + i] = pc.xg[i]; out[12 + i] = pc.xxg[i]; }
    out[18] = pc.ig11; out[19] = pc.ig03; out[20] = pc.ig33; out[21] = pc.ig55;
    return TF_OK;
}

extern "C" size_t tf_farneback_workspace_bytes(int n_pairs, int H, int W, const tf_fb_params* p) {
    if (validate_params(p) != TF_OK || n_pairs <= 0 || H <= 0 || W <= 0) return 0;
    return carve(nullptr, n_pairs, H, W, make_level_plan(H, W, to_config(*p))).total;
}

extern "C" int tf_fb_pyramid_level(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, const tf_fb_params* p,
                                   int level, float* out, void* workspace, size_t workspace_bytes, int flags, void* stream) {
    if (n_pairs == 0) return TF_OK;
    int rc = validate_params(p);
    if (rc != TF_OK) return rc;
    return pyramid_level_impl(q0, q1, n_pairs, H, W, to_config(*p), level, out, workspace, workspace_bytes, flags, stream);
}

extern "C" long long tf_fb_r_stride(int h, int w) { return r_img_stride(h, w); }

extern "C" int tf_fb_polyexp(const float* I, int n_img, int h, int w, const tf_fb_params* p, float* R, void* stream) {
    if (n_img == 0) return TF_OK;
    int rc = validate_params(p);
    if (rc != TF_OK) return rc;
    return polyexp_impl(I, n_img, h, w, to_config(*p), R, stream);
}

extern "C" int tf_farneback_pairs(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                                  long long bwd_stride, int n_pairs, int H, int W, const tf_fb_params* p, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    if (n_pairs == 0) return TF_OK;
    int rc = validate_params(p);
    if (rc != TF_OK) return rc;
    return farneback_pairs_impl(q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W, to_config(*p), workspace,
                                workspace_bytes, stream);
}

extern "C" void tf_fb_config_default(tf_fb_config* c) {
    if (!c) return;
    tf_fb_params p;
    tf_fb_default_params(&p);
    *c = to_config(p);
}

extern "C" int tf_fb_config_level_plan(int H, int W, const tf_fb_config* c, int* hs, int* ws) {
    int rc = validate_config(c);
    if (rc != TF_OK) return rc;
    if (H <= 0 || W <= 0) { set_error("tf_fb_config_level_plan: invalid frame size"); return TF_ERR_INVALID_ARGUMENT; }
    return level_plan_impl(H, W, *c, hs, ws);
}

extern "C" size_t tf_fb_config_workspace_bytes(int n_pairs, int H, int W, const tf_fb_config* c) {
    if (validate_config(c) != TF_OK || n_pairs <= 0 || H <= 0 || W <= 0) return 0;
    return carve(nullptr, n_pairs, H, W, make_level_plan(H, W, *c)).total;
}

extern "C" int tf_fb_config_pyramid_level(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W,
                                          const tf_fb_config* c, int level, float* out, void* workspace,
                                          size_t workspace_bytes, int flags, void* stream) {
    if (n_pairs == 0) return TF_OK;
    int rc = validate_config(c);
    if (rc != TF_OK) return rc;
    return pyramid_level_impl(q0, q1, n_pairs, H, W, *c, level, out, workspace, workspace_bytes, flags, stream);
}

extern "C" int tf_fb_config_polyexp(const float* I, int n_img, int h, int w, const tf_fb_config* c, float* R, void* stream) {
    if (n_img == 0) return TF_OK;
    int rc = validate_config(c);
    if (rc != TF_OK) return rc;
    return polyexp_impl(I, n_img, h, w, *c, R, stream);
}

extern "C" int tf_farneback_config_pairs(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                                         long long bwd_stride, int n_pairs, int H, int W, const tf_fb_config* c,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    if (n_pairs == 0) return TF_OK;
    int rc = validate_config(c);
    if (rc != TF_OK) return rc;
    return farneback_pairs_impl(q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W, *c, workspace, workspace_bytes,
                                stream);
}

namespace tf {

static int farneback_pairs_impl(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                                long long bwd_stride, int n_pairs, int H, int W, const tf_fb_config& c, void* workspace,
                                size_t workspace_bytes, void* stream) {
    const tf_fb_config* p = &c;
    int rc;
    if (!q0 || !q1 || !fwd || !bwd || !workspace || n_pairs < 0 || H <= 0 || W <= 0) {
        set_error("tf_farneback_pairs: invalid argument");
        return TF_ERR_INVALID_ARGUMENT;
    }
    if ((long long)H * W > 0x3fffffffLL) { set_error("tf_farneback_pairs: frame too large"); return TF_ERR_INVALID_ARGUMENT; }
    cudaStream_t s = (cudaStream_t)stream;
    const LevelPlan lp = make_level_plan(H, W, *p);
    const Workspace ws = carve(workspace, n_pairs, H, W, lp);
    if (ws.total > workspace_bytes) {
        set_error("tf_farneback_pairs: workspace too small (%zu < %zu)", workspace_bytes, ws.total);
        return TF_ERR_WORKSPACE_TOO_SMALL;
    }
    const PolyConsts pc = make_poly_consts(p->poly_n, p->poly_sigma);
    // the default kernel (fb_iter.cu) is built for the 13 x 13 box window only; every other window runs the general one
    const bool default_kernel = p->win_size == 13 && p->flags == 0;
    const bool gaussian = p->flags == TF_FB_GAUSSIAN;
    auto iterate = [&](const float* f_in, float* o_fwd, long long o_fwd_stride, float* o_bwd, long long o_bwd_stride,
                       int h, int w, float clamp, bool full_res, const UpArgs* upp) {
        if (default_kernel)
            return launch_fb_iteration(ws.R, r_img_stride(h, w), f_in, o_fwd, o_fwd_stride, o_bwd, o_bwd_stride, n_pairs, h,
                                       w, p->win_size, clamp, full_res, s, upp);
        return launch_fb_iteration_general(ws.R, r_img_stride(h, w), f_in, o_fwd, o_fwd_stride, o_bwd, o_bwd_stride,
                                           n_pairs, h, w, p->win_size, gaussian, clamp, full_res, s);
    };

    float* prev_flow = nullptr;  // flow of the previous (coarser) level
    int ph = 0, pw = 0;
    int cur = 0;                 // index of the buffer holding the current level's flow
    for (int li = 0; li < lp.n; ++li) {
        const int h = lp.h[li], w = lp.w[li];
        const bool last_level = (li == lp.n - 1);
        // level images + polynomial expansion for the 2*n_pairs images
        rc = launch_pyramid_level(q0, q1, n_pairs, H, W, h, w, lp.ksize[li], lp.sigma[li], ws.tmp, ws.I, s);
        if (rc != TF_OK) return rc;
        const long long rs = r_img_stride(h, w);
        rc = launch_polyexp(ws.I, ws.R, rs, 2 * n_pairs, h, w, pc, s);
        if (rc != TF_OK) return rc;
        // initial flow: zeros at the coarsest level, else resize(prev) * (1 / pyr_scale) -- formed inside the first
        // iteration from the previous level's result (UpArgs) when the default kernel runs, else by its own kernel
        float* f_in = ws.flow[cur];
        const bool fuse_up = prev_flow != nullptr && default_kernel && fb_iteration_can_fuse_upsample();
        UpArgs up{};
        if (fuse_up) {
            up.coarse = prev_flow;
            up.x0 = ws.tab; up.fx = reinterpret_cast<float*>(ws.tab + W);
            up.y0 = ws.tab + 2 * W; up.fy = reinterpret_cast<float*>(ws.tab + 2 * W + H);
            up.sh = ph; up.sw = pw; up.mul = (float)(1.0 / p->pyr_scale);
            rc = launch_resize_tables(ws.tab, reinterpret_cast<float*>(ws.tab + W), w, pw, ws.tab + 2 * W,
                                      reinterpret_cast<float*>(ws.tab + 2 * W + H), h, ph, s);
        } else {
            rc = launch_flow_upsample(prev_flow, f_in, 2 * n_pairs, ph, pw, h, w, (float)(1.0 / p->pyr_scale), s);
        }
        if (rc != TF_OK) return rc;
        float* f_a = f_in;
        float* f_b = ws.flow[(cur + 1) % 3];
        const long long lvl_stride = (long long)2 * h * w * 2;  // [pair] stride of the (P, 2, h, w, 2) buffers
        for (int it = 0; it < p->num_iters; ++it) {
            const bool final_write = last_level && it == p->num_iters - 1;
            const UpArgs* upp = (fuse_up && it == 0) ? &up : nullptr;
            if (final_write) rc = iterate(f_a, fwd, fwd_stride, bwd, bwd_stride, h, w, p->max_value, last_level, upp);
            else rc = iterate(f_a, f_b, lvl_stride, f_b + (long long)h * w * 2, lvl_stride, h, w, 0.f, last_level, upp);
            if (rc != TF_OK) return rc;
            float* t = f_a; f_a = f_b; f_b = t;
        }
        // f_a now holds this level's result (unless it went straight to fwd/bwd)
        prev_flow = f_a;
        ph = h; pw = w;
        // choose a buffer for the next level that is neither prev_flow nor its ping-pong partner-in-use
        int idx_a = 0;
        for (int i = 0; i < 3; ++i) if (ws.flow[i] == f_a) idx_a = i;
        cur = (idx_a + 1) % 3;
    }
    return TF_OK;
}

}  // namespace tf
