// Shared pieces of the fused Farneback iteration kernels (fb_iter.cu: the default TMA / tensor-memory / packed-fp32 kernel;
// fb_iter_scalar.cu: the round-1 scalar kernel kept as the A/B and cross-check reference).
#pragma once
#include "farneback_internal.cuh"

namespace tf {

constexpr int IT_HALO = 6, IT_WIN = 13, IT_RB = 4;    // window radius, window size, rows per M-phase batch

__device__ __forceinline__ float border_factor(int p, int n) {
    // border[] = {0.14, 0.14, 0.4472, 0.4472, 0.4472} applied from both sides
    float s = 1.f;
    if (p < 5) s *= (p < 2 ? 0.14f : 0.4472f);
    const int q = n - 1 - p;
    if (q < 5) s *= (q < 2 ? 0.14f : 0.4472f);
    return s;
}

// Tensor memory as thread-private scratch: with the 32x32b shape lane i of warp w addresses TMEM lane 32 * (w % 4) + i,
// so a column is one private 32-bit word per thread.  The prefix-sum ring of the vertical window lives there: its
// loads and stores then use the TMEM datapath (LDTM / STTM) instead of shared-memory wavefronts of the L1 data pipe,
// which is the unit that limits this kernel.
__device__ __forceinline__ void tm_ld5(float v[5], uint32_t a) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=f"(v[4]) : "r"(a + 4) : "memory");
}
__device__ __forceinline__ void tm_st5(uint32_t a, const float v[5]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(a), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(a + 4), "f"(v[4]) : "memory");
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// a*b - c*d with one rounding error in the result (Kahan)
__device__ __forceinline__ float diff_of_products(float a, float b, float c, float d) {
    const float cd = c * d;
    const float err = fmaf(-c, d, cd);
    const float dop = fmaf(a, b, -cd);
    return dop + err;
}


// The arithmetic of FarnebackUpdateMatrices after the bilinear blend, written with explicit roundings so that every kernel
// (scalar or packed, whatever its instruction schedule) forms the same bits: the compiler may otherwise contract
// a * b + c * d into an FMA around either product, differently from one instantiation to the next.
//   r[0..4] = (r2, r3, r4, r5, r6) blended and averaged with R0; (dx, dy) the flow; sc the border scale (1 inside)
__device__ __forceinline__ void terms_from_blend(float r2, float r3, float r4, float r5, float r6, float dx, float dy,
                                                 float sc, float m[5]) {
    r2 = __fadd_rn(r2, fmaf(r4, dy, __fmul_rn(r6, dx)));
    r3 = __fadd_rn(r3, fmaf(r6, dy, __fmul_rn(r5, dx)));
    if (sc != 1.f) {
        r2 = __fmul_rn(r2, sc); r3 = __fmul_rn(r3, sc); r4 = __fmul_rn(r4, sc); r5 = __fmul_rn(r5, sc); r6 = __fmul_rn(r6, sc);
    }
    const float r66 = __fmul_rn(r6, r6);
    m[0] = fmaf(r4, r4, r66);
    m[1] = __fmul_rn(__fadd_rn(r4, r5), r6);
    m[2] = fmaf(r5, r5, r66);
    m[3] = fmaf(r4, r2, __fmul_rn(r6, r3));
    m[4] = fmaf(r6, r2, __fmul_rn(r5, r3));
}
// bilinear weights of the four taps from the fractions
__device__ __forceinline__ void bilinear_weights(float fx, float fy, float& a00, float& a01, float& a10, float& a11) {
    const float gx = __fsub_rn(1.f, fx), gy = __fsub_rn(1.f, fy);
    a00 = __fmul_rn(gx, gy); a01 = __fmul_rn(fx, gy); a10 = __fmul_rn(gx, fy); a11 = __fmul_rn(fx, fy);
}
// one blended channel: ((a00 p00 + a01 p01) + a10 p10) + a11 p11 as a chain of FMAs
__device__ __forceinline__ float blend4(float a00, float a01, float a10, float a11, float p00, float p01, float p10, float p11) {
    return fmaf(a11, p11, fmaf(a10, p10, fmaf(a01, p01, __fmul_rn(a00, p00))));
}
// OpenCV's test for the attenuated band along one axis, (unsigned)(p - 5) >= (unsigned)(n - 10): p < 5 || p >= n - 5
// when n >= 10.  For n < 10 the right-hand side wraps and only n - 5 <= p < 5 passes, so on a side of 6..9 px some
// pixels within 5 px of an edge are left unattenuated unless the other axis selects them.
__device__ __forceinline__ bool border_band(int p, int n) { return (unsigned)(p - 5) >= (unsigned)(n - 10); }
// The scale of FarnebackUpdateMatrices: 1 unless either axis' band test holds, else the four edge factors multiplied
// left to right in fp32; sc_x = border_factor(x, w) is the product of the first two.
__device__ __forceinline__ float border_scale(float sc_x, bool band_x, int y, int h) {
    if (!band_x && !border_band(y, h)) return 1.f;
    float s = sc_x;
    if (y < 5) s = __fmul_rn(s, y < 2 ? 0.14f : 0.4472f);
    const int q = h - 1 - y;
    if (q < 5) s = __fmul_rn(s, q < 2 ? 0.14f : 0.4472f);
    return s;
}

// Non-caching loads of data a CTA touches once
__device__ __forceinline__ float4 ld_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ld_stream(const float2* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// Everything one pixel's FarnebackUpdateMatrices reads: R0 at the pixel, the four bilinear taps of R1 at p + flow.
struct Taps {
    float4 c;  float c4;                 // R0: (c0..c3), c4
    float4 p00, p01, p10, p11;           // R1 float4 plane taps
    float q00, q01, q10, q11;            // R1 c4 plane taps
    float fx, fy, dx, dy;                // bilinear fractions and the flow
    int y;                               // image row (replicate-clamped)
    bool inside;
};

struct RPlanes {
    const float4* R0a; const float* R0b; const float4* R1a; const float* R1b;
};

// issue the loads of one pixel (addresses are always valid; `inside` says whether the R1 taps are used)
__device__ __forceinline__ void issue_taps(Taps& t, const RPlanes& R, int w, int h, int x, int y, float2 f) {
    const int o = y * w + x;
    t.y = y;
    t.dx = f.x;
    t.dy = f.y;
    const float fx = __fadd_rn((float)x, f.x), fy = __fadd_rn((float)y, f.y);
    const float flx = floorf(fx), fly = floorf(fy);
    const int x1 = (int)flx, y1 = (int)fly;
    t.fx = __fsub_rn(fx, flx);
    t.fy = __fsub_rn(fy, fly);
    t.inside = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
    // out-of-image positions read a clamped (valid) 2x2 footprint whose values are then ignored
    const int xc = max(min(x1, w - 2), 0), yc = max(min(y1, h - 2), 0);
    const float4* a0 = R.R1a + (yc * w + xc);
    const float4* a1 = a0 + w;
    const float* b0 = R.R1b + (yc * w + xc);
    const float* b1 = b0 + w;
    t.c = ld_stream(R.R0a + o);      // touched once by this CTA: do not displace the gather footprint in L1
    t.c4 = ld_stream1(R.R0b + o);
    t.p00 = __ldg(a0);
    t.p01 = __ldg(a0 + 1);
    t.p10 = __ldg(a1);
    t.p11 = __ldg(a1 + 1);
    t.q00 = __ldg(b0);
    t.q01 = __ldg(b0 + 1);
    t.q10 = __ldg(b1);
    t.q11 = __ldg(b1 + 1);
}

// FarnebackUpdateMatrices for one pixel from its loaded taps (explicit roundings: see terms_from_blend)
__device__ __forceinline__ void matrix_from_taps(const Taps& t, int h, float sc_x, bool band_x, float m[5]) {
    float r2, r3, r4, r5, r6;
    if (t.inside) {
        float a00, a01, a10, a11;
        bilinear_weights(t.fx, t.fy, a00, a01, a10, a11);
        r2 = blend4(a00, a01, a10, a11, t.p00.x, t.p01.x, t.p10.x, t.p11.x);
        r3 = blend4(a00, a01, a10, a11, t.p00.y, t.p01.y, t.p10.y, t.p11.y);
        r4 = blend4(a00, a01, a10, a11, t.p00.z, t.p01.z, t.p10.z, t.p11.z);
        r5 = blend4(a00, a01, a10, a11, t.p00.w, t.p01.w, t.p10.w, t.p11.w);
        r6 = blend4(a00, a01, a10, a11, t.q00, t.q01, t.q10, t.q11);
        r4 = __fmul_rn(__fadd_rn(t.c.z, r4), 0.5f);
        r5 = __fmul_rn(__fadd_rn(t.c.w, r5), 0.5f);
        r6 = __fmul_rn(__fadd_rn(t.c4, r6), 0.25f);
    } else {
        r2 = r3 = 0.f;
        r4 = t.c.z;
        r5 = t.c.w;
        r6 = __fmul_rn(t.c4, 0.5f);
    }
    r2 = __fmul_rn(__fsub_rn(t.c.x, r2), 0.5f);
    r3 = __fmul_rn(__fsub_rn(t.c.y, r3), 0.5f);
    terms_from_blend(r2, r3, r4, r5, r6, t.dx, t.dy, border_scale(sc_x, band_x, t.y, h), m);
}

// Chunk grid of the strip march: rows per chunk minimising (waves of resident CTAs) x (rows a CTA marches, including its
// 2 * halo warm-up rows), for `strips` strips x 2 directions x n_pairs pairs and `slots` resident CTAs on the device.
inline int plan_chunk_rows(int h, int strips, int n_pairs, long long slots, int* n_chunks, int halo = IT_HALO) {
    int chunks = 1;
    long long best = -1;
    for (int c = 1; c <= (h / 16 > 1 ? h / 16 : 1); ++c) {
        const long long ctas = 2LL * strips * c * n_pairs;
        const long long cost = ((ctas + slots - 1) / slots) * (cdiv(h, c) + 2 * halo);
        if (best < 0 || cost < best) { best = cost; chunks = c; }
    }
    const int chunk_rows = cdiv(h, chunks);
    *n_chunks = cdiv(h, chunk_rows);
    return chunk_rows;
}

// the two kernels (selected in launch_fb_iteration)
void launch_fb_v3(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                  float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, int pf, cudaStream_t s,
                  const UpArgs* up);

// cv::resize INTER_LINEAR of one flow vector from its four source vectors, times mul; shared by flow_upsample_kernel and by
// the first iteration's fused up-sampling so that both give the same bits (explicit roundings, no contraction choices)
__device__ __forceinline__ float lerp_rn(float a, float b, float f) { return fmaf(b, f, __fmul_rn(a, __fsub_rn(1.f, f))); }
__device__ __forceinline__ float2 upsample_vec(float2 a, float2 b, float2 c, float2 d, float fx, float fy, float mul) {
    const float ax = lerp_rn(a.x, b.x, fx), ay = lerp_rn(a.y, b.y, fx);
    const float cx = lerp_rn(c.x, d.x, fx), cy = lerp_rn(c.y, d.y, fx);
    return make_float2(__fmul_rn(lerp_rn(ax, cx, fy), mul), __fmul_rn(lerp_rn(ay, cy, fy), mul));
}
void launch_fb_scalar(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                      float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, bool tmem_ring,
                      cudaStream_t s);

}  // namespace tf
