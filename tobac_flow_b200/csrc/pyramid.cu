// K2: one pyramid level = convertTo(CV_32F) -> GaussianBlur(ksize, sigma, REFLECT_101) -> resize(INTER_LINEAR),
// always from the full-resolution u8 image (OpenCV FarnebackOpticalFlow::calc, fastPyramids = false).
// K6: bilinear flow up-sampling (resize(prevFlow) * 1/pyrScale).
//
// Only the source rows/columns the bilinear resize actually reads are blurred: pass A blurs vertically at the
// (at most two) source rows of every destination row, pass B blurs those rows horizontally at the (at most two)
// source columns of every destination pixel and combines the four values with OpenCV's resize weights.
#include <stdlib.h>

#include "tf_common.cuh"
#include "farneback_internal.cuh"
#include "fb_iter_common.cuh"

namespace tf {

__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) {
        if (i < 0) i = -i;
        if (i >= n) i = 2 * (n - 1) - i;
    }
    return i;
}

// cv::resize INTER_LINEAR source coordinate: index of the first tap and fp32 weight of the second
__device__ __forceinline__ void resize_coord(int d, double scale, int src_n, int& i0, int& i1, float& f) {
    float fx = (float)((d + 0.5) * scale - 0.5);
    int ix = (int)floorf(fx);
    fx -= (float)ix;
    if (ix < 0) { fx = 0.f; ix = 0; }
    if (ix >= src_n - 1) { fx = 0.f; ix = src_n - 1; }
    i0 = ix;
    i1 = min(ix + 1, src_n - 1);
    f = fx;
}

// pass A.  tmp: (n_img, h*rp, W) fp32, rp = rows per destination row (1 when h == H, else 2)
// (Taps: BlurTaps, or WideBlurTaps for the blurs wider than kMaxBlurTaps)
template <class Taps>
__global__ void __launch_bounds__(256) blur_v_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                     float* __restrict__ tmp, int H, int W, int h, int rp,
                                                     double scale_y, Taps taps) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    const int img = blockIdx.z;  // 2*pair + which
    if (x >= W) return;
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    int sy;
    if (rp == 1) {
        sy = r;
    } else {
        int y0, y1; float fy;
        resize_coord(r >> 1, scale_y, H, y0, y1, fy);
        sy = (r & 1) ? y1 : y0;
    }
    const int rad = taps.ksize >> 1;
    float acc = 0.f;
    for (int k = 0; k < taps.ksize; ++k) {
        int yy = reflect101(sy + k - rad, H);
        acc += taps.w[k] * (float)src[(long long)yy * W + x];
    }
    tmp[((long long)img * (h * rp) + r) * W + x] = acc;
}

// exact u8 -> fp32 without the quarter-rate I2F: splice the byte into the mantissa of 2^23 and subtract 2^23
__device__ __forceinline__ float byte_to_float(unsigned v, unsigned sel) {
    return __uint_as_float(__byte_perm(v, 0x4B000000u, sel)) - 8388608.f;
}

// pass A, 4 columns per thread (W % 4 == 0): one 32-bit load per tap row, float4 store.  For a down-sampled level
// (rp == 2) a thread produces both source rows of its destination row: they are neighbours (y1 == y0 + 1) except at the
// bottom clamp, so one walk over ksize + 1 image rows feeds both accumulators (tap k of row y0 is tap k - 1 of row y1).
__global__ void __launch_bounds__(256) blur_v4_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                      float* __restrict__ tmp, int H, int W, int h, int rp,
                                                      double scale_y, BlurTaps taps) {
    const int x4 = blockIdx.x * blockDim.x + threadIdx.x;   // group of 4 columns
    const int r = blockIdx.y;                               // source row (rp == 1) or destination row (rp == 2)
    const int img = blockIdx.z;
    const int W4 = W >> 2;
    if (x4 >= W4) return;
    const unsigned* src = reinterpret_cast<const unsigned*>(((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W);
    const int rad = taps.ksize >> 1;
    int y0 = r, y1 = r;
    if (rp == 2) { float fy; resize_coord(r, scale_y, H, y0, y1, fy); }
    float4* dst = reinterpret_cast<float4*>(tmp + ((long long)img * (h * rp) + (long long)r * rp) * W) + x4;
    if (rp == 2 && y1 == y0 + 1 && y0 - rad >= 0 && y1 + rad < H) {
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
        const unsigned* p = src + (long long)(y0 - rad) * W4 + x4;
        float wprev = 0.f;
#pragma unroll 4
        for (int k = 0; k <= taps.ksize; ++k) {
            const unsigned c = __ldg(p + (long long)k * W4);
            const float wk = k < taps.ksize ? taps.w[k] : 0.f;
            const float v0 = byte_to_float(c, 0x7540u), v1 = byte_to_float(c, 0x7541u);
            const float v2 = byte_to_float(c, 0x7542u), v3 = byte_to_float(c, 0x7543u);
            a0.x += wk * v0; a0.y += wk * v1; a0.z += wk * v2; a0.w += wk * v3;
            a1.x += wprev * v0; a1.y += wprev * v1; a1.z += wprev * v2; a1.w += wprev * v3;
            wprev = wk;
        }
        dst[0] = a0;
        dst[W4] = a1;
        return;
    }
    for (int which = 0; which < rp; ++which) {
        const int sy = which ? y1 : y0;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool interior = sy - rad >= 0 && sy + rad < H;
#pragma unroll 4
        for (int k = 0; k < taps.ksize; ++k) {
            const int yy = interior ? sy + k - rad : reflect101(sy + k - rad, H);
            const unsigned c = __ldg(src + (long long)yy * W4 + x4);
            const float wk = taps.w[k];
            acc.x += wk * byte_to_float(c, 0x7540u);
            acc.y += wk * byte_to_float(c, 0x7541u);
            acc.z += wk * byte_to_float(c, 0x7542u);
            acc.w += wk * byte_to_float(c, 0x7543u);
        }
        dst[which * W4] = acc;
    }
}

// Levels whose blur has 3 taps (the full-resolution level and the first half-resolution one) in ONE pass, straight from
// the u8 image: no intermediate rows in HBM.  Same arithmetic as the two-pass path: vertical 3-tap sums first
// (accumulated in tap order), then the horizontal ones, then OpenCV's bilinear resize weights.
__device__ __forceinline__ float u8f(unsigned v) { return __uint_as_float(0x4B000000u | v) - 8388608.f; }

// full resolution: 4 adjacent outputs per thread (W % 4 == 0), FR_ROWS consecutive rows per thread: the three source rows
// of an output row slide down in registers (one 32-bit load per new row; the two neighbour bytes come from the adjacent
// lanes' words), so a row costs one load, six byte conversions and the 18 + 12 multiply-adds of the two 3-tap passes.
constexpr int FR_ROWS = 8;
__global__ void __launch_bounds__(128) blur3_fullres_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                            float* __restrict__ out, int H, int W, float w0, float w1,
                                                            float w2) {
    const int x4 = blockIdx.x * blockDim.x + threadIdx.x;
    const int yb = blockIdx.y * FR_ROWS;
    const int img = blockIdx.z;
    const int W4 = W >> 2;
    const bool active = x4 < W4;
    const int x4c = min(x4, W4 - 1);
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    const int xb = 4 * x4c;
    const int lane = threadIdx.x & 31;
    // the bytes left / right of this thread's word: the neighbouring lanes' words, except at the warp / image edges
    const bool left_edge = lane == 0 || x4c == 0, right_edge = lane == 31 || x4c == W4 - 1;
    const int xl = reflect101(xb - 1, W), xr = reflect101(xb + 4, W);
    float r[3][6];                                       // converted source rows y-1, y, y+1 at columns xb-1 .. xb+4
    auto load_row = [&](int y, float dst[6]) {
        const uint8_t* row = src + (long long)reflect101(y, H) * W;
        const unsigned c = __ldg(reinterpret_cast<const unsigned*>(row) + x4c);
        const unsigned cl = __shfl_up_sync(0xffffffffu, c, 1), cr = __shfl_down_sync(0xffffffffu, c, 1);
        dst[0] = left_edge ? u8f(__ldg(row + xl)) : byte_to_float(cl, 0x7543u);
        dst[1] = byte_to_float(c, 0x7540u);
        dst[2] = byte_to_float(c, 0x7541u);
        dst[3] = byte_to_float(c, 0x7542u);
        dst[4] = byte_to_float(c, 0x7543u);
        dst[5] = right_edge ? u8f(__ldg(row + xr)) : byte_to_float(cr, 0x7540u);
    };
    load_row(yb - 1, r[0]);
    load_row(yb, r[1]);
    float4* dst = reinterpret_cast<float4*>(out + ((long long)img * H + yb) * W) + x4c;
#pragma unroll
    for (int i = 0; i < FR_ROWS; ++i) {
        if (yb + i >= H) break;                          // uniform across the block
        load_row(yb + i + 1, r[(i + 2) % 3]);
        const float* ra = r[i % 3];
        const float* rb = r[(i + 1) % 3];
        const float* rc = r[(i + 2) % 3];
        float v[6];
#pragma unroll
        for (int c = 0; c < 6; ++c) {
            float a = 0.f;
            a += w0 * ra[c];
            a += w1 * rb[c];
            a += w2 * rc[c];
            v[c] = a;
        }
        float4 o;
        o.x = (w0 * v[0] + w1 * v[1]) + w2 * v[2];
        o.y = (w0 * v[1] + w1 * v[2]) + w2 * v[3];
        o.z = (w0 * v[2] + w1 * v[3]) + w2 * v[4];
        o.w = (w0 * v[3] + w1 * v[4]) + w2 * v[5];
        if (active) dst[(long long)i * W4] = o;
    }
}

// down-sampled level with a 3-tap blur: one output per thread from its 4 x 4 source footprint
__global__ void __launch_bounds__(256) blur3_resize_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                           float* __restrict__ out, int H, int W, int h, int w,
                                                           double scale_x, double scale_y, float w0, float w1, float w2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    const int img = blockIdx.z;
    if (i >= w) return;
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    int x0, x1, y0, y1; float fx, fy;
    resize_coord(i, scale_x, W, x0, x1, fx);
    resize_coord(j, scale_y, H, y0, y1, fy);
    float b[2][2];
    if (x1 == x0 + 1 && x0 >= 1 && x1 + 1 < W && y1 == y0 + 1 && y0 >= 1 && y1 + 1 < H) {
        // interior: one 4 x 4 byte footprint feeds both rows and both columns
        const uint8_t* p = src + (long long)(y0 - 1) * W + (x0 - 1);
        float P[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) P[r][c] = u8f(__ldg(p + r * W + c));
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float V[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float a = 0.f;
                a += w0 * P[r][c];
                a += w1 * P[r + 1][c];
                a += w2 * P[r + 2][c];
                V[c] = a;
            }
            float s0 = 0.f, s1 = 0.f;
            s0 += w0 * V[0]; s0 += w1 * V[1]; s0 += w2 * V[2];
            s1 += w0 * V[1]; s1 += w1 * V[2]; s1 += w2 * V[3];
            b[r][0] = s0;
            b[r][1] = s1;
        }
    } else {
    // vertical sums of the two source rows at the three columns around x0 and around x1
    float va[2][3], vb[2][3];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int sy = r ? y1 : y0;
#pragma unroll
        for (int c = 0; c < 3; ++c) { va[r][c] = 0.f; vb[r][c] = 0.f; }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const uint8_t* row = src + (long long)reflect101(sy + k - 1, H) * W;
            const float wk = k == 0 ? w0 : (k == 1 ? w1 : w2);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                va[r][c] += wk * u8f(__ldg(row + reflect101(x0 + c - 1, W)));
                vb[r][c] += wk * u8f(__ldg(row + reflect101(x1 + c - 1, W)));
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float wk = k == 0 ? w0 : (k == 1 ? w1 : w2);
            s0 += wk * va[r][k];
            s1 += wk * vb[r][k];
        }
        b[r][0] = s0;
        b[r][1] = s1;
    }
    }
    const float r0 = b[0][0] * (1.f - fx) + b[0][1] * fx;
    const float r1 = b[1][0] * (1.f - fx) + b[1][1] * fx;
    out[((long long)img * h + j) * w + i] = r0 * (1.f - fy) + r1 * fy;
}

// Down-sampled level in ONE pass (any blur width): a CTA owns a TW x TH tile of the level image.
//   1. the u8 footprint of the tile (REFLECT_101 applied while loading) goes to shared memory;
//   2. vertical blur at the two source rows of every destination row, 4 columns per thread, the two rows sharing one
//      walk over ksize + 1 footprint rows (they are neighbours; at the bottom clamp they coincide);
//   3. horizontal blur at the two source columns of every destination pixel + OpenCV's bilinear weights.
// Same arithmetic, in the same order, as the two-pass kernels above (fp32, taps accumulated in k order), but nothing
// round-trips through HBM and the image rows come from shared memory instead of L2.  The rows of vertical sums are
// skewed by one float per 32 columns so that the stride-`scale` reads of step 3 are bank-conflict free.
__device__ __forceinline__ int skew32(int c) { return c + (c >> 5); }

template <int TW, int TH, int KS>
__global__ void __launch_bounds__(256, 6) blur_resize_tile_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                               float* __restrict__ out, int H, int W, int h, int w,
                                                               double scale_x, double scale_y, int FWp, int FH,
                                                               BlurTaps taps) {
    extern __shared__ __align__(16) unsigned char pyr_smem[];
    const int VP = skew32(FWp) + 1;                              // pitch of a row of vertical sums
    unsigned* foot = reinterpret_cast<unsigned*>(pyr_smem);      // [FH][FWp / 4] words of 4 pixels
    float* V = reinterpret_cast<float*>(pyr_smem + (size_t)FH * FWp);   // [2 * TH][VP]
    // resize coordinates of the tile's columns / rows (cv::resize works them out in double; once per tile, not per use)
    __shared__ int s_x0[TW], s_y0[TH];
    __shared__ float s_fx[TW], s_fy[TH];
    __shared__ unsigned char s_x1[TW], s_y1[TH];                 // 1: second tap = first + 1; 0: clamped onto the first
    const int tid = threadIdx.x;
    const int img = blockIdx.z;
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    const int i0 = blockIdx.x * TW, j0 = blockIdx.y * TH;
    const int ni = min(TW, w - i0), nj = min(TH, h - j0);
    const int ksize = KS > 0 ? KS : taps.ksize;                  // KS > 0: compile-time blur width (loops fully unrolled)
    const int rad = ksize >> 1;
    if (tid < TW) {
        int a, b2; float f;
        resize_coord(min(i0 + tid, w - 1), scale_x, W, a, b2, f);
        s_x0[tid] = a; s_x1[tid] = (unsigned char)(b2 - a); s_fx[tid] = f;
    } else if (tid >= 128 && tid < 128 + TH) {
        int a, b2; float f;
        resize_coord(min(j0 + tid - 128, h - 1), scale_y, H, a, b2, f);
        s_y0[tid - 128] = a; s_y1[tid - 128] = (unsigned char)(b2 - a); s_fy[tid - 128] = f;
    }
    __syncthreads();
    const int xa = s_x0[0] - rad, ya = s_y0[0] - rad;
    const int xal = xa & ~3;                                     // footprint starts at a 4-pixel boundary (may be < 0)
    const int fw4 = min((s_x0[ni - 1] + s_x1[ni - 1] + rad - xal) / 4 + 1, FWp / 4);   // words per footprint row in use
    const int fh = min(s_y0[nj - 1] + s_y1[nj - 1] + rad - ya + 1, FH);
    const int W4 = FWp >> 2;
    const float inv_fw4 = 1.f / (float)fw4;                      // idx / fw4 == (int)((idx + 0.5f) * inv_fw4) for idx < 2^20

    // 1. footprint (measured: a warp per row with 16-byte loads is slower -- the wider, 16-aligned footprint costs a CTA
    // per SM at the deep levels)
    const bool rows_aligned = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 3) == 0;
    for (int idx = tid; idx < fh * fw4; idx += 256) {
        const int r = (int)(((float)idx + 0.5f) * inv_fw4), c4 = idx - r * fw4;
        int gy = ya + r;
        if ((unsigned)gy >= (unsigned)H) gy = reflect101(gy, H);
        const int gx = xal + 4 * c4;
        const uint8_t* row = src + (long long)gy * W;
        unsigned v;
        if (rows_aligned && gx >= 0 && gx + 3 < W) {
            v = __ldg(reinterpret_cast<const unsigned*>(row + gx));
        } else {
            v = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) v |= (unsigned)__ldg(row + reflect101(gx + b, W)) << (8 * b);
        }
        foot[r * W4 + c4] = v;
    }
    __syncthreads();

    // 2. vertical blur: task = (destination row, 4 columns)
    for (int idx = tid; idx < nj * fw4; idx += 256) {
        const int j = (int)(((float)idx + 0.5f) * inv_fw4), c4 = idx - j * fw4;
        const unsigned* p = foot + (s_y0[j] - rad - ya) * W4 + c4;
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
        if (s_y1[j]) {
            float wprev = 0.f;
#pragma unroll (KS > 0 ? KS + 1 : 4)
            for (int k = 0; k <= ksize; ++k) {
                const unsigned c = p[k * W4];
                const float wk = k < ksize ? taps.w[k] : 0.f;
                const float v0 = byte_to_float(c, 0x7540u), v1 = byte_to_float(c, 0x7541u);
                const float v2 = byte_to_float(c, 0x7542u), v3 = byte_to_float(c, 0x7543u);
                a0.x += wk * v0; a0.y += wk * v1; a0.z += wk * v2; a0.w += wk * v3;
                a1.x += wprev * v0; a1.y += wprev * v1; a1.z += wprev * v2; a1.w += wprev * v3;
                wprev = wk;
            }
        } else {
#pragma unroll (KS > 0 ? KS + 1 : 4)
            for (int k = 0; k < ksize; ++k) {
                const unsigned c = p[k * W4];
                const float wk = taps.w[k];
                a0.x += wk * byte_to_float(c, 0x7540u);
                a0.y += wk * byte_to_float(c, 0x7541u);
                a0.z += wk * byte_to_float(c, 0x7542u);
                a0.w += wk * byte_to_float(c, 0x7543u);
            }
            a1 = a0;                                             // y1 == y0: the same source row
        }
        float* v0p = V + (2 * j) * VP + skew32(4 * c4);
        float* v1p = v0p + VP;
        v0p[0] = a0.x; v0p[1] = a0.y; v0p[2] = a0.z; v0p[3] = a0.w;
        v1p[0] = a1.x; v1p[1] = a1.y; v1p[2] = a1.z; v1p[3] = a1.w;
    }
    __syncthreads();

    // 3. horizontal blur at the two source columns + bilinear weights: one destination pixel per thread
    for (int idx = tid; idx < nj * TW; idx += 256) {
        const int j = idx / TW, ii = idx - j * TW;
        if (ii >= ni) continue;
        const float fx = s_fx[ii], fy = s_fy[j];
        const float* row0 = V + (2 * j) * VP;
        const float* row1 = row0 + VP;
        const int c0 = s_x0[ii] - rad - xal;
        float b00 = 0.f, b01 = 0.f, b10 = 0.f, b11 = 0.f;
        if (s_x1[ii]) {
            float a0 = row0[skew32(c0)], a1 = row1[skew32(c0)];
#pragma unroll (KS > 0 ? KS + 1 : 4)
            for (int k = 0; k < ksize; ++k) {
                const float wk = taps.w[k];
                const int cs = skew32(c0 + k + 1);
                const float n0 = row0[cs], n1 = row1[cs];
                b00 += wk * a0;
                b01 += wk * n0;
                b10 += wk * a1;
                b11 += wk * n1;
                a0 = n0;
                a1 = n1;
            }
        } else {
            for (int k = 0; k < ksize; ++k) {
                const float wk = taps.w[k];
                const int cs = skew32(c0 + k);
                b00 += wk * row0[cs];
                b10 += wk * row1[cs];
            }
            b01 = b00;                                           // x1 == x0: the same source column
            b11 = b10;
        }
        const float r0 = b00 * (1.f - fx) + b01 * fx;
        const float r1 = b10 * (1.f - fx) + b11 * fx;
        out[((long long)img * h + (j0 + j)) * w + (i0 + ii)] = r0 * (1.f - fy) + r1 * fy;
    }
}

// Down-sampled level, one CTA per destination row (the default for W % 4 == 0).
// Blur followed by bilinear resize is one separable filter per destination pixel: with y0 / y0 + 1 the two source rows of
// destination row j and fy the weight of the second,
//     (1 - fy) * sum_k g[k] S(y0 - r + k) + fy * sum_k g[k] S(y0 + 1 - r + k) = sum_{c = 0 .. ksize} cw[c] S(y0 - r + c),
//     cw[c] = g[c] + fy * (g[c - 1] - g[c])          (g[-1] = g[ksize] = 0)
// and the same along x.  So a destination row needs ONE vertical pass over ksize + 1 image rows (not two blurred rows),
// and a destination pixel ONE horizontal pass over ksize + 1 vertical sums (not four blurred values):
//   1. vertical: the CTA forms the W vertical sums of its row, a thread eight columns at a time (two 32-bit words of four
//      pixels, packed fp32 conversions and multiply-adds), into shared memory;
//   2. horizontal: a thread per destination pixel walks its ksize + 1 sums with its own combined taps.
// No halo, no intermediate rows in HBM, about half the multiply-adds of blurring both source rows / columns, and the
// image rows are read straight from L2 (neighbouring destination rows share 60 % of them).  fp32 sums in a different
// association than the two-pass kernels: the level images agree to ~1e-5 of the 0..255 range (tests/test_gpu_stages.py).
struct RowTaps {
    int ksize;
    float g[kMaxBlurTaps + 1];    // g[ksize] = 0
    float dg[kMaxBlurTaps + 1];   // dg[c] = g[c - 1] - g[c]
};

__device__ __forceinline__ float2 bytes_to_float2(unsigned v, unsigned sel_lo, unsigned sel_hi) {
    const float2 m = make_float2(__uint_as_float(__byte_perm(v, 0x4B000000u, sel_lo)),
                                 __uint_as_float(__byte_perm(v, 0x4B000000u, sel_hi)));
    return __fadd2_rn(m, make_float2(-8388608.f, -8388608.f));
}

template <int NT>
__global__ void __launch_bounds__(NT) pyr_row_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                     float* __restrict__ out, int H, int W, int h, int w, double scale_x,
                                                     double scale_y, RowTaps taps) {
    extern __shared__ __align__(16) float pr_smem[];
    float* V = pr_smem;                                          // skew32(W) vertical sums of this destination row
    __shared__ float s_cv[kMaxBlurTaps + 1], s_g[kMaxBlurTaps + 1], s_dg[kMaxBlurTaps + 1];
    __shared__ int s_row[kMaxBlurTaps + 1];
    const int tid = threadIdx.x;
    const int j = blockIdx.x, img = blockIdx.y;
    const int ksize = taps.ksize, rad = ksize >> 1;
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    int y0, y1; float fy;
    resize_coord(j, scale_y, H, y0, y1, fy);
    const int ys = y0 - rad;
    for (int c = tid; c <= ksize; c += NT) {
        const float g = taps.g[c], dg = taps.dg[c];
        s_g[c] = g; s_dg[c] = dg;
        s_cv[c] = fmaf(fy, dg, g);
        s_row[c] = reflect101(ys + c, H);
    }
    __syncthreads();
    const bool rows_inside = ys >= 0 && ys + ksize < H;
    const int W4 = W >> 2;
    const unsigned* src32 = reinterpret_cast<const unsigned*>(src);

    // 1. vertical
    for (int cg0 = tid; cg0 < W4; cg0 += 2 * NT) {
        const bool has1 = cg0 + NT < W4;
        float2 a0 = make_float2(0.f, 0.f), a1 = a0, b0 = a0, b1 = a0;
        if (rows_inside) {
            const unsigned* p = src32 + (long long)ys * W4 + cg0;
#pragma unroll 6
            for (int r = 0; r <= ksize; ++r) {
                const float2 wr = make_float2(s_cv[r], s_cv[r]);
                const unsigned u = __ldg(p), v = has1 ? __ldg(p + NT) : 0u;
                p += W4;
                a0 = __ffma2_rn(wr, bytes_to_float2(u, 0x7540u, 0x7541u), a0);
                a1 = __ffma2_rn(wr, bytes_to_float2(u, 0x7542u, 0x7543u), a1);
                b0 = __ffma2_rn(wr, bytes_to_float2(v, 0x7540u, 0x7541u), b0);
                b1 = __ffma2_rn(wr, bytes_to_float2(v, 0x7542u, 0x7543u), b1);
            }
        } else {
#pragma unroll 2
            for (int r = 0; r <= ksize; ++r) {
                const float2 wr = make_float2(s_cv[r], s_cv[r]);
                const unsigned* p = src32 + (long long)s_row[r] * W4 + cg0;
                const unsigned u = __ldg(p), v = has1 ? __ldg(p + NT) : 0u;
                a0 = __ffma2_rn(wr, bytes_to_float2(u, 0x7540u, 0x7541u), a0);
                a1 = __ffma2_rn(wr, bytes_to_float2(u, 0x7542u, 0x7543u), a1);
                b0 = __ffma2_rn(wr, bytes_to_float2(v, 0x7540u, 0x7541u), b0);
                b1 = __ffma2_rn(wr, bytes_to_float2(v, 0x7542u, 0x7543u), b1);
            }
        }
        float* d = V + skew32(4 * cg0);
        d[0] = a0.x; d[1] = a0.y; d[2] = a1.x; d[3] = a1.y;
        if (has1) {
            float* e = V + skew32(4 * (cg0 + NT));
            e[0] = b0.x; e[1] = b0.y; e[2] = b1.x; e[3] = b1.y;
        }
    }
    __syncthreads();

    // 2. horizontal
    float* orow = out + ((long long)img * h + j) * w;
    for (int i = tid; i < w; i += NT) {
        int x0, x1; float fx;
        resize_coord(i, scale_x, W, x0, x1, fx);
        const int xs = x0 - rad;
        float acc = 0.f;
        if (xs >= 0 && xs + ksize < W) {
#pragma unroll 6
            for (int c = 0; c <= ksize; ++c) acc = fmaf(fmaf(fx, s_dg[c], s_g[c]), V[skew32(xs + c)], acc);
        } else {
            for (int c = 0; c <= ksize; ++c) acc = fmaf(fmaf(fx, s_dg[c], s_g[c]), V[skew32(reflect101(xs + c, W))], acc);
        }
        orow[i] = acc;
    }
}

// The first down-sampled level when the image halves exactly (W == 2 w, H == 2 h, 3-tap blur): every destination pixel
// is the same 4 x 4 separable filter (combined taps c = g + dg / 2) of the source pixels (2j - 1 .. 2j + 2) x (2i - 1 ..
// 2i + 2).  A thread owns eight source columns = four destination columns and walks down the source rows: per row one
// 64-bit load (the two edge bytes come from the neighbouring lanes), the four horizontal sums, and two vertical updates
// (a source row feeds the destination row it opens and the one it closes).  ~5 instructions per source pixel instead of the
// ~40 the general row kernel spends at this level (its per-pixel coordinate and loop overheads dominate a 4-tap filter).
constexpr int HALF_RJ = 16;      // destination rows per thread
__global__ void __launch_bounds__(128) pyr_half_kernel(const uint8_t* __restrict__ q0, const uint8_t* __restrict__ q1,
                                                       float* __restrict__ out, int H, int W, int h, int w, float c0, float c1,
                                                       float c2, float c3) {
    const int W8 = (W + 7) >> 3;
    const int t = blockIdx.x * 128 + threadIdx.x;
    const bool active = t < W8;
    const int tc = min(t, W8 - 1);
    const int xb = 8 * tc;
    const int img = blockIdx.z;
    const uint8_t* src = ((img & 1) ? q1 : q0) + (long long)(img >> 1) * H * W;
    const int j0 = blockIdx.y * HALF_RJ;
    const int nj = min(HALF_RJ, h - j0);
    const bool has_hi = xb + 4 < W;                              // W % 4 == 0: the last thread may own one word only
    const int lane = threadIdx.x & 31;
    const bool left_edge = lane == 0 || tc == 0, right_edge = lane == 31 || tc == W8 - 1;
    const int xl = reflect101(xb - 1, W), xr = reflect101(xb + 8, W), xm = reflect101(xb + 4, W);
    float prev[4] = {0.f, 0.f, 0.f, 0.f}, cur[4] = {0.f, 0.f, 0.f, 0.f};
    float* orow = out + ((long long)img * h + j0) * w + 4 * tc;
    const int n_out = max(0, min(4, w - 4 * tc));
    const bool vec2 = (w & 1) == 0 && n_out == 4;
    // source rows 2 j0 - 1 .. 2 (j0 + nj): row s (0-based) opens destination row s / 2 with tap s % 2 and feeds row
    // s / 2 - 1 with tap s % 2 + 2
    for (int s = 0; s < 2 * nj + 2; ++s) {
        const uint8_t* row = src + (long long)reflect101(2 * j0 - 1 + s, H) * W;
        const unsigned lo = __ldg(reinterpret_cast<const unsigned*>(row + xb));
        const unsigned hi = has_hi ? __ldg(reinterpret_cast<const unsigned*>(row + xb + 4)) : (unsigned)__ldg(row + xm);
        const unsigned nl = __shfl_up_sync(0xffffffffu, hi, 1), nr = __shfl_down_sync(0xffffffffu, lo, 1);
        float p[10];
        p[0] = left_edge ? u8f(__ldg(row + xl)) : byte_to_float(nl, 0x7543u);
        p[1] = byte_to_float(lo, 0x7540u); p[2] = byte_to_float(lo, 0x7541u);
        p[3] = byte_to_float(lo, 0x7542u); p[4] = byte_to_float(lo, 0x7543u);
        p[5] = byte_to_float(hi, 0x7540u); p[6] = byte_to_float(hi, 0x7541u);
        p[7] = byte_to_float(hi, 0x7542u); p[8] = byte_to_float(hi, 0x7543u);
        p[9] = right_edge ? u8f(__ldg(row + xr)) : byte_to_float(nr, 0x7540u);
        const bool odd = s & 1;
        const float wa = odd ? c1 : c0, wb = odd ? c3 : c2;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float hsum = fmaf(c3, p[2 * k + 3], fmaf(c2, p[2 * k + 2], fmaf(c1, p[2 * k + 1], c0 * p[2 * k])));
            cur[k] = fmaf(wa, hsum, cur[k]);
            prev[k] = fmaf(wb, hsum, prev[k]);
        }
        if (odd) {
            const int jl = (s >> 1) - 1;                         // the destination row this source row closes
            if (jl >= 0 && active) {
                float* o = orow + (long long)jl * w;
                if (vec2) {
                    *reinterpret_cast<float2*>(o) = make_float2(prev[0], prev[1]);
                    *reinterpret_cast<float2*>(o + 2) = make_float2(prev[2], prev[3]);
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k < n_out) o[k] = prev[k];
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) { prev[k] = cur[k]; cur[k] = 0.f; }
        }
    }
}

// pass B at the full-resolution level (w == W, no resize), 4 outputs per thread (W % 4 == 0)
__global__ void __launch_bounds__(256) blur_h4_fullres_kernel(const float* __restrict__ tmp, float* __restrict__ out, int W,
                                                              int h, BlurTaps taps) {
    const int x4 = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    const int img = blockIdx.z;
    const int W4 = W >> 2;
    if (x4 >= W4) return;
    const float* row = tmp + ((long long)img * h + j) * W;
    const int rad = taps.ksize >> 1;
    const int xb = 4 * x4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (taps.ksize == 3 && xb >= 1 && xb + 4 < W) {
        const float4 m = reinterpret_cast<const float4*>(row)[x4];
        const float l = row[xb - 1], rr = row[xb + 4];
        const float w0 = taps.w[0], w1 = taps.w[1], w2 = taps.w[2];
        acc.x = (w0 * l + w1 * m.x) + w2 * m.y;
        acc.y = (w0 * m.x + w1 * m.y) + w2 * m.z;
        acc.z = (w0 * m.y + w1 * m.z) + w2 * m.w;
        acc.w = (w0 * m.z + w1 * m.w) + w2 * rr;
    } else {
        for (int k = 0; k < taps.ksize; ++k) {
            const float wk = taps.w[k];
            acc.x += wk * row[reflect101(xb + k - rad, W)];
            acc.y += wk * row[reflect101(xb + 1 + k - rad, W)];
            acc.z += wk * row[reflect101(xb + 2 + k - rad, W)];
            acc.w += wk * row[reflect101(xb + 3 + k - rad, W)];
        }
    }
    reinterpret_cast<float4*>(out + ((long long)img * h + j) * W)[x4] = acc;
}

// pass B.  out: (n_img, h, w) fp32
template <class Taps>
__global__ void __launch_bounds__(256) blur_h_resize_kernel(const float* __restrict__ tmp, float* __restrict__ out, int W,
                                                            int h, int w, int rp, double scale_x, double scale_y,
                                                            int H, Taps taps) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    const int img = blockIdx.z;
    if (i >= w) return;
    const int rad = taps.ksize >> 1;
    const float* rows = tmp + ((long long)img * (h * rp) + (long long)j * rp) * W;
    float res;
    if (w == W && rp == 1) {
        float acc = 0.f;
        for (int k = 0; k < taps.ksize; ++k) acc += taps.w[k] * rows[reflect101(i + k - rad, W)];
        res = acc;
    } else {
        int x0, x1, y0, y1; float fx, fy;
        resize_coord(i, scale_x, W, x0, x1, fx);
        resize_coord(j, scale_y, H, y0, y1, fy);
        const float* row0 = rows;
        const float* row1 = rp == 2 ? rows + W : rows;
        float b00 = 0.f, b01 = 0.f, b10 = 0.f, b11 = 0.f;
        if (x1 == x0 + 1 && x0 - rad >= 0 && x1 + rad < W) {
            // interior: the two column positions are neighbours, so one pass over ksize+1 values feeds both
            const float* p0 = row0 + x0 - rad;
            const float* p1 = row1 + x0 - rad;
            float a0 = p0[0], a1 = p1[0];
#pragma unroll 4
            for (int k = 0; k < taps.ksize; ++k) {
                const float wk = taps.w[k];
                const float n0 = p0[k + 1], n1 = p1[k + 1];
                b00 += wk * a0;
                b01 += wk * n0;
                b10 += wk * a1;
                b11 += wk * n1;
                a0 = n0;
                a1 = n1;
            }
        } else {
            for (int k = 0; k < taps.ksize; ++k) {
                const float wk = taps.w[k];
                const int xa = reflect101(x0 + k - rad, W), xb = reflect101(x1 + k - rad, W);
                b00 += wk * row0[xa];
                b01 += wk * row0[xb];
                b10 += wk * row1[xa];
                b11 += wk * row1[xb];
            }
        }
        const float r0 = b00 * (1.f - fx) + b01 * fx;
        const float r1 = b10 * (1.f - fx) + b11 * fx;
        res = r0 * (1.f - fy) + r1 * fy;
    }
    out[((long long)img * h + j) * w + i] = res;
}

// K6: dst (n_fields, h, w, 2) = resize_linear(src (n_fields, sh, sw, 2)) * mul ; zero-fill when src == nullptr.
// Two adjacent outputs per thread (one 16-byte store); the row coordinate is computed once per thread.
__device__ __forceinline__ float2 upsample_one(const float2* __restrict__ r0, const float2* __restrict__ r1, int x0, int x1,
                                               float fx, float fy, float mul) {
    return upsample_vec(r0[x0], r0[x1], r1[x0], r1[x1], fx, fy, mul);
}

// A block of 256 threads covers 512 columns x UP_ROWS rows of one field: cv::resize's double-precision source coordinates
// are worked out once per block column / row into shared memory instead of per output.
constexpr int UP_ROWS = 4;
__global__ void __launch_bounds__(256) flow_upsample_kernel(const float2* __restrict__ src, float2* __restrict__ dst, int sh,
                                                            int sw, int h, int w, double scale_x, double scale_y,
                                                            float mul) {
    __shared__ int s_x0[512], s_x1[512], s_y0[UP_ROWS], s_y1[UP_ROWS];
    __shared__ float s_fx[512], s_fy[UP_ROWS];
    const int tid = threadIdx.x;
    const int i = 2 * (blockIdx.x * blockDim.x + tid);
    const int jb = blockIdx.y * UP_ROWS;
    const int f = blockIdx.z;
    if (src != nullptr) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c = 2 * tid + q;                   // block column
            int a0, a1; float fr;
            resize_coord(min(2 * (int)(blockIdx.x * blockDim.x) + c, w - 1), scale_x, sw, a0, a1, fr);
            s_x0[c] = a0; s_x1[c] = a1; s_fx[c] = fr;
        }
        if (tid < UP_ROWS) {
            int a0, a1; float fr;
            resize_coord(min(jb + tid, h - 1), scale_y, sh, a0, a1, fr);
            s_y0[tid] = a0; s_y1[tid] = a1; s_fy[tid] = fr;
        }
        __syncthreads();
    }
    if (i >= w) return;
    const float2* s = src ? src + (long long)f * sh * sw : nullptr;
#pragma unroll
    for (int r = 0; r < UP_ROWS; ++r) {
        const int j = jb + r;
        if (j >= h) break;
        float2 o0 = make_float2(0.f, 0.f), o1 = o0;
        if (src != nullptr) {
            const float2* r0 = s + (long long)s_y0[r] * sw;
            const float2* r1 = s + (long long)s_y1[r] * sw;
            const float fy = s_fy[r];
            o0 = upsample_one(r0, r1, s_x0[2 * tid], s_x1[2 * tid], s_fx[2 * tid], fy, mul);
            if (i + 1 < w) o1 = upsample_one(r0, r1, s_x0[2 * tid + 1], s_x1[2 * tid + 1], s_fx[2 * tid + 1], fy, mul);
        }
        float2* d = dst + ((long long)f * h + j) * w + i;
        if (i + 1 < w && (reinterpret_cast<uintptr_t>(d) & 15) == 0) {
            *reinterpret_cast<float4*>(d) = make_float4(o0.x, o0.y, o1.x, o1.y);
        } else {
            d[0] = o0;
            if (i + 1 < w) d[1] = o1;
        }
    }
}

// cv::getGaussianKernel(ksize, sigma, CV_32F)
template <class Taps>
static void gaussian_taps(Taps& taps, int ksize, double sigma) {
    taps.ksize = ksize;
    if (sigma <= 0 && ksize == 3) {
        taps.w[0] = 0.25f; taps.w[1] = 0.5f; taps.w[2] = 0.25f;
    } else {
        if (sigma <= 0) sigma = 0.3 * ((ksize - 1) * 0.5 - 1) + 0.8;
        double sum = 0, v[sizeof(taps.w) / sizeof(float)];
        for (int i = 0; i < ksize; ++i) {
            double x = i - (ksize - 1) * 0.5;
            v[i] = exp(-0.5 * x * x / (sigma * sigma));
            sum += v[i];
        }
        for (int i = 0; i < ksize; ++i) taps.w[i] = (float)(v[i] / sum);
    }
}

// A level whose blur is wider than kMaxBlurTaps (deep levels, small pyr_scale): the separable two-pass kernels with the
// taps in a larger parameter block.  Such levels are small (at most 1/20 of the frame per side), so the ksize
// multiply-adds per pixel and pass cost little next to the full-resolution level.
static int launch_pyramid_level_wide(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, int h, int w,
                                     int ksize, double sigma, float* tmp, float* out, cudaStream_t s) {
    if (ksize > kMaxWideBlurTaps) { set_error("pyramid: blur kernel too wide (%d)", ksize); return TF_ERR_UNSUPPORTED; }
    WideBlurTaps taps;
    gaussian_taps(taps, ksize, sigma);
    const int rp = (h == H) ? 1 : 2;
    const double sx = (double)W / w, sy = (double)H / h;
    const int n_img = 2 * n_pairs;
    LaunchTimer lt(KC_PYRAMID, (2.0 * H * W + 8.0 * h * w) * n_pairs, s, 2 * cdiv(n_img, 65534));
    for (int z0 = 0; z0 < n_img; z0 += 65534) {
        const int nz = min(n_img - z0, 65534);
        const uint8_t* a0 = q0 + (long long)(z0 / 2) * H * W;
        const uint8_t* a1 = q1 + (long long)(z0 / 2) * H * W;
        float* tz = tmp + (long long)z0 * h * rp * W;
        dim3 ga(cdiv(W, 256), h * rp, nz);
        blur_v_kernel<<<ga, 256, 0, s>>>(a0, a1, tz, H, W, h, rp, sy, taps);
        dim3 gb(cdiv(w, 256), h, nz);
        blur_h_resize_kernel<<<gb, 256, 0, s>>>(tz, out + (long long)z0 * h * w, W, h, w, rp, sx, sy, H, taps);
    }
    return check_launch("pyramid level (wide blur)");
}

int launch_pyramid_level(const uint8_t* q0, const uint8_t* q1, int n_pairs, int H, int W, int h, int w, int ksize,
                         double sigma, float* tmp, float* out, cudaStream_t s, bool two_pass) {
    if (ksize > kMaxBlurTaps) return launch_pyramid_level_wide(q0, q1, n_pairs, H, W, h, w, ksize, sigma, tmp, out, s);
    BlurTaps taps;
    gaussian_taps(taps, ksize, sigma);
    const int rp = (h == H) ? 1 : 2;
    const double sx = (double)W / w, sy = (double)H / h;
    const int n_img = 2 * n_pairs;
    static const char* env_two_pass = getenv("TF_PYR_TWO_PASS");
    two_pass = two_pass || env_two_pass != nullptr;
    static const char* env_tile = getenv("TF_PYR_TILE");     // A/B: the tile kernels instead of the row kernel
    if (rp == 2 && !two_pass && env_tile == nullptr && (W & 3) == 0 && (((uintptr_t)q0 | (uintptr_t)q1) & 3) == 0 &&
        ((long long)H * W & 3) == 0) {
        RowTaps rt;
        rt.ksize = ksize;
        for (int c = 0; c <= ksize; ++c) {
            const float gc = c < ksize ? taps.w[c] : 0.f, gm = c > 0 ? taps.w[c - 1] : 0.f;
            rt.g[c] = gc;
            rt.dg[c] = gm - gc;
        }
        for (int c = ksize + 1; c <= kMaxBlurTaps; ++c) rt.g[c] = rt.dg[c] = 0.f;
        static const char* env_half = getenv("TF_PYR_NO_HALF");   // A/B: the general row kernel at the half-resolution level
        if (ksize == 3 && W == 2 * w && H == 2 * h && env_half == nullptr) {
            const float c0 = rt.g[0] + 0.5f * rt.dg[0], c1 = rt.g[1] + 0.5f * rt.dg[1], c2 = rt.g[2] + 0.5f * rt.dg[2],
                        c3 = rt.g[3] + 0.5f * rt.dg[3];
            LaunchTimer lt(KC_PYRAMID, (2.0 * H * W + 8.0 * h * w) * n_pairs, s, cdiv(n_img, 65534));
            for (int z0 = 0; z0 < n_img; z0 += 65534) {
                const int nz = min(n_img - z0, 65534);
                dim3 g(cdiv((W + 7) / 8, 128), cdiv(h, HALF_RJ), nz);
                pyr_half_kernel<<<g, 128, 0, s>>>(q0 + (long long)(z0 / 2) * H * W, q1 + (long long)(z0 / 2) * H * W,
                                                  out + (long long)z0 * h * w, H, W, h, w, c0, c1, c2, c3);
            }
            return check_launch("pyramid level (half)");
        }
        const int W4 = W >> 2;
        const size_t smem = (size_t)(W + W / 32 + 8) * sizeof(float);
        // threads: the W / 4 column words in an even number of rounds of two words per thread
        const int rounds = cdiv(W4, 2 * 320);
        const int nt_want = cdiv(cdiv(W4, 2 * rounds), 32) * 32;
        const int n_launch = cdiv(n_img, 65534);
        LaunchTimer lt(KC_PYRAMID, (2.0 * H * W + 8.0 * h * w) * n_pairs, s, n_launch);
        for (int z0 = 0; z0 < n_img; z0 += 65534) {
            const int nz = min(n_img - z0, 65534);
            const uint8_t* a0 = q0 + (long long)(z0 / 2) * H * W;
            const uint8_t* a1 = q1 + (long long)(z0 / 2) * H * W;
            float* oz = out + (long long)z0 * h * w;
            dim3 g(h, nz);
#define TF_ROW_LAUNCH(NT_)                                                                                             \
    do {                                                                                                               \
        cudaFuncSetAttribute(pyr_row_kernel<NT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
        pyr_row_kernel<NT_><<<g, NT_, smem, s>>>(a0, a1, oz, H, W, h, w, sx, sy, rt);                                   \
    } while (0)
            if (nt_want <= 128) TF_ROW_LAUNCH(128);
            else if (nt_want <= 192) TF_ROW_LAUNCH(192);
            else if (nt_want <= 256) TF_ROW_LAUNCH(256);
            else TF_ROW_LAUNCH(320);
#undef TF_ROW_LAUNCH
        }
        return check_launch("pyramid level (row)");
    }
    if (rp == 2 && !two_pass) {
        // one fused pass per down-sampled level; tile shape by down-sampling factor (bigger footprints, smaller tiles)
        const int n_launch = cdiv(n_img, 65534);
        LaunchTimer lt(KC_PYRAMID, (2.0 * H * W + 8.0 * h * w) * n_pairs, s, n_launch);
        const bool wide = sx < 3.0;                              // half resolution: 64 x 16 tiles, else 32 x 8 / 16 x 8 / 8 x 4
        // (deep levels: few rows per tile, so that the footprint leaves room for 5-6 CTAs per SM)
        const int TW = wide ? 64 : (sx < 6.0 ? 32 : (sx < 24.0 ? 16 : 8));
        const int TH = wide ? 16 : (sx < 12.0 ? 8 : (sx < 24.0 ? 4 : 2));
        const int FWp = (((int)ceil((TW - 1) * sx) + 2 + ksize + 3 + 3) / 4 + 1) * 4;   // + alignment slack
        const int FH = (int)ceil((TH - 1) * sy) + 3 + ksize;
        const size_t smem = (size_t)FH * FWp + (size_t)2 * TH * (FWp + FWp / 32 + 2) * sizeof(float);
        if (smem <= 200 * 1024) {
            for (int z0 = 0; z0 < n_img; z0 += 65534) {
                const int nz = min(n_img - z0, 65534);
                const uint8_t* a0 = q0 + (long long)(z0 / 2) * H * W;
                const uint8_t* a1 = q1 + (long long)(z0 / 2) * H * W;
                float* oz = out + (long long)z0 * h * w;
                dim3 g(cdiv(w, TW), cdiv(h, TH), nz);
#define TF_TILE_LAUNCH(TW_, TH_, KS_)                                                                                  \
    do {                                                                                                               \
        cudaFuncSetAttribute(blur_resize_tile_kernel<TW_, TH_, KS_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        blur_resize_tile_kernel<TW_, TH_, KS_><<<g, 256, smem, s>>>(a0, a1, oz, H, W, h, w, sx, sy, FWp, FH, taps);   \
    } while (0)
                if (TW == 64 && ksize == 3) TF_TILE_LAUNCH(64, 16, 3);
                else if (TW == 64) TF_TILE_LAUNCH(64, 16, 0);
                else if (TW == 32 && ksize == 9) TF_TILE_LAUNCH(32, 8, 9);
                else if (TW == 32) TF_TILE_LAUNCH(32, 8, 0);
                else if (TW == 16 && TH == 8) TF_TILE_LAUNCH(16, 8, 0);
                else if (TW == 16) TF_TILE_LAUNCH(16, 4, 0);
                else TF_TILE_LAUNCH(8, 2, 0);
#undef TF_TILE_LAUNCH
            }
            return check_launch("pyramid level (tile)");
        }
    }
    const bool fused3 = ksize == 3 && !two_pass && ((h == H && w == W && W % 4 == 0) || rp == 2);
    LaunchTimer lt(KC_PYRAMID, (2.0 * H * W + 8.0 * h * w) * n_pairs, s, (fused3 ? 1 : 2) * cdiv(n_img, 65534));
    for (int z0 = 0; z0 < n_img; z0 += 65534) {
        const int nz = min(n_img - z0, 65534);  // even, so image parity is preserved
        const uint8_t* a0 = q0 + (long long)(z0 / 2) * H * W;
        const uint8_t* a1 = q1 + (long long)(z0 / 2) * H * W;
        float* tz = tmp + (long long)z0 * h * rp * W;
        if (fused3) {
            float* o3 = out + (long long)z0 * h * w;
            if (h == H && w == W && W % 4 == 0 && (((uintptr_t)a0 | (uintptr_t)a1) % 4 == 0) && (uintptr_t)o3 % 16 == 0) {
                dim3 g(cdiv(W / 4, 128), cdiv(H, FR_ROWS), nz);
                blur3_fullres_kernel<<<g, 128, 0, s>>>(a0, a1, o3, H, W, taps.w[0], taps.w[1], taps.w[2]);
                continue;
            }
            if (rp == 2) {
                dim3 g(cdiv(w, 256), h, nz);
                blur3_resize_kernel<<<g, 256, 0, s>>>(a0, a1, o3, H, W, h, w, sx, sy, taps.w[0], taps.w[1], taps.w[2]);
                continue;
            }
        }
        const bool vec4 = (W % 4 == 0) && (((uintptr_t)a0 | (uintptr_t)a1) % 4 == 0) && ((uintptr_t)tz % 16 == 0);
        if (vec4) {
            dim3 ga(cdiv(W / 4, 128), h, nz);
            blur_v4_kernel<<<ga, 128, 0, s>>>(a0, a1, tz, H, W, h, rp, sy, taps);
        } else {
            dim3 ga(cdiv(W, 256), h * rp, nz);
            blur_v_kernel<<<ga, 256, 0, s>>>(a0, a1, tz, H, W, h, rp, sy, taps);
        }
        float* oz = out + (long long)z0 * h * w;
        if (vec4 && w == W && rp == 1 && (uintptr_t)oz % 16 == 0) {
            dim3 gb(cdiv(W / 4, 128), h, nz);
            blur_h4_fullres_kernel<<<gb, 128, 0, s>>>(tz, oz, W, h, taps);
        } else {
            dim3 gb(cdiv(w, 256), h, nz);
            blur_h_resize_kernel<<<gb, 256, 0, s>>>(tz, oz, W, h, w, rp, sx, sy, H, taps);
        }
    }
    return check_launch("pyramid level");
}

// cv::resize's source coordinates of a (sh, sw) -> (h, w) up-sampling, tabulated once per level for the first iteration's
// fused up-sampling
__global__ void resize_tables_kernel(int* __restrict__ x0, float* __restrict__ fx, int w, int sw, double scale_x,
                                     int* __restrict__ y0, float* __restrict__ fy, int h, int sh, double scale_y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int a, b; float f;
    if (i < w) { resize_coord(i, scale_x, sw, a, b, f); x0[i] = a; fx[i] = f; }
    if (i < h) { resize_coord(i, scale_y, sh, a, b, f); y0[i] = a; fy[i] = f; }
}

int launch_resize_tables(int* x0, float* fx, int w, int sw, int* y0, float* fy, int h, int sh, cudaStream_t s) {
    const int n = w > h ? w : h;
    resize_tables_kernel<<<cdiv(n, 256), 256, 0, s>>>(x0, fx, w, sw, (double)sw / w, y0, fy, h, sh, (double)sh / h);
    return check_launch("resize tables");
}

int launch_flow_upsample(const float* src, float* dst, int n_fields, int sh, int sw, int h, int w, float mul,
                         cudaStream_t s) {
    const double sx = sw > 0 ? (double)sw / w : 1.0, sy = sh > 0 ? (double)sh / h : 1.0;
    LaunchTimer lt(KC_UPSAMPLE, (8.0 * h * w + 8.0 * sh * sw) * n_fields, s, cdiv(n_fields, 65535));
    for (int z0 = 0; z0 < n_fields; z0 += 65535) {
        const int nz = min(n_fields - z0, 65535);
        dim3 g(cdiv(cdiv(w, 2), 256), cdiv(h, UP_ROWS), nz);
        flow_upsample_kernel<<<g, 256, 0, s>>>(
            src ? reinterpret_cast<const float2*>(src) + (long long)z0 * sh * sw : nullptr,
            reinterpret_cast<float2*>(dst) + (long long)z0 * h * w, sh, sw, h, w, sx, sy, mul);
    }
    return check_launch("flow upsample");
}

}  // namespace tf
