// K11: DIS (Dense Inverse Search) optical flow, the arithmetic of cv::DISOpticalFlow::calc
// (opencv/modules/video/src/dis_flow.cpp, restated and pinned in oracle/dis_np.py) for patch size 8 with mean
// normalisation and spatial propagation, batched over pairs; both directions of a pair share one pyramid.
//
// Per call: INTER_AREA u8 pyramid of both frames (all scales), then per scale, coarsest to finest, for the 2n
// (pair, direction) images: Sobel gradients of I0, the per-patch structure tensors (float running sums in OpenCV's
// order), the patch inverse search, the densification, the scale's variational refinement (the library's
// tf_variational_refinement on the scale images) and the x2 bilinear up-sampling.  The last up-sampling to the frame
// is fused with the x2^finest scaling, the optional clamp and the store into the caller's strided outputs.
//
// Patch search: OpenCV cuts the patch rows into 8 stripes of ceil(hs / 8) rows (whatever its thread count) and runs
// each stripe serially: pass 1 in raster order with the left and upper neighbours as candidates, pass 2 in reverse
// order with the right and lower ones; nothing propagates across stripes.  The patches of one anti-diagonal of a
// stripe are independent, so one CTA per (image, stripe) walks the diagonals with a barrier between them, one thread
// per patch.  Every float operation uses the _rn intrinsics in OpenCV's evaluation order (no contraction into FMA):
// the 8x8 sums accumulate in four lanes (lane k += column k + column k + 4, row by row) reduced as (l0+l2)+(l1+l3),
// as OpenCV's SSE build does, so the propagation choices are the same.
#include <climits>

#include "tf_common.cuh"

namespace tf {

constexpr int DIS_PS = 8;         // patch size (the presets' value; the only one built)
constexpr int DIS_BORDER = 16;    // replicate border of I1 in OpenCV (the clamps of the patch positions depend on it)
constexpr int DIS_STRIPES = 8;
constexpr int DIS_MAX_SCALES = 16;

__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }

__device__ __forceinline__ uint8_t sat_u8(float v) { return (uint8_t)min(max(__float2int_rn(v), 0), 255); }

// ---- resize(INTER_AREA), u8, downscale: fast integer path or the general area-weight path -------------------------
__global__ void dis_area_kernel(const uint8_t* __restrict__ src, long long src_img_stride, int sh, int sw,
                                uint8_t* __restrict__ dst, long long dst_img_stride, int h, int w) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const uint8_t* S = src + blockIdx.z * src_img_stride;
    uint8_t* D = dst + blockIdx.z * dst_img_stride;
    const double scx = (double)sw / w, scy = (double)sh / h;
    const int kx = (int)rint(scx), ky = (int)rint(scy);
    if (fabs(scx - kx) < 2.220446049250313e-16 && fabs(scy - ky) < 2.220446049250313e-16) {
        int sum = 0;
        for (int dy = 0; dy < ky; ++dy)
            for (int dx = 0; dx < kx; ++dx) sum += S[(long long)(y * ky + dy) * sw + x * kx + dx];
        D[(long long)y * w + x] = (kx == 2 && ky == 2) ? (uint8_t)((sum + 2) >> 2)
                                                       : sat_u8(fm((float)sum, 1.f / (float)(kx * ky)));
        return;
    }
    // computeResizeAreaTab entries of this row / column, in table order
    const double fy1 = y * scy, fy2 = fy1 + scy, cy = fmin(scy, sh - fy1);
    int sy1 = (int)ceil(fy1), sy2 = (int)floor(fy2);
    sy2 = min(sy2, sh - 1); sy1 = min(sy1, sy2);
    const double fx1 = x * scx, fx2 = fx1 + scx, cx = fmin(scx, sw - fx1);
    int sx1 = (int)ceil(fx1), sx2 = (int)floor(fx2);
    sx2 = min(sx2, sw - 1); sx1 = min(sx1, sx2);
    const bool xl = sx1 - fx1 > 1e-3, xr = fx2 - sx2 > 1e-3;
    const float axl = (float)((sx1 - fx1) / cx), axm = (float)(1.0 / cx), axr = (float)(fmin(fmin(fx2 - sx2, 1.), cx) / cx);
    const bool yl = sy1 - fy1 > 1e-3, yr = fy2 - sy2 > 1e-3;
    const float byl = (float)((sy1 - fy1) / cy), bym = (float)(1.0 / cy), byr = (float)(fmin(fmin(fy2 - sy2, 1.), cy) / cy);
    float acc = 0.f;
    bool first = true;
    auto row = [&](int sy, float beta) {
        const uint8_t* r = S + (long long)sy * sw;
        float buf = 0.f;
        if (xl) buf = fa(buf, fm((float)r[sx1 - 1], axl));
        for (int sx = sx1; sx < sx2; ++sx) buf = fa(buf, fm((float)r[sx], axm));
        if (xr) buf = fa(buf, fm((float)r[sx2], axr));
        acc = first ? fm(beta, buf) : fa(acc, fm(beta, buf));
        first = false;
    };
    if (yl) row(sy1 - 1, byl);
    for (int sy = sy1; sy < sy2; ++sy) row(sy, bym);
    if (yr) row(sy2, byr);
    D[(long long)y * w + x] = sat_u8(acc);
}

// ---- spatialGradient: 3x3 Sobel, BORDER_REFLECT_101, int16 --------------------------------------------------------
__device__ __forceinline__ int refl101(int i, int n) {
    if (n == 1) return 0;
    if (i < 0) return -i;
    if (i >= n) return 2 * n - 2 - i;
    return i;
}

__global__ void dis_sobel_kernel(const uint8_t* __restrict__ img, int h, int w, int16_t* __restrict__ gx,
                                 int16_t* __restrict__ gy) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const long long o = (long long)blockIdx.z * h * w;
    const uint8_t* I = img + o;
    const int xm = refl101(x - 1, w), xp = refl101(x + 1, w), ym = refl101(y - 1, h), yp = refl101(y + 1, h);
    auto P = [&](int yy, int xx) { return (int)I[yy * w + xx]; };
    const int ix = (P(ym, xp) - P(ym, xm)) + 2 * (P(y, xp) - P(y, xm)) + (P(yp, xp) - P(yp, xm));
    const int iy = (P(yp, xm) - P(ym, xm)) + 2 * (P(yp, x) - P(ym, x)) + (P(yp, xp) - P(ym, xp));
    gx[o + y * w + x] = (int16_t)ix;
    gy[o + y * w + x] = (int16_t)iy;
}

// ---- precomputeStructureTensor: horizontal running sums per row, then vertical running sums per patch column ------
// planes: xx, yy, xy, x, y
__global__ void dis_struct_h_kernel(const int16_t* __restrict__ gx, const int16_t* __restrict__ gy, int h, int w,
                                    int stride, int wsn, float* __restrict__ aux, int n_img) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_img * h) return;
    const int z = t / h, i = t % h;
    const int16_t* X = gx + ((long long)z * h + i) * w;
    const int16_t* Y = gy + ((long long)z * h + i) * w;
    const long long plane = (long long)n_img * h * wsn;
    float* A = aux + ((long long)z * h + i) * wsn;
    float sxx = 0.f, syy = 0.f, sxy = 0.f, sx = 0.f, sy = 0.f;
    for (int j = 0; j < DIS_PS; ++j) {
        const int a = X[j], b = Y[j];
        sxx = fa(sxx, (float)(a * a)); syy = fa(syy, (float)(b * b)); sxy = fa(sxy, (float)(a * b));
        sx = fa(sx, (float)a); sy = fa(sy, (float)b);
    }
    A[0] = sxx; A[plane] = syy; A[2 * plane] = sxy; A[3 * plane] = sx; A[4 * plane] = sy;
    int js = 1;
    for (int j = DIS_PS; j < w; ++j) {
        const int a = X[j], b = Y[j], a0 = X[j - DIS_PS], b0 = Y[j - DIS_PS];
        sxx = fa(sxx, (float)(a * a - a0 * a0)); syy = fa(syy, (float)(b * b - b0 * b0));
        sxy = fa(sxy, (float)(a * b - a0 * b0)); sx = fa(sx, (float)(a - a0)); sy = fa(sy, (float)(b - b0));
        if ((j - DIS_PS + 1) % stride == 0) {
            A[js] = sxx; A[plane + js] = syy; A[2 * plane + js] = sxy; A[3 * plane + js] = sx; A[4 * plane + js] = sy;
            ++js;
        }
    }
}

__global__ void dis_struct_v_kernel(const float* __restrict__ aux, int h, int stride, int hsn, int wsn,
                                    float* __restrict__ st, int n_img) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_img * wsn * 5) return;
    const int c = t / (n_img * wsn), r = t % (n_img * wsn), z = r / wsn, js = r % wsn;
    const float* A = aux + (long long)c * n_img * h * wsn + (long long)z * h * wsn + js;
    float* O = st + (long long)c * n_img * hsn * wsn + (long long)z * hsn * wsn + js;
    float s = 0.f;
    for (int i = 0; i < DIS_PS; ++i) s = fa(s, A[(long long)i * wsn]);
    O[0] = s;
    int is = 1;
    for (int i = DIS_PS; i < h; ++i) {
        s = fa(s, fs(A[(long long)i * wsn], A[(long long)(i - DIS_PS) * wsn]));
        if ((i - DIS_PS + 1) % stride == 0) { O[(long long)is * wsn] = s; ++is; }
    }
}

// ---- patch inverse search --------------------------------------------------------------------------------------
struct DisImg {
    const uint8_t* I0; const uint8_t* I1; const int16_t* gx; const int16_t* gy;
    int h, w;
};

// bilinear I1 patch at (i, j) + (ux, uy) minus the I0 patch; sums in OpenCV's SSE lane order.  With grads, also the
// I0x / I0y weighted sums (processPatchMeanNorm); returns the mean-normalised SSD.
template <bool GRAD>
__device__ float dis_patch(const DisImg& m, int i, int j, float ux, float uy, float xg, float yg, float* dux,
                           float* duy) {
    const float ii = fminf(fmaxf(fa(fa((float)i, uy), (float)DIS_BORDER), (float)(DIS_BORDER - DIS_PS + 1)),
                           (float)(DIS_BORDER + m.h - 1));
    const float jj = fminf(fmaxf(fa(fa((float)j, ux), (float)DIS_BORDER), (float)(DIS_BORDER - DIS_PS + 1)),
                           (float)(DIS_BORDER + m.w - 1));
    const float di = fs(ii, floorf(ii)), dj = fs(jj, floorf(jj));
    const float w11 = fm(di, dj), w10 = fm(di, fs(1.f, dj)), w01 = fm(fs(1.f, di), dj), w00 = fm(fs(1.f, di), fs(1.f, dj));
    const int bi = (int)ii - DIS_BORDER, bj = (int)jj - DIS_BORDER;   // window origin in I1 (replicate outside)
    int cols[DIS_PS + 1];
#pragma unroll
    for (int c = 0; c <= DIS_PS; ++c) cols[c] = min(max(bj + c, 0), m.w - 1);
    float s[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f}, sx[4] = {0.f, 0.f, 0.f, 0.f},
          sy[4] = {0.f, 0.f, 0.f, 0.f};
    float top[DIS_PS + 1];
    {
        const uint8_t* r = m.I1 + (long long)min(max(bi, 0), m.h - 1) * m.w;
#pragma unroll
        for (int c = 0; c <= DIS_PS; ++c) top[c] = (float)r[cols[c]];
    }
#pragma unroll 1
    for (int r = 0; r < DIS_PS; ++r) {
        float bot[DIS_PS + 1];
        const uint8_t* rr = m.I1 + (long long)min(max(bi + r + 1, 0), m.h - 1) * m.w;
#pragma unroll
        for (int c = 0; c <= DIS_PS; ++c) bot[c] = (float)rr[cols[c]];
        const uint8_t* i0 = m.I0 + (long long)(i + r) * m.w + j;
        float d[DIS_PS];
#pragma unroll
        for (int c = 0; c < DIS_PS; ++c)
            d[c] = fs(fa(fa(fa(fm(w00, top[c]), fm(w01, top[c + 1])), fm(w10, bot[c])), fm(w11, bot[c + 1])),
                      (float)i0[c]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            s[k] = fa(s[k], fa(d[k], d[k + 4]));
            q[k] = fa(q[k], fa(fm(d[k], d[k]), fm(d[k + 4], d[k + 4])));
        }
        if (GRAD) {
            const int16_t* X = m.gx + (long long)(i + r) * m.w + j;
            const int16_t* Y = m.gy + (long long)(i + r) * m.w + j;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                sx[k] = fa(sx[k], fa(fm(d[k], (float)X[k]), fm(d[k + 4], (float)X[k + 4])));
                sy[k] = fa(sy[k], fa(fm(d[k], (float)Y[k]), fm(d[k + 4], (float)Y[k + 4])));
            }
        }
#pragma unroll
        for (int c = 0; c <= DIS_PS; ++c) top[c] = bot[c];
    }
    const float n = (float)(DIS_PS * DIS_PS);
    const float S = fa(fa(s[0], s[2]), fa(s[1], s[3]));
    const float Q = fa(fa(q[0], q[2]), fa(q[1], q[3]));
    if (GRAD) {
        const float SX = fa(fa(sx[0], sx[2]), fa(sx[1], sx[3]));
        const float SY = fa(fa(sy[0], sy[2]), fa(sy[1], sy[3]));
        *dux = fs(SX, __fdiv_rn(fm(S, xg), n));
        *duy = fs(SY, __fdiv_rn(fm(S, yg), n));
    }
    return fs(Q, __fdiv_rn(fm(S, S), n));
}

struct DisSearchArgs {
    const uint8_t* pyr; int n_img;      // scale images: image z = I0 of (pair, direction) z, its I1 is (z + n_img/2) % n_img
    const int16_t* gx; const int16_t* gy;
    const float* st;                    // 5 planes (n_img, hs, ws)
    const float* U;                     // (n_img, h, w, 2) initial flow at this scale
    float* Sx; float* Sy;               // (n_img, hs, ws)
    int h, w, hs, ws, stride, stripe, inner;
};

__global__ void __launch_bounds__(64) dis_search_kernel(DisSearchArgs a) {
    const int stripe = blockIdx.x, z = blockIdx.y;
    const int r0 = min(stripe * a.stripe, a.hs), r1 = min((stripe + 1) * a.stripe, a.hs);
    const int rows = r1 - r0;
    if (rows <= 0) return;
    const long long hw = (long long)a.h * a.w, sp = (long long)a.hs * a.ws;
    const int half = a.n_img / 2;
    DisImg m;
    m.I0 = a.pyr + z * hw; m.I1 = a.pyr + ((z + half) % a.n_img) * hw;
    m.gx = a.gx + z * hw; m.gy = a.gy + z * hw; m.h = a.h; m.w = a.w;
    float* Sx = a.Sx + z * sp;
    float* Sy = a.Sy + z * sp;
    const long long plane = (long long)a.n_img * sp;
    const float* XX = a.st + z * sp; const float* YY = XX + plane; const float* XY = XX + 2 * plane;
    const float* GX = XX + 3 * plane; const float* GY = XX + 4 * plane;
    const float2* U = reinterpret_cast<const float2*>(a.U) + z * hw;
    for (int t = threadIdx.x; t < rows * a.ws; t += blockDim.x) {
        const int is = r0 + t / a.ws, js = t % a.ws;
        const float2 u = U[(long long)(is * a.stride + DIS_PS / 2) * a.w + js * a.stride + DIS_PS / 2];
        Sx[is * a.ws + js] = u.x; Sy[is * a.ws + js] = u.y;
    }
    __syncthreads();
    const int n_diag = rows + a.ws - 1;
    for (int pass = 0; pass < 2; ++pass) {
        const int dir = pass == 0 ? 1 : -1;
        for (int dg = 0; dg < n_diag; ++dg) {
            // local row lr of the pass order, column from the diagonal
            for (int lr = threadIdx.x; lr < rows; lr += blockDim.x) {
                const int lc = dg - lr;
                if (lc < 0 || lc >= a.ws) continue;
                const int is = pass == 0 ? r0 + lr : r1 - 1 - lr;
                const int js = pass == 0 ? lc : a.ws - 1 - lc;
                const int i = is * a.stride, j = js * a.stride, o = is * a.ws + js;
                float cx = Sx[o], cy = Sy[o];
                float best = dis_patch<false>(m, i, j, cx, cy, 0.f, 0.f, nullptr, nullptr);
                if (lc > 0) {
                    const int on = o - dir;
                    const float nx = Sx[on], ny = Sy[on];
                    const float c = dis_patch<false>(m, i, j, nx, ny, 0.f, 0.f, nullptr, nullptr);
                    if (c < best) { best = c; cx = nx; cy = ny; }
                }
                if (lr > 0) {
                    const int on = o - dir * a.ws;
                    const float nx = Sx[on], ny = Sy[on];
                    const float c = dis_patch<false>(m, i, j, nx, ny, 0.f, 0.f, nullptr, nullptr);
                    if (c < best) { best = c; cx = nx; cy = ny; }
                }
                const float sx0 = cx, sy0 = cy;
                const float xx = XX[o], yy = YY[o], xy = XY[o];
                float det = fs(fm(xx, yy), fm(xy, xy));
                if (fabsf(det) < 0.001f) det = 0.001f;
                const float h11 = __fdiv_rn(yy, det), h12 = __fdiv_rn(-xy, det), h22 = __fdiv_rn(xx, det);
                const float xg = GX[o], yg = GY[o];
                float prev = 1e10f;
                for (int t = 0; t < a.inner; ++t) {
                    float dux, duy;
                    const float ssd = dis_patch<true>(m, i, j, cx, cy, xg, yg, &dux, &duy);
                    cx = fs(cx, fa(fm(h11, dux), fm(h12, duy)));
                    cy = fs(cy, fa(fm(h12, dux), fm(h22, duy)));
                    if (ssd >= prev) break;
                    prev = ssd;
                }
                const double ex = (double)fs(cx, sx0), ey = (double)fs(cy, sy0);
                if (sqrt(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey))) <= (double)DIS_PS) { Sx[o] = cx; Sy[o] = cy; }
                else { Sx[o] = sx0; Sy[o] = sy0; }
            }
            __syncthreads();
        }
    }
}

// ---- densification ----------------------------------------------------------------------------------------------
__global__ void dis_densify_kernel(const uint8_t* __restrict__ pyr, int n_img, const float* __restrict__ Sx_all,
                                   const float* __restrict__ Sy_all, int h, int w, int hs, int ws, int stride,
                                   float* __restrict__ U_all) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
    if (x >= w || y >= h) return;
    const long long hw = (long long)h * w, sp = (long long)hs * ws;
    const uint8_t* I0 = pyr + z * hw;
    const uint8_t* I1 = pyr + ((z + n_img / 2) % n_img) * hw;
    const float* Sx = Sx_all + z * sp;
    const float* Sy = Sy_all + z * sp;
    // patches covering (y, x), as Densification_ParBody's incremental bounds give them
    const int ie = min(y / stride, hs - 1), is0 = min(y < DIS_PS ? 0 : (y - DIS_PS) / stride + 1, ie);
    const int je = min(x / stride, ws - 1), js0 = min(x < DIS_PS ? 0 : (x - DIS_PS) / stride + 1, je);
    const float i0 = (float)I0[y * w + x];
    const float wl = fs(fs((float)w, 1.f), 0.001f), hl = fs(fs((float)h, 1.f), 0.001f);
    float sum_x = 0.f, sum_y = 0.f, sum_c = 0.f;
    for (int is = is0; is <= ie; ++is)
        for (int js = js0; js <= je; ++js) {
            const float sx = Sx[is * ws + js], sy = Sy[is * ws + js];
            const float jm = fminf(fmaxf(fa((float)x, sx), 0.f), wl);
            const float im = fminf(fmaxf(fa((float)y, sy), 0.f), hl);
            const int jl = (int)jm, il = (int)im, ju = jl + 1, iu = il + 1;
            const float a = fs(jm, (float)jl), b = fs(im, (float)il), c = fs((float)ju, jm), d = fs((float)iu, im);
            float diff = fm(fm(a, b), (float)I1[iu * w + ju]);
            diff = fa(diff, fm(fm(c, b), (float)I1[iu * w + jl]));
            diff = fa(diff, fm(fm(a, d), (float)I1[il * w + ju]));
            diff = fa(diff, fm(fm(c, d), (float)I1[il * w + jl]));
            diff = fs(diff, i0);
            const float coef = __fdiv_rn(1.f, fmaxf(1.f, fabsf(diff)));
            sum_x = fa(sum_x, fm(coef, sx));
            sum_y = fa(sum_y, fm(coef, sy));
            sum_c = fa(sum_c, coef);
        }
    reinterpret_cast<float2*>(U_all)[z * hw + (long long)y * w + x] =
        make_float2(__fdiv_rn(sum_x, sum_c), __fdiv_rn(sum_y, sum_c));
}

// ---- resize(INTER_LINEAR) of a flow, times `factor`; columns clamp the weight at the edges, rows keep it ----------
__device__ __forceinline__ void lin_coord(int d, int dn, int sn, int* i0, int* i1, float* f, bool clamp_w) {
    const float fv = (float)(((double)d + 0.5) * (1.0 / ((double)dn / sn)) - 0.5);
    int i = (int)floorf(fv);
    float fr = fs(fv, (float)i);
    if (clamp_w) {
        if (i < 0 || i >= sn - 1) { fr = 0.f; i = min(max(i, 0), sn - 1); }
        *i0 = i; *i1 = min(i + 1, sn - 1);
    } else {
        *i0 = min(max(i, 0), sn - 1); *i1 = min(max(i + 1, 0), sn - 1);
    }
    *f = fr;
}

// z < n_out_dirs * ... : image z reads U + z*sh*sw*2; output pointer chosen per image (fwd for z < half, else bwd)
__global__ void dis_upsample_kernel(const float* __restrict__ U, int sh, int sw, int h, int w, float factor,
                                    float* out0, long long stride0, float* out1, long long stride1, int half,
                                    float max_value) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
    if (x >= w || y >= h) return;
    const float2* S = reinterpret_cast<const float2*>(U) + (long long)z * sh * sw;
    float2 v;
    if (sh == h && sw == w) {
        v = S[(long long)y * sw + x];
    } else {
        int x0, x1, y0, y1;
        float fx, fy;
        lin_coord(x, w, sw, &x0, &x1, &fx, true);
        lin_coord(y, h, sh, &y0, &y1, &fy, false);
        const float gx = fs(1.f, fx), gy = fs(1.f, fy);
        const float2 a = S[(long long)y0 * sw + x0], b = S[(long long)y0 * sw + x1];
        const float2 c = S[(long long)y1 * sw + x0], d = S[(long long)y1 * sw + x1];
        const float r0x = fa(fm(a.x, gx), fm(b.x, fx)), r0y = fa(fm(a.y, gx), fm(b.y, fx));
        const float r1x = fa(fm(c.x, gx), fm(d.x, fx)), r1y = fa(fm(c.y, gx), fm(d.y, fx));
        v.x = fa(fm(r0x, gy), fm(r1x, fy));
        v.y = fa(fm(r0y, gy), fm(r1y, fy));
    }
    v.x = fm(v.x, factor); v.y = fm(v.y, factor);
    if (max_value > 0.f) {
        v.x = fminf(fmaxf(v.x, -max_value), max_value);
        v.y = fminf(fmaxf(v.y, -max_value), max_value);
    }
    float* o = z < half ? out0 + (long long)z * stride0 : out1 + (long long)(z - half) * stride1;
    reinterpret_cast<float2*>(o)[(long long)y * w + x] = v;
}

// ---- host side --------------------------------------------------------------------------------------------------
struct DisPlan {
    int finest, coarsest;
    int h[DIS_MAX_SCALES], w[DIS_MAX_SCALES];
};

int dis_plan(int H, int W, const tf_dis_params& p, DisPlan* out) {
    if (H <= 0 || W <= 0) { set_error("DIS: empty frame"); return TF_ERR_INVALID_ARGUMENT; }
    if (p.finest_scale < 0 || p.patch_stride < 1 || p.patch_stride > DIS_PS || p.gradient_descent_iterations < 0 ||
        p.variational_refinement_iterations < 0) {
        set_error("DIS: invalid parameters (finest_scale >= 0, 1 <= patch_stride <= 8, iterations >= 0)");
        return TF_ERR_INVALID_ARGUMENT;
    }
    // calc(): the coarsest scale keeps a maximal motion of a quarter of the frame and a pyramid no smaller than a patch
    const int mn = min(W, H) / DIS_PS;
    const int c_deep = mn > 0 ? (int)(log((double)mn) / log(2.0)) : INT_MIN;
    int coarsest = min((int)(log(max(W, H) / (4.0 * DIS_PS)) / log(2.0) + 0.5), c_deep);
    int finest = p.finest_scale;
    if (coarsest < 0) {
        set_error("DIS: the frame (%d x %d) is too small (OpenCV: \"The input image must have either width or height >= 12\")", H, W);
        return TF_ERR_INVALID_ARGUMENT;
    }
    if (coarsest < finest) {
        // autoSelectPatchSizeAndScales: finest scales 0..2 keep patch size 8 (3, 4 would switch to 12)
        if (finest > 2) { set_error("DIS: finest_scale > 2 on a small frame selects patch size 12 (not built)"); return TF_ERR_UNSUPPORTED; }
        coarsest = max(0, (int)floorf(log2f((2.0f * (float)W) / (5.0f * 8.0f))));
        finest = max(coarsest - 2, 0);
    }
    if (coarsest >= DIS_MAX_SCALES) { set_error("DIS: frame too large"); return TF_ERR_INVALID_ARGUMENT; }
    out->finest = finest; out->coarsest = coarsest;
    out->h[finest] = H / (1 << finest); out->w[finest] = W / (1 << finest);
    for (int s = finest + 1; s <= coarsest; ++s) { out->h[s] = out->h[s - 1] / 2; out->w[s] = out->w[s - 1] / 2; }
    for (int s = finest; s <= coarsest; ++s)
        if (out->h[s] < DIS_PS || out->w[s] < DIS_PS) {
            set_error("DIS: scale %d of a %d x %d frame is %d x %d, smaller than a patch", s, H, W, out->h[s], out->w[s]);
            return TF_ERR_INVALID_ARGUMENT;
        }
    return TF_OK;
}

struct DisLayout {
    size_t pyr[DIS_MAX_SCALES], gx, gy, aux, st, sx, sy, u0, u1, vr, total;
};

DisLayout dis_layout(int n, const DisPlan& pl, int stride) {
    DisLayout L{};
    size_t o = 0;
    auto take = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
    for (int s = pl.finest; s <= pl.coarsest; ++s) L.pyr[s] = take((size_t)2 * n * pl.h[s] * pl.w[s]);
    const size_t hf = pl.h[pl.finest], wf = pl.w[pl.finest];
    const size_t hsf = 1 + (hf - DIS_PS) / stride, wsf = 1 + (wf - DIS_PS) / stride;
    L.gx = take(2 * n * hf * wf * 2);
    L.gy = take(2 * n * hf * wf * 2);
    L.aux = take(5 * 2 * n * hf * wsf * 4);
    L.st = take(5 * 2 * n * hsf * wsf * 4);
    L.sx = take(2 * n * hsf * wsf * 4);
    L.sy = take(2 * n * hsf * wsf * 4);
    L.u0 = take(2 * n * hf * wf * 8);
    L.u1 = take(2 * n * hf * wf * 8);
    L.vr = take(tf_vr_workspace_bytes(n, (int)hf, (int)wf));
    L.total = o;
    return L;
}

// pyramid of the 2n images (q0 block then q1 block) at every scale
void dis_pyramid(const uint8_t* q0, const uint8_t* q1, int n, int H, int W, const DisPlan& pl, const DisLayout& L,
                uint8_t* ws, cudaStream_t s) {
    const dim3 blk(32, 8);
    const int f = pl.finest;
    const long long hw = (long long)pl.h[f] * pl.w[f];
    uint8_t* P = ws + L.pyr[f];
    if (f == 0) {
        cudaMemcpyAsync(P, q0, (size_t)n * hw, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(P + n * hw, q1, (size_t)n * hw, cudaMemcpyDeviceToDevice, s);
    } else {
        const dim3 g(cdiv(pl.w[f], 32), cdiv(pl.h[f], 8), n);
        dis_area_kernel<<<g, blk, 0, s>>>(q0, (long long)H * W, H, W, P, hw, pl.h[f], pl.w[f]);
        dis_area_kernel<<<g, blk, 0, s>>>(q1, (long long)H * W, H, W, P + n * hw, hw, pl.h[f], pl.w[f]);
    }
    for (int sc = f + 1; sc <= pl.coarsest; ++sc) {
        const dim3 g(cdiv(pl.w[sc], 32), cdiv(pl.h[sc], 8), 2 * n);
        dis_area_kernel<<<g, blk, 0, s>>>(ws + L.pyr[sc - 1], (long long)pl.h[sc - 1] * pl.w[sc - 1], pl.h[sc - 1],
                                          pl.w[sc - 1], ws + L.pyr[sc], (long long)pl.h[sc] * pl.w[sc], pl.h[sc], pl.w[sc]);
    }
}

}  // namespace tf

using namespace tf;

extern "C" void tf_dis_default_params(tf_dis_params* p, int preset) {
    if (!p) return;
    p->finest_scale = 2; p->patch_stride = 4; p->gradient_descent_iterations = 16;
    p->variational_refinement_iterations = 5;
    if (preset == 0) { p->gradient_descent_iterations = 12; p->variational_refinement_iterations = 0; }
    if (preset == 2) { p->finest_scale = 1; p->patch_stride = 3; p->gradient_descent_iterations = 25; }
    p->vr_alpha = 20.f; p->vr_delta = 5.f; p->vr_gamma = 10.f; p->vr_epsilon = 0.01f;
    p->max_value = 0.f;
}

extern "C" int tf_dis_scale_plan(int H, int W, const tf_dis_params* p, int* finest, int* coarsest, int* hs, int* ws) {
    if (!p) { set_error("tf_dis_scale_plan: invalid argument"); return TF_ERR_INVALID_ARGUMENT; }
    DisPlan pl;
    const int rc = dis_plan(H, W, *p, &pl);
    if (rc != TF_OK) return rc;
    if (finest) *finest = pl.finest;
    if (coarsest) *coarsest = pl.coarsest;
    for (int s = pl.finest; s <= pl.coarsest; ++s) {
        if (hs) hs[s] = pl.h[s];
        if (ws) ws[s] = pl.w[s];
    }
    return TF_OK;
}

extern "C" size_t tf_dis_workspace_bytes(int n_pairs, int H, int W, const tf_dis_params* p) {
    if (!p || n_pairs <= 0) return 0;
    DisPlan pl;
    if (dis_plan(H, W, *p, &pl) != TF_OK) return 0;
    return dis_layout(n_pairs, pl, p->patch_stride).total;
}

extern "C" int tf_dis_scale_images(const uint8_t* q, int n_img, int H, int W, const tf_dis_params* p, int scale,
                                   uint8_t* img, int16_t* gx, int16_t* gy, void* workspace, size_t workspace_bytes,
                                   void* stream) {
    if (!q || !p || !img || !gx || !gy || !workspace || n_img <= 0 || n_img > 32767) {
        set_error("tf_dis_scale_images: invalid argument");
        return TF_ERR_INVALID_ARGUMENT;
    }
    DisPlan pl;
    int rc = dis_plan(H, W, *p, &pl);
    if (rc != TF_OK) return rc;
    if (scale < pl.finest || scale > pl.coarsest) { set_error("tf_dis_scale_images: scale %d outside the plan [%d, %d]", scale, pl.finest, pl.coarsest); return TF_ERR_INVALID_ARGUMENT; }
    // the n_img images as both halves of an n_img-pair batch (the second half is not read back)
    const DisLayout L = dis_layout(n_img, pl, p->patch_stride);
    if (workspace_bytes < L.total) { set_error("tf_dis_scale_images: workspace too small (%zu < %zu)", workspace_bytes, L.total); return TF_ERR_WORKSPACE_TOO_SMALL; }
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    dis_pyramid(q, q, n_img, H, W, pl, L, ws, s);
    const long long hw = (long long)pl.h[scale] * pl.w[scale];
    const uint8_t* P = ws + L.pyr[scale];
    cudaMemcpyAsync(img, P, (size_t)n_img * hw, cudaMemcpyDeviceToDevice, s);
    const dim3 g(cdiv(pl.w[scale], 32), cdiv(pl.h[scale], 8), n_img);
    dis_sobel_kernel<<<g, dim3(32, 8), 0, s>>>(P, pl.h[scale], pl.w[scale], gx, gy);
    return check_launch("tf_dis_scale_images");
}

extern "C" int tf_dis_pairs(const uint8_t* q0, const uint8_t* q1, float* fwd, long long fwd_stride, float* bwd,
                            long long bwd_stride, int n_pairs, int H, int W, const tf_dis_params* p, void* workspace,
                            size_t workspace_bytes, void* stream) {
    if (n_pairs == 0) return TF_OK;
    if (!q0 || !q1 || !fwd || !bwd || !p || !workspace || n_pairs < 0 || n_pairs > 32767) {
        set_error("tf_dis_pairs: invalid argument");
        return TF_ERR_INVALID_ARGUMENT;
    }
    if ((long long)H * W > 0x3fffffffLL) { set_error("tf_dis_pairs: frame too large"); return TF_ERR_INVALID_ARGUMENT; }
    DisPlan pl;
    int rc = dis_plan(H, W, *p, &pl);
    if (rc != TF_OK) return rc;
    const int n = n_pairs, nz = 2 * n, stride = p->patch_stride;
    const DisLayout L = dis_layout(n, pl, stride);
    if (workspace_bytes < L.total) { set_error("tf_dis_pairs: workspace too small (%zu < %zu)", workspace_bytes, L.total); return TF_ERR_WORKSPACE_TOO_SMALL; }
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    int16_t* gx = reinterpret_cast<int16_t*>(ws + L.gx);
    int16_t* gy = reinterpret_cast<int16_t*>(ws + L.gy);
    float* aux = reinterpret_cast<float*>(ws + L.aux);
    float* st = reinterpret_cast<float*>(ws + L.st);
    float* Sx = reinterpret_cast<float*>(ws + L.sx);
    float* Sy = reinterpret_cast<float*>(ws + L.sy);
    float* Ucur = reinterpret_cast<float*>(ws + L.u0);
    float* Unext = reinterpret_cast<float*>(ws + L.u1);
    const size_t vr_bytes = tf_vr_workspace_bytes(n, pl.h[pl.finest], pl.w[pl.finest]);
    dis_pyramid(q0, q1, n, H, W, pl, L, ws, s);
    const dim3 blk(32, 8);
    {
        const int c = pl.coarsest;
        cudaMemsetAsync(Ucur, 0, (size_t)nz * pl.h[c] * pl.w[c] * 8, s);
    }
    tf_vr_params vp;
    tf_vr_default_params(&vp);
    vp.alpha = p->vr_alpha; vp.delta = p->vr_delta; vp.gamma = p->vr_gamma; vp.epsilon = p->vr_epsilon;
    vp.fixed_point_iterations = p->variational_refinement_iterations; vp.sor_iterations = 5;
    for (int sc = pl.coarsest; sc >= pl.finest; --sc) {
        const int h = pl.h[sc], w = pl.w[sc];
        const int hsn = 1 + (h - DIS_PS) / stride, wsn = 1 + (w - DIS_PS) / stride;
        const uint8_t* P = ws + L.pyr[sc];
        const dim3 g(cdiv(w, 32), cdiv(h, 8), nz);
        {
            dis_sobel_kernel<<<g, blk, 0, s>>>(P, h, w, gx, gy);
            dis_struct_h_kernel<<<cdiv(nz * h, 128), 128, 0, s>>>(gx, gy, h, w, stride, wsn, aux, nz);
            dis_struct_v_kernel<<<cdiv(nz * wsn * 5, 128), 128, 0, s>>>(aux, h, stride, hsn, wsn, st, nz);
            DisSearchArgs a;
            a.pyr = P; a.n_img = nz; a.gx = gx; a.gy = gy; a.st = st; a.U = Ucur; a.Sx = Sx; a.Sy = Sy;
            a.h = h; a.w = w; a.hs = hsn; a.ws = wsn; a.stride = stride;
            a.stripe = (int)ceil(hsn / (double)DIS_STRIPES);
            a.inner = (int)floorf(p->gradient_descent_iterations / 2.0f);
            dis_search_kernel<<<dim3(DIS_STRIPES, nz), 64, 0, s>>>(a);
            dis_densify_kernel<<<g, blk, 0, s>>>(P, nz, Sx, Sy, h, w, hsn, wsn, stride, Ucur);
        }
        if (p->variational_refinement_iterations > 0) {
            const long long hw2 = (long long)h * w * 2;
            rc = tf_variational_refinement(P, P + (long long)n * h * w, Ucur, hw2, Ucur + n * hw2, hw2, n, h, w, &vp,
                                           ws + L.vr, vr_bytes, s);
            if (rc != TF_OK) return rc;
        }
        if (sc > pl.finest) {
            const int h2 = pl.h[sc - 1], w2 = pl.w[sc - 1];
            const long long o2 = (long long)h2 * w2 * 2;
            dis_upsample_kernel<<<dim3(cdiv(w2, 32), cdiv(h2, 8), nz), blk, 0, s>>>(
                Ucur, h, w, h2, w2, 2.f, Unext, o2, Unext + n * o2, o2, n, 0.f);
            float* t = Ucur; Ucur = Unext; Unext = t;
        } else {
            dis_upsample_kernel<<<dim3(cdiv(W, 32), cdiv(H, 8), nz), blk, 0, s>>>(
                Ucur, h, w, H, W, (float)(1 << pl.finest), fwd, fwd_stride, bwd, bwd_stride, n, p->max_value);
        }
    }
    return check_launch("tf_dis_pairs");
}
