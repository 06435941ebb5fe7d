// The Farneback Jacobi iteration for any window OpenCV offers that the GPU reproduces: FarnebackUpdateFlow_Blur with a
// box of 3..63 and FarnebackUpdateFlow_GaussianBlur with a Gaussian window of 4..63.  UpdateMatrices, the window sums
// and the 2x2 solve for n_pairs pairs x 2 directions, with the launch contract of launch_fb_iteration (without the fused
// up-sampling).  The default 13 x 13 box runs the specialised kernel of fb_iter.cu instead.
//
// A CTA marches down a strip of 128 - 2m output columns (m = win_size / 2) and a chunk of rows, in batches of 4 rows:
//   M phase: two threads per region column form UpdateMatrices' five products of two rows each into a shared-memory
//            ring that holds the last 2m + 4 rows;
//   V phase: the vertical window sums of the batch's rows, each summed directly from the 2m + 1 ring rows;
//   H phase: the horizontal window sums of those rows, the solve, the (clamped) flow store.
// Every window sum is formed fresh in a fixed order (no running sums, whose fp32 rounding drifts down a column), so a
// result depends neither on the chunk grid nor on the batch of pairs.  Box: plain sums top to bottom / left to right,
// with OpenCV's 1 / win_size^2 scale folded into the regulariser (numerator and determinant are both quadratic in the
// sums).  Gaussian: k0 r[y] + sum_i k_i (r[y + i] + r[y - i]) in fp32, as OpenCV orders it, first along y, then x.
// Both borders replicate: the ring rows and region columns are read at clamped image positions.
#include "fb_iter_common.cuh"

namespace tf {

constexpr int GI_COLS = 128;   // region columns: the output strip plus m halo columns on either side
constexpr int GI_NT = 256;     // threads per CTA
constexpr int GI_RB = 4;       // rows per batch
constexpr int GI_MAX_M = 31;   // window radius of win_size 63

struct WinTaps {
    float k[GI_MAX_M + 1];     // Gaussian taps k[0..m] (normalised); unused for the box
};

static int gi_smem_bytes(int m) { return (2 * m + 2 * GI_RB) * 5 * GI_COLS * (int)sizeof(float); }

template <bool GAUSS>
__global__ void __launch_bounds__(GI_NT)
fb_iter_general_kernel(const float* __restrict__ R, long long img_stride, const float* __restrict__ flow_in,
                       float* __restrict__ out_fwd, long long fwd_stride, float* __restrict__ out_bwd, long long bwd_stride,
                       int h, int w, int m, int chunk_rows, float reg, float clampv, const __grid_constant__ WinTaps taps) {
    constexpr int CH = 5 * GI_COLS;                    // floats per row of five channel planes
    extern __shared__ __align__(16) float gi_smem[];
    const int ring_rows = 2 * m + GI_RB;
    float* ring = gi_smem;                             // [image row % ring_rows][channel][column]: the products M
    float* vs = gi_smem + ring_rows * CH;              // [batch row][channel][column]: vertical window sums
    const int tid = threadIdx.x;
    const int dir = blockIdx.x & 1, strip = blockIdx.x >> 1, pair = blockIdx.z;
    const int yc0 = blockIdx.y * chunk_rows, yc1 = min(yc0 + chunk_rows, h);
    const int plane = h * w;
    const float* Rp = R + (long long)(2 * pair) * img_stride;
    const float* Rn = Rp + img_stride;
    const float* R0 = dir ? Rn : Rp;
    const float* R1 = dir ? Rp : Rn;
    RPlanes RP;
    RP.R0a = reinterpret_cast<const float4*>(R0);
    RP.R0b = R0 + 4 * (long long)plane;
    RP.R1a = reinterpret_cast<const float4*>(R1);
    RP.R1b = R1 + 4 * (long long)plane;
    const float2* fin = reinterpret_cast<const float2*>(flow_in) + (long long)(2 * pair + dir) * plane;
    float2* fout = reinterpret_cast<float2*>(dir ? out_bwd + (long long)pair * bwd_stride
                                                 : out_fwd + (long long)pair * fwd_stride);
    const int xs = strip * (GI_COLS - 2 * m) - m;      // image column of region column 0
    // M phase identity: region column c, batch rows `half` and `half + 2`
    const int c = tid & (GI_COLS - 1), half = tid >> 7;
    const int gx = min(max(xs + c, 0), w - 1);
    const float sc_x = border_factor(gx, w);
    const bool band_x = border_band(gx, w);
    // region row i is image row yc0 - m + i (clamped); output row yc0 + o has its window in region rows o .. o + 2m
    const int n_rows = (yc1 - yc0) + 2 * m;
    const int n_batches = (n_rows + GI_RB - 1) / GI_RB;

    for (int b = 0; b < n_batches; ++b) {
        // ---- M phase ----------------------------------------------------------------------------------------------
        Taps t[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int y = min(max(yc0 - m + b * GI_RB + half + 2 * q, 0), h - 1);
            issue_taps(t[q], RP, w, h, gx, y, ld_stream(fin + (long long)y * w + gx));
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            float mm[5];
            matrix_from_taps(t[q], h, sc_x, band_x, mm);
            float* dst = ring + ((b * GI_RB + half + 2 * q) % ring_rows) * CH + c;
#pragma unroll
            for (int k = 0; k < 5; ++k) dst[k * GI_COLS] = mm[k];
        }
        __syncthreads();
        const int o0 = b * GI_RB - 2 * m;              // output row (relative to yc0) of batch row 0
        if (o0 + GI_RB <= 0) continue;                 // no window complete yet (uniform across the CTA)
        // ---- V phase ----------------------------------------------------------------------------------------------
        for (int e = tid; e < GI_RB * CH; e += GI_NT) {
            const int j = e / CH, kc = e - j * CH;
            const int o = o0 + j;
            if (o < 0 || yc0 + o >= yc1) continue;
            const float* col = ring + kc;
            float acc;
            if (GAUSS) {
                int up = (o + m) % ring_rows, dn = up;
                acc = col[up * CH] * taps.k[0];
                for (int i = 1; i <= m; ++i) {
                    up = (up == ring_rows - 1) ? 0 : up + 1;
                    dn = (dn == 0) ? ring_rows - 1 : dn - 1;
                    acc = fmaf(col[up * CH] + col[dn * CH], taps.k[i], acc);
                }
            } else {
                int s = o % ring_rows;
                acc = col[s * CH];
                for (int i = 1; i <= 2 * m; ++i) {
                    s = (s == ring_rows - 1) ? 0 : s + 1;
                    acc += col[s * CH];
                }
            }
            vs[e] = acc;
        }
        __syncthreads();
        // ---- H phase: batch row tid / 64, region columns m + tid % 64 + 64 i ------------------------------------------
        const int j = tid >> 6;
        const int y = yc0 + o0 + j;
        if (o0 + j < 0 || y >= yc1) continue;
        for (int cc = m + (tid & 63); cc < GI_COLS - m; cc += 64) {
            const int x = xs + cc;
            if (x >= w) break;
            float g[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float* v = vs + (j * 5 + k) * GI_COLS + cc;
                float acc;
                if (GAUSS) {
                    acc = v[0] * taps.k[0];
                    for (int i = 1; i <= m; ++i) acc = fmaf(v[-i] + v[i], taps.k[i], acc);
                } else {
                    acc = v[-m];
                    for (int i = 1 - m; i <= m; ++i) acc += v[i];
                }
                g[k] = acc;
            }
            const float g11 = g[0], g12 = g[1], g22 = g[2], h1 = g[3], h2 = g[4];
            const float idet = 1.f / (diff_of_products(g11, g22, g12, g12) + reg);
            float fx = diff_of_products(g11, h2, g12, h1) * idet;
            float fy = diff_of_products(g22, h1, g12, h2) * idet;
            if (clampv > 0.f) {
                fx = fminf(fmaxf(fx, -clampv), clampv);
                fy = fminf(fmaxf(fy, -clampv), clampv);
            }
            fout[(long long)y * w + x] = make_float2(fx, fy);
        }
    }
}

int launch_fb_iteration_general(const float* R, long long img_stride, const float* flow_in, float* out_fwd,
                                long long fwd_stride, float* out_bwd, long long bwd_stride, int n_pairs, int h, int w,
                                int win, bool gaussian, float clamp, bool full_res, cudaStream_t s) {
    const int m = win / 2;
    if (win < (gaussian ? 4 : 3) || m > GI_MAX_M) {
        set_error("fb iteration: win_size %d is outside the built range (box 3..63, Gaussian 4..63)", win);
        return TF_ERR_UNSUPPORTED;
    }
    if ((long long)h * w > 0x3fffffffLL) { set_error("fb iteration: level too large"); return TF_ERR_INVALID_ARGUMENT; }
    WinTaps taps{};
    float reg;
    if (gaussian) {
        // FarnebackUpdateFlow_GaussianBlur: sigma = 0.3 m, fp32 taps normalised by their sum taken in double
        const double sigma = m * 0.3;
        double sum = 1;
        float k[GI_MAX_M + 1];
        k[0] = 1.f;
        for (int i = 1; i <= m; ++i) {
            k[i] = (float)exp(-i * i / (2 * sigma * sigma));
            sum += k[i] * 2.0;
        }
        for (int i = 0; i <= m; ++i) taps.k[i] = (float)(k[i] * (1. / sum));
        reg = 1e-3f;
    } else {
        reg = 1e-3f * (float)(win * win) * (float)(win * win);
    }
    const int smem = gi_smem_bytes(m);
    auto kern = gaussian ? fb_iter_general_kernel<true> : fb_iter_general_kernel<false>;
    // (the attribute is per device: set it on every call, it is cheap)
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const int strips = cdiv(w, GI_COLS - 2 * m);
    const int per_sm = max(1, min(2048 / GI_NT, 228 * 1024 / (smem + 1024)));
    int chunks;
    const int chunk_rows = plan_chunk_rows(h, strips, n_pairs, 148LL * per_sm, &chunks, m);
    // algorithmic bytes: the 56 B per pixel-iteration of the default kernel's model
    LaunchTimer lt(full_res ? KC_FB_ITER_L0 : KC_FB_ITER, 56.0 * h * w * 2 * n_pairs, s, cdiv(n_pairs, 65535));
    for (int p0 = 0; p0 < n_pairs; p0 += 65535) {
        const int np = min(n_pairs - p0, 65535);
        dim3 g(2 * strips, chunks, np);
        kern<<<g, GI_NT, smem, s>>>(R + (long long)(2 * p0) * img_stride, img_stride, flow_in + (long long)(2 * p0) * 2 * h * w,
                                    out_fwd + p0 * fwd_stride, fwd_stride, out_bwd + p0 * bwd_stride, bwd_stride, h, w, m,
                                    chunk_rows, reg, clamp, taps);
    }
    return check_launch("fb iteration (general window)");
}

}  // namespace tf
