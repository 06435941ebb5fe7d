// K3: Farneback polynomial expansion (OpenCV FarnebackPolyExp, polyN = 5 or 7): separable (2N+1)-tap tile convolution
// with replicate borders.  Input level image I (h, w) fp32 -> per image a float4 plane (c0..c3) followed by a float plane
// (c4), so the iteration kernel's bilinear gathers are one 16-byte and one 4-byte coalesced load per tap.
// Shared-memory tile with an N-pixel halo; both passes are register-blocked (vertical: a (16 + 2N)-row column window per
// thread for 16 outputs; horizontal: 4 + 2N values of each moment row per thread for 4 outputs).
// HBM traffic: 4 B/px read (+ halo re-reads that hit L2) and 20 B/px written.
#include "farneback_internal.cuh"

namespace tf {

template <int N>
struct PeCfg {
    static constexpr int SW = 128;                 // region columns incl. halo (also the shared-memory pitch)
    static constexpr int TW = SW - 2 * N;          // output columns per tile
    static constexpr int TH = 32;                  // output rows per tile
    static constexpr int SH = TH + 2 * N;          // rows incl. halo
    static constexpr int VSEG = 16;                // rows per thread in the vertical pass
    static constexpr int NV = (4 + 2 * N + 3) / 4; // float4 loads of a moment row per thread in the horizontal pass
    static constexpr int GROUPS = (TW + 3) / 4;    // groups of 4 output columns (the last one may overhang TW)
    // +4: the last group's loads overhang
    static constexpr int SMEM_BYTES = (SH * SW + 3 * TH * SW + 4) * (int)sizeof(float);
    static_assert(4 * (GROUPS - 1) + 4 * NV <= SW + 4, "horizontal loads stay inside the tile + pad");
};

template <int N>
__global__ void __launch_bounds__(256) polyexp_kernel(const float* __restrict__ I, float* __restrict__ R,
                                                      long long img_stride, int h, int w, PolyConsts pc) {
    using C = PeCfg<N>;
    constexpr int PE_N = N, PE_SW = C::SW, PE_TW = C::TW, PE_TH = C::TH, PE_SH = C::SH, PE_VSEG = C::VSEG;
    extern __shared__ __align__(16) float pe_smem[];
    float (*s_in)[PE_SW] = reinterpret_cast<float (*)[PE_SW]>(pe_smem);
    float (*s_v)[PE_TH][PE_SW] = reinterpret_cast<float (*)[PE_TH][PE_SW]>(pe_smem + PE_SH * PE_SW);
    const int img = blockIdx.z;
    const int x0 = blockIdx.x * PE_TW, y0 = blockIdx.y * PE_TH;
    const float* src = I + (long long)img * h * w;
    const int tid = threadIdx.x;

    // tile + N-px halo, replicate-clamped (the clamp IS OpenCV's border rule for both passes)
    // (all loads of a thread are issued before the first shared-memory store: one memory round trip, not one per load)
    {
        static_assert((PE_SH * PE_SW) % 256 == 0 && PE_SW == 128, "tile load: 2 rows per pass of the 256 threads");
        constexpr int PASSES = PE_SH * PE_SW / 256;
        const int c = tid & (PE_SW - 1), r0 = tid >> 7;
        const int gx = min(max(x0 + c - PE_N, 0), w - 1);
        float v[PASSES];
#pragma unroll
        for (int p = 0; p < PASSES; ++p) {
            const int gy = min(max(y0 + r0 + 2 * p - PE_N, 0), h - 1);
            v[p] = __ldg(src + gy * w + gx);
        }
#pragma unroll
        for (int p = 0; p < PASSES; ++p) s_in[r0 + 2 * p][c] = v[p];
    }
    __syncthreads();

    // vertical pass: one thread per (column, 16-row segment), the 26 input rows it needs held in registers;
    // fp32, accumulation order of OpenCV (k = 1..n)
    {
        const int c = tid & (PE_SW - 1), seg = tid >> 7;
        float in[PE_VSEG + 2 * PE_N];
#pragma unroll
        for (int i = 0; i < PE_VSEG + 2 * PE_N; ++i) in[i] = s_in[seg * PE_VSEG + i][c];
#pragma unroll
        for (int r = 0; r < PE_VSEG; ++r) {
            float t0 = in[r + PE_N] * pc.g[0], t1 = 0.f, t2 = 0.f;
#pragma unroll
            for (int k = 1; k <= PE_N; ++k) {
                const float a = in[r + PE_N - k], b = in[r + PE_N + k];
                const float p = a + b;
                t0 = t0 + pc.g[k] * p;
                t1 = t1 + pc.xg[k] * (b - a);
                t2 = t2 + pc.xxg[k] * p;
            }
            s_v[0][seg * PE_VSEG + r][c] = t0;
            s_v[1][seg * PE_VSEG + r][c] = t1;
            s_v[2][seg * PE_VSEG + r][c] = t2;
        }
    }
    __syncthreads();

    // horizontal pass: one thread per (row, 4 adjacent outputs): 16 values of each moment row via LDS.128
    const int plane = h * w;
    float4* dst_a = reinterpret_cast<float4*>(R + (long long)img * img_stride);
    float* dst_b = R + (long long)img * img_stride + 4 * (long long)plane;
    constexpr int GROUPS = C::GROUPS, NV = C::NV;
    const bool wide_ok = (w & 1) == 0 && (reinterpret_cast<uintptr_t>(dst_a) & 31) == 0;   // 32-byte aligned texel pairs
    for (int task = tid; task < PE_TH * GROUPS; task += 256) {
        const int r = task / GROUPS, cgp = task - r * GROUPS;
        const int c0 = 4 * cgp;               // first output column (tile-relative); its region column is c0 + PE_N
        const int gy = y0 + r;
        if (gy >= h || x0 + c0 >= w) continue;
        float v0[4 * NV], v1[4 * NV], v2[4 * NV];   // region columns c0 .. c0+4NV-1  (outputs need c0 .. c0+3+2N)
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const float4 a = *reinterpret_cast<const float4*>(&s_v[0][r][c0 + 4 * q]);
            const float4 b = *reinterpret_cast<const float4*>(&s_v[1][r][c0 + 4 * q]);
            const float4 d = *reinterpret_cast<const float4*>(&s_v[2][r][c0 + 4 * q]);
            v0[4 * q] = a.x; v0[4 * q + 1] = a.y; v0[4 * q + 2] = a.z; v0[4 * q + 3] = a.w;
            v1[4 * q] = b.x; v1[4 * q + 1] = b.y; v1[4 * q + 2] = b.z; v1[4 * q + 3] = b.w;
            v2[4 * q] = d.x; v2[4 * q + 1] = d.y; v2[4 * q + 2] = d.z; v2[4 * q + 3] = d.w;
        }
        float4 oa[4];
        float ob[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = i + PE_N;           // index of the output's own column in v*
            float b1 = v0[m] * pc.g[0], b2 = 0.f, b3 = v1[m] * pc.g[0], b4 = 0.f, b5 = v2[m] * pc.g[0], b6 = 0.f;
#pragma unroll
            for (int k = 1; k <= PE_N; ++k) {
                const float tg = v0[m + k] + v0[m - k];
                b1 += tg * pc.g[k];
                b4 += tg * pc.xxg[k];
                b2 += (v0[m + k] - v0[m - k]) * pc.xg[k];
                b3 += (v1[m + k] + v1[m - k]) * pc.g[k];
                b6 += (v1[m + k] - v1[m - k]) * pc.xg[k];
                b5 += (v2[m + k] + v2[m - k]) * pc.g[k];
            }
            oa[i] = make_float4(b3 * pc.ig11, b2 * pc.ig11, b1 * pc.ig03 + b5 * pc.ig33, b1 * pc.ig03 + b4 * pc.ig33);
            ob[i] = b6 * pc.ig55;
        }
        // A thread's four texels are 64 contiguous bytes of the float4 plane.  Lanes are 64 bytes apart, so four 16-byte
        // stores touch every 128-byte line of the warp's 2 KB span four times; Blackwell's 256-bit stores (STG.256) halve
        // that.  Tile width and group offset are even, so with an even w the pairs (0, 1) and (2, 3) are 32-byte aligned
        // and inside / outside the image together.
        const int gx0 = x0 + c0;
        const long long o = (long long)gy * w + gx0;
        const int nvalid = max(0, min(4, min(PE_TW - c0, w - gx0)));
        if (wide_ok && (nvalid & 1) == 0) {
#pragma unroll
            for (int i = 0; i < 4; i += 2) {
                if (i >= nvalid) break;
                asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                             ::"l"(dst_a + o + i), "f"(oa[i].x), "f"(oa[i].y), "f"(oa[i].z), "f"(oa[i].w), "f"(oa[i + 1].x),
                               "f"(oa[i + 1].y), "f"(oa[i + 1].z), "f"(oa[i + 1].w) : "memory");
            }
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (i < nvalid) dst_a[o + i] = oa[i];
        }
        if (nvalid == 4 && ((reinterpret_cast<uintptr_t>(dst_b + o)) & 15) == 0) {
            *reinterpret_cast<float4*>(dst_b + o) = make_float4(ob[0], ob[1], ob[2], ob[3]);
        } else if ((nvalid & 1) == 0 && ((reinterpret_cast<uintptr_t>(dst_b + o)) & 7) == 0) {
#pragma unroll
            for (int i = 0; i < 4; i += 2)
                if (i < nvalid) *reinterpret_cast<float2*>(dst_b + o + i) = make_float2(ob[i], ob[i + 1]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (i < nvalid) dst_b[o + i] = ob[i];
        }
    }
}

template <int N>
static void launch_polyexp_n(const float* I, float* R, long long img_stride, int n_img, int h, int w, const PolyConsts& pc,
                             cudaStream_t s) {
    using C = PeCfg<N>;
    // (the attribute is per device: set it on every call, it is cheap)
    cudaFuncSetAttribute(polyexp_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    for (int z0 = 0; z0 < n_img; z0 += 65535) {
        const int nz = min(n_img - z0, 65535);
        dim3 g(cdiv(w, C::TW), cdiv(h, C::TH), nz);
        polyexp_kernel<N><<<g, 256, C::SMEM_BYTES, s>>>(I + (long long)z0 * h * w, R + (long long)z0 * img_stride,
                                                        img_stride, h, w, pc);
    }
}

int launch_polyexp(const float* I, float* R, long long img_stride, int n_img, int h, int w, const PolyConsts& pc,
                   cudaStream_t s) {
    if (pc.n != 5 && pc.n != 7) { set_error("polyexp: poly_n %d is not built (5 or 7)", pc.n); return TF_ERR_UNSUPPORTED; }
    LaunchTimer lt(KC_POLYEXP, 24.0 * h * w * n_img, s, cdiv(n_img, 65535));
    if (pc.n == 5) launch_polyexp_n<5>(I, R, img_stride, n_img, h, w, pc, s);
    else launch_polyexp_n<7>(I, R, img_stride, n_img, h, w, pc, s);
    return check_launch("polyexp");
}

// FarnebackPrepareGaussian: fp32 taps, fp64 moment matrix inverse (closed form for the sparse 6x6)
PolyConsts make_poly_consts(int n, double sigma) {
    PolyConsts pc{};
    pc.n = n;
    if (sigma < 1.1920929e-07) sigma = n * 0.3;
    float g[15];
    double s = 0;
    for (int x = -n; x <= n; ++x) {
        g[x + n] = (float)exp(-x * x / (2 * sigma * sigma));
        s += g[x + n];
    }
    s = 1. / s;
    for (int x = -n; x <= n; ++x) g[x + n] = (float)(g[x + n] * s);
    for (int k = 0; k <= n; ++k) {
        pc.g[k] = g[n + k];
        pc.xg[k] = (float)(k * g[n + k]);
        pc.xxg[k] = (float)(k * k * g[n + k]);
    }
    double G00 = 0, G11 = 0, G33 = 0, G55 = 0;
    for (int y = -n; y <= n; ++y)
        for (int x = -n; x <= n; ++x) {
            const double gg = (double)g[y + n] * g[x + n];
            G00 += gg;
            G11 += gg * x * x;
            G33 += gg * x * x * x * x;
            G55 += gg * x * x * y * y;
        }
    // G = [[G00,0,0,G11,G11,0],[0,G11,..],[..G11..],[G11,0,0,G33,G55,0],[G11,0,0,G55,G33,0],[0,..,G55]]
    // inverse entries needed: (1,1), (0,3), (3,3), (5,5).  The {0,3,4} block is
    //   A = [[a, b, b], [b, c, d], [b, d, c]] with a=G00, b=G11, c=G33, d=G55.
    const double a = G00, b = G11, c = G33, d = G55;
    const double det = a * (c * c - d * d) - 2 * b * b * (c - d);
    pc.ig11 = (float)(1.0 / G11);
    pc.ig03 = (float)(-(b * (c - d)) / det);   // cofactor(3,0)/det = -(b*c - b*d)/det
    pc.ig33 = (float)((a * c - b * b) / det);
    pc.ig55 = (float)(1.0 / G55);
    return pc;
}

}  // namespace tf
