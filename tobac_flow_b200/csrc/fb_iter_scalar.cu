// The fused Farneback iteration in plain LDG / shared-memory / scalar-fp32 form: the round-1 kernel, kept as the A/B
// baseline and cross-check of the default kernel in fb_iter.cu (same strip march, same batches, same window sums bit for
// bit; see that file for the design).  tf_fb_select_kernel(0) -- or TF_TMA=0 in the environment -- selects it;
// tf_fb_select_kernel(1) the same kernel with its prefix-sum ring in tensor memory instead of shared memory.
//
// M phase: software-pipelined one row ahead (the next row's ten gather loads, its R0 and four rows of flow are in flight
// while the current row is computed).  127 registers without spills, 4 CTAs x 128 threads per SM, 43.5 KB shared memory
// per CTA.  Measured at 4.43 TB/s (0.68 of the copy bandwidth) against 5.1-5.2 TB/s for the default kernel: 40 % of its
// warp time is long-scoreboard wait at the first use of a row's taps (profiles/README.md has the variants tried on it:
// deeper lookahead, L2 prefetch, tap inheritance, persistent row-space grid, 256-column strips).
#include "fb_iter_common.cuh"

namespace tf {

template <bool TM>
struct ScalarCfg {
    static constexpr int NT = 128, HK = 4, OUT_W = NT - 2 * IT_HALO;
    // 3 batches x prefix sums P0..P2 x 5 channels; TM: the ring lives in tensor memory (thread-private columns)
    static constexpr int RING_FLOATS = TM ? 0 : 3 * 3 * 5 * NT;
    static constexpr int TM_COLS = 64;                       // 45 used; allocations are powers of two >= 32
    static constexpr int VBUF_FLOATS = 8 * 5 * NT;           // 2 buffers x 4 rows of vertical sums
    static constexpr int SMEM_BYTES = (RING_FLOATS + VBUF_FLOATS) * (int)sizeof(float);
};

template <bool TM>
__global__ void __launch_bounds__(128, 4)
fb_iter_scalar_kernel(const float* __restrict__ R, long long img_stride, const float* __restrict__ flow_in,
                      float* __restrict__ out_fwd, long long fwd_stride, float* __restrict__ out_bwd,
                      long long bwd_stride, int h, int w, int chunk_rows, float clampv) {
    using C = ScalarCfg<TM>;
    constexpr int NT = C::NT, HK = C::HK;
    extern __shared__ __align__(16) float smem[];
    float* ring = smem;                       // [batch % 3][P0..P2][k][col]: prefix sums of the batch's rows
    float* vbuf = smem + C::RING_FLOATS;      // [buf][row][k][NT]
    const int tid = threadIdx.x;
    uint32_t tm_base = 0;                     // TM: this warp's lane quarter, column 0 of the CTA's allocation
    if constexpr (TM) {
        __shared__ uint32_t tm_addr_s;
        if (tid < 32) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"((uint32_t)__cvta_generic_to_shared(&tm_addr_s)), "n"(C::TM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tm_base = tm_addr_s + ((uint32_t)(tid >> 5) << 21);      // lane (bits 31:16) = 32 * warp
    }
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
    const int x0 = strip * C::OUT_W;
    // M-phase identity: one column of the strip (replicate-clamped = the box filter's border rule)
    const int gx = min(max(x0 - IT_HALO + tid, 0), w - 1);
    const float sc_x = border_factor(gx, w);
    const bool band_x = border_band(gx, w);
    // H-phase identity: a warp owns one row of the batch, a lane four adjacent outputs
    const int hr = tid >> 5, cg = tid & 31;

    if constexpr (TM) {
        const float z[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int s = 0; s < 9; ++s) tm_st5(tm_base + 5 * s, z);
        tm_wait_st();
    } else {
#pragma unroll
        for (int s = 0; s < 3 * 3 * 5; ++s) ring[s * NT + tid] = 0.f;
    }
    // the 13-row window of row r0+j is: rows j..3 of batch b-3 (its full sum minus its prefix P_{j-1}, kept in the
    // ring) + batches b-2, b-1 + prefix P_j of batch b.  Every partial sum is formed fresh from at most 4 values, so
    // rounding never accumulates down the chunk.
    float B1[5], B2[5], B3[5];   // full sums of batches b-1, b-2, b-3
#pragma unroll
    for (int k = 0; k < 5; ++k) B1[k] = B2[k] = B3[k] = 0.f;
    // batches of 4 rows are aligned to absolute image rows, so the partial sums a window is built from (and hence
    // the result bits) do not depend on where the chunk starts, i.e. on the launch geometry / batch size
    const int r_begin = (((yc0 - IT_HALO + 8) >> 2) << 2) - 8;
    const int n_rows = (yc1 + IT_HALO) - r_begin;
    const int n_batches = (n_rows + IT_RB - 1) / IT_RB;
    int rb = 0;                  // ring slot of batch b (b % 3): overwritten at the end of the batch, read as b-3 first

    // software pipeline: the current row's taps are in registers, the next row's taps and four rows of flow in flight
    auto row_y = [&](int i) { return min(max(r_begin + i, 0), h - 1); };
    Taps cur;
    issue_taps(cur, RP, w, h, gx, row_y(0), ld_stream(fin + row_y(0) * w + gx));
    float2 fq[4];                // flows of rows i+1 .. i+4 (a DRAM round trip ahead of their use)
#pragma unroll
    for (int j = 0; j < 4; ++j) fq[j] = ld_stream(fin + row_y(1 + j) * w + gx);
    __syncthreads();

    for (int b = 0; b < n_batches; ++b) {
        float* vbm = vbuf + (b & 1) * (IT_RB * 5 * NT);
        float* rg = ring + rb * (3 * 5 * NT) + tid;
        float P[5], pold[5];
        // ---- M phase: 4 rows of this thread's column -------------------------------------------------------------
#pragma unroll
        for (int j = 0; j < IT_RB; ++j) {
            const int i = b * IT_RB + j;
            Taps nxt;
            issue_taps(nxt, RP, w, h, gx, row_y(i + 1), fq[j]);
            fq[j] = ld_stream(fin + row_y(i + 5) * w + gx);
            float m[5];
            matrix_from_taps(cur, h, sc_x, band_x, m);
            if constexpr (TM) {
                float xold[5];
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    P[k] = (j == 0) ? m[k] : P[k] + m[k];
                    xold[k] = B3[k];
                    if (j > 0) xold[k] -= pold[k];
                }
                const uint32_t slot = tm_base + (uint32_t)((rb * 3 + j) * 5);
                if (j < IT_RB - 1) tm_ld5(pold, slot);
#pragma unroll
                for (int k = 0; k < 5; ++k) vbm[(j * 5 + k) * NT + tid] = (xold[k] + B2[k]) + (B1[k] + P[k]);
                if (j < IT_RB - 1) {
                    tm_wait_ld();
                    tm_st5(slot, P);
                }
            } else {
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    P[k] = (j == 0) ? m[k] : P[k] + m[k];
                    // rows j..3 of batch b-3 = its full sum minus its prefix P_{j-1}; the slot is then reused for batch b
                    float xold = B3[k];
                    if (j > 0) xold -= pold[k];
                    if (j < IT_RB - 1) {
                        pold[k] = rg[(j * 5 + k) * NT];   // P_j of batch b-3, needed by the next row
                        rg[(j * 5 + k) * NT] = P[k];
                    }
                    vbm[(j * 5 + k) * NT + tid] = (xold + B2[k]) + (B1[k] + P[k]);
                }
            }
            cur = nxt;
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            B3[k] = B2[k];
            B2[k] = B1[k];
            B1[k] = P[k];
        }
        rb = (rb == 2) ? 0 : rb + 1;
        if constexpr (TM) tm_wait_st();
        __syncthreads();
        // ---- H phase: row hr of the batch, outputs 4 cg .. 4 cg + 3 ------------------------------------------------
        const int y = r_begin + b * IT_RB + hr - IT_HALO;
        if (y >= yc0 && y < yc1) {
            float g[5][HK];
            constexpr unsigned FULL = 0xffffffffu;
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float4 q = *reinterpret_cast<const float4*>(vbm + (hr * 5 + k) * NT + HK * cg);
                const float p2 = q.x + q.y, s2 = q.z + q.w;
                const float T = p2 + s2, p3 = p2 + q.z, s3 = q.y + s2;
                const float Tm1 = __shfl_up_sync(FULL, T, 1), Tp1 = __shfl_down_sync(FULL, T, 1);
                const float s2m2 = __shfl_up_sync(FULL, s2, 2), s1m2 = __shfl_up_sync(FULL, q.w, 2);
                const float s3m1 = __shfl_up_sync(FULL, s3, 1), p3p1 = __shfl_down_sync(FULL, p3, 1);
                const float p1p2 = __shfl_down_sync(FULL, q.x, 2), p2p2 = __shfl_down_sync(FULL, p2, 2);
                const float U = Tm1 + T;
                g[k][0] = (s2m2 + U) + p3p1;        // columns 4cg-6 .. 4cg+6
                g[k][1] = (s1m2 + U) + Tp1;         //         4cg-5 .. 4cg+7
                g[k][2] = (U + Tp1) + p1p2;         //         4cg-4 .. 4cg+8
                g[k][3] = (s3m1 + T) + (Tp1 + p2p2);  //       4cg-3 .. 4cg+9
            }
            // OpenCV scales the five sums by 1/169 before the solve; numerator and determinant are both quadratic in
            // them, so the scale folds into the regulariser: 1e-3 * 169^2
            const float reg = 1e-3f * (float)(IT_WIN * IT_WIN) * (float)(IT_WIN * IT_WIN);
            float2 o[HK];
#pragma unroll
            for (int i = 0; i < HK; ++i) {
                const float g11 = g[0][i], g12 = g[1][i], g22 = g[2][i];
                const float h1 = g[3][i], h2 = g[4][i];
                const float idet = 1.f / (diff_of_products(g11, g22, g12, g12) + reg);
                float fx = diff_of_products(g11, h2, g12, h1) * idet;
                float fy = diff_of_products(g22, h1, g12, h2) * idet;
                if (clampv > 0.f) {
                    fx = fminf(fmaxf(fx, -clampv), clampv);
                    fy = fminf(fmaxf(fy, -clampv), clampv);
                }
                o[i] = make_float2(fx, fy);
            }
            const int c0 = HK * cg;                        // region column of o[0]
            const int xg = x0 - IT_HALO + c0;              // image column of o[0]
            float2* dst = fout + (long long)y * w + xg;
#pragma unroll
            for (int i = 0; i < HK; ++i) {
                const int c = c0 + i;
                if (c >= IT_HALO && c < NT - IT_HALO && xg + i < w) dst[i] = o[i];
            }
        }
    }
    if constexpr (TM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid < 32)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tm_base), "n"(C::TM_COLS) : "memory");
    }
}

template <bool TM>
static void launch_scalar_tm(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                             float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, cudaStream_t s) {
    using C = ScalarCfg<TM>;
    cudaFuncSetAttribute(fb_iter_scalar_kernel<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    const int strips = cdiv(w, C::OUT_W);
    int chunks;
    const int chunk_rows = plan_chunk_rows(h, strips, n_pairs, 148LL * 4, &chunks);
    for (int p0 = 0; p0 < n_pairs; p0 += 65535) {
        const int np = min(n_pairs - p0, 65535);
        dim3 g(2 * strips, chunks, np);
        fb_iter_scalar_kernel<TM><<<g, C::NT, C::SMEM_BYTES, s>>>(R + (long long)(2 * p0) * img_stride, img_stride,
                                                                  flow_in + (long long)(2 * p0) * 2 * h * w,
                                                                  out_fwd + p0 * fwd_stride, fwd_stride,
                                                                  out_bwd + p0 * bwd_stride, bwd_stride, h, w, chunk_rows,
                                                                  clamp);
    }
}

void launch_fb_scalar(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                      float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, bool tmem_ring,
                      cudaStream_t s) {
    if (tmem_ring) launch_scalar_tm<true>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s);
    else launch_scalar_tm<false>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s);
}

}  // namespace tf
