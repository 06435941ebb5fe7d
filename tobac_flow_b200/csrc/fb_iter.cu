// K4+K5: one fused Farneback iteration = FarnebackUpdateMatrices + FarnebackUpdateFlow_Blur (box window).
//
// OpenCV's sweep is a pure Jacobi update (the matrices it refreshes behind the sliding window are never re-read in the
// same sweep), so flow buffers ping-pong and M is never materialised in HBM.
//
// Strip-marching design (the shape of OpenCV's own sliding window, mapped to a CTA):
//   * a CTA of 128 threads owns a strip of 128 columns (116 outputs + a 6-column halo on each side) and marches down a
//     chunk of rows; there is no row halo re-read apart from a 12-row warm-up per chunk;
//   * M phase, one thread per column: flow (8 B), R0 (float4 + float) and the bilinear R1 gather at p + flow
//     (4 x (float4 + float)) -> the five normal-equation terms.  Rows are handled in batches of 4; the vertical 13-row
//     window sum is assembled from fresh partial sums (prefix sums of batch b-3 kept in a ring and subtracted from its
//     full sum, the full sums of batches b-3..b-1 in registers, the running prefix of batch b), so rounding never
//     accumulates down the chunk (OpenCV uses fp64 running sums; plain fp32 running sums drifted visibly);
//   * H phase, every 4 rows: the vertical sums of 4 rows are exchanged through shared memory; a warp owns a row, a lane 4
//     adjacent outputs: it reads only its own quad of vertical sums and builds the four 13-column windows from prefix /
//     suffix / full quad sums of its neighbouring lanes (eight shuffles per channel), solves the 2x2 systems in registers
//     and stores the new flow;
//   * forward and backward CTAs of the same pair and strip are adjacent in launch order, so the second reader of the
//     shared R planes hits L2;
//   * work distribution: a grid of (strip, row chunk, pair) CTAs, the chunk count chosen to minimise waves x rows.
// Algorithmic HBM bytes per pixel-iteration: flow 8 + R0 20 + R1 20 read, flow 8 written = 56 B.
//
// This file holds the default kernel (v3).  What it adds to that structure, and why (measurements in profiles/README.md:
// the plain LDG / shared-memory form, fb_iter_scalar.cu, stalls 40 % of its warp time on long-scoreboard waits although
// the memory system delivers the same access pattern at the copy bandwidth when the arithmetic is stripped):
//   * the address-regular streams of a strip -- R0 (float4 + float) and the flow, 28 of the 48 bytes a pixel reads --
//     are staged a batch (4 rows) ahead into shared memory by bulk async copies (cp.async.bulk -> UBLKCP, TMA engine,
//     one mbarrier per ring slot).  They no longer occupy LSU issue slots, L1 miss-queue entries, scoreboards or
//     destination registers, and their lookahead is a whole batch instead of one row;
//   * the prefix-sum ring of the vertical window lives in tensor memory (tcgen05.ld / .st, 32x32b shape: a TMEM column is
//     one private word per thread), which takes its traffic off the L1 data pipe and frees the shared memory the staging
//     ring needs at 4 CTAs per SM;
//   * the R1 bilinear gather stays on the L1-cached LDG path (its addresses depend on the flow), two rows ahead: a row's
//     tap registers are re-loaded for the row after next as soon as they are blended;
//   * packed fp32 (FFMA2 / FADD2 / FMUL2: one issue slot for two IEEE fp32 operations) for the blend and for the five
//     terms, which travel as A = (M0, M2) -> (g11, g22), B = (M3, M4) -> (h1, h2), C = M1 -> g12 through prefix sums,
//     vertical window, shared memory and the H phase's horizontal window: the same IEEE operations in the same order as the
//     scalar kernel, so the window sums are bit-identical to its;
//   * one MUFU.RCP (<= 1 ulp) for the reciprocal of the regularised, always normal determinant.
#include <stdlib.h>

#include "fb_iter_common.cuh"

namespace tf {

// ---- async-copy / mbarrier plumbing -------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

struct TsCfg {
    static constexpr int NT = 128, HK = 4, OUT_W = NT - 2 * IT_HALO, SLOTS = 2;
    static constexpr int A_ROW = NT * 16;                    // R0 float4 plane: bytes per staged row
    static constexpr int B_ROW = (NT + 4) * 4;               // R0 c4 plane (+ up to 3 floats of alignment skew)
    static constexpr int F_ROW = (NT + 2) * 8;               // flow (+ 1 float2 of alignment skew)
    static constexpr int A_OFF = 0, B_OFF = IT_RB * A_ROW, F_OFF = B_OFF + IT_RB * B_ROW;
    static constexpr int SLOT_BYTES = F_OFF + IT_RB * F_ROW;
    static constexpr int VBUF_FLOATS = 8 * 5 * NT;
    static constexpr int VBUF_OFF = SLOTS * SLOT_BYTES;
    static constexpr int MBAR_OFF = VBUF_OFF + VBUF_FLOATS * 4;
    static constexpr int SMEM_BYTES = MBAR_OFF + SLOTS * 8;
    static constexpr int TM_COLS = 64;
    static_assert(A_ROW % 16 == 0 && B_ROW % 16 == 0 && F_ROW % 16 == 0 && SLOT_BYTES % 16 == 0, "bulk copies: 16-byte granules");
};


// ---- packed fp32 ------------------------------------------------------------------------------------------------------
#ifndef TF_RCP_EXACT
#define TF_RCP_EXACT 0
#endif
typedef float2 f2;
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 dup2(float a) { return make_float2(a, a); }
__device__ __forceinline__ f2 lo2(float4 v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ f2 hi2(float4 v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ f2 shfl_up2(f2 v, int d) {
    return make_float2(__shfl_up_sync(0xffffffffu, v.x, d), __shfl_up_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ f2 shfl_down2(f2 v, int d) {
    return make_float2(__shfl_down_sync(0xffffffffu, v.x, d), __shfl_down_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ float rcp_fast(float x) {
#if TF_RCP_EXACT
    return 1.f / x;
#else
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}

__device__ __forceinline__ void tm_ld_abc(f2& a, f2& b, float& c, uint32_t addr) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y) : "r"(addr) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=f"(c) : "r"(addr + 4) : "memory");
}
__device__ __forceinline__ void tm_st_abc(uint32_t addr, f2 a, f2 b, float c) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(addr), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y) : "memory");
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(addr + 4), "f"(c) : "memory");
}


struct TapsV3 {
    float4 p00, p01, p10, p11;
    float q00, q01, q10, q11;
    float fx, fy;
    bool inside;
};

__device__ __forceinline__ void issue_taps_v3(TapsV3& t, const float4* __restrict__ R1a, const float* __restrict__ R1b,
                                              int w, int h, int x, int y, float2 f) {
    const float px = __fadd_rn((float)x, f.x), py = __fadd_rn((float)y, f.y);
    const float flx = floorf(px), fly = floorf(py);
    const int x1 = (int)flx, y1 = (int)fly;
    t.fx = __fsub_rn(px, flx);
    t.fy = __fsub_rn(py, fly);
    t.inside = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
    // the taps of a position outside the image are never used: predicated loads instead of clamped addresses
    if (t.inside) {
        const float4* a0 = R1a + (y1 * w + x1);
        const float4* a1 = a0 + w;
        const float* b0 = R1b + (y1 * w + x1);
        const float* b1 = b0 + w;
        t.p00 = __ldg(a0);
        t.p01 = __ldg(a0 + 1);
        t.p10 = __ldg(a1);
        t.p11 = __ldg(a1 + 1);
        t.q00 = __ldg(b0);
        t.q01 = __ldg(b0 + 1);
        t.q10 = __ldg(b1);
        t.q11 = __ldg(b1 + 1);
    }
}

// FarnebackUpdateMatrices for one pixel: (A, B, C) = ((M0, M2), (M3, M4), M1); c / c4 = R0 at the pixel, f = its flow.
// The (c0, c1) and (c2, c3) halves of every float4 tap are blended with packed FMAs: per lane exactly the chain of
// blend4() (fb_iter_common.cuh), so the terms carry the same bits as the scalar kernel's.
__device__ __forceinline__ void matrix_v3(const TapsV3& t, float4 c, float c4, float2 f, int y, int h, float sc_x,
                                          bool band_x, f2& mA, f2& mB, float& mC) {
    f2 r23, r45;
    float r6;
    const f2 half2 = make_float2(0.5f, 0.5f), minus1 = make_float2(-1.f, -1.f);
    if (t.inside) {
        float a00, a01, a10, a11;
        bilinear_weights(t.fx, t.fy, a00, a01, a10, a11);
        const f2 w00 = dup2(a00), w01 = dup2(a01), w10 = dup2(a10), w11 = dup2(a11);
        r23 = fma2(w11, lo2(t.p11), fma2(w10, lo2(t.p10), fma2(w01, lo2(t.p01), mul2(w00, lo2(t.p00)))));
        r45 = fma2(w11, hi2(t.p11), fma2(w10, hi2(t.p10), fma2(w01, hi2(t.p01), mul2(w00, hi2(t.p00)))));
        r6 = blend4(a00, a01, a10, a11, t.q00, t.q01, t.q10, t.q11);
        r45 = mul2(add2(hi2(c), r45), half2);
        r6 = __fmul_rn(__fadd_rn(c4, r6), 0.25f);
    } else {
        r23 = make_float2(0.f, 0.f);
        r45 = hi2(c);
        r6 = __fmul_rn(c4, 0.5f);
    }
    r23 = mul2(fma2(r23, minus1, lo2(c)), half2);                // (c - r) * 0.5: the FMA with -1 is the exact subtraction
    float m[5];
    terms_from_blend(r23.x, r23.y, r45.x, r45.y, r6, f.x, f.y, border_scale(sc_x, band_x, y, h), m);
    mA = make_float2(m[0], m[2]);
    mC = m[1];
    mB = make_float2(m[3], m[4]);
}

// WAL = 2: w % 4 == 0 -- every row of the 4-byte / 8-byte streams then starts at the same offset from a 16-byte
// boundary, so the alignment skews of the staged rows are constants of the strip (hoisted) and the outputs can go out as
// 16-byte stores.  WAL = 1: w even -- the same for the 8-byte streams (flow in, flow out) only.  WAL = 0: any w.
// UP = 1: the level's first iteration -- the initial flow is not read from flow_in but up-sampled from the previous level's
// result (UpArgs) into the staging ring's flow rows by the CTA itself, a batch ahead like the bulk copies it replaces.
template <int PF, int WAL, int UP>
__global__ void __launch_bounds__(TsCfg::NT, 4)
fb_iter_v3_kernel(const float* __restrict__ R, long long img_stride, const float* __restrict__ flow_in,
                  float* __restrict__ out_fwd, long long fwd_stride, float* __restrict__ out_bwd, long long bwd_stride,
                  int h, int w, int chunk_rows, float clampv, UpArgs up) {
    using C = TsCfg;
    constexpr int NT = C::NT, HK = C::HK, ROWF = 5 * NT;         // a row of vertical sums: [A: NT x f2][B: NT x f2][C: NT]
    static_assert(PF == 1 || PF == 2, "rows of R1 taps in flight");
    extern __shared__ __align__(128) unsigned char ts_smem[];
    float* vbuf = reinterpret_cast<float*>(ts_smem + C::VBUF_OFF);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(ts_smem + C::MBAR_OFF);
    __shared__ uint32_t tm_addr_s;
    const int tid = threadIdx.x;
    const int dir = blockIdx.x & 1, strip = blockIdx.x >> 1, pair = blockIdx.z;
    const int yc0 = blockIdx.y * chunk_rows, yc1 = min(yc0 + chunk_rows, h);
    const int plane = h * w;
    const float* Rp = R + (long long)(2 * pair) * img_stride;
    const float* Rn = Rp + img_stride;
    const float* R0 = dir ? Rn : Rp;
    const float* R1 = dir ? Rp : Rn;
    const float4* R0a = reinterpret_cast<const float4*>(R0);
    const float* R0b = R0 + 4 * (long long)plane;
    const float4* R1a = reinterpret_cast<const float4*>(R1);
    const float* R1b = R1 + 4 * (long long)plane;
    const float2* fin = reinterpret_cast<const float2*>(flow_in) + (UP ? 0LL : (long long)(2 * pair + dir) * plane);
    const float2* coarse = reinterpret_cast<const float2*>(up.coarse) + (UP ? (long long)(2 * pair + dir) * up.sh * up.sw : 0LL);
    float2* fout = reinterpret_cast<float2*>(dir ? out_bwd + (long long)pair * bwd_stride
                                                 : out_fwd + (long long)pair * fwd_stride);
    const int x0 = strip * C::OUT_W;
    const int xs = x0 - IT_HALO;
    const int cx0 = max(xs, 0), cx1 = min(xs + NT, w), ncol = cx1 - cx0;
    const int gx = min(max(xs + tid, 0), w - 1);
    const int gxs = gx - cx0;
    const float sc_x = border_factor(gx, w);
    const bool band_x = border_band(gx, w);
    const int hr = tid >> 5, cg = tid & 31;
    const unsigned skb0 = (unsigned)(reinterpret_cast<uintptr_t>(R0b) >> 2), skf0 = (unsigned)(reinterpret_cast<uintptr_t>(fin) >> 3);

    if (tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tm_addr_s)), "n"(C::TM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        if (tid == 0) {
            mbar_init(&mbar[0], 1);
            mbar_init(&mbar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tm_base = tm_addr_s + ((uint32_t)(tid >> 5) << 21);
    const f2 zero2 = make_float2(0.f, 0.f), minus1 = make_float2(-1.f, -1.f);
#pragma unroll
    for (int s = 0; s < 9; ++s) tm_st_abc(tm_base + 5 * s, zero2, zero2, 0.f);
    tm_wait_st();
    f2 B1a = zero2, B1b = zero2, B2a = zero2, B2b = zero2, B3a = zero2, B3b = zero2;
    float B1c = 0.f, B2c = 0.f, B3c = 0.f;
    const int r_begin = (((yc0 - IT_HALO + 8) >> 2) << 2) - 8;
    const int n_rows = (yc1 + IT_HALO) - r_begin;
    const int n_batches = (n_rows + IT_RB - 1) / IT_RB;
    int rb = 0;
    auto row_y = [&](int i) { return min(max(r_begin + i, 0), h - 1); };

    // Staging of batch bb (rows 4bb .. 4bb+3, replicate-clamped) into ring slot bb & 1: warp r copies row r, its lanes
    // 0..2 one stream each (cp.async.bulk takes warp-uniform operands, so the copies of a warp issue one after the other:
    // three per warp keeps the four warps level at the batch barrier -- one warp issuing all twelve left 17 % of all warp
    // samples waiting there).  Byte counts are constants of the strip -- the 4-byte / 8-byte streams start at the 16-byte
    // boundary below their first element and always move the padded row -- so thread 0 arms the barrier with a constant.
    const int swarp = tid >> 5, slane = tid & 31;
    const uint32_t bytes_a = (uint32_t)ncol * 16u, bytes_b = (((uint32_t)ncol + 6u) & ~3u) * 4u,
                   bytes_f = (((uint32_t)ncol + 2u) & ~1u) * 8u;
    const uint32_t stage_tx = IT_RB * (bytes_a + bytes_b + (UP ? 0u : bytes_f));
    const char* st_base = slane == 0 ? reinterpret_cast<const char*>(R0a)
                        : (slane == 1 ? reinterpret_cast<const char*>(R0b) : reinterpret_cast<const char*>(fin));
    const int st_esz = slane == 0 ? 16 : (slane == 1 ? 4 : 8);
    const uint32_t st_bytes = slane == 0 ? bytes_a : (slane == 1 ? bytes_b : bytes_f);
    const uint32_t st_dst = smem_u32(ts_smem) + (slane == 0 ? C::A_OFF + swarp * C::A_ROW + (cx0 - xs) * 16
                                                 : (slane == 1 ? C::B_OFF + swarp * C::B_ROW : C::F_OFF + swarp * C::F_ROW));
    auto stage_batch = [&](int bb) {
        const uint32_t bar = smem_u32(&mbar[bb & 1]);
        if (slane < (UP ? 2 : 3)) {
            const int y = row_y(IT_RB * bb + swarp);
            const uintptr_t src = (reinterpret_cast<uintptr_t>(st_base) + (long long)(y * w + cx0) * st_esz) & ~(uintptr_t)15;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st_dst + (uint32_t)(bb & 1) * C::SLOT_BYTES), "l"(src), "r"(st_bytes), "r"(bar) : "memory");
        }
        if (tid == 0) mbar_arrive_expect_tx(&mbar[bb & 1], stage_tx);
    };
    const unsigned skb_c = (skb0 + (unsigned)cx0) & 3u, skf_c = (skf0 + (unsigned)cx0) & 1u;   // WA: the skews of every row
    // UP: the four flow rows of batch bb, up-sampled from the coarse field, written by every thread for its own column
    // (no alignment skew); called where the bulk copies of that batch are issued
    auto upsample_batch = [&](int bb) {
        const int x0 = __ldg(up.x0 + gx), x1 = min(x0 + 1, up.sw - 1);
        const float fx = __ldg(up.fx + gx), gxw = __fsub_rn(1.f, fx);
        float2* dst = reinterpret_cast<float2*>(ts_smem + (bb & 1) * C::SLOT_BYTES + C::F_OFF) + gxs;
        int y0_prev = -1;
        float2 top = make_float2(0.f, 0.f), bot = top;           // the two source rows blended along x
#pragma unroll
        for (int j = 0; j < IT_RB; ++j) {
            const int y = row_y(IT_RB * bb + j);
            const int y0 = __ldg(up.y0 + y);
            const float fy = __ldg(up.fy + y);
            if (y0 != y0_prev) {                                 // (uniform: neighbouring rows often share their source rows)
                const float2* r0 = coarse + y0 * up.sw;
                const float2* r1 = coarse + min(y0 + 1, up.sh - 1) * up.sw;
                const float2 a = __ldg(r0 + x0), b = __ldg(r0 + x1), c = __ldg(r1 + x0), d = __ldg(r1 + x1);
                top = make_float2(fmaf(b.x, fx, __fmul_rn(a.x, gxw)), fmaf(b.y, fx, __fmul_rn(a.y, gxw)));
                bot = make_float2(fmaf(d.x, fx, __fmul_rn(c.x, gxw)), fmaf(d.y, fx, __fmul_rn(c.y, gxw)));
                y0_prev = y0;
            }
            const float gyw = __fsub_rn(1.f, fy);
            dst[j * (C::F_ROW / 8)] = make_float2(__fmul_rn(fmaf(bot.x, fy, __fmul_rn(top.x, gyw)), up.mul),
                                                  __fmul_rn(fmaf(bot.y, fy, __fmul_rn(top.y, gyw)), up.mul));
        }
    };
    auto staged_flow = [&](int bb, int j) {
        unsigned sk = UP ? 0u : skf_c;
        if (WAL == 0 && !UP) sk = (skf0 + (unsigned)(row_y(IT_RB * bb + j) * w + cx0)) & 1u;
        return reinterpret_cast<const float2*>(ts_smem + (bb & 1) * C::SLOT_BYTES + C::F_OFF + j * C::F_ROW)[sk + gxs];
    };

    stage_batch(0);
    if (n_batches > 1) stage_batch(1);
    if (UP) {
        upsample_batch(0);
        if (n_batches > 1) upsample_batch(1);
        __syncthreads();
    }
    mbar_wait(&mbar[0], 0u);
    TapsV3 S0, S1;
    issue_taps_v3(S0, R1a, R1b, w, h, gx, row_y(0), staged_flow(0, 0));
    if (PF == 2) issue_taps_v3(S1, R1a, R1b, w, h, gx, row_y(1), staged_flow(0, 1));

    for (int b = 0; b < n_batches; ++b) {
        float* vbm = vbuf + (b & 1) * (IT_RB * ROWF);
        const unsigned char* slot = ts_smem + (b & 1) * C::SLOT_BYTES;
        f2 Pa, Pb, olda, oldb;
        float Pc, oldc;
#pragma unroll
        for (int j = 0; j < IT_RB; ++j) {
            const int i = b * IT_RB + j;
            const int y_cur = row_y(i);
            // R0 and the flow of this row from the staging ring
            const float4 c = reinterpret_cast<const float4*>(slot + C::A_OFF + j * C::A_ROW)[gx - xs];
            unsigned skb = skb_c, skf = UP ? 0u : skf_c;
            if (WAL < 2) {
                const unsigned e_cur = (unsigned)(y_cur * w + cx0);
                skb = (skb0 + e_cur) & 3u;
                if (WAL == 0 && !UP) skf = (skf0 + e_cur) & 1u;
            }
            const float c4 = reinterpret_cast<const float*>(slot + C::B_OFF + j * C::B_ROW)[skb + gxs];
            const float2 fcur = reinterpret_cast<const float2*>(slot + C::F_OFF + j * C::F_ROW)[skf + gxs];
            // the flow of row i + PF (from row 4 - PF on it lives in the next batch's slot, staged a batch ago)
            const int jn = j + PF;
            const int bn = b + (jn >= IT_RB ? 1 : 0);
            if (jn == IT_RB && bn < n_batches) mbar_wait(&mbar[bn & 1], (uint32_t)((bn >> 1) & 1));
            float2 fnext = make_float2(0.f, 0.f);
            if (bn < n_batches) fnext = staged_flow(bn, jn & (IT_RB - 1));
            f2 mA, mB;
            float mC;
            if (PF == 1) {
                issue_taps_v3(S1, R1a, R1b, w, h, gx, row_y(i + 1), fnext);
                matrix_v3(S0, c, c4, fcur, y_cur, h, sc_x, band_x, mA, mB, mC);
            } else {
                TapsV3& st = (j & 1) ? S1 : S0;
                matrix_v3(st, c, c4, fcur, y_cur, h, sc_x, band_x, mA, mB, mC);
                issue_taps_v3(st, R1a, R1b, w, h, gx, row_y(i + 2), fnext);
            }
            if (j == 0) { Pa = mA; Pb = mB; Pc = mC; }
            else { Pa = add2(Pa, mA); Pb = add2(Pb, mB); Pc = Pc + mC; }
            f2 xa = B3a, xb = B3b;
            float xc = B3c;
            if (j > 0) { xa = fma2(olda, minus1, xa); xb = fma2(oldb, minus1, xb); xc -= oldc; }
            const uint32_t tslot = tm_base + (uint32_t)((rb * 3 + j) * 5);
            if (j < IT_RB - 1) tm_ld_abc(olda, oldb, oldc, tslot);
            float* vr = vbm + j * ROWF;
            reinterpret_cast<f2*>(vr)[tid] = add2(add2(xa, B2a), add2(B1a, Pa));
            reinterpret_cast<f2*>(vr + 2 * NT)[tid] = add2(add2(xb, B2b), add2(B1b, Pb));
            vr[4 * NT + tid] = (xc + B2c) + (B1c + Pc);
            if (j < IT_RB - 1) {
                tm_wait_ld();
                tm_st_abc(tslot, Pa, Pb, Pc);
            }
            if (PF == 1) S0 = S1;
        }
        B3a = B2a; B3b = B2b; B3c = B2c;
        B2a = B1a; B2b = B1b; B2c = B1c;
        B1a = Pa; B1b = Pb; B1c = Pc;
        rb = (rb == 2) ? 0 : rb + 1;
        tm_wait_st();
        __syncthreads();
        if (b + 2 < n_batches) {
            stage_batch(b + 2);
            if (UP) upsample_batch(b + 2);     // (visible to its readers through the barriers of batches b + 1 / b + 2)
        }
        // ---- H phase: a warp owns row hr of the batch, a lane four adjacent outputs ---------------------------------
        const int y = r_begin + b * IT_RB + hr - IT_HALO;
        if (y >= yc0 && y < yc1) {
            const float* vr = vbm + hr * ROWF;
            f2 gA[HK], gB[HK];
            float gC[HK];
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) {
                const float4* src = reinterpret_cast<const float4*>(vr + pr * 2 * NT) + 2 * cg;
                const float4 u = src[0], v = src[1];
                const f2 q0 = lo2(u), q1 = hi2(u), q2 = lo2(v), q3 = hi2(v);
                const f2 p2 = add2(q0, q1), s2 = add2(q2, q3);
                const f2 T = add2(p2, s2), p3 = add2(p2, q2), s3 = add2(q1, s2);
                const f2 Tm1 = shfl_up2(T, 1), Tp1 = shfl_down2(T, 1);
                const f2 s2m2 = shfl_up2(s2, 2), s1m2 = shfl_up2(q3, 2);
                const f2 s3m1 = shfl_up2(s3, 1), p3p1 = shfl_down2(p3, 1);
                const f2 p1p2 = shfl_down2(q0, 2), p2p2 = shfl_down2(p2, 2);
                const f2 U = add2(Tm1, T);
                f2* g = pr ? gB : gA;
                g[0] = add2(add2(s2m2, U), p3p1);
                g[1] = add2(add2(s1m2, U), Tp1);
                g[2] = add2(add2(U, Tp1), p1p2);
                g[3] = add2(add2(s3m1, T), add2(Tp1, p2p2));
            }
            {
                constexpr unsigned FULL = 0xffffffffu;
                const float4 q = reinterpret_cast<const float4*>(vr + 4 * NT)[cg];
                const float p2 = q.x + q.y, s2 = q.z + q.w;
                const float T = p2 + s2, p3 = p2 + q.z, s3 = q.y + s2;
                const float Tm1 = __shfl_up_sync(FULL, T, 1), Tp1 = __shfl_down_sync(FULL, T, 1);
                const float s2m2 = __shfl_up_sync(FULL, s2, 2), s1m2 = __shfl_up_sync(FULL, q.w, 2);
                const float s3m1 = __shfl_up_sync(FULL, s3, 1), p3p1 = __shfl_down_sync(FULL, p3, 1);
                const float p1p2 = __shfl_down_sync(FULL, q.x, 2), p2p2 = __shfl_down_sync(FULL, p2, 2);
                const float U = Tm1 + T;
                gC[0] = (s2m2 + U) + p3p1;
                gC[1] = (s1m2 + U) + Tp1;
                gC[2] = (U + Tp1) + p1p2;
                gC[3] = (s3m1 + T) + (Tp1 + p2p2);
            }
            const float reg = 1e-3f * (float)(IT_WIN * IT_WIN) * (float)(IT_WIN * IT_WIN);
            float2 o[HK];
#pragma unroll
            for (int i = 0; i < HK; ++i) {
                const float g11 = gA[i].x, g22 = gA[i].y, g12 = gC[i];
                const float h1 = gB[i].x, h2 = gB[i].y;
                const float idet = rcp_fast(diff_of_products(g11, g22, g12, g12) + reg);
                float fx = diff_of_products(g11, h2, g12, h1) * idet;
                float fy = diff_of_products(g22, h1, g12, h2) * idet;
                if (clampv > 0.f) {
                    fx = fminf(fmaxf(fx, -clampv), clampv);
                    fy = fminf(fmaxf(fy, -clampv), clampv);
                }
                o[i] = make_float2(fx, fy);
            }
            const int c0 = HK * cg;
            const int xg = xs + c0;
            float2* dst = fout + (long long)y * w + xg;
            if (WAL >= 1 && (reinterpret_cast<uintptr_t>(fout) & 15) == 0) {
                // xg and w are even: the output pairs (0, 1) and (2, 3) are 16-byte aligned and valid / invalid together
#pragma unroll
                for (int i = 0; i < HK; i += 2) {
                    const int cc = c0 + i;
                    if (cc >= IT_HALO && cc < NT - IT_HALO && xg + i < w)
                        *reinterpret_cast<float4*>(dst + i) = make_float4(o[i].x, o[i].y, o[i + 1].x, o[i + 1].y);
                }
            } else {
#pragma unroll
                for (int i = 0; i < HK; ++i) {
                    const int cc = c0 + i;
                    if (cc >= IT_HALO && cc < NT - IT_HALO && xg + i < w) dst[i] = o[i];
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tm_addr_s), "n"(C::TM_COLS) : "memory");
}

template <int PF, int UP>
static void launch_v3_pf(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                         float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, cudaStream_t s,
                         const UpArgs* upp) {
    using C = TsCfg;
    auto kern = (w & 3) == 0 ? fb_iter_v3_kernel<PF, 2, UP> : ((w & 1) == 0 ? fb_iter_v3_kernel<PF, 1, UP> : fb_iter_v3_kernel<PF, 0, UP>);
    UpArgs up{};
    if (upp) up = *upp;
    // (the attribute is per device: set it on every call, it is cheap)
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    const int strips = cdiv(w, C::OUT_W);
    int chunks;
    const int chunk_rows = plan_chunk_rows(h, strips, n_pairs, 148LL * 4, &chunks);
    for (int p0 = 0; p0 < n_pairs; p0 += 65535) {
        const int np = min(n_pairs - p0, 65535);
        dim3 g(2 * strips, chunks, np);
        UpArgs upz = up;
        if (UP) upz.coarse = up.coarse + (long long)(2 * p0) * 2 * up.sh * up.sw;
        kern<<<g, C::NT, C::SMEM_BYTES, s>>>(R + (long long)(2 * p0) * img_stride, img_stride,
                                             UP ? nullptr : flow_in + (long long)(2 * p0) * 2 * h * w, out_fwd + p0 * fwd_stride,
                                             fwd_stride, out_bwd + p0 * bwd_stride, bwd_stride, h, w, chunk_rows, clamp, upz);
    }
}

void launch_fb_v3(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                  float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, float clamp, int pf, cudaStream_t s,
                  const UpArgs* up) {
    if (up) {
        if (pf == 1) launch_v3_pf<1, 1>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s, up);
        else launch_v3_pf<2, 1>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s, up);
        return;
    }
    if (pf == 1) launch_v3_pf<1, 0>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s, nullptr);
    else launch_v3_pf<2, 0>(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, s, nullptr);
}

// which iteration kernel runs: 3 = v3 with two rows of taps in flight (default), 4 = v3 with one, 5 = 3 with the flow
// up-sampling in its own kernel instead of the first iteration, 0 = the scalar kernel with its ring in shared memory,
// 1 = the scalar kernel with the ring in tensor memory.  TF_TMA in the environment sets
// the initial choice; tf_fb_select_kernel changes it (A/B runs, cross-check tests).
static int g_kernel_choice = -1;

static int kernel_choice() {
    if (g_kernel_choice < 0) {
        const char* e = getenv("TF_TMA");
        g_kernel_choice = e ? atoi(e) : 3;
    }
    return g_kernel_choice;
}

// the fused up-sampling exists in the default (v3) kernels only; TF_UPSAMPLE_FUSED=0 keeps the separate kernel (A/B)
bool fb_iteration_can_fuse_upsample() {
    static const char* e = getenv("TF_UPSAMPLE_FUSED");
    if (e && atoi(e) == 0) return false;
    const int k = kernel_choice();
    return k != 0 && k != 1 && k != 5;
}

int launch_fb_iteration(const float* R, long long img_stride, const float* flow_in, float* out_fwd, long long fwd_stride,
                        float* out_bwd, long long bwd_stride, int n_pairs, int h, int w, int win, float clamp,
                        bool full_res, cudaStream_t s, const UpArgs* up) {
    if (win != IT_WIN) {
        set_error("fb iteration: only winSize 13 is built (got %d)", win);
        return TF_ERR_UNSUPPORTED;
    }
    if ((long long)h * w > 0x3fffffffLL) { set_error("fb iteration: level too large"); return TF_ERR_INVALID_ARGUMENT; }
    // algorithmic bytes: 56 B per pixel-iteration; a first iteration that also up-samples its initial flow carries the
    // bytes the separate up-sampling kernel accounts for (coarse field read, up-sampled field written: SURVEY 8d's 20 S term)
    double bytes = 56.0 * h * w * 2 * n_pairs;
    if (up) bytes += (8.0 * h * w + 8.0 * up->sh * up->sw) * 2 * n_pairs;
    LaunchTimer lt(full_res ? KC_FB_ITER_L0 : KC_FB_ITER, bytes, s, cdiv(n_pairs, 65535));
    const int choice = kernel_choice();
    if (up && (choice == 0 || choice == 1)) { set_error("fb iteration: the scalar kernels have no fused up-sampling"); return TF_ERR_UNSUPPORTED; }
    switch (choice) {
        case 0: launch_fb_scalar(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, false, s); break;
        case 1: launch_fb_scalar(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, true, s); break;
        case 4: launch_fb_v3(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, 1, s, up); break;
        default: launch_fb_v3(R, img_stride, flow_in, out_fwd, fwd_stride, out_bwd, bwd_stride, n_pairs, h, w, clamp, 2, s, up);
    }
    return check_launch("fb iteration");
}

}  // namespace tf

extern "C" int tf_fb_select_kernel(int which) {
    if (which != 0 && which != 1 && which != 3 && which != 4 && which != 5) {
        tf::set_error("tf_fb_select_kernel: unknown kernel %d (0, 1: scalar; 3, 4: v3; 5: v3 with the separate up-sampling kernel)", which);
        return TF_ERR_INVALID_ARGUMENT;
    }
    tf::g_kernel_choice = which;
    return TF_OK;
}
