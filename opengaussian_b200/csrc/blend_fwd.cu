// blend_fwd.cu -- per-tile front-to-back alpha compositing of C = 3 + n_extra channels plus depth
// and alpha in ONE pass.
//
// Replaces upstream renderCUDA<3> forward (ashawkey variant with depth/alpha outputs) that
// gaussian_renderer/__init__.py:104-112 calls, and -- through the extra channels -- the three
// additional passes of gaussian_renderer/__init__.py:129-163 (ins_feat[:, :3], ins_feat[:, 3:6],
// silhouette).  Semantics follow SURVEY.md section 8c / oracle/raster_oracle.c:
// power > 0 skip; alpha = min(0.99, o * exp(power)); alpha < 1/255 skip; T' = T (1 - alpha);
// T' < 1e-4 stops BEFORE applying; colour = sum c alpha T + T_final bg; depth = sum z alpha T;
// alpha_out = 1 - T_final.
//
// Layout: one CTA per 16x16 tile (the tile size is part of the bit-exact binning contract).  A warp
// owns an 8 x (8*PAIRS) pixel block and every lane 2*PAIRS pixels (rows y, y+4, ...).  The pixels
// of a lane are processed as PACKED PAIRS with Blackwell's two-wide FP32 instructions
// (fma.rn.f32x2 / mul.f32x2 / add.f32x2 -> FFMA2/FMUL2/FADD2): the kernel is FP32-issue bound
// (SURVEY.md section 8d) and a scalar FFMA occupies the issue slot as long as an FFMA2 that does
// two.  Contributions are masked arithmetically (w = 0) instead of branched, so both halves of a
// pair always run the same instruction stream; a finished pixel is encoded in the SIGN of its
// transmittance (T <= 0: done, |T| = final T), which makes every later test fail by itself.
// Gaussians are staged 256 per round in shared memory as pre-scaled records (common.cuh:
// ogs_stage -- the exponent comes out in the log2 domain, one MUFU.EX2 per pixel) followed by
// their C colours + depth; per group of 32 staged Gaussians lane l tests Gaussian l against the
// warp's block (ogs_rect_hit_s) and only the ballot survivors are blended.
// SUBSETS = true (ogs_raster_forward_subsets): blockIdx.z is a subset; its tile lists start at
// ranges + z * tiles and its images at z * C * H * W (colour) and z * H * W (depth, alpha; depth may be
// NULL).  final_T / n_contrib (ogs_raster_forward_subsets_state) go to z * H * W + pixel when set, n_contrib
// counted inside the slot's own tile segment; NULL (ogs_raster_forward_subsets) writes no state.
#include "common.cuh"
#include <stdlib.h>

namespace ogs {

#define BATCH 256

template <int C, int PAIRS, bool SUBSETS>
__global__ void __launch_bounds__(128 / PAIRS) blend_fwd_kernel(BlendFwdArgs a) {
    constexpr int THREADS = 128 / PAIRS;      // 4 / PAIRS warps
    constexpr int NPX = 2 * PAIRS;            // pixels per lane
    constexpr int CH = (C + 1 + 3) & ~3;      // colours + depth, padded to float4
    __shared__ float4 s_a[BATCH];
    __shared__ float2 s_b[BATCH];
    __shared__ __align__(16) float s_ch[BATCH * CH];

    const int gx = (a.W + 15) / 16;
    const int tile = blockIdx.y * gx + blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bxi = blockIdx.x * 16 + (warp & 1) * 8, byi = blockIdx.y * 16 + (warp >> 1) * 8 * PAIRS;
    const int px = bxi + (lane & 7);
    const float pxf = (float)px;
    const float bx0 = (float)bxi, by0 = (float)byi;

    const uint2* ranges = a.ranges;
    if constexpr (SUBSETS) ranges += (size_t)blockIdx.z * gx * gridDim.y;
    const uint2 range = ranges[tile];
    int todo = (int)(range.y - range.x);
    const int rounds = (todo + BATCH - 1) / BATCH;

    uint32_t last[NPX];
    float2 npy[PAIRS], T2[PAIRS], acc[PAIRS][C + 1];
#pragma unroll
    for (int p = 0; p < PAIRS; p++) {
        const int ya = byi + (lane >> 3) + 8 * p, yb = ya + 4;
        npy[p] = make_float2(-(float)ya, -(float)yb);
        last[2 * p] = last[2 * p + 1] = 0;
        T2[p] = make_float2((px < a.W && ya < a.H) ? 1.0f : -1.0f, (px < a.W && yb < a.H) ? 1.0f : -1.0f);
#pragma unroll
        for (int c = 0; c <= C; c++) acc[p][c] = s2(0.0f);
    }
    auto all_done = [&]() {
        bool d = true;
#pragma unroll
        for (int p = 0; p < PAIRS; p++) d = d && !(T2[p].x > 0.0f) && !(T2[p].y > 0.0f);
        return d;
    };

    for (int r = 0; r < rounds; r++, todo -= BATCH) {
        if (__syncthreads_count(all_done()) == THREADS) break;
#pragma unroll
        for (int h = 0; h < BATCH / THREADS; h++) {
            const int slot = threadIdx.x + h * THREADS;
            const int idx = r * BATCH + slot;
            if (range.x + idx < range.y) {
                const uint32_t g = a.point_list[range.x + idx];
                const float4 r1 = __ldg(a.rec1 + g);
                ogs_stage(__ldg(a.rec0 + g), r1, s_a[slot], s_b[slot]);
                float* ch = s_ch + slot * CH;
#pragma unroll
                for (int c = 0; c < 3; c++) ch[c] = __ldg(a.base + 3 * (size_t)g + c);
#pragma unroll
                for (int c = 3; c < C; c++) ch[c] = __ldg(a.extra + (size_t)(C - 3) * g + (c - 3));
                ch[C] = r1.z;
            }
        }
        __syncthreads();
        const int n = todo < BATCH ? todo : BATCH;
        if (!__all_sync(0xffffffffu, all_done())) {
            for (int grp = 0; grp < n; grp += 32) {
                const int idx = grp + lane;
                bool hit = false;
                if (idx < n) hit = ogs_rect_hit_s(s_a[idx], s_b[idx], bx0, by0, bx0 + 7.0f, by0 + (float)(8 * PAIRS - 1));
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                while (mask) {
                    const int j = grp + __ffs(mask) - 1;
                    mask &= mask - 1;
                    const float4 ra = s_a[j];
                    const float2 rb = s_b[j];
                    float chv[CH];
#pragma unroll
                    for (int q = 0; q < CH / 4; q++) {
                        const float4 t = reinterpret_cast<const float4*>(s_ch + j * CH)[q];
                        chv[4 * q] = t.x; chv[4 * q + 1] = t.y; chv[4 * q + 2] = t.z; chv[4 * q + 3] = t.w;
                    }
                    const float dx = ra.x - pxf;
                    const float adx = __fmul_rn(__fmul_rn(ra.z, dx), dx), bdx = __fmul_rn(ra.w, dx);
                    const uint32_t pos = (uint32_t)(r * BATCH + j + 1);
#pragma unroll
                    for (int p = 0; p < PAIRS; p++) {
                        float2 dy;
                        const float2 pw = ogs_pair_power(adx, bdx, rb.x, ra.y, npy[p], dy);
                        float2 al = __fmul2_rn(s2(rb.y), make_float2(ogs_ex2(pw.x), ogs_ex2(pw.y)));
                        al.x = fminf(0.99f, al.x);
                        al.y = fminf(0.99f, al.y);
                        const bool oka = pw.x <= 0.0f && al.x >= (1.0f / 255.0f);
                        const bool okb = pw.y <= 0.0f && al.y >= (1.0f / 255.0f);
                        // a skipped entry gets alpha 0, so tT = T exactly and the one floor test below also covers it
                        const float2 alm = make_float2(oka ? al.x : 0.0f, okb ? al.y : 0.0f);
                        const float2 T = T2[p];
                        const float2 tT = __fmul2_rn(T, __fadd2_rn(s2(1.0f), make_float2(-alm.x, -alm.y)));
                        const float2 w = __fmul2_rn(alm, T);
                        // live: the pixel stays above the transmittance floor (false once T <= 0); a live skipped entry
                        // adds w = 0 and keeps T, a valid alpha that reaches the floor stops the pixel without being
                        // applied (T <- -|T|, which leaves a finished pixel's T as it is)
                        const bool lva = tT.x >= 0.0001f, lvb = tT.y >= 0.0001f;
                        const float2 wm = make_float2(lva ? w.x : 0.0f, lvb ? w.y : 0.0f);
#pragma unroll
                        for (int c = 0; c <= C; c++) acc[p][c] = __ffma2_rn(s2(chv[c]), wm, acc[p][c]);
                        T2[p] = make_float2(lva ? tT.x : -fabsf(T.x), lvb ? tT.y : -fabsf(T.y));
                        last[2 * p] = (oka && lva) ? pos : last[2 * p];
                        last[2 * p + 1] = (okb && lvb) ? pos : last[2 * p + 1];
                    }
                }
                if (__all_sync(0xffffffffu, all_done())) break;
            }
        }
    }
    const size_t HW = (size_t)a.H * a.W;
#pragma unroll
    for (int k = 0; k < NPX; k++) {
        const int p = k >> 1;
        const int py = byi + (lane >> 3) + 8 * p + 4 * (k & 1);
        if (px < a.W && py < a.H) {
            const size_t pix = (size_t)py * a.W + px;
            const float T = fabsf((k & 1) ? T2[p].y : T2[p].x);
            if constexpr (SUBSETS) {
                const size_t z = blockIdx.z;
#pragma unroll
                for (int c = 0; c < C; c++)
                    a.out_color[(z * C + c) * HW + pix] = ((k & 1) ? acc[p][c].y : acc[p][c].x) + T * __ldg(a.bg + c);
                if (a.out_depth) a.out_depth[z * HW + pix] = (k & 1) ? acc[p][C].y : acc[p][C].x;
                a.out_alpha[z * HW + pix] = 1.0f - T;
                if (a.final_T) {
                    a.final_T[z * HW + pix] = T;
                    a.n_contrib[z * HW + pix] = last[k];
                }
            } else {
                a.final_T[pix] = T;
                a.n_contrib[pix] = last[k];
#pragma unroll
                for (int c = 0; c < C; c++)
                    a.out_color[c * HW + pix] = ((k & 1) ? acc[p][c].y : acc[p][c].x) + T * __ldg(a.bg + c);
                a.out_depth[pix] = (k & 1) ? acc[p][C].y : acc[p][C].x;
                a.out_alpha[pix] = 1.0f - T;
            }
        }
    }
}

template <int C>
static int launch_c(const BlendFwdArgs& a, cudaStream_t s) {
    dim3 grid((a.W + 15) / 16, (a.H + 15) / 16);
    static const int pairs = getenv("OGS_FWD_PAIRS") ? atoi(getenv("OGS_FWD_PAIRS")) : OGS_FWD_PAIRS;  // tuning knob
    if (pairs == 2) blend_fwd_kernel<C, 2, false><<<grid, 64, 0, s>>>(a);
    else blend_fwd_kernel<C, 1, false><<<grid, 128, 0, s>>>(a);
    return 0;
}

template <int C>
static int launch_subsets_c(const BlendFwdArgs& a, int S, cudaStream_t s) {
    blend_fwd_kernel<C, OGS_FWD_PAIRS, true><<<dim3((a.W + 15) / 16, (a.H + 15) / 16, S), 128 / OGS_FWD_PAIRS, 0, s>>>(a);
    return 0;
}

int launch_blend_forward(const BlendFwdArgs& a, cudaStream_t s) {
    switch (a.C) {
        case 3: return launch_c<3>(a, s);
        case 4: return launch_c<4>(a, s);
        case 6: return launch_c<6>(a, s);
        case 9: return launch_c<9>(a, s);
        case 12: return launch_c<12>(a, s);
        case 16: return launch_c<16>(a, s);
    }
    set_error("blend forward: unsupported channel count %d (supported: 3,4,6,9,12,16)", a.C);
    return -4;
}

int launch_blend_forward_subsets(const BlendFwdArgs& a, int S, cudaStream_t s) {
    switch (a.C) {
        case 3: return launch_subsets_c<3>(a, S, s);
        case 4: return launch_subsets_c<4>(a, S, s);
        case 6: return launch_subsets_c<6>(a, S, s);
        case 9: return launch_subsets_c<9>(a, S, s);
        case 12: return launch_subsets_c<12>(a, S, s);
        case 16: return launch_subsets_c<16>(a, S, s);
    }
    set_error("blend forward: unsupported channel count %d (supported: 3,4,6,9,12,16)", a.C);
    return -4;
}

}  // namespace ogs
