// blend_bwd.cu -- per-tile back-to-front gradient pass of the alpha compositing.
//
// Replaces upstream renderCUDA<3> backward (ashawkey variant: colour + depth + alpha gradients) of
// the external rasterizer reached from loss.backward() at train.py:497-498.  Math follows
// SURVEY.md section 8c / oracle/raster_oracle.c (ogs_oracle_blend_backward).
//
// B200 design points (vs upstream's ~10 global float atomics per contributing (pixel, Gaussian)):
//  * the "colour behind" recursion is carried as ONE scalar per pixel: with d_i = <c_i, g> (dot of
//    the Gaussian's channel vector incl. depth and 1 with the pixel's incoming gradients),
//    dL/dalpha = (d_i - S) T, then S <- a_i d_i + (1 - a_i) S -- C-independent state, one register per pixel;
//  * 128 threads per 16x16 tile, warp = 8x8 pixel block, TWO pixels per lane evaluated as a packed
//    pair (FADD2/FMUL2/FFMA2, same staged records and exponent arithmetic as blend_fwd.cu, so the
//    skip decisions are bit-identical); non-contributing pixels are masked arithmetically
//    (alpha = G = 0 leaves T, S and every sum unchanged) so both halves share one instruction stream;
//  * geometry gradients are reduced as the raw moments of u = G dL/dalpha (sum u, u dx, u dy,
//    u dx^2, u dx dy, u dy^2): dL/dmean2D and dL/dconic are linear in them with per-Gaussian
//    factors, which preprocess_bwd applies once per Gaussian instead of once per (pixel, Gaussian);
//  * per (warp, Gaussian) the lanes' sums are combined with a recursive-halving (transpose)
//    reduction over power-of-two chunks of the value vector: V values cost ~V + 5 shuffles;
//  * warp-level culling (ogs_rect_hit_s): lane l tests Gaussian l of a 32-group against the warp's
//    block; only ballot survivors are evaluated;
//  * each warp stores into its own shared-memory rows (a (warp, Gaussian) pair is visited once per
//    batch: plain stores, no read-modify-write); once per batch of 64 Gaussians the 4 warp rows are
//    summed and ONE red.global.add per value per (tile, Gaussian) is issued, skipping zeros;
//  * GEOM=false specialisation (OpenGaussian stages 1-2 detach geometry, train.py:431-436): only
//    w = alpha T and dL/dc are evaluated.
// SUBSETS = true (ogs_raster_backward_subsets): blockIdx.z is a subset; its tile lists start at ranges + z * tiles
// (the partitioned lists of ogs_raster_forward_subsets_state), its final_T / n_contrib and depth / alpha gradients at
// z * H * W, its colour gradients at z * (3 or C) * H * W and its feature gradients at z * (C - 3) * H * W.  The
// subsets are disjoint, so a Gaussian's accumulator row only receives its own subset's contributions.
#include "common.cuh"
#include <stdlib.h>

namespace ogs {

#ifndef BB
#define BB 64            // Gaussians per backward batch
#endif

template <int CUR, int M>
struct HalvingReduce {
    template <int VP>
    __device__ __forceinline__ static void run(float (&v)[VP], int lane) {
        if constexpr (M >= 1) {
            if constexpr (CUR > 1) {
                constexpr int HALF = CUR / 2;
                const bool upper = (lane & M) != 0;
                if constexpr (HALF == 1) {
                    const float send = upper ? v[0] : v[1];
                    const float keep = upper ? v[1] : v[0];
                    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, M);
                } else {
                    // two values per FADD2
#pragma unroll
                    for (int k = 0; k < HALF; k += 2) {
                        const float2 keep = upper ? make_float2(v[k + HALF], v[k + 1 + HALF]) : make_float2(v[k], v[k + 1]);
                        const float2 send = upper ? make_float2(v[k], v[k + 1]) : make_float2(v[k + HALF], v[k + 1 + HALF]);
                        const float2 sum = __fadd2_rn(keep, make_float2(__shfl_xor_sync(0xffffffffu, send.x, M),
                                                                        __shfl_xor_sync(0xffffffffu, send.y, M)));
                        v[k] = sum.x;
                        v[k + 1] = sum.y;
                    }
                }
                HalvingReduce<HALF, M / 2>::run(v, lane);
            } else {
                v[0] += __shfl_xor_sync(0xffffffffu, v[0], M);
                HalvingReduce<1, M / 2>::run(v, lane);
            }
        }
    }
};

constexpr int floor_pow2(int v) { return v >= 16 ? 16 : (v >= 8 ? 8 : (v >= 4 ? 4 : (v >= 2 ? 2 : 1))); }
constexpr int log2c(int v) { return v <= 1 ? 0 : 1 + log2c(v / 2); }

// Sums v[BASE..BASE+N) over the 32 lanes, chunk by chunk (largest power of two first), and stores
// the totals to row[BASE..BASE+N): after a chunk of S values, every lane l holds the total of value
// l / (32/S) (the last log2(32/S) steps are butterflies, and the 32/S lanes of a value add the same
// partial sums in commuted order, so their totals are bit-identical).  They all store it: no predicate
// and no lane test per store.
template <int N, int BASE>
struct ChunkReduceStore {
    template <int VT>
    __device__ __forceinline__ static void run(const float (&v)[VT], int lane, uint32_t row) {   // row: shared address
        if constexpr (N > 0) {
            constexpr int S = floor_pow2(N);
            constexpr int SH = 5 - log2c(S);
            float t[S];
#pragma unroll
            for (int k = 0; k < S; k++) t[k] = v[BASE + k];
            HalvingReduce<S, 16>::run(t, lane);
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(row + 4u * (BASE + (lane >> SH))), "f"(t[0]) : "memory");
            ChunkReduceStore<N - S, BASE + S>::run(v, lane, row);
        }
    }
};

int blend_bwd_stride(int C, int geom) { return geom ? C + 7 : C; }

// PAIRS packed pixel pairs per lane: the warp's block is 8 x (8 * PAIRS) pixels and a 16x16 tile takes
// 4 / PAIRS warps.  More pixels per lane amortise the cross-lane reduction and the per-entry loop
// overhead (about half of the instructions at PAIRS = 1) at the price of coarser culling.
// Register cap: with the recursion state trimmed to one scalar per pixel the 3- and 4-channel kernels fit 80
// registers without spills, which lets 12 CTAs of 64 threads share an SM instead of 10.  Measured on B200 (ncu,
// profiles/r2_kernels_full.csv): warps active 28 -> 33 %, issue active 67 -> 70 %, but 7 % more instructions
// (rematerialisation), so the net is small: 0.517 ms capped vs 0.531 ms uncapped in the same bench run.
// The per-warp survivor records (below) make ptxas take 4-9 more registers where it is not capped.  The instantiations
// that launch_cg picks by default are held to the CTAs per SM they had without the records (register-limited, 64 or
// 128 threads): 12 for the 3- and 4-channel geometry backward, 14 / 16 / 10 / 14 / 12 for the colour backwards, 4 for
// the 12- and 16-channel geometry backward and 5-7 for their colour backwards.  The 6- and 9-channel geometry
// backwards keep 6 CTAs on their own.
constexpr int bwd_min_blocks(int C, int C0, bool geom, int pairs) {
    if (pairs == 2 && C <= 9) {
        if (geom) return C <= 4 ? 12 : 1;
        if (C0 > 0) return C - C0 <= 1 ? 16 : (C - C0 <= 3 ? 14 : 12);
        return C <= 4 ? 14 : 10;
    }
    if (pairs == 1 && C >= 12) {
        if (geom) return 4;
        return C0 > 0 ? (C <= 12 ? 7 : 5) : (C <= 12 ? 6 : 5);
    }
    return 1;   // the other combinations are reached only through OGS_BWD_PAIRS
}

// C0 > 0 (colour-only backward, GEOM = false): channels [0, C0) carry no incoming gradient -- OpenGaussian's Stage 1
// back-propagates through the 6 feature channels only (train.py:441-456), the RGB planes of the fused pass have no
// loss -- so their pixel gradients are not loaded, their weighted sums not formed and not reduced across the lanes
// (6 of 9 values: a third of the FFMA2s and of the reduction of every evaluated entry).  The accumulator rows keep
// their C columns (preprocess_bwd reads them by column); columns [0, C0) stay zero.
template <int C, bool GEOM, int PAIRS, int C0 = 0, bool SUBSETS = false>
__global__ void __launch_bounds__(128 / PAIRS, bwd_min_blocks(C, C0, GEOM, PAIRS)) blend_bwd_kernel(BlendBwdArgs a) {
    static_assert(C0 == 0 || !GEOM, "the geometry gradients need every channel");
    constexpr int BWD_THREADS = 128 / PAIRS, BWD_WARPS = 4 / PAIRS, NPX = 2 * PAIRS;
    constexpr int V = GEOM ? C + 7 : C;
    constexpr int CG = C - C0;            // channels with an incoming gradient
    constexpr int VG = GEOM ? V : CG;     // values reduced per evaluated entry
    constexpr int CH = (C + 1 + 3) & ~3;  // colours + depth, padded to float4
    // everything is double-buffered by batch parity: batch b-1 is staged while batch b is traversed,
    // and batch b is flushed (after the ONE barrier per batch) while the fast warps start on b-1
    extern __shared__ float s_dyn[];      // [2][BWD_WARPS][BB][V] per-warp sums
    __shared__ float4 s_a2[2][BB];
    __shared__ float2 s_b2[2][BB];
    __shared__ __align__(16) float s_ch2[2][BB * CH];
    __shared__ uint32_t s_id3[3][BB];     // ids live until the batch's flush, i.e. while batch b-2 is already being staged: 3 slots
    // per warp, the current group's surviving entries back to front, two float4 each: the staged sa and {sb, list
    // position, shared addresses of the entry's accumulator row and channels}.  The entry loop walks consecutive
    // records instead of locating each set bit of the ballot and re-deriving the addresses from it.
    __shared__ float4 s_hit[BWD_WARPS][32 * 2];
    __shared__ int s_max_last;

    const int gx = (a.W + 15) / 16;
    const int tile = blockIdx.y * gx + blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bxi = blockIdx.x * 16 + (warp & 1) * 8, byi = blockIdx.y * 16 + (warp >> 1) * 8 * PAIRS;
    const int px = bxi + (lane & 7);
    const float pxf = (float)px;
    const float bx0 = (float)bxi, by0 = (float)byi;
    const size_t HW = (size_t)a.H * a.W;
    const size_t z = SUBSETS ? blockIdx.z : 0;                       // 0 folds every offset below away
    const size_t zc = SUBSETS ? z * (a.dL_dfeat ? 3 : C) * HW : 0;  // colour planes per subset: 3 with dL_dfeat, else C
    const uint2 range = a.ranges[tile + z * gx * gridDim.y];

    // per-lane state of the pixel pairs (.x: row y + 8 p, .y: row y + 8 p + 4)
    float2 T2[PAIRS], S2[PAIRS], gd2[PAIRS], ga2[PAIRS], tfbg2[PAIRS], npy[PAIRS];
    float2 g2[PAIRS][CG];
    int last[NPX];
#pragma unroll
    for (int p = 0; p < PAIRS; p++) {
        float Tf[2], gdv[2] = {0.f, 0.f}, gav[2] = {0.f, 0.f}, bgd[2] = {0.f, 0.f};
        float gv[2][CG];
        const int y0 = byi + (lane >> 3) + 8 * p;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int py = y0 + 4 * k;
            const bool inside = px < a.W && py < a.H;
            const size_t pix = (size_t)py * a.W + px;
            last[2 * p + k] = inside ? (int)a.n_contrib[z * HW + pix] : 0;
            Tf[k] = inside ? a.final_T[z * HW + pix] : 0.f;
#pragma unroll
            for (int cc = 0; cc < CG; cc++) {
                const int c = C0 + cc;
                const float* plane = (a.dL_dfeat && c >= 3) ? a.dL_dfeat + (z * (C - 3) + (size_t)(c - 3)) * HW
                                                            : (a.dL_dcolor ? a.dL_dcolor + zc + (size_t)c * HW : nullptr);
                gv[k][cc] = (inside && plane) ? __ldg(plane + pix) : 0.f;
                if constexpr (GEOM) bgd[k] = fmaf(__ldg(a.bg + c), gv[k][cc], bgd[k]);
            }
            if constexpr (GEOM) {
                gdv[k] = (inside && a.dL_ddepth) ? __ldg(a.dL_ddepth + z * HW + pix) : 0.f;
                gav[k] = (inside && a.dL_dalpha) ? __ldg(a.dL_dalpha + z * HW + pix) : 0.f;
            }
        }
        npy[p] = make_float2(-(float)y0, -(float)(y0 + 4));
        T2[p] = make_float2(Tf[0], Tf[1]);
        S2[p] = s2(0.f);
#pragma unroll
        for (int c = 0; c < CG; c++) g2[p][c] = make_float2(gv[0][c], gv[1][c]);
        gd2[p] = make_float2(gdv[0], gdv[1]);
        ga2[p] = make_float2(gav[0], gav[1]);
        tfbg2[p] = make_float2(Tf[0] * bgd[0], Tf[1] * bgd[1]);
    }

    // block / warp maxima of the last contributor
    if (threadIdx.x == 0) s_max_last = 0;
    for (int e = threadIdx.x; e < 2 * BWD_WARPS * BB * V; e += BWD_THREADS) s_dyn[e] = 0.f;
    __syncthreads();
    int wmax = 0;
#pragma unroll
    for (int k = 0; k < NPX; k++) wmax = max(wmax, last[k]);
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, m));
    if (lane == 0 && wmax > 0) atomicMax(&s_max_last, wmax);
    __syncthreads();
    const int max_last = s_max_last;
    if (max_last == 0) return;
    // ---- stage one batch (pre-scaled records, colours + depth) into buffer `sb` ----
    auto stage = [&](int b, int sb) {
        const int start = b * BB;
        const int n = min(BB, max_last - start);
        for (int t = threadIdx.x; t < n; t += BWD_THREADS) {
            const uint32_t gid = a.point_list[range.x + start + t];
            s_id3[b % 3][t] = gid;
            const float4 r1 = __ldg(a.rec1 + gid);
            ogs_stage(__ldg(a.rec0 + gid), r1, s_a2[sb][t], s_b2[sb][t]);
            if constexpr (GEOM) s_ch2[sb][t * CH + C] = r1.z;
        }
        if constexpr (GEOM) {          // the channel values enter dL/dalpha only; the colour-only backward never reads them
            for (int e = threadIdx.x; e < n * C; e += BWD_THREADS) {
                const int j = e / C, c = e - j * C;
                const uint32_t gid = a.point_list[range.x + start + j];
                s_ch2[sb][j * CH + c] = (c < 3) ? __ldg(a.base + 3 * (size_t)gid + c) : __ldg(a.extra + (size_t)(C - 3) * gid + (c - 3));
            }
        }
    };
    const int b_first = (max_last - 1) / BB;
    stage(b_first, b_first & 1);
    __syncthreads();

    for (int b = b_first; b >= 0; b--) {
        const int start = b * BB;
        const int n = min(BB, max_last - start);
        const int sb = b & 1;
        if (b > 0) stage(b - 1, sb ^ 1);     // its loads are in flight while this batch is traversed
        const float4* s_a = s_a2[sb];
        const float2* s_b = s_b2[sb];
        const float* s_ch = s_ch2[sb];
        float* acc_b = s_dyn + (size_t)sb * BWD_WARPS * BB * V;
        float* my_acc = acc_b + (size_t)warp * BB * V;
        // ---- traverse back to front ----
        if (start < wmax) {
            const int nw = min(n, wmax - start);
            for (int grp = ((nw - 1) >> 5) << 5; grp >= 0; grp -= 32) {
                const int idx = grp + lane;
                bool hit = false;
                if (idx < nw) hit = ogs_rect_hit_s(s_a[idx], s_b[idx], bx0, by0, bx0 + 7.0f, by0 + (float)(8 * PAIRS - 1));
                const unsigned mask = __ballot_sync(0xffffffffu, hit);
                float4* hits = s_hit[warp];
                if (hit) {   // (re-read: keeping the record live across the test costs spills at the 80-register cap)
                    float4* h = hits + 2 * __popc(mask & ~((2u << lane) - 1u));   // rank among the later survivors
                    const float2 rb = s_b[idx];
                    // shared addresses of the accumulator row (4-byte aligned, < 2^18) and of the channels (16-byte
                    // aligned), packed into one word: the loop loads and stores through them with no base to rebuild
                    const uint32_t row = (uint32_t)__cvta_generic_to_shared(my_acc + idx * V + C0);
                    const uint32_t chs = GEOM ? (uint32_t)__cvta_generic_to_shared(s_ch + idx * CH) : 0u;   // unread without GEOM: s_ch2 stays unallocated
                    h[0] = s_a[idx];
                    h[1] = make_float4(rb.x, rb.y, __int_as_float(start + idx), __uint_as_float((row >> 2) | ((chs >> 4) << 16)));
                }
                __syncwarp();
                const float4* const hend = hits + 2 * __popc(mask);
                for (const float4* h = hits; h != hend; h += 2) {
                    const float4 ra = h[0];
                    const float4 rb = h[1];
                    const int pos = __float_as_int(rb.z);
                    const float dx = ra.x - pxf;
                    const float adx = __fmul_rn(__fmul_rn(ra.z, dx), dx), bdx = __fmul_rn(ra.w, dx);
                    float2 dy[PAIRS], G[PAIRS], al[PAIRS];
                    bool ok[NPX];
                    bool any = false;
#pragma unroll
                    for (int p = 0; p < PAIRS; p++) {
                        const float2 pw = ogs_pair_power(adx, bdx, rb.x, ra.y, npy[p], dy[p]);
                        G[p] = make_float2(ogs_ex2(pw.x), ogs_ex2(pw.y));
                        al[p] = __fmul2_rn(s2(rb.y), G[p]);
                        al[p].x = fminf(0.99f, al[p].x);
                        al[p].y = fminf(0.99f, al[p].y);
                        ok[2 * p] = pos < last[2 * p] && pw.x <= 0.0f && al[p].x >= (1.0f / 255.0f);
                        ok[2 * p + 1] = pos < last[2 * p + 1] && pw.y <= 0.0f && al[p].y >= (1.0f / 255.0f);
                        any = any || ok[2 * p] || ok[2 * p + 1];
                    }
                    if (!__any_sync(0xffffffffu, any)) continue;
                    float chv[CH];
                    if constexpr (GEOM) {
#pragma unroll
                        for (int q = 0; q < CH / 4; q++) {
                            // s_ch2[sb] is written by stage() before the __syncthreads that precedes this traversal;
                            // the "memory" clobber keeps the load behind that barrier if the staging ever moves
                            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                         : "=f"(chv[4 * q]), "=f"(chv[4 * q + 1]), "=f"(chv[4 * q + 2]), "=f"(chv[4 * q + 3])
                                         : "r"(((__float_as_uint(rb.w) >> 16) << 4) + 16u * q) : "memory");
                        }
                    }
                    // packed sums over the lane's pairs; .x + .y is taken once at the end
                    float2 vc[CG], vd = s2(0.f), su2 = s2(0.f), suy2 = s2(0.f), suyy2 = s2(0.f);
#pragma unroll
                    for (int c = 0; c < CG; c++) vc[c] = s2(0.f);
#pragma unroll
                    for (int p = 0; p < PAIRS; p++) {
                        const float2 alm = make_float2(ok[2 * p] ? al[p].x : 0.f, ok[2 * p + 1] ? al[p].y : 0.f);
                        const float2 om = __fadd2_rn(s2(1.0f), make_float2(-alm.x, -alm.y));
                        const float2 inv = make_float2(ogs_rcp(om.x), ogs_rcp(om.y));
                        T2[p] = __fmul2_rn(T2[p], inv);
                        const float2 w = __fmul2_rn(alm, T2[p]);
#pragma unroll
                        for (int c = 0; c < CG; c++) vc[c] = __ffma2_rn(w, g2[p][c], vc[c]);
                        if constexpr (GEOM) {
                            float2 dot = __ffma2_rn(s2(chv[0]), g2[p][0], ga2[p]);
#pragma unroll
                            for (int c = 1; c < C; c++) dot = __ffma2_rn(s2(chv[c]), g2[p][c], dot);
                            dot = __ffma2_rn(s2(chv[C]), gd2[p], dot);
                            const float2 dS = __fadd2_rn(dot, make_float2(-S2[p].x, -S2[p].y));
                            // S <- a d + (1 - a) S, applied as soon as this entry's dS is taken (a masked entry has
                            // a = 0: S unchanged), so no per-pixel state other than S crosses entries
                            S2[p] = __ffma2_rn(om, S2[p], __fmul2_rn(alm, dot));
                            const float2 dLda = __ffma2_rn(make_float2(-tfbg2[p].x, -tfbg2[p].y), inv, __fmul2_rn(dS, T2[p]));
                            const float2 Gm = make_float2(ok[2 * p] ? G[p].x : 0.f, ok[2 * p + 1] ? G[p].y : 0.f);
                            const float2 u = __fmul2_rn(Gm, dLda);
                            const float2 uy = __fmul2_rn(u, dy[p]);
                            su2 = __fadd2_rn(su2, u);
                            suy2 = __fadd2_rn(suy2, uy);
                            suyy2 = __ffma2_rn(uy, dy[p], suyy2);
                            vd = __ffma2_rn(w, gd2[p], vd);
                        }
                    }
                    float v[VG];
#pragma unroll
                    for (int c = 0; c < CG; c++) v[c] = vc[c].x + vc[c].y;
                    if constexpr (GEOM) {
                        const float su = su2.x + su2.y, suy = suy2.x + suy2.y;
                        const float sux = su * dx;
                        v[C + 0] = vd.x + vd.y;
                        v[C + 1] = su;
                        v[C + 2] = sux;
                        v[C + 3] = suy;
                        v[C + 4] = sux * dx;
                        v[C + 5] = suy * dx;
                        v[C + 6] = suyy2.x + suyy2.y;
                    }
                    ChunkReduceStore<VG, 0>::run(v, lane, (__float_as_uint(rb.w) & 0xffffu) << 2);
                }
                __syncwarp();   // the records are read before the next group overwrites them
            }
        }
        __syncthreads();   // batch b fully traversed by every warp; batch b-1 fully staged
        // ---- flush: sum the warp rows, one red per value per (tile, Gaussian) ----
        for (int e0 = threadIdx.x; e0 < n * VG; e0 += BWD_THREADS) {
            const int j = e0 / VG, k = C0 + (e0 - j * VG);
            const int e = j * V + k;
            float sum = 0.f;
#pragma unroll
            for (int w8 = 0; w8 < BWD_WARPS; w8++) {
                sum += acc_b[(size_t)w8 * BB * V + e];
                acc_b[(size_t)w8 * BB * V + e] = 0.f;
            }
            if (sum != 0.f) atomicAdd(a.acc + (size_t)s_id3[b % 3][j] * a.stride + k, sum);
        }
    }
}

template <int C, bool GEOM, int C0, bool SUBSETS>
static int launch_cg(const BlendBwdArgs& a, int S, cudaStream_t s) {
    constexpr int V = GEOM ? C + 7 : C;
    // two pairs per lane pay off while the pixel state fits the register file comfortably (measured: C <= 9)
    static const int env_pairs = getenv("OGS_BWD_PAIRS") ? atoi(getenv("OGS_BWD_PAIRS")) : 0;  // tuning knob
    const int pairs = env_pairs ? env_pairs : (C <= 9 ? 2 : 1);
    dim3 grid((a.W + 15) / 16, (a.H + 15) / 16, S);
    const size_t smem = (size_t)2 * (4 / (pairs == 2 ? 2 : 1)) * BB * V * sizeof(float);
    static PerDeviceOnce attr_done[2];
    if (smem > 24 * 1024 && attr_done[pairs == 2].todo()) {   // static + dynamic shared memory may pass the 48 KB default
        if (pairs == 2) OGS_CUDA(cudaFuncSetAttribute(blend_bwd_kernel<C, GEOM, 2, C0, SUBSETS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        else OGS_CUDA(cudaFuncSetAttribute(blend_bwd_kernel<C, GEOM, 1, C0, SUBSETS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr_done[pairs == 2].done();
    }
    if (pairs == 2) blend_bwd_kernel<C, GEOM, 2, C0, SUBSETS><<<grid, 64, smem, s>>>(a);
    else blend_bwd_kernel<C, GEOM, 1, C0, SUBSETS><<<grid, 128, smem, s>>>(a);
    return 0;
}

template <int C, bool SUBSETS>
static int launch_c(const BlendBwdArgs& a, int S, cudaStream_t s) {
    if (a.geom) return launch_cg<C, true, 0, SUBSETS>(a, S, s);
    if constexpr (C > 3) {
        if (!a.dL_dcolor && a.dL_dfeat) return launch_cg<C, false, 3, SUBSETS>(a, S, s);   // only the feature channels carry a gradient
    }
    return launch_cg<C, false, 0, SUBSETS>(a, S, s);
}

template <bool SUBSETS>
static int launch_any(const BlendBwdArgs& a, int S, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(a.acc, 0, (size_t)a.P * a.stride * sizeof(float), s);
    if (e != cudaSuccess) return cuda_fail(e, "memset acc");
    switch (a.C) {
        case 3: return launch_c<3, SUBSETS>(a, S, s);
        case 4: return launch_c<4, SUBSETS>(a, S, s);
        case 6: return launch_c<6, SUBSETS>(a, S, s);
        case 9: return launch_c<9, SUBSETS>(a, S, s);
        case 12: return launch_c<12, SUBSETS>(a, S, s);
        case 16: return launch_c<16, SUBSETS>(a, S, s);
    }
    set_error("blend backward: unsupported channel count %d", a.C);
    return -4;
}

int launch_blend_backward(const BlendBwdArgs& a, cudaStream_t s) { return launch_any<false>(a, 1, s); }

int launch_blend_backward_subsets(const BlendBwdArgs& a, int S, cudaStream_t s) { return launch_any<true>(a, S, s); }

}  // namespace ogs
