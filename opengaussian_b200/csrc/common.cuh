// common.cuh -- shared declarations of libogs_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/ogs_b200.h"

#ifndef OGS_FWD_PAIRS
#define OGS_FWD_PAIRS 1            // packed pixel pairs per lane in blend_fwd (1: 8x8 px per warp, 2: 8x16)
#endif
#define OGS_NUM_SMS 148

namespace ogs {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);   // records + returns (int)e

#define OGS_CUDA(call)                                                \
    do {                                                              \
        cudaError_t _e = (call);                                      \
        if (_e != cudaSuccess) return ogs::cuda_fail(_e, #call);      \
    } while (0)

#define OGS_KERNEL_CHECK(name, dbg, stream)                           \
    do {                                                              \
        cudaError_t _e = cudaGetLastError();                          \
        if (_e == cudaSuccess && (dbg)) _e = cudaStreamSynchronize(stream); \
        if (_e != cudaSuccess) return ogs::cuda_fail(_e, name);       \
    } while (0)

// Function attributes (cudaFuncSetAttribute) belong to a device: "already done" flags are kept per device so that
// one process driving several GPUs (or several host threads) sets them on each.  Racing threads may both set the
// attribute; that is harmless.
#define OGS_MAX_DEVICES 64
inline int current_device() {
    int d = 0;
    cudaGetDevice(&d);
    return d & (OGS_MAX_DEVICES - 1);
}
struct PerDeviceOnce {
    std::atomic<uint64_t> mask{0};
    bool todo() const { return !((mask.load(std::memory_order_relaxed) >> current_device()) & 1ull); }
    void done() { mask.fetch_or(1ull << current_device(), std::memory_order_relaxed); }
};

// Frees stream-ordered scratch on every exit path of a launcher.
struct AsyncScratch {
    void* p = nullptr;
    cudaStream_t s = nullptr;
    explicit AsyncScratch(cudaStream_t s_) : s(s_) {}
    AsyncScratch(const AsyncScratch&) = delete;
    AsyncScratch& operator=(const AsyncScratch&) = delete;
    cudaError_t alloc(size_t bytes) { release(); return cudaMallocAsync(&p, bytes, s); }
    void release() { if (p) { cudaFreeAsync(p, s); p = nullptr; } }
    ~AsyncScratch() { release(); }
};

// ---- optional per-family device timing (CUDA events on the launching stream) ----
enum ProfFamily { PF_PREPROCESS_FWD = 0, PF_DEPTH_SORT_SCAN, PF_EMIT, PF_TILE_SORT, PF_RANGES, PF_BLEND_FWD,
                  PF_BLEND_BWD, PF_PREPROCESS_BWD, PF_KMEANS_ASSIGN, PF_MASK_STATS, PF_ADAM, PF_FOOTPRINT, PF_COUNT };
void prof_begin(int family, cudaStream_t s);
void prof_end(int family, cudaStream_t s);
struct ProfScope {
    int f; cudaStream_t s;
    ProfScope(int family, cudaStream_t st) : f(family), s(st) { prof_begin(f, s); }
    ~ProfScope() { prof_end(f, s); }
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- geometry state layout (one caller-owned block, see ogs_raster_state::geom) ----
struct GeomLayout {
    size_t rec0, rec1, rgb, clamped, tiles, feat, total;
    __host__ static GeomLayout make(int P, bool has_sh, int n_feat_act = 0) {
        GeomLayout g;
        size_t o = 0;
        size_t n = (size_t)(P > 0 ? P : 1);
        g.rec0 = o; o = align_up(o + n * 16, 256);
        g.rec1 = o; o = align_up(o + n * 16, 256);
        g.rgb = o; if (has_sh) o = align_up(o + n * 12, 256);
        g.clamped = o; if (has_sh) o = align_up(o + n, 256);
        g.tiles = o; o = align_up(o + n * 4, 256);
        g.feat = o; if (n_feat_act > 0) o = align_up(o + n * 4 * (size_t)n_feat_act, 256);   // activated extra channels
        g.total = o;
        return g;
    }
};

struct GeomPtrs {
    float4* rec0;      // x, y, conic.a, conic.b
    float4* rec1;      // conic.c, opacity, depth, radius (int bits)
    float* rgb;        // [P,3] SH colours (only with shs)
    uint8_t* clamped;  // bit c set: channel c was clamped at 0
    uint32_t* tiles;   // tiles_touched
    float* feat;       // [P,n_extra] activated extra channels (raw-parameter mode only)
    __host__ static GeomPtrs from(void* base, const GeomLayout& l) {
        char* b = (char*)base;
        GeomPtrs p;
        p.rec0 = (float4*)(b + l.rec0);
        p.rec1 = (float4*)(b + l.rec1);
        p.rgb = (float*)(b + l.rgb);
        p.clamped = (uint8_t*)(b + l.clamped);
        p.tiles = (uint32_t*)(b + l.tiles);
        p.feat = (float*)(b + l.feat);
        return p;
    }
};

struct BinLayout {
    size_t point_list, ranges, total;
    __host__ static BinLayout make(int64_t N, int tiles) {
        BinLayout b;
        size_t o = 0;   // ranges first: their offset must not depend on the (speculative) capacity
        b.ranges = o; o = align_up(o + (size_t)tiles * 8, 256);
        b.point_list = o; o = align_up(o + (size_t)(N > 0 ? N : 1) * 4, 256);
        b.total = o;
        return b;
    }
};

struct ImgLayout {
    size_t final_T, n_contrib, total;
    __host__ static ImgLayout make(int W, int H) {
        ImgLayout l;
        size_t o = 0, n = (size_t)W * H;
        l.final_T = o; o = align_up(o + n * 4, 256);
        l.n_contrib = o; o = align_up(o + n * 4, 256);
        l.total = o;
        return l;
    }
};

// Exact e / d for the staging loops (e < 2^16, d < 2^10): one multiply-high instead of the ~20-instruction runtime
// division.  floor(e * ceil(2^32 / d) / 2^32) == floor(e / d) while e * d < 2^32.
struct SmallDiv {
    uint32_t inv;
    __device__ __forceinline__ explicit SmallDiv(int d) : inv(0xFFFFFFFFu / (uint32_t)d + 1u) {}
    __device__ __forceinline__ int operator()(int e) const { return (int)__umulhi((uint32_t)e, inv); }
};

// ---- kernels launchers (defined in the per-family .cu files) ----
struct PreprocessArgs {
    int P, D, M, W, H;
    int act_flags, n_extra;         // raw-parameter mode (OGS_ACT_*), extra channel count
    const float *shs_rest, *extra;  // split SH (see ogs_raster_inputs), raw extra channels
    const float *means3D, *scales, *rotations, *cov3D_precomp, *opacities, *shs;
    float scale_modifier, tanfovx, tanfovy;
    const float *view, *proj, *campos;
    int32_t* radii;
    GeomPtrs g;
    uint32_t* depth_keys;   // [P] depth bits, 0xFFFFFFFF when culled
    uint32_t* depth_vals;   // [P] identity
};
int launch_preprocess_forward(const PreprocessArgs& a, cudaStream_t s);
int launch_feat_refresh(int P, int n_extra, const float4* rec1, const float* extra, float* feat, cudaStream_t s);
int launch_mark_visible(int P, const float* means3D, const float* view, uint8_t* present, cudaStream_t s);

// binning (binning.cu)
struct BinScratch {
    uint32_t *dkeys_in, *dvals_in, *dkeys_out, *dvals_out;  // [P]
    uint32_t* offsets;                                      // [P + 2]: inclusive scan in depth order over the visible
                                                            // slots, then N and the overflow flag
    const uint32_t* nvis_ptr;                               // device count of visible Gaussians (= sorted slots in use)
    void* cub_temp; size_t cub_temp_bytes;
};
size_t binning_temp_bytes(int P, int64_t N_cap);
int depth_sort_and_scan(int P, const GeomPtrs& g, BinScratch& sc, cudaStream_t s, int debug);
int emit_sort_ranges(int P, int W, int H, const uint32_t* n_ptr, int64_t cap, const GeomPtrs& g, BinScratch& sc,
                     uint16_t* tkeys_a, uint32_t* tvals_a, uint16_t* tkeys_b,
                     uint32_t* point_list, uint2* ranges, cudaStream_t s, int debug);
size_t tile_sort_temp_bytes(int64_t N);
size_t depth_sort_temp_bytes(int P);

// blend (blend_fwd.cu / blend_bwd.cu)
struct BlendFwdArgs {
    int W, H, C;                // C = 3 + n_extra
    const uint2* ranges; const uint32_t* point_list;
    const float4 *rec0, *rec1;
    const float* base;          // [P,3] rgb (SH) or colors_precomp
    const float* extra;         // [P,C-3] or NULL
    const float* bg;            // [C]
    float *out_color, *out_depth, *out_alpha, *final_T; uint32_t* n_contrib;
};
int launch_blend_forward(const BlendFwdArgs& a, cudaStream_t s);

struct BlendBwdArgs {
    int P, W, H, C;
    const uint2* ranges; const uint32_t* point_list;
    const float4 *rec0, *rec1;
    const float* base; const float* extra; const float* bg;
    const float* final_T; const uint32_t* n_contrib;
    const float *dL_dcolor, *dL_ddepth, *dL_dalpha;
    const float* dL_dfeat;      // NULL: dL_dcolor holds all C planes; else dL_dcolor = 3 planes (or NULL = 0), this = C - 3 planes
    int geom;                   // 1: all gradients, 0: colour/feature gradients only
    float* acc;                 // [P][stride] accumulators (zeroed by the launcher)
    int stride;                 // floats per Gaussian in acc
};
// acc layout per Gaussian: [0..C) dL_dcolors, then (geom) C+0 dL_ddepth and the raw moments of
// u = G dL/dalpha over the contributing pixels (d = mean2D - pixel):
// C+1 sum u (= dL_dopacity), C+2 sum u dx, C+3 sum u dy, C+4 sum u dx^2, C+5 sum u dx dy, C+6 sum u dy^2.
// preprocess_bwd turns them into dL_dmean2D / dL_dconic (linear in the moments, per-Gaussian factors).
int blend_bwd_stride(int C, int geom);
int launch_blend_backward(const BlendBwdArgs& a, cudaStream_t s);

struct PreprocessBwdArgs {
    int P, D, M, C, W, H;
    int act_flags;
    int accumulate;                 // bit 0: parameter gradients are ADDED to (invisible Gaussians skipped); bit 1: dL_dmeans2D too
    const float *shs_rest, *extra, *opacities;
    float* dL_dshs_rest;
    const float *means3D, *scales, *rotations, *cov3D_precomp, *shs;
    float scale_modifier, tanfovx, tanfovy;
    const float *view, *proj, *campos;
    GeomPtrs g;
    const float* acc; int stride; int geom;
    float *dL_dmeans3D, *dL_dmeans2D, *dL_dopacities, *dL_dshs, *dL_dcolors_precomp, *dL_dscales,
        *dL_drotations, *dL_dcov3D, *dL_dextra;
};
int launch_preprocess_backward(const PreprocessBwdArgs& a, cudaStream_t s);

#ifdef __CUDACC__
// ---- blend kernels: staged (pre-scaled) Gaussian records and packed two-pixel arithmetic ----
// The blend kernels stage each list entry in shared memory with the conic pre-multiplied so that
// the exponent comes out directly in the log2 domain (one MUFU.EX2, no range fix-up):
//   sa = {x, y, A' = -0.5 log2(e) A, B' = -log2(e) B},  sb = {C' = -0.5 log2(e) C, opacity}
//   power2 = (A' dx) dx + (C' dy) dy + (B' dx) dy  ( = log2(e) * power ),  G = 2^power2.
// Two pixels of a lane (same column, rows y and y+4) are evaluated with Blackwell's packed FP32
// instructions (FADD2 / FMUL2 / FFMA2).  Forward and backward share ogs_stage/ogs_pair_power/
// ogs_ex2 so that they take bit-identical skip / contribute decisions.
#define OGS_LOG2E 1.44269504088896340736f
__device__ __forceinline__ float2 s2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float ogs_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float ogs_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void ogs_stage(const float4 r0, const float4 r1, float4& sa, float2& sb) {
    sa = make_float4(r0.x, r0.y, __fmul_rn(-0.5f * OGS_LOG2E, r0.z), __fmul_rn(-OGS_LOG2E, r0.w));
    sb = make_float2(__fmul_rn(-0.5f * OGS_LOG2E, r1.x), r1.y);
}
// adx = (A' dx) dx, bdx = B' dx (per column); npy = -(pixel rows); returns power2 of the two pixels, dy by reference
__device__ __forceinline__ float2 ogs_pair_power(float adx, float bdx, float Cs, float y, float2 npy, float2& dy) {
    dy = __fadd2_rn(s2(y), npy);
    const float2 t = __fmul2_rn(s2(Cs), dy);
    const float2 q = __ffma2_rn(t, dy, s2(adx));
    return __ffma2_rn(s2(bdx), dy, q);
}
// Conservative test on a staged record: "can this Gaussian reach alpha >= 1/255 anywhere in the pixel
// rectangle [x0,x1] x [y0,y1]?"  That needs q'(d) = a dx^2 + 2 hb dx dy + c dy^2 <= log2(255 opacity)
// with a = -A', hb = -B'/2, c = -C'.  q' is convex, so its minimum over the rectangle is 0 if the centre
// is inside, else the smallest of the four clamped 1-D edge minima.  A small margin keeps the test
// conservative under fp32 rounding: an entry is dropped only if every pixel would have skipped it.
__device__ __forceinline__ bool ogs_rect_hit_s(const float4 sa, const float2 sb, float x0, float y0, float x1, float y1) {
    const float A = -sa.z, B = -0.5f * sa.w, C = -sb.x;
    const float o255 = 255.0f * sb.y;
    if (!(o255 >= 1.0f)) return false;
    if (!(A > 0.f && C > 0.f)) return true;
    const float tau = __log2f(o255);
    const float dxl = sa.x - x1, dxh = sa.x - x0, dyl = sa.y - y1, dyh = sa.y - y0;
    if (dxl <= 0.f && dxh >= 0.f && dyl <= 0.f && dyh >= 0.f) return true;
    const float nbc = -B / C, nba = -B / A;
    float q = 3.0e38f;
    {
        const float c = dxl, d = fminf(dyh, fmaxf(dyl, nbc * c));
        q = fminf(q, A * c * c + 2.f * B * c * d + C * d * d);
    }
    {
        const float c = dxh, d = fminf(dyh, fmaxf(dyl, nbc * c));
        q = fminf(q, A * c * c + 2.f * B * c * d + C * d * d);
    }
    {
        const float c = dyl, d = fminf(dxh, fmaxf(dxl, nba * c));
        q = fminf(q, A * d * d + 2.f * B * d * c + C * c * c);
    }
    {
        const float c = dyh, d = fminf(dxh, fmaxf(dxl, nba * c));
        q = fminf(q, A * d * d + 2.f * B * d * c + C * c * c);
    }
    return q <= tau * 1.001f + 1e-3f;
}
#endif

// kmeans (kmeans.cu)
int launch_kmeans_assign(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b,
                         const float* centers, int k, const int64_t* select_ids, int64_t selected, int64_t id_offset,
                         int64_t* ids_out, float* sums, float* counts, cudaStream_t s);
int launch_kmeans_gather_st(int64_t N, const float* feat, int Dout, const float* centers, int Dc, const int64_t* ids,
                            float* out, cudaStream_t s);
size_t kmeans_lloyd_workspace_bytes(int k, int D);
size_t kmeans_seg_lloyd_workspace_bytes(int k1, int k2, int D);
int launch_kmeans_lloyd_pass(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b, float* centers, int k,
                             int k_out, const int64_t* select_ids, int64_t selected, int64_t id_offset, int64_t* ids_out,
                             float* counts_state, float eps_add, const ogs_peer_comm* comm, void* workspace, cudaStream_t s);
int launch_kmeans_seg_lloyd_pass(int64_t N, const float* a, int D, const int64_t* coarse_ids, float* seg_centers,
                                 const int32_t* seg_k, int k1, int k2, int64_t* ids_out, int fix_bits, float* counts_state,
                                 float eps_add, const ogs_peer_comm* comm, void* workspace, cudaStream_t s);
int launch_kmeans_assign_segmented(int64_t N, const float* a, int D, const int64_t* coarse_ids, const float* seg_centers,
                                   const int32_t* seg_k, int k1, int k2, int64_t* ids_out, int64_t* acc, int fix_bits,
                                   cudaStream_t s);
int launch_kmeans_seg_finalize(int rows, int D, const int64_t* acc, int fix_bits, float eps_add, float* counts_state,
                               float* centers, cudaStream_t s);


// mask statistics (mask_stats.cu)
int launch_mask_mean_forward(int M, int C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids, const int32_t* overlap, const float* img, float* sums,
                             float* counts, cudaStream_t s);
int launch_mask_mean_backward(int M, int C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids, const int32_t* overlap, const float* img, const float* G,
                              const float* K, float* dfeat, float* dimg, cudaStream_t s);
int launch_mask_var_forward(int M, int C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids, const int32_t* overlap, const float* img, const float* mean,
                            float* sq, cudaStream_t s);
int launch_cohesion_forward(int M, int C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids, const int32_t* overlap, const float* mean, float* dsum,
                            float* npix, cudaStream_t s);
int launch_cohesion_backward(int M, int C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids, const int32_t* overlap, const float* mean, const float* coef,
                             float* dfeat, float* dmean, cudaStream_t s);


int launch_sam_masks(int M, int64_t HW, const int32_t* level_ids, int offset, int64_t* mask_id, uint8_t* invalid_pix,
                     int16_t* ids, uint8_t* masks, cudaStream_t s);
int launch_mask_id_map(int M, int64_t HW, const uint8_t* masks, int16_t* ids, int32_t* overlap, cudaStream_t s);

// inter-mask contrastive loss (separation.cu)
int launch_separation_loss(int N, int C, const float* mean, int small_weights, float* scratch, float* loss_out, float* dmean,
                           cudaStream_t s);

// pairwise mask intersections (mask_iou.cu)
int64_t mask_iou_scratch_bytes(int n1, int n2, int64_t HW);
int launch_mask_pair_counts(int n1, int n2, int64_t HW, const uint8_t* masks1, const uint8_t* masks2, uint32_t* scratch,
                            int32_t* inter, int32_t* counts, cudaStream_t s);


// single-splat footprint votes (footprint.cu)
int launch_footprint_votes(int P, int W, int H, const GeomPtrs& g, const int32_t* sam_ids, int empty_id, float color,
                           int32_t* dominant_id, int32_t* dominant_weight, int32_t* footprint_pixels, int32_t* q_max,
                           int32_t* overflow, cudaStream_t s);

// optimiser step (adam.cu)
int launch_adam_step(int n_tensors, const ogs_adam_tensor* tensors, float grad_scale, cudaStream_t s);

}  // namespace ogs
