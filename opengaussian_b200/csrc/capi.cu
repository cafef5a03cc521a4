// capi.cu -- the extern "C" boundary of libogs_b200.so (declared in include/ogs_b200.h).
// Orchestrates the kernel families; owns no long-lived memory: per-call state lives in buffers
// obtained through the caller's allocation callback (same role as upstream's resize functionals),
// transient sort scratch comes from the stream-ordered CUDA memory pool.
#include <stdarg.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace ogs {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return (int)e > 0 ? (int)e : 999;
}

// ---- profiling: event pairs per family, drained by ogs_profile_read ----
struct ProfPair { cudaEvent_t a, b; int fam; };
static bool g_prof_on = false;
static std::vector<ProfPair> g_prof_pairs;
static std::vector<cudaEvent_t> g_prof_free;
static cudaEvent_t g_prof_open[PF_COUNT];
static std::mutex g_prof_mu;      // the profile is a per-process measurement aid; the lock keeps it consistent

static cudaEvent_t prof_event() {
    if (!g_prof_free.empty()) { cudaEvent_t e = g_prof_free.back(); g_prof_free.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
void prof_begin(int family, cudaStream_t s) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEvent_t e = prof_event();
    cudaEventRecord(e, s);
    g_prof_open[family] = e;
}
void prof_end(int family, cudaStream_t s) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (!g_prof_open[family]) return;
    cudaEvent_t e = prof_event();
    cudaEventRecord(e, s);
    g_prof_pairs.push_back({g_prof_open[family], e, family});
    g_prof_open[family] = nullptr;
}

static int ensure_pool(void) {
    static thread_local int done_dev = -1;
    int dev = 0;
    OGS_CUDA(cudaGetDevice(&dev));
    if (done_dev == dev) return 0;
    cudaMemPool_t pool;
    OGS_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t thr = UINT64_MAX;
    OGS_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    done_dev = dev;
    return 0;
}

// Per host thread AND per device: running estimate of num_rendered (+25 %, see ogs_raster_forward), the pinned
// word the scan total is copied to, and the event that marks that copy.  (Events and pinned allocations belong to
// the device/context that was current when they were made.)
#define OGS_MAX_PENDING 64
struct PendingFrame {
    cudaEvent_t ev = nullptr;      // marks the copy of [N, overflow flag] into the slot's pinned words
    int64_t cap = 0;               // the capacity the frame was binned with
    bool live = false;
};
struct ForwardCtx {
    uint64_t cap_hint = 0;
    uint32_t* pinned = nullptr;    // 2 words for the synchronous check + 2 per pending slot
    cudaEvent_t ev = nullptr;
    PendingFrame pending[OGS_MAX_PENDING];
    void grow_hint(int64_t N) {
        const uint64_t want = (uint64_t)N + (uint64_t)N / 4 + 65536;
        const uint64_t decay = cap_hint - cap_hint / 32;
        cap_hint = want > decay ? want : decay;
    }
};
static ForwardCtx& forward_ctx(void) {
    static thread_local ForwardCtx ctx[OGS_MAX_DEVICES];
    return ctx[current_device()];
}

static uint32_t* pinned_scalar(ForwardCtx& fc) {
    if (!fc.pinned) {
        if (cudaMallocHost((void**)&fc.pinned, 8 * (1 + OGS_MAX_PENDING)) != cudaSuccess) fc.pinned = nullptr;
    }
    return fc.pinned;
}

__global__ void export_keys_kernel(int tiles, const uint2* __restrict__ ranges, const uint32_t* __restrict__ point_list,
                                   const float4* __restrict__ rec1, uint64_t* __restrict__ keys) {
    const int t = blockIdx.x;
    if (t >= tiles) return;
    const uint2 r = ranges[t];
    for (uint32_t i = r.x + threadIdx.x; i < r.y; i += blockDim.x) {
        const uint32_t g = point_list[i];
        keys[i] = ((uint64_t)(uint32_t)t << 32) | (uint64_t)__float_as_uint(rec1[g].z);
    }
}

__global__ void export_geom_kernel(int P, GeomPtrs g, bool has_rgb, float* xy, float* depth, float* conic_opacity,
                                   float* rgb, uint32_t* tiles) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float4 a = g.rec0[i], b = g.rec1[i];
    if (xy) { xy[2 * i] = a.x; xy[2 * i + 1] = a.y; }
    if (depth) depth[i] = b.z;
    if (conic_opacity) {
        conic_opacity[4 * i] = a.z; conic_opacity[4 * i + 1] = a.w; conic_opacity[4 * i + 2] = b.x;
        conic_opacity[4 * i + 3] = b.y;
    }
    if (rgb && has_rgb) { rgb[3 * i] = g.rgb[3 * i]; rgb[3 * i + 1] = g.rgb[3 * i + 1]; rgb[3 * i + 2] = g.rgb[3 * i + 2]; }
    if (tiles) tiles[i] = g.tiles[i];
}

static int validate_inputs(const ogs_raster_inputs* in) {
    if (!in) { set_error("inputs is NULL"); return -1; }
    if (in->P < 0 || in->W <= 0 || in->H <= 0) { set_error("bad sizes P=%d W=%d H=%d", in->P, in->W, in->H); return -1; }
    if ((in->shs != nullptr) == (in->colors_precomp != nullptr) && in->P > 0) {
        set_error("Please provide excatly one of either SHs or precomputed colors!");
        return -2;
    }
    const bool sr = in->scales != nullptr && in->rotations != nullptr;
    if (in->P > 0 && (sr == (in->cov3D_precomp != nullptr) || ((in->scales != nullptr) != (in->rotations != nullptr)))) {
        set_error("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
        return -2;
    }
    if (in->n_extra < 0 || 3 + in->n_extra > OGS_MAX_CHANNELS) { set_error("n_extra=%d out of range", in->n_extra); return -1; }
    if (in->n_extra > 0 && !in->extra && in->P > 0) { set_error("n_extra > 0 but extra is NULL"); return -1; }
    if (in->shs && (in->sh_degree < 0 || in->sh_degree > 3 || (in->sh_degree + 1) * (in->sh_degree + 1) > in->M)) {
        set_error("sh_degree=%d incompatible with M=%d", in->sh_degree, in->M);
        return -1;
    }
    if (in->prefiltered) { set_error("prefiltered=True is not supported"); return -1; }
    if (in->shs_rest && (!in->shs || in->M < 2)) { set_error("shs_rest needs shs (= _features_dc) and M >= 2"); return -1; }
    if ((in->act_flags & (OGS_ACT_SCALE_EXP | OGS_ACT_ROT_NORMALIZE)) && !(in->scales && in->rotations)) {
        set_error("scale/rotation activations need scales and rotations");
        return -1;
    }
    if ((in->act_flags & OGS_ACT_EXTRA_UNIT_HALF) && in->n_extra <= 0) { set_error("extra activation needs n_extra > 0"); return -1; }
    const int gx = (in->W + 15) / 16, gy = (in->H + 15) / 16;
    if ((int64_t)gx * gy > 65536) { set_error("image too large: %d tiles (max 65536: the tile id is a 16-bit sort key)", gx * gy); return -1; }
    if (!in->bg || !in->viewmatrix || !in->projmatrix || !in->campos) { set_error("bg/viewmatrix/projmatrix/campos must be set"); return -1; }
    return 0;
}

}  // namespace ogs

using namespace ogs;

extern "C" {

int ogs_abi_version(void) { return OGS_ABI_VERSION; }

void ogs_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = on != 0;
    if (g_prof_on && g_prof_free.size() < 2048) {   // pre-create so that recording costs no driver allocation
        for (int i = 0; i < 2048; i++) {
            cudaEvent_t e = nullptr;
            if (cudaEventCreate(&e) == cudaSuccess) g_prof_free.push_back(e);
        }
    }
}

int ogs_profile_read(float* ms_out, int32_t* launches_out, int32_t n) {
    float ms[PF_COUNT] = {0};
    int cnt[PF_COUNT] = {0};
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& p : g_prof_pairs) {
        cudaError_t e = cudaEventSynchronize(p.b);
        float t = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&t, p.a, p.b);
        if (e != cudaSuccess) return cuda_fail(e, "profile_read");
        ms[p.fam] += t;
        cnt[p.fam]++;
        g_prof_free.push_back(p.a);
        g_prof_free.push_back(p.b);
    }
    g_prof_pairs.clear();
    for (int i = 0; i < n && i < PF_COUNT; i++) {
        if (ms_out) ms_out[i] = ms[i];
        if (launches_out) launches_out[i] = cnt[i];
    }
    return 0;
}
const char* ogs_last_error(void) { return g_err; }

size_t ogs_raster_backward_scratch_floats(int32_t P, int32_t n_extra) {
    return (size_t)(P > 0 ? P : 1) * (size_t)(3 + n_extra + 7);
}

int ogs_raster_forward(const ogs_raster_inputs* in, const ogs_raster_outputs* out, ogs_alloc_fn alloc,
                       void* alloc_user, ogs_raster_state* st, void* stream_) {
    int rc = validate_inputs(in);
    if (rc) return rc;
    if (!out || !out->color || !out->depth || !out->alpha || (!out->radii && in->P > 0) || !alloc || !st) {
        set_error("outputs/alloc/state must be set");
        return -1;
    }
    cudaStream_t s = (cudaStream_t)stream_;
    if ((rc = ensure_pool())) return rc;
    const int P = in->P, W = in->W, H = in->H, C = 3 + in->n_extra;
    const int gx = (W + 15) / 16, gy = (H + 15) / 16, tiles = gx * gy;
    const bool has_sh = in->shs != nullptr;

    const int n_feat_act = (in->act_flags & OGS_ACT_EXTRA_UNIT_HALF) ? in->n_extra : 0;
    const GeomLayout gl = GeomLayout::make(P, has_sh, n_feat_act);
    const ImgLayout il = ImgLayout::make(W, H);
    memset(st, 0, sizeof *st);
    st->geom = alloc(alloc_user, gl.total, "geom");
    st->image = alloc(alloc_user, il.total, "image");
    st->geom_bytes = (int64_t)gl.total;
    st->image_bytes = (int64_t)il.total;
    if (!st->geom || !st->image) { set_error("allocation callback returned NULL"); return -6; }
    const GeomPtrs g = GeomPtrs::from(st->geom, gl);
    float* final_T = (float*)((char*)st->image + il.final_T);
    uint32_t* n_contrib = (uint32_t*)((char*)st->image + il.n_contrib);

    int64_t N = 0, cap = 0;
    bool speculative = false;
    uint32_t* h = nullptr;
    const uint32_t* n_ptr = nullptr;
    cudaEvent_t n_event = nullptr;
    ForwardCtx& fc = forward_ctx();
    PendingFrame* deferred = nullptr;
    AsyncScratch scratch1(s);          // freed (stream-ordered) on every exit path
    BinScratch sc;
    memset(&sc, 0, sizeof sc);
    if (P > 0) {
        const size_t pw = align_up((size_t)(P + 2) * 4, 256);      // offsets carries two extra words: N and the overflow flag
        sc.cub_temp_bytes = align_up(depth_sort_temp_bytes(P), 256);
        OGS_CUDA(scratch1.alloc(pw * 5 + sc.cub_temp_bytes));
        char* s1 = (char*)scratch1.p;
        sc.dkeys_in = (uint32_t*)(s1);
        sc.dvals_in = (uint32_t*)(s1 + pw);
        sc.dkeys_out = (uint32_t*)(s1 + 2 * pw);
        sc.dvals_out = (uint32_t*)(s1 + 3 * pw);
        sc.offsets = (uint32_t*)(s1 + 4 * pw);
        sc.cub_temp = s1 + 5 * pw;

        PreprocessArgs pa;
        pa.P = P; pa.D = in->sh_degree; pa.M = in->M; pa.W = W; pa.H = H;
        pa.act_flags = in->act_flags; pa.n_extra = in->n_extra; pa.shs_rest = in->shs_rest; pa.extra = in->extra;
        pa.means3D = in->means3D; pa.scales = in->scales; pa.rotations = in->rotations;
        pa.cov3D_precomp = in->cov3D_precomp; pa.opacities = in->opacities; pa.shs = in->shs;
        pa.scale_modifier = in->scale_modifier; pa.tanfovx = in->tanfovx; pa.tanfovy = in->tanfovy;
        pa.view = in->viewmatrix; pa.proj = in->projmatrix; pa.campos = in->campos;
        pa.radii = out->radii; pa.g = g; pa.depth_keys = sc.dkeys_in; pa.depth_vals = sc.dvals_in;
        prof_begin(PF_PREPROCESS_FWD, s);
        rc = launch_preprocess_forward(pa, s);
        prof_end(PF_PREPROCESS_FWD, s);
        if (rc) return rc;
        OGS_KERNEL_CHECK("preprocess_forward", in->debug, s);
        prof_begin(PF_DEPTH_SORT_SCAN, s);
        rc = depth_sort_and_scan(P, g, sc, s, in->debug);
        prof_end(PF_DEPTH_SORT_SCAN, s);
        if (rc) return rc;
        h = pinned_scalar(fc);
        if (!h) { set_error("cudaMallocHost failed"); return 2; }
        if (in->defer_capacity_check && fc.cap_hint != 0 && !in->debug) {
            for (int k = 0; k < OGS_MAX_PENDING && !deferred; k++)
                if (!fc.pending[k].live) deferred = &fc.pending[k];
            if (deferred) h += 2 * (1 + (deferred - fc.pending));
        }
        n_ptr = sc.offsets + P;
        OGS_CUDA(cudaMemcpyAsync(h, n_ptr, 8, cudaMemcpyDeviceToHost, s));     // [N, overflow flag]
        // Capacity speculation: the binning buffers are sized from the running estimate cap_hint and
        // the N-dependent kernels take N from device memory, so emit/sort/blend are queued WITHOUT
        // waiting for the scan; the host reads N only after everything is launched (the scan has long
        // finished by then).  If the estimate was too small the binning + blend are redone (rare).
        if (fc.cap_hint == 0 || in->debug) {
            OGS_CUDA(cudaStreamSynchronize(s));
            if (h[1]) { set_error("more than 2^32 - 1 (Gaussian, tile) duplicates in one frame: 32-bit offsets overflow"); return -7; }
            N = (int64_t)*h;
            cap = N;
        } else if (deferred) {
            if (!deferred->ev) OGS_CUDA(cudaEventCreateWithFlags(&deferred->ev, cudaEventDisableTiming));
            OGS_CUDA(cudaEventRecord(deferred->ev, s));
            cap = (int64_t)fc.cap_hint;
            deferred->cap = cap;
            deferred->live = true;
            speculative = true;
        } else {
            if (!fc.ev) OGS_CUDA(cudaEventCreateWithFlags(&fc.ev, cudaEventDisableTiming));
            OGS_CUDA(cudaEventRecord(fc.ev, s));
            n_event = fc.ev;
            cap = (int64_t)fc.cap_hint;
            speculative = true;
        }
    }
    uint32_t* point_list = nullptr;
    uint2* ranges = nullptr;
    for (;;) {
        const BinLayout bl = BinLayout::make(cap, tiles);
        st->binning = alloc(alloc_user, bl.total, "binning");
        st->binning_bytes = (int64_t)bl.total;
        if (!st->binning) { set_error("allocation callback returned NULL"); return -6; }
        point_list = (uint32_t*)((char*)st->binning + bl.point_list);
        ranges = (uint2*)((char*)st->binning + bl.ranges);
        if (cap > 0 && P > 0) {
            AsyncScratch scratch2(s);
            const size_t k2 = align_up((size_t)cap * 2, 256), v4 = align_up((size_t)cap * 4, 256);
            const size_t tb = align_up(tile_sort_temp_bytes(cap), 256);
            OGS_CUDA(scratch2.alloc(2 * k2 + v4 + tb));
            char* s2 = (char*)scratch2.p;
            sc.cub_temp = s2 + 2 * k2 + v4;
            sc.cub_temp_bytes = tb;
            rc = emit_sort_ranges(P, W, H, n_ptr, cap, g, sc, (uint16_t*)s2, (uint32_t*)(s2 + 2 * k2),
                                  (uint16_t*)(s2 + k2), point_list, ranges, s, in->debug);
        } else {
            cudaError_t e = cudaMemsetAsync(ranges, 0, (size_t)tiles * sizeof(uint2), s);
            if (e != cudaSuccess) rc = cuda_fail(e, "memset ranges");
        }
        if (rc) return rc;

        BlendFwdArgs ba;
        ba.W = W; ba.H = H; ba.C = C;
        ba.ranges = ranges; ba.point_list = point_list; ba.rec0 = g.rec0; ba.rec1 = g.rec1;
        ba.base = has_sh ? g.rgb : in->colors_precomp;
        ba.extra = n_feat_act ? g.feat : in->extra; ba.bg = in->bg;
        ba.out_color = out->color; ba.out_depth = out->depth; ba.out_alpha = out->alpha;
        ba.final_T = final_T; ba.n_contrib = n_contrib;
        prof_begin(PF_BLEND_FWD, s);
        rc = launch_blend_forward(ba, s);
        prof_end(PF_BLEND_FWD, s);
        if (rc) return rc;
        OGS_KERNEL_CHECK("blend_forward", in->debug, s);
        if (!speculative) break;
        if (deferred) {                // the caller resolves this frame in ogs_raster_capacity_check
            N = -1;
            break;
        }
        OGS_CUDA(cudaEventSynchronize(n_event));
        if (h[1]) { set_error("more than 2^32 - 1 (Gaussian, tile) duplicates in one frame: 32-bit offsets overflow"); return -7; }
        N = (int64_t)*h;
        speculative = false;
        if (N <= cap) break;
        cap = N;                       // estimate too small: redo binning + blend with the exact size
    }
    scratch1.release();
    if (P > 0 && N >= 0) fc.grow_hint(N);
    st->num_rendered = N;
    return 0;
}

int ogs_raster_cached_bytes(const ogs_raster_inputs* in, int64_t num_rendered, int64_t* geom_bytes, int64_t* binning_bytes) {
    if (!in || num_rendered < 0 || in->P < 0 || in->W <= 0 || in->H <= 0) { set_error("cached_bytes: bad arguments"); return -1; }
    const int tiles = ((in->W + 15) / 16) * ((in->H + 15) / 16);
    if (geom_bytes) *geom_bytes = (int64_t)GeomLayout::make(in->P, in->shs != nullptr, 0).total;
    if (binning_bytes) *binning_bytes = (int64_t)BinLayout::make(num_rendered, tiles).total;
    return 0;
}

int ogs_raster_forward_cached(const ogs_raster_inputs* in, const ogs_raster_outputs* out, ogs_alloc_fn alloc,
                              void* alloc_user, const ogs_raster_state* cached, ogs_raster_state* st, void* stream_) {
    int rc = validate_inputs(in);
    if (rc) return rc;
    if (!out || !out->color || !out->depth || !out->alpha || !alloc || !st || !cached) {
        set_error("outputs/alloc/state must be set");
        return -1;
    }
    cudaStream_t s = (cudaStream_t)stream_;
    const int P = in->P, W = in->W, H = in->H, C = 3 + in->n_extra;
    const int gx = (W + 15) / 16, gy = (H + 15) / 16, tiles = gx * gy;
    const bool has_sh = in->shs != nullptr;
    const int n_feat_act = (in->act_flags & OGS_ACT_EXTRA_UNIT_HALF) ? in->n_extra : 0;
    // the activated channels sit last in the geometry layout: every other offset is the same with and without them
    const GeomLayout gl = GeomLayout::make(P, has_sh, 0);
    const ImgLayout il = ImgLayout::make(W, H);
    if (!cached->geom || !cached->binning || cached->num_rendered < 0 || cached->geom_bytes < (int64_t)gl.total ||
        cached->binning_bytes < (int64_t)BinLayout::make(cached->num_rendered, tiles).total) {
        set_error("cached state does not belong to a finished forward of these sizes (P=%d, %d tiles, N=%lld)", P, tiles,
                  (long long)cached->num_rendered);
        return -1;
    }
    *st = *cached;
    st->image = alloc(alloc_user, il.total, "image");
    st->image_bytes = (int64_t)il.total;
    st->feat = nullptr;
    if (!st->image) { set_error("allocation callback returned NULL"); return -6; }
    const GeomPtrs g = GeomPtrs::from(st->geom, gl);
    const BinLayout bl = BinLayout::make(st->num_rendered, tiles);
    if (n_feat_act && P > 0) {
        st->feat = alloc(alloc_user, (size_t)P * n_feat_act * sizeof(float), "feat");
        if (!st->feat) { set_error("allocation callback returned NULL"); return -6; }
        prof_begin(PF_PREPROCESS_FWD, s);
        rc = launch_feat_refresh(P, n_feat_act, g.rec1, in->extra, (float*)st->feat, s);
        prof_end(PF_PREPROCESS_FWD, s);
        if (rc) return rc;
        OGS_KERNEL_CHECK("feat_refresh", in->debug, s);
    }
    if (out->radii && P > 0) {          // radius = rec1.w as int bits; culled Gaussians hold 0 there
        cudaError_t e = cudaMemcpy2DAsync(out->radii, 4, &g.rec1[0].w, 16, 4, (size_t)P, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) return cuda_fail(e, "radii copy");
    }
    BlendFwdArgs ba;
    ba.W = W; ba.H = H; ba.C = C;
    ba.ranges = (uint2*)((char*)st->binning + bl.ranges);
    ba.point_list = (uint32_t*)((char*)st->binning + bl.point_list);
    ba.rec0 = g.rec0; ba.rec1 = g.rec1;
    ba.base = has_sh ? g.rgb : in->colors_precomp;
    ba.extra = n_feat_act ? (const float*)st->feat : in->extra; ba.bg = in->bg;
    ba.out_color = out->color; ba.out_depth = out->depth; ba.out_alpha = out->alpha;
    ba.final_T = (float*)((char*)st->image + il.final_T);
    ba.n_contrib = (uint32_t*)((char*)st->image + il.n_contrib);
    prof_begin(PF_BLEND_FWD, s);
    rc = launch_blend_forward(ba, s);
    prof_end(PF_BLEND_FWD, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("blend_forward", in->debug, s);
    return 0;
}

int64_t ogs_raster_capacity_hint(int64_t new_hint) {
    ForwardCtx& fc = forward_ctx();
    const int64_t old = (int64_t)fc.cap_hint;
    if (new_hint >= 0) fc.cap_hint = (uint64_t)new_hint;
    return old;
}

int ogs_raster_capacity_check(void) {
    ForwardCtx& fc = forward_ctx();
    int result = 0;
    for (int k = 0; k < OGS_MAX_PENDING; k++) {
        PendingFrame& pf = fc.pending[k];
        if (!pf.live) continue;
        pf.live = false;
        cudaError_t e = cudaEventSynchronize(pf.ev);
        if (e != cudaSuccess) { result = cuda_fail(e, "capacity check"); continue; }
        const uint32_t* h = fc.pinned + 2 * (1 + k);
        if (h[1]) {
            set_error("more than 2^32 - 1 (Gaussian, tile) duplicates in one frame: 32-bit offsets overflow");
            result = -7;
            continue;
        }
        const int64_t N = (int64_t)h[0];
        fc.grow_hint(N);
        if (N > pf.cap && result == 0) result = 1;
    }
    return result;
}

int ogs_raster_backward(const ogs_raster_inputs* in, const ogs_raster_state* st, const ogs_raster_grads_in* gin,
                        const ogs_raster_grads_out* go, void* stream_) {
    int rc = validate_inputs(in);
    if (rc) return rc;
    if (!st || !gin || !go || (!gin->dL_dcolor && !gin->dL_dfeat) || !go->scratch) { set_error("state/grads/scratch must be set"); return -1; }
    if (gin->dL_dfeat && in->n_extra <= 0) { set_error("dL_dfeat needs n_extra > 0"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    const int P = in->P, W = in->W, H = in->H, C = 3 + in->n_extra;
    if (P == 0) return 0;
    const int gx = (W + 15) / 16, gy = (H + 15) / 16, tiles = gx * gy;
    const bool has_sh = in->shs != nullptr;
    const int n_feat_act = (in->act_flags & OGS_ACT_EXTRA_UNIT_HALF) ? in->n_extra : 0;
    const GeomLayout gl = GeomLayout::make(P, has_sh, n_feat_act);
    const ImgLayout il = ImgLayout::make(W, H);
    const BinLayout bl = BinLayout::make(st->num_rendered, tiles);
    const GeomPtrs g = GeomPtrs::from(st->geom, gl);

    const int geom = (go->dL_dmeans3D || go->dL_dmeans2D || go->dL_dopacities || go->dL_dshs || go->dL_dshs_rest ||
                      go->dL_dscales || go->dL_drotations || go->dL_dcov3D) ? 1 : 0;
    if (go->dL_dshs_rest && !go->dL_dshs) { set_error("dL_dshs_rest needs dL_dshs"); return -1; }
    BlendBwdArgs ba;
    ba.P = P; ba.W = W; ba.H = H; ba.C = C;
    ba.ranges = (const uint2*)((char*)st->binning + bl.ranges);
    ba.point_list = (const uint32_t*)((char*)st->binning + bl.point_list);
    ba.rec0 = g.rec0; ba.rec1 = g.rec1;
    ba.base = has_sh ? g.rgb : in->colors_precomp;
    ba.extra = n_feat_act ? (st->feat ? (const float*)st->feat : g.feat) : in->extra; ba.bg = in->bg;
    ba.final_T = (const float*)((char*)st->image + il.final_T);
    ba.n_contrib = (const uint32_t*)((char*)st->image + il.n_contrib);
    ba.dL_dcolor = gin->dL_dcolor; ba.dL_ddepth = gin->dL_ddepth; ba.dL_dalpha = gin->dL_dalpha; ba.dL_dfeat = gin->dL_dfeat;
    ba.geom = geom;
    ba.acc = (float*)go->scratch;
    ba.stride = blend_bwd_stride(C, geom);
    prof_begin(PF_BLEND_BWD, s);
    rc = launch_blend_backward(ba, s);
    prof_end(PF_BLEND_BWD, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("blend_backward", in->debug, s);

    PreprocessBwdArgs pa;
    pa.P = P; pa.D = in->sh_degree; pa.M = in->M; pa.C = C; pa.W = W; pa.H = H;
    pa.act_flags = in->act_flags; pa.shs_rest = in->shs_rest; pa.extra = in->extra; pa.opacities = in->opacities;
    pa.dL_dshs_rest = go->dL_dshs_rest; pa.accumulate = go->accumulate;
    pa.means3D = in->means3D; pa.scales = in->scales; pa.rotations = in->rotations;
    pa.cov3D_precomp = in->cov3D_precomp; pa.shs = in->shs;
    pa.scale_modifier = in->scale_modifier; pa.tanfovx = in->tanfovx; pa.tanfovy = in->tanfovy;
    pa.view = in->viewmatrix; pa.proj = in->projmatrix; pa.campos = in->campos;
    pa.g = g; pa.acc = ba.acc; pa.stride = ba.stride; pa.geom = geom;
    pa.dL_dmeans3D = go->dL_dmeans3D; pa.dL_dmeans2D = go->dL_dmeans2D; pa.dL_dopacities = go->dL_dopacities;
    pa.dL_dshs = go->dL_dshs; pa.dL_dcolors_precomp = go->dL_dcolors_precomp; pa.dL_dscales = go->dL_dscales;
    pa.dL_drotations = go->dL_drotations; pa.dL_dcov3D = go->dL_dcov3D; pa.dL_dextra = go->dL_dextra;
    prof_begin(PF_PREPROCESS_BWD, s);
    rc = launch_preprocess_backward(pa, s);
    prof_end(PF_PREPROCESS_BWD, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("preprocess_backward", in->debug, s);
    return 0;
}

int ogs_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, uint8_t* present, void* stream_) {
    if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) { set_error("mark_visible: bad arguments"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    int rc = launch_mark_visible(P, means3D, viewmatrix, present, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mark_visible", 0, s);
    return 0;
}

int ogs_raster_export(const ogs_raster_inputs* in, const ogs_raster_state* st, uint64_t* keys, uint32_t* point_list,
                      uint32_t* ranges, float* xy, float* depth, float* conic_opacity, float* rgb,
                      uint32_t* tiles_touched, float* final_T, uint32_t* n_contrib, void* stream_) {
    if (!in || !st) { set_error("export: NULL inputs/state"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    const int P = in->P, W = in->W, H = in->H;
    const int gx = (W + 15) / 16, gy = (H + 15) / 16, tiles = gx * gy;
    const bool has_sh = in->shs != nullptr;
    const GeomLayout gl = GeomLayout::make(P, has_sh, (in->act_flags & OGS_ACT_EXTRA_UNIT_HALF) ? in->n_extra : 0);
    const ImgLayout il = ImgLayout::make(W, H);
    const BinLayout bl = BinLayout::make(st->num_rendered, tiles);
    const GeomPtrs g = GeomPtrs::from(st->geom, gl);
    const uint32_t* pl = (const uint32_t*)((char*)st->binning + bl.point_list);
    const uint2* rg = (const uint2*)((char*)st->binning + bl.ranges);
    const int64_t N = st->num_rendered;
    if (keys && N > 0) export_keys_kernel<<<tiles, 128, 0, s>>>(tiles, rg, pl, g.rec1, keys);
    if (point_list && N > 0) OGS_CUDA(cudaMemcpyAsync(point_list, pl, (size_t)N * 4, cudaMemcpyDeviceToDevice, s));
    if (ranges) OGS_CUDA(cudaMemcpyAsync(ranges, rg, (size_t)tiles * 8, cudaMemcpyDeviceToDevice, s));
    if (P > 0 && (xy || depth || conic_opacity || rgb || tiles_touched))
        export_geom_kernel<<<(P + 255) / 256, 256, 0, s>>>(P, g, has_sh, xy, depth, conic_opacity, rgb, tiles_touched);
    if (final_T) OGS_CUDA(cudaMemcpyAsync(final_T, (char*)st->image + il.final_T, (size_t)W * H * 4, cudaMemcpyDeviceToDevice, s));
    if (n_contrib) OGS_CUDA(cudaMemcpyAsync(n_contrib, (char*)st->image + il.n_contrib, (size_t)W * H * 4, cudaMemcpyDeviceToDevice, s));
    OGS_KERNEL_CHECK("export", 0, s);
    return 0;
}

int ogs_kmeans_assign(int64_t N, const float* a, int32_t Da, const float* b, int32_t Db, float scale_b,
                      const float* centers, int32_t k, const int64_t* select_ids, int64_t selected,
                      int64_t id_offset, int64_t* ids_out, float* sums, float* counts, void* stream_) {
    if (N < 0 || Da < 0 || Db < 0 || Da + Db < 1 || k < 1 || !centers || (N > 0 && (!a || !ids_out)) || (Db > 0 && !b)) {
        set_error("kmeans_assign: bad arguments");
        return -1;
    }
    if (N == 0) return 0;
    int rc = ensure_pool();
    if (rc) return rc;
    ProfScope ps(PF_KMEANS_ASSIGN, (cudaStream_t)stream_);
    return launch_kmeans_assign(N, a, Da, b, Db, scale_b, centers, k, select_ids, selected, id_offset, ids_out, sums,
                                counts, (cudaStream_t)stream_);
}

int ogs_kmeans_gather_st(int64_t N, const float* feat, int32_t Dout, const float* centers, int32_t Dc,
                         const int64_t* ids, float* out, void* stream_) {
    if (N < 0 || Dout < 1 || Dc < Dout || (N > 0 && (!feat || !centers || !ids || !out))) {
        set_error("kmeans_gather_st: bad arguments");
        return -1;
    }
    int rc = launch_kmeans_gather_st(N, feat, Dout, centers, Dc, ids, out, (cudaStream_t)stream_);
    if (rc) return rc;
    OGS_KERNEL_CHECK("kmeans_gather_st", 0, (cudaStream_t)stream_);
    return 0;
}

int ogs_kmeans_assign_segmented(int64_t N, const float* a, int32_t D, const int64_t* coarse_ids, const float* seg_centers,
                                const int32_t* seg_k, int32_t k1, int32_t k2, int64_t* ids_out, int64_t* acc,
                                int32_t fix_bits, void* stream_) {
    if (N < 0 || D < 1 || k1 < 1 || k2 < 1 || !seg_centers || !seg_k || fix_bits < 0 || fix_bits > 40 ||
        (N > 0 && (!a || !coarse_ids || !ids_out))) {
        set_error("kmeans_assign_segmented: bad arguments");
        return -1;
    }
    if (N == 0) return 0;
    int rc = ensure_pool();
    if (rc) return rc;
    ProfScope ps(PF_KMEANS_ASSIGN, (cudaStream_t)stream_);
    return launch_kmeans_assign_segmented(N, a, D, coarse_ids, seg_centers, seg_k, k1, k2, ids_out, acc, fix_bits,
                                          (cudaStream_t)stream_);
}

size_t ogs_kmeans_lloyd_segmented_workspace_bytes(int32_t k1, int32_t k2, int32_t D) {
    return kmeans_seg_lloyd_workspace_bytes(k1, k2, D);
}

int ogs_kmeans_lloyd_pass_segmented(int64_t N, const float* a, int32_t D, const int64_t* coarse_ids, float* seg_centers,
                                    const int32_t* seg_k, int32_t k1, int32_t k2, int64_t* ids_out, int32_t fix_bits,
                                    float* counts_state, float eps_add, ogs_peer_comm* comm, void* workspace, void* stream_) {
    if (N < 0 || D < 1 || k1 < 1 || k2 < 1 || !seg_centers || !seg_k || !counts_state || !workspace || fix_bits < 0 ||
        fix_bits > 40 || (N > 0 && (!a || !coarse_ids || !ids_out))) {
        set_error("kmeans_lloyd_pass_segmented: bad arguments");
        return -1;
    }
    ProfScope ps(PF_KMEANS_ASSIGN, (cudaStream_t)stream_);
    return launch_kmeans_seg_lloyd_pass(N, a, D, coarse_ids, seg_centers, seg_k, k1, k2, ids_out, fix_bits, counts_state,
                                        eps_add, comm, workspace, (cudaStream_t)stream_);
}

size_t ogs_kmeans_lloyd_workspace_bytes(int32_t k, int32_t D) { return kmeans_lloyd_workspace_bytes(k, D); }

int ogs_kmeans_lloyd_pass(int64_t N, const float* a, int32_t Da, const float* b, int32_t Db, float scale_b, float* centers,
                          int32_t k, int32_t k_out, const int64_t* select_ids, int64_t selected, int64_t id_offset,
                          int64_t* ids_out, float* counts_state, float eps_add, ogs_peer_comm* comm, void* workspace,
                          void* stream_) {
    if (N < 0 || Da < 0 || Db < 0 || Da + Db < 1 || k < 1 || k_out < k || !centers || !counts_state || !workspace ||
        (N > 0 && (!a || !ids_out)) || (Db > 0 && N > 0 && !b)) {
        set_error("kmeans_lloyd_pass: bad arguments");
        return -1;
    }
    ProfScope ps(PF_KMEANS_ASSIGN, (cudaStream_t)stream_);
    return launch_kmeans_lloyd_pass(N, a, Da, b, Db, scale_b, centers, k, k_out, select_ids, selected, id_offset, ids_out,
                                    counts_state, eps_add, comm, workspace, (cudaStream_t)stream_);
}

int ogs_kmeans_finalize_fixed(int32_t rows, int32_t D, const int64_t* acc, int32_t fix_bits, float eps_add,
                              float* counts_state, float* centers, void* stream_) {
    if (rows < 0 || D < 1 || !acc || !counts_state || !centers || fix_bits < 0 || fix_bits > 40) {
        set_error("kmeans_finalize_fixed: bad arguments");
        return -1;
    }
    return launch_kmeans_seg_finalize(rows, D, acc, fix_bits, eps_add, counts_state, centers, (cudaStream_t)stream_);
}

#define OGS_MASK_ARGS_OK(what)                                                                          \
    if (M < 0 || HW < 0 || ((M > 0 || HW > 0) && !feat) || (M > 0 && HW > 0 && !masks) ||                \
        (ids && !ids_overlap)) {                                                                         \
        set_error(what ": bad arguments");                                                               \
        return -1;                                                                                       \
    }

int ogs_mask_mean_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                          const float* image_mask, float* sums, float* counts, void* stream_) {
    OGS_MASK_ARGS_OK("mask_mean_forward");
    if (M > 0 && (!sums || !counts)) { set_error("mask_mean_forward: outputs must be set"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_mask_mean_forward(M, C, HW, feat, masks, ids, ids_overlap, image_mask, sums, counts, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mask_mean_forward", 0, s);
    return 0;
}

int ogs_mask_mean_backward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                           const float* image_mask, const float* G, const float* K, float* dfeat,
                           float* dimg, void* stream_) {
    OGS_MASK_ARGS_OK("mask_mean_backward");
    if ((M > 0 && (!G || !K)) || (HW > 0 && !dfeat)) { set_error("mask_mean_backward: G/K/dfeat must be set"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_mask_mean_backward(M, C, HW, feat, masks, ids, ids_overlap, image_mask, G, K, dfeat, image_mask ? dimg : nullptr, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mask_mean_backward", 0, s);
    return 0;
}

int ogs_mask_var_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                         const float* image_mask, const float* mean, float* sq, void* stream_) {
    OGS_MASK_ARGS_OK("mask_var_forward");
    if (M > 0 && (!mean || !sq)) { set_error("mask_var_forward: mean/sq must be set"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_mask_var_forward(M, C, HW, feat, masks, ids, ids_overlap, image_mask, mean, sq, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mask_var_forward", 0, s);
    return 0;
}

int ogs_cohesion_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                         const float* mean, float* dsum, float* npix, void* stream_) {
    OGS_MASK_ARGS_OK("cohesion_forward");
    if (M > 0 && (!mean || !dsum || !npix)) { set_error("cohesion_forward: mean/outputs must be set"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_cohesion_forward(M, C, HW, feat, masks, ids, ids_overlap, mean, dsum, npix, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("cohesion_forward", 0, s);
    return 0;
}

int ogs_cohesion_backward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                          const float* mean, const float* coef, float* dfeat, float* dmean, void* stream_) {
    OGS_MASK_ARGS_OK("cohesion_backward");
    if ((M > 0 && (!mean || !coef || !dmean)) || (HW > 0 && !dfeat)) { set_error("cohesion_backward: inputs/outputs must be set"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_cohesion_backward(M, C, HW, feat, masks, ids, ids_overlap, mean, coef, dfeat, dmean, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("cohesion_backward", 0, s);
    return 0;
}

int ogs_sam_masks(int32_t M, int64_t HW, const int32_t* level_ids, int32_t offset, int64_t* mask_id, uint8_t* invalid_pix,
                  int16_t* ids, uint8_t* masks, void* stream_) {
    if (M < 0 || HW < 0 || (HW > 0 && (!level_ids || !mask_id || !invalid_pix || !ids || (M > 0 && !masks)))) {
        set_error("sam_masks: bad arguments");
        return -1;
    }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_sam_masks(M, HW, level_ids, offset, mask_id, invalid_pix, ids, masks, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("sam_masks", 0, s);
    return 0;
}

int ogs_mask_id_map(int32_t M, int64_t HW, const uint8_t* masks, int16_t* ids, int32_t* ids_overlap, void* stream_) {
    if (M < 0 || HW < 0 || (M > 0 && HW > 0 && !masks) || (HW > 0 && !ids) || !ids_overlap) {
        set_error("mask_id_map: bad arguments");
        return -1;
    }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_mask_id_map(M, HW, masks, ids, ids_overlap, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mask_id_map", 0, s);
    return 0;
}

int ogs_separation_loss(int32_t N, int32_t C, const float* mean, int32_t small_weights, float* scratch, float* loss_out,
                        float* dmean, void* stream_) {
    if (N < 2 || !mean || !scratch || !loss_out || !dmean) { set_error("separation_loss: needs N >= 2 and all pointers"); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    return launch_separation_loss(N, C, mean, small_weights, scratch, loss_out, dmean, s);
}

int64_t ogs_mask_iou_scratch_bytes(int32_t n1, int32_t n2, int64_t HW) {
    if (n1 < 0 || n2 < 0 || HW < 0) return -1;
    return mask_iou_scratch_bytes(n1, n2, HW);
}

int ogs_mask_pair_counts(int32_t n1, int32_t n2, int64_t HW, const uint8_t* masks1, const uint8_t* masks2,
                         void* scratch, int32_t* inter, int32_t* counts, void* stream_) {
    if (n1 < 0 || n2 < 0 || HW < 0 || (HW > 0 && ((n1 > 0 && !masks1) || (n2 > 0 && !masks2))) ||
        (n1 + n2 > 0 && !counts) || (n1 > 0 && n2 > 0 && !inter) || (n1 + n2 > 0 && HW > 0 && !scratch)) {
        set_error("mask_pair_counts: bad arguments");
        return -1;
    }
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_MASK_STATS, s);
    int rc = launch_mask_pair_counts(n1, n2, HW, masks1, masks2, (uint32_t*)scratch, inter, counts, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("mask_pair_counts", 0, s);
    return 0;
}

int ogs_splat_footprint_votes(const ogs_footprint_inputs* in, int32_t* dominant_id, int32_t* dominant_weight,
                              int32_t* footprint_pixels, int32_t* q_max, int32_t* radii, int32_t* overflow_host,
                              void* stream_) {
    if (!in) { set_error("footprint_votes: inputs is NULL"); return -1; }
    if (in->P < 0 || in->W <= 0 || in->H <= 0) { set_error("footprint_votes: bad sizes P=%d W=%d H=%d", in->P, in->W, in->H); return -1; }
    if (overflow_host) *overflow_host = 0;
    const int P = in->P;
    if (P == 0) return 0;
    if (!in->means3D || !in->opacities || !in->scales || !in->rotations || !in->viewmatrix || !in->projmatrix || !in->sam_ids ||
        !dominant_id || !dominant_weight || !footprint_pixels || !q_max || !radii) {
        set_error("footprint_votes: all inputs and outputs must be set");
        return -1;
    }
    if (in->act_flags & ~(OGS_ACT_SCALE_EXP | OGS_ACT_ROT_NORMALIZE | OGS_ACT_OPACITY_SIGMOID)) {
        set_error("footprint_votes: only the scale / rotation / opacity activations apply");
        return -1;
    }
    const int gx = (in->W + 15) / 16, gy = (in->H + 15) / 16;
    if ((int64_t)gx * gy > 65535) { set_error("image too large: %d tiles (max 65535)", gx * gy); return -1; }
    cudaStream_t s = (cudaStream_t)stream_;
    int rc = ensure_pool();
    if (rc) return rc;
    ProfScope ps(PF_FOOTPRINT, s);
    const GeomLayout gl = GeomLayout::make(P, false, 0);
    const size_t pw = align_up((size_t)P * 4, 256);
    char* scratch = nullptr;
    OGS_CUDA(cudaMallocAsync((void**)&scratch, gl.total + 2 * pw + 256, s));
    const GeomPtrs g = GeomPtrs::from(scratch, gl);
    int32_t* d_over = (int32_t*)(scratch + gl.total + 2 * pw);
    cudaError_t e = cudaMemsetAsync(d_over, 0, 4, s);
    if (e != cudaSuccess) { cudaFreeAsync(scratch, s); return cuda_fail(e, "footprint_votes memset"); }
    PreprocessArgs pa;
    memset(&pa, 0, sizeof pa);
    pa.P = P; pa.D = 0; pa.M = 0; pa.W = in->W; pa.H = in->H;
    pa.act_flags = in->act_flags;
    pa.means3D = in->means3D; pa.scales = in->scales; pa.rotations = in->rotations; pa.opacities = in->opacities;
    pa.scale_modifier = in->scale_modifier; pa.tanfovx = in->tanfovx; pa.tanfovy = in->tanfovy;
    pa.view = in->viewmatrix; pa.proj = in->projmatrix;
    pa.radii = radii; pa.g = g;
    pa.depth_keys = (uint32_t*)(scratch + gl.total);
    pa.depth_vals = (uint32_t*)(scratch + gl.total + pw);
    rc = launch_preprocess_forward(pa, s);
    if (!rc) rc = launch_footprint_votes(P, in->W, in->H, g, in->sam_ids, in->empty_id, in->color, dominant_id, dominant_weight,
                                         footprint_pixels, q_max, d_over, s);
    int32_t over = 0;
    if (!rc) {
        e = cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "footprint_votes");
    }
    cudaFreeAsync(scratch, s);
    if (rc) return rc;
    if (overflow_host) *overflow_host = over;
    return 0;
}

int ogs_adam_step(int32_t n_tensors, const ogs_adam_tensor* tensors, float grad_scale, void* stream_) {
    if (n_tensors < 0 || (n_tensors > 0 && !tensors)) { set_error("adam_step: bad arguments"); return -1; }
    if (n_tensors == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream_;
    ProfScope ps(PF_ADAM, s);
    int rc = launch_adam_step(n_tensors, tensors, grad_scale, s);
    if (rc) return rc;
    OGS_KERNEL_CHECK("adam_step", 0, s);
    return 0;
}

}  // extern "C"
