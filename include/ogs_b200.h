/*
 * ogs_b200.h -- C ABI of libogs_b200.so, the B200 (sm_100a) hot path of OpenGaussian:
 * the tile-based differentiable Gaussian rasterizer and the k-means codebook kernels.
 *
 * Every entry point: plain pointers and sizes, no torch types, returns int
 * (0 = ok, < 0 = argument error, > 0 = cudaError_t), never throws.  ogs_last_error()
 * returns a thread-local message for the last non-zero return.
 * All pointers are DEVICE pointers unless the name ends in _host.  All kernels are enqueued on
 * `stream` (a cudaStream_t passed as void*).  Arrays are contiguous, row-major, fp32 unless said.
 *
 * What each entry point replaces in the reference (paths under /root/reference):
 *   ogs_raster_forward / ogs_raster_backward
 *       the external package `ashawkey_diff_gaussian_rasterization` that
 *       gaussian_renderer/__init__.py:15,55-70,104-163,203-225,327-345 and
 *       utils/sam_refinement_utils.py:21,347-403,431-486 import and call (upstream pybind
 *       symbols rasterize_gaussians / rasterize_gaussians_backward).  The C ABI additionally
 *       composites `n_extra` per-Gaussian feature channels (OpenGaussian's ins_feat) in the same
 *       pass, which replaces the 2x3-channel feature passes + silhouette pass of
 *       gaussian_renderer/__init__.py:125-163.
 *       Raw-parameter mode (act_flags / shs_rest) additionally folds the GaussianModel getters of
 *       scene/gaussian_model.py:122-169 and the (normalize(ins_feat)+1)/2 of
 *       gaussian_renderer/__init__.py:127 into the same kernels (SURVEY.md 8a9).
 *   ogs_raster_forward_subsets   the per-subset rasterizer forwards of the coarse-cluster and leaf loops of
 *                                gaussian_renderer/__init__.py:174-236,245-356 (one per cluster or leaf, each
 *                                with its own gather, preprocess, sorts and blend), for all subsets of a view
 *                                in one call: one preprocess and binning, then a stable per-tile partition by
 *                                subset and one blend over (tiles x subsets).
 *   ogs_raster_forward_subsets_state / ogs_raster_backward_subsets
 *                                the same with the reference's backward through those passes (the gradient-carrying
 *                                cluster pass of train.py:475-489): a forward that keeps its state and one blend
 *                                backward over (tiles x subsets).
 *   ogs_mark_visible             upstream GaussianRasterizer.markVisible (mark_visible symbol)
 *   ogs_raster_export            debug view of the geometry records and the sorted (tile|depth) keys
 *                                (upstream geomState / binningState)
 *   ogs_kmeans_assign            scene/kmeans_quantize.py:38-55 (get_dist) + :181-182,:200-201,
 *                                :223-224,:237-238 (argmin) fused with :82-87,:183-187,:202-205
 *                                (one-hot centroid sums and counts)
 *   ogs_kmeans_gather_st         scene/kmeans_quantize.py:273-275 (gather centres, straight-through)
 *   ogs_kmeans_assign_segmented, ogs_kmeans_finalize_fixed
 *                                scene/kmeans_quantize.py:196-214,233-238 (leaf mode) for all coarse clusters at once
 *   ogs_multimem_allreduce_f32   no reference counterpart: the view-parallel step's gradient all-reduce, reduced inside
 *                                the NVSwitch
 *   ogs_peer_*                   no reference counterpart (the reference is single-GPU): the all-reduce of the
 *                                sharded k-means' centroid partials over NVLink peer memory
 *   ogs_mask_pair_counts         utils/opengs_utlis.py:90-123 (calculate_iou)
 *   ogs_splat_footprint_votes    utils/sam_refinement_utils.py:902-913 (get_splat_id_and_weights, batched)
 *   ogs_adam_step                train.py:609 (gaussians.optimizer.step(), the torch.optim.Adam of
 *                                scene/gaussian_model.py:215-230)
 *   ogs_sam_masks                utils/opengs_utlis.py:125-182 (get_SAM_mask_and_feat: id map -> mask_id, one-hot masks, invalid_pix)
 *   ogs_mask_id_map              the inverse (one-hot masks -> id map) for mask sets that arrive as [M,H,W] tensors
 *   ogs_mask_mean_forward/backward, ogs_mask_var_forward
 *                                utils/opengs_utlis.py:240-283 (mask_feature_mean incl. return_var) and
 *                                :184-201 (pair_mask_feature_mean)
 *   ogs_cohesion_forward/backward
 *                                train.py:102-121 (cohesion_loss)
 *   ogs_separation_loss          train.py:123-155 (separation_loss)
 *   ogs_knn_segmented            pytorch3d.ops.knn_points, which gaussian_renderer/__init__.py's post_process calls once
 *                                per leaf (:315-322): here for all leaves of a view, or all clouds of a batch, at once
 */
#ifndef OGS_B200_H
#define OGS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OGS_ABI_VERSION 7
#define OGS_TILE 16
#define OGS_MAX_CHANNELS 16 /* 3 colour channels + n_extra <= OGS_MAX_CHANNELS */

/* Allocation callback (same role as upstream's resize functional): returns a device pointer to
 * `bytes` bytes (>= 256-byte aligned) owned by the caller, alive until the matching backward
 * has run.  `tag` names the buffer ("geom", "binning", "image"). */
typedef void* (*ogs_alloc_fn)(void* user, size_t bytes, const char* tag);

typedef struct ogs_raster_inputs {
    int32_t P;              /* number of Gaussians */
    int32_t sh_degree;      /* active SH degree (0..3) */
    int32_t M;              /* SH coefficients per Gaussian in `shs` (e.g. 16), 0 if shs == NULL */
    int32_t n_extra;        /* extra feature channels composited beside RGB (0 or e.g. 6) */
    int32_t W, H;           /* image size in pixels */
    float tanfovx, tanfovy;
    float scale_modifier;
    int32_t prefiltered;    /* kept for API parity; must be 0 */
    int32_t debug;          /* != 0: synchronise and check for errors after every kernel */
    const float* bg;        /* [3 + n_extra] background (device) */
    const float* viewmatrix;/* [16] raw floats of the transposed world->view tensor (device) */
    const float* projmatrix;/* [16] raw floats of the transposed full projection tensor (device) */
    const float* campos;    /* [3] (device) */
    const float* means3D;   /* [P,3] */
    const float* opacities; /* [P] */
    const float* shs;       /* [P,M,3] or NULL */
    const float* colors_precomp; /* [P,3] or NULL (exactly one of shs / colors_precomp) */
    const float* scales;    /* [P,3] or NULL */
    const float* rotations; /* [P,4] or NULL (scales+rotations, or cov3D_precomp) */
    const float* cov3D_precomp;  /* [P,6] or NULL */
    const float* extra;     /* [P,n_extra] or NULL when n_extra == 0 */
    /* ---- raw-parameter mode (SURVEY.md 8a9): the GaussianModel getters of
     * scene/gaussian_model.py:122-169 folded into preprocess.  act_flags == 0 and shs_rest == NULL:
     * every tensor is ACTIVATED, as the reference rasterizer receives them. ---- */
    int32_t act_flags;      /* OGS_ACT_* bits */
    int32_t defer_capacity_check; /* != 0: do not wait for this frame's duplicate count (see ogs_raster_capacity_check) */
    const float* shs_rest;  /* if != NULL: `shs` is _features_dc [P,1,3] and this is _features_rest [P,M-1,3]
                               (get_features' torch.cat is never materialised) */
} ogs_raster_inputs;

#define OGS_ACT_SCALE_EXP 1        /* scales are log-scales: exp() (get_scaling, :123-125) */
#define OGS_ACT_ROT_NORMALIZE 2    /* rotations are unnormalised: x / max(|x|, 1e-12) (get_rotation, :131-133) */
#define OGS_ACT_OPACITY_SIGMOID 4  /* opacities are logits: sigmoid() (get_opacity, :155-157) */
#define OGS_ACT_EXTRA_UNIT_HALF 8  /* extra is raw ins_feat: (normalize(x) + 1) / 2 (get_ins_feat :161-169 and
                                      gaussian_renderer/__init__.py:127) */

typedef struct ogs_raster_outputs {
    float* color;    /* [3 + n_extra, H, W] planar */
    float* depth;    /* [H, W]  sum depth*alpha*T (no background, not normalised) */
    float* alpha;    /* [H, W]  1 - T_final */
    int32_t* radii;  /* [P] */
} ogs_raster_outputs;

/* Opaque-to-the-caller state filled by forward and consumed by backward / export. */
typedef struct ogs_raster_state {
    void* geom;      /* per-Gaussian records (rec0/rec1 float4, rgb, clamped, tiles_touched) */
    void* binning;   /* point_list uint32[N] followed by ranges uint2[tiles] */
    void* image;     /* final_T float[H*W], n_contrib uint32[H*W] */
    int64_t num_rendered; /* N = number of (Gaussian, tile) duplicates */
    int64_t geom_bytes, binning_bytes, image_bytes;
    void* feat;      /* NULL, or the activated extra channels [P,n_extra] of THIS call when they do not live in `geom`
                        (ogs_raster_forward_cached: `geom` is shared by every call that reuses the view) */
} ogs_raster_state;

typedef struct ogs_raster_grads_in {
    const float* dL_dcolor;  /* [3 + n_extra, H, W]; with dL_dfeat set: [3, H, W] or NULL (= zero) */
    const float* dL_ddepth;  /* [H, W] or NULL */
    const float* dL_dalpha;  /* [H, W] or NULL */
    const float* dL_dfeat;   /* NULL, or [n_extra, H, W]: the gradient of the extra channels as a separate image (the two
                                images an autograd graph hands back for the colour and the feature map need not be
                                copied into one; Stage 1 has no colour gradient at all) */
} ogs_raster_grads_in;

/* Any output pointer may be NULL: that gradient is then not produced.  If all of the geometry
 * gradients (means3D, means2D, opacities, scales, rotations, cov3D, shs) are NULL the cheap
 * colour-only backward is used (OpenGaussian stages 1-2, train.py:431-436). */
typedef struct ogs_raster_grads_out {
    float* dL_dmeans3D;   /* [P,3] */
    float* dL_dmeans2D;   /* [P,3]  (x,y in NDC-scaled units, z = 0) */
    float* dL_dopacities; /* [P] */
    float* dL_dshs;       /* [P,M,3] */
    float* dL_dcolors_precomp; /* [P,3] */
    float* dL_dscales;    /* [P,3] */
    float* dL_drotations; /* [P,4] */
    float* dL_dcov3D;     /* [P,6] */
    float* dL_dextra;     /* [P,n_extra] */
    float* dL_dshs_rest;  /* [P,M-1,3] when shs_rest is used (dL_dshs is then [P,1,3]) */
    void* scratch;        /* ogs_raster_backward_scratch_floats(P, n_extra) floats of caller workspace */
    int32_t accumulate;   /* bit 0: the parameter-gradient outputs hold the gradients of earlier views and are ADDED to
                             (summing the views of a step costs one read of the old gradient instead of a separate
                             add pass); bit 1: dL_dmeans2D is added to as well (otherwise it is written) */
    int32_t reserved_;
} ogs_raster_grads_out;

int ogs_abi_version(void);
const char* ogs_last_error(void);

/* Optional device timing of the kernel families (CUDA events recorded on the launching stream).
 * Families: 0 preprocess_fwd, 1 depth_sort_scan, 2 emit, 3 tile_sort, 4 tile_ranges, 5 blend_fwd,
 * 6 blend_bwd, 7 preprocess_bwd, 8 kmeans_assign, 9 mask_stats, 10 adam, 11 footprint.  ogs_profile_read synchronises the recorded
 * events, writes the summed milliseconds and launch counts of the first n families and resets. */
#define OGS_PROFILE_FAMILIES 12
void ogs_profile_enable(int on);
int ogs_profile_read(float* ms_out_host, int32_t* launches_out_host, int32_t n);

int ogs_raster_forward(const ogs_raster_inputs* in, const ogs_raster_outputs* out,
                       ogs_alloc_fn alloc, void* alloc_user, ogs_raster_state* state, void* stream);

int ogs_raster_backward(const ogs_raster_inputs* in, const ogs_raster_state* state,
                        const ogs_raster_grads_in* gin, const ogs_raster_grads_out* gout,
                        void* stream);

/* Frozen-geometry view reuse.  From Stage 1 on OpenGaussian detaches xyz / scaling / rotation / opacity / SH
 * (train.py:431-436) and only `_ins_feat` trains, yet every render() call of the reference re-runs preprocess, the
 * duplicate emission and the 64-bit sort for a camera whose per-Gaussian records and tile lists cannot have changed.
 * ogs_raster_forward_cached composites a frame from the `geom` and `binning` buffers an EARLIER ogs_raster_forward
 * of the same camera and the same geometry inputs left in `cached` (the caller keeps them alive and decides validity:
 * opengaussian_b200/rasterizer.py::ViewCache keys on the tensors' storage and version counters; ~95 MB per 1 M-Gaussian
 * view, i.e. hundreds of training views of a scene fit the 180 GB of one B200).  Per call it allocates only the image
 * state (final_T, n_contrib: tag "image") and, in raw-parameter mode, the activated extra channels (tag "feat"),
 * recomputes those from in->extra, and runs the forward blend; `state` receives cached's geometry / binning pointers
 * plus the new buffers and is what ogs_raster_backward takes.  in->extra, in->colors_precomp and in->bg may differ
 * from the first call; everything else must be identical (not checked beyond the buffer sizes).  out->radii may be
 * NULL (the caller kept the first call's).  Results are bit-identical to a fresh ogs_raster_forward. */
int ogs_raster_forward_cached(const ogs_raster_inputs* in, const ogs_raster_outputs* out, ogs_alloc_fn alloc,
                              void* alloc_user, const ogs_raster_state* cached, ogs_raster_state* state, void* stream);
/* The leading bytes of a finished forward's `geom` and `binning` buffers that ogs_raster_forward_cached reads (the
 * forward sizes `binning` for an estimate above N and `geom` may end with the activated extra channels): what a cache
 * needs to keep. */
int ogs_raster_cached_bytes(const ogs_raster_inputs* in, int64_t num_rendered, int64_t* geom_bytes, int64_t* binning_bytes);

/* Deferred capacity check.  ogs_raster_forward sizes the (Gaussian, tile) buffers from a running estimate of N and, by
 * default, waits for the frame's real N before it returns -- the one host<->device synchronisation of a frame (the
 * reference's rasterizer has the same one: a blocking read of num_rendered).  With in->defer_capacity_check != 0 the
 * forward returns as soon as its kernels are queued (state->num_rendered = -1) and remembers the frame; the caller
 * MUST call ogs_raster_capacity_check from the same host thread, with the same current device, before it trusts
 * anything computed from those frames.  Returns 0: every deferred frame fitted; 1: at least one did not -- its outputs
 * are truncated, and so is everything derived from them: discard and redo the work (the estimate has been raised);
 * < 0: error (ogs_last_error).  A step-level transaction built on this: opengaussian_b200/dist.py::render_views_backward.
 * At most 64 frames can be pending per thread and device; further forwards fall back to the synchronous check. */
int ogs_raster_capacity_check(void);
/* The calling thread's running estimate of N on the current device (entries the next speculative forward is sized
 * for); new_hint >= 0 replaces it (0: forget -- the next forward waits for its count and re-seeds the estimate, e.g.
 * after switching scenes), new_hint < 0 only reads.  Returns the previous value. */
int64_t ogs_raster_capacity_hint(int64_t new_hint);

size_t ogs_raster_backward_scratch_floats(int32_t P, int32_t n_extra);

/* ---- all subsets of a view in one call (render()'s cluster / leaf passes) ----
 * subset int32 [P]: slot in [0, S) or -1 (not rendered; any value outside [0, S) is treated as -1).  Every slot's
 * images equal, bit for bit, an ogs_raster_forward of the rows with subset == slot (in increasing index order):
 * a pass over a subset sorts its rows stably by depth, then stably by tile, so its tile lists are the frame's lists
 * restricted to the subset, in the same order.  The call runs one preprocess and one binning over the Gaussians
 * that belong to a slot, partitions each tile's list stably by slot and blends all (tile, slot) pairs in one launch.
 * Inputs as for ogs_raster_forward, activated (act_flags == 0).  No radii; ogs_raster_forward_subsets keeps no state
 * (forward only), ogs_raster_forward_subsets_state below does.
 * Reads the frame's duplicate count synchronously (one host wait per call) and leaves the running capacity
 * estimate of ogs_raster_capacity_hint untouched.  Temporaries come from `alloc` (tags "geom", "binning") and the
 * stream-ordered pool.  1 <= S <= OGS_MAX_SUBSETS (the partition kernel keeps S counters in shared memory). */
#define OGS_MAX_SUBSETS 4096
typedef struct ogs_subset_outputs {
    float* color;   /* [S, 3 + n_extra, H, W] planar, background composited as in ogs_raster_forward */
    float* depth;   /* [S, H, W] or NULL */
    float* alpha;   /* [S, H, W] 1 - T_final */
} ogs_subset_outputs;
int ogs_raster_forward_subsets(const ogs_raster_inputs* in, const int32_t* subset, int32_t S,
                               const ogs_subset_outputs* out, ogs_alloc_fn alloc, void* alloc_user, void* stream);
/* ogs_raster_forward_subsets that also fills `state` for ogs_raster_backward_subsets: the same images, bit for bit, plus
 * an "image" buffer from `alloc` (final_T float[S][H][W], then n_contrib uint32[S][H][W]: S * H * W * 8 bytes) that
 * stays alive with "geom" and "binning" (which holds the frame's and the partitioned tile lists) until the backward
 * has run.  state->num_rendered = N of the frame. */
int ogs_raster_forward_subsets_state(const ogs_raster_inputs* in, const int32_t* subset, int32_t S,
                                     const ogs_subset_outputs* out, ogs_alloc_fn alloc, void* alloc_user,
                                     ogs_raster_state* state, void* stream);
/* Backward of ogs_raster_forward_subsets_state (same inputs, same S).  gin holds every slot's image gradients:
 * dL_dcolor [S, 3 + n_extra, H, W], or with dL_dfeat set [S, 3, H, W] or NULL; dL_dfeat [S, n_extra, H, W];
 * dL_ddepth, dL_dalpha [S, H, W] or NULL.  gout as for ogs_raster_backward, per Gaussian: the subsets are disjoint, so
 * each Gaussian's gradient is that of its own slot's images, and Gaussians of no slot get zero.  accumulate must be 0.
 * A state whose buffer sizes do not match P, S, W and H (a state of another call) is an argument error. */
int ogs_raster_backward_subsets(const ogs_raster_inputs* in, int32_t S, const ogs_raster_state* state,
                                const ogs_raster_grads_in* gin, const ogs_raster_grads_out* gout, void* stream);

int ogs_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, uint8_t* present,
                     void* stream);

/* Debug/export: geometry records and the sorted (tile << 32 | depth bits) keys rebuilt from the
 * state.  Any output may be NULL.  keys/point_list: [N]; ranges: [tiles][2] uint32;
 * xy [P,2]; depth [P]; conic_opacity [P,4]; rgb [P,3]; tiles_touched uint32 [P];
 * final_T [H*W]; n_contrib uint32 [H*W]. */
int ogs_raster_export(const ogs_raster_inputs* in, const ogs_raster_state* state, uint64_t* keys,
                      uint32_t* point_list, uint32_t* ranges, float* xy, float* depth,
                      float* conic_opacity, float* rgb, uint32_t* tiles_touched, float* final_T,
                      uint32_t* n_contrib, void* stream);

/* ---- k-means codebook ----
 * A point is the concatenation [a (Da floats) | b (Db floats) * scale_b]  (b may be NULL, Db = 0).
 * ids are int64 (the reference's torch.argmin dtype).  If select_ids != NULL only points with
 * select_ids[i] == selected take part (leaf mode); others keep ids_out[i] untouched.
 * sums [k, Da+Db] and counts [k] are ACCUMULATED into (caller zeroes them); either may be NULL
 * to skip the centroid-sum fusion (pure reassign). */
int ogs_kmeans_assign(int64_t N, const float* a, int32_t Da, const float* b, int32_t Db,
                      float scale_b, const float* centers, int32_t k, const int64_t* select_ids,
                      int64_t selected, int64_t id_offset, int64_t* ids_out, float* sums,
                      float* counts, void* stream);

/* out[i, :] = feat[i, :] - feat[i, :] + centers[ids[i], :Dout]  evaluated as the reference does
 * (x - x + c in fp32), i.e. the forward value of the straight-through quantised feature. */
int ogs_kmeans_gather_st(int64_t N, const float* feat, int32_t Dout, const float* centers,
                         int32_t Dc, const int64_t* ids, float* out, void* stream);

/* ---- fine level of the two-level codebook, ALL coarse clusters in one launch ----
 * Replaces k1 calls of the reference's leaf mode (scene/kmeans_quantize.py:196-206 assign + :82-87,:202-205
 * centroid sums, :233-238 reassign; one coarse cluster per call, driven by train.py:322-332).
 * Point i (a [N,D] floats) with coarse id c = coarse_ids[i] in [0, k1) competes among the rows
 * [c*k2, c*k2 + seg_k[c]) of seg_centers [>= k1*k2, D] (= leaf_centers; seg_k = iLeafSubNum, int32 [k1]) and gets
 * ids_out[i] = c*k2 + argmin (same fmaf chain and tie rule as ogs_kmeans_assign); points whose coarse id is outside
 * [0, k1) or whose cluster has seg_k <= 0 keep ids_out[i] untouched.
 * acc (int64 [k1*k2, D+1], ADDED to, caller zeroes; NULL = pure reassign): exact fixed-point centroid sums and
 * counts: acc[r][d] += llrint(x_d * 2^fix_bits), acc[r][D] += 1.  Integer sums do not depend on the summation
 * order, the grid or the sharding; the caller picks fix_bits so that max|x| * 2^fix_bits < 2^32 and
 * N * max|x| * 2^fix_bits < 2^63. */
int ogs_kmeans_assign_segmented(int64_t N, const float* a, int32_t D, const int64_t* coarse_ids,
                                const float* seg_centers, const int32_t* seg_k, int32_t k1, int32_t k2,
                                int64_t* ids_out, int64_t* acc, int32_t fix_bits, void* stream);

/* One Lloyd update of all rows from the exact sums with the reference's count bookkeeping
 * (scene/kmeans_quantize.py:167,186,208-214): counts_state[r] += acc[r][D] + eps_add;
 * centers[r, :] = (acc[r, :D] * 2^-fix_bits) / counts_state[r]; counts_state[r] = 0 where it exceeds 0.1. */
int ogs_kmeans_finalize_fixed(int32_t rows, int32_t D, const int64_t* acc, int32_t fix_bits, float eps_add,
                              float* counts_state, float* centers, void* stream);

/* ---- one whole Lloyd iteration in ONE launch (scene/kmeans_quantize.py:180-214 for the root mode, :196-214 for one
 * leaf call): assign every point (ogs_kmeans_assign's arithmetic and tie rule), accumulate the centroid sums and
 * counts, and -- in the LAST CTA to finish -- sum the per-CTA partials in a fixed order, all-reduce the [k, D+1] vector
 * over the peers' memory when `comm` is given (points sharded over GPUs; ogs_peer_* below), and update the centres the
 * way the reference does:  counts_state[j] += count_j + eps_add;  centers[j, :] = sum_j / counts_state[j];
 * counts_state[j] = 0 where it exceeds 0.1, for j < k_out (rows in [k, k_out) have no members and become 0).
 * centers [>= max(k, k_out), D] is read (rows < k) and updated IN PLACE; counts_state float [k_out].
 * workspace: ogs_kmeans_lloyd_workspace_bytes(k, D) bytes of device memory, zero-initialised ONCE by the caller and
 * reusable by consecutive calls on one stream.  An empty shard (N = 0) still takes part in the collective. */
typedef struct ogs_peer_comm ogs_peer_comm;
size_t ogs_kmeans_lloyd_workspace_bytes(int32_t k, int32_t D);
int ogs_kmeans_lloyd_pass(int64_t N, const float* a, int32_t Da, const float* b, int32_t Db, float scale_b,
                          float* centers, int32_t k, int32_t k_out, const int64_t* select_ids, int64_t selected,
                          int64_t id_offset, int64_t* ids_out, float* counts_state, float eps_add,
                          ogs_peer_comm* comm, void* workspace, void* stream);

/* The same for the fine level of ALL coarse clusters (ogs_kmeans_assign_segmented + the integer all-reduce +
 * ogs_kmeans_finalize_fixed in one launch): seg_centers [>= k1*k2, D] is read and updated in place, counts_state float
 * [k1*k2]; workspace: ogs_kmeans_lloyd_segmented_workspace_bytes(k1, k2, D) bytes, zero-initialised once. */
size_t ogs_kmeans_lloyd_segmented_workspace_bytes(int32_t k1, int32_t k2, int32_t D);
int ogs_kmeans_lloyd_pass_segmented(int64_t N, const float* a, int32_t D, const int64_t* coarse_ids, float* seg_centers,
                                    const int32_t* seg_k, int32_t k1, int32_t k2, int64_t* ids_out, int32_t fix_bits,
                                    float* counts_state, float eps_add, ogs_peer_comm* comm, void* workspace,
                                    void* stream);

/* ---- small all-reduce over NVLink peer memory in ONE kernel (SURVEY.md 8e: the [k, D+1] centroid partials of
 * the sharded k-means; the reference has no distributed code) ----
 * One communicator per process (one process per GPU, same node).  create: allocates this rank's inbox (2 parities x
 * world slots of max_bytes) and returns its 64-byte cudaIpc handle in handle_out; the caller exchanges the handles
 * (e.g. torch.distributed.all_gather_object) and passes all `world` of them, in rank order, to connect.
 * allreduce: in-place sum of buf [n] (dtype 0 = float32, 1 = int64) over the ranks, enqueued on `stream`; every rank
 * adds the contributions in rank order, so all ranks end with bit-identical results.  All ranks must issue the same
 * sequence of calls.  error: 1 if a call gave up waiting for a peer (~20 s) since the last check. */
int ogs_peer_comm_create(int32_t rank, int32_t world, int64_t max_bytes, ogs_peer_comm** out, void* handle_out);
int ogs_peer_comm_connect(ogs_peer_comm* comm, const void* all_handles);
int ogs_peer_allreduce(ogs_peer_comm* comm, void* buf, int64_t n, int32_t dtype, void* stream);
int ogs_peer_comm_error(ogs_peer_comm* comm, void* stream);
int ogs_peer_comm_destroy(ogs_peer_comm* comm);

/* ---- per-mask feature statistics and the Stage-1 cohesion loss (SURVEY.md section 8f rank 1) ----
 * Replace utils/opengs_utlis.py::mask_feature_mean (:240-283) and train.py::cohesion_loss (:102-121).
 * feat [C,H*W] float (C = 3 or 6), masks [M,H*W] bytes (torch.bool storage, non-zero = inside),
 * image_mask [H*W] float or NULL (the rendered silhouette, :253-255).  All device pointers.
 *   mean forward : sums [M,C] = sum_p feat * mask * image_mask, counts [M] = sum_p mask * image_mask
 *   mean backward: G [M,C] = dL/dmean / max(count,1), K [M] = (count > 1) ? sum_c G * mean : 0;
 *                  writes dfeat [C,H*W] and (if image_mask) dimg [H*W]
 *   var forward  : sq [M,C] = sum_p mask * (feat * image_mask - mean)^2
 *   cohesion fwd : dsum [M] = sum_p mask * ||feat[:,p] - mean[m]||_2, npix [M] = sum_p mask
 *   cohesion bwd : coef [M] = dL/dloss / (M * max(npix,1)); writes dfeat [C,H*W], dmean [M,C]
 * ids / ids_overlap (both NULL, or both set): the id map of ogs_mask_id_map for THESE masks.  SAM masks are a partition
 * of the image (get_SAM_mask_and_feat one-hot-encodes an id map, utils/opengs_utlis.py:144-148); when *ids_overlap == 0
 * the passes read 2 B per pixel from ids instead of M B from masks, with identical results up to summation order.  When
 * the flag is 1 (overlapping masks) ids is ignored.  The flag is read on the device: no host synchronisation. */
int ogs_mask_mean_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                          const float* image_mask, float* sums, float* counts, void* stream);
int ogs_mask_mean_backward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                           const float* image_mask, const float* G, const float* K, float* dfeat,
                           float* dimg, void* stream);
int ogs_mask_var_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                         const float* image_mask, const float* mean, float* sq, void* stream);
int ogs_cohesion_forward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                         const float* mean, float* dsum, float* npix, void* stream);
int ogs_cohesion_backward(int32_t M, int32_t C, int64_t HW, const float* feat, const uint8_t* masks, const int16_t* ids,
        const int32_t* ids_overlap,
                          const float* mean, const float* coef, float* dfeat, float* dmean,
                          void* stream);
/* get_SAM_mask_and_feat (utils/opengs_utlis.py:125-182) for one level of a view's SAM id map: level_ids [H*W] int32
 * (gt_sam_mask[level]), offset = previous level's largest id + 1 (0 at level 0).  Per pixel v = max(level_id - offset, -1):
 * mask_id [H*W] int64 = v + 1 (0 = invalid), invalid_pix [H*W] bytes = (v < 0), ids [H*W] int16 = v (the id map of
 * the passes above), masks [M,H*W] bytes = the one-hot expansion (mask m = pixels with v == m).  At most 32767 masks. */
int ogs_sam_masks(int32_t M, int64_t HW, const int32_t* level_ids, int32_t offset, int64_t* mask_id,
                  uint8_t* invalid_pix, int16_t* ids, uint8_t* masks, void* stream);
/* Per-pixel id map of a mask set: ids [H*W] int16 = the (last) mask that holds the pixel, -1 = none; *ids_overlap
 * (device int32) = 1 when some pixel lies in two or more masks, else 0.  At most 32767 masks. */
int ogs_mask_id_map(int32_t M, int64_t HW, const uint8_t* masks, int16_t* ids, int32_t* ids_overlap, void* stream);

/* ---- inter-mask contrastive loss of Stage 1: train.py:123-155 (separation_loss), value AND gradient in two launches ----
 * mean [N,C] (the per-mask feature means, N >= 2, C <= 16); small_weights != 0 is the reference's `iteration > 35000`
 * branch (weights below 0.9 become 0.1).  loss_out [1] receives sum_{i != j} w_ij / (|m_i - m_j|^2 + 1) / (N (N - 1)) with
 * w_ij = rank_ij / (N - 1) * 0.9 + 0.1, rank_ij = position of the term inside row i in ascending order (ties by column);
 * dmean [N,C] its gradient w.r.t. mean (the weights are constants, as in the reference's autograd graph).
 * scratch: N * N + N floats of device memory. */
int ogs_separation_loss(int32_t N, int32_t C, const float* mean, int32_t small_weights, float* scratch,
                        float* loss_out, float* dmean, void* stream);

/* ---- pairwise mask intersections: utils/opengs_utlis.py::calculate_iou (:90-123) ----
 * masks1 [n1,H*W], masks2 [n2,H*W] bytes (torch.bool storage, non-zero = inside), device pointers.
 * Writes inter int32 [n2,n1] = |masks2[j] & masks1[i]| and counts int32 [n1+n2] = pixel count of every row
 * (masks1 rows first); the union is counts[i] + counts[n1+j] - inter[j][i].  scratch: device buffer of
 * ogs_mask_iou_scratch_bytes(n1, n2, H*W) bytes (the bit-packed rows).  Outputs are zeroed by the call. */
int64_t ogs_mask_iou_scratch_bytes(int32_t n1, int32_t n2, int64_t HW);
int ogs_mask_pair_counts(int32_t n1, int32_t n2, int64_t HW, const uint8_t* masks1, const uint8_t* masks2,
                         void* scratch, int32_t* inter, int32_t* counts, void* stream);

/* ---- gradient all-reduce through the NVSwitch multicast mapping (SURVEY.md 8e: "Gaussian-parameter gradients are
 * allreduced"; the reference has no distributed code) ----
 * multicast_ptr: the MULTICAST address of a float32 buffer that every rank of the node maps at the same offset
 * (e.g. torch.distributed._symmetric_memory: rendezvous(...).multicast_ptr + byte offset), 16-byte aligned;
 * n_floats a multiple of 4.  Rank r reduces slice r with multimem.ld_reduce (the switch adds the ranks' copies in
 * flight) and writes the sums to every copy with multimem.st: afterwards all ranks hold the element-wise sum.
 * The caller must place a cross-rank barrier on the stream before the call (all gradients written) and after it
 * (all slices stored). */
int ogs_multimem_allreduce_f32(void* multicast_ptr, int64_t n_floats, int32_t rank, int32_t world, void* stream);

/* ---- batched single-splat footprints and their SAM-id votes: utils/sam_refinement_utils.py::
 * MultiViewSAMMaskRefiner.get_splat_id_and_weights (:902-913) = render_single_gaussian (:330-403, white
 * view-independent SH, black background) + fix_image (:143-176) + rgb_to_weight_map (:103-141) +
 * get_most_common_id_in_mask_weighted (:645-702), for P selected Gaussians in ONE camera ----
 * means3D [P,3], opacities [P], scales [P,3], rotations [P,4]: the (gathered) rows of the selected Gaussians,
 * activated unless act_flags says otherwise; camera as in ogs_raster_inputs; sam_ids int32 [H*W]; empty_id = the id
 * reported for an empty footprint (the reference's argmax over all-zero counts: the smallest id if that is
 * negative or the only one, else 0); color = the
 * splat's constant colour (0.28209479177387814f + 0.5f for the white SH).  Per splat i:
 *   dominant_id[i]      id with the largest sum of q = uint8(color * alpha * 255) under the footprint (ties: lowest)
 *   dominant_weight[i]  that sum (-1: see overflow);   footprint_pixels[i]  pixels with q > 0;   q_max[i]  largest q (the normaliser
 *   of rgb_to_weight_map);   radii[i]  as the rasterizer reports it (0 = culled).
 * *overflow_host receives the number of splats whose footprint touched more than 128 distinct ids (their
 * dominant id is then unreliable; the caller falls back for those).  Synchronises the stream. */
typedef struct ogs_footprint_inputs {
    int32_t P, W, H, act_flags;
    const float* means3D;
    const float* opacities;
    const float* scales;
    const float* rotations;
    float scale_modifier, tanfovx, tanfovy, color;
    const float* viewmatrix;
    const float* projmatrix;
    const int32_t* sam_ids;
    int32_t empty_id, reserved_;
} ogs_footprint_inputs;
int ogs_splat_footprint_votes(const ogs_footprint_inputs* in, int32_t* dominant_id, int32_t* dominant_weight,
                              int32_t* footprint_pixels, int32_t* q_max, int32_t* radii,
                              int32_t* overflow_host, void* stream);

/* ---- optimiser step: gaussians.optimizer.step() (train.py:609) for torch.optim.Adam(l, lr=0.0, eps=1e-15)
 * (scene/gaussian_model.py:215-230) -- all parameter tensors in one launch ----
 * One entry per parameter tensor (float32, contiguous, device pointers).  step_size = lr / (1 - beta1^t) and
 * bias_correction2_sqrt = sqrt(1 - beta2^t) for the tensor's step count t AFTER the increment, as
 * torch/optim/adam.py::_single_tensor_adam computes them; no weight decay, no amsgrad.  `tensors` is a HOST
 * array; grad_scale multiplies every gradient on load (1 for the reference's semantics). */
typedef struct ogs_adam_tensor {
    float* param;
    const float* grad;
    float* exp_avg;
    float* exp_avg_sq;
    int64_t n;
    float step_size;
    float bias_correction2_sqrt;
    float beta1;
    float beta2;
    float one_minus_beta1;           /* computed in double on the host, like torch's Python scalars */
    float one_minus_beta2;
    float eps;
    float reserved_;
} ogs_adam_tensor;
int ogs_adam_step(int32_t n_tensors, const ogs_adam_tensor* tensors, float grad_scale, void* stream);

/* ---- exact k-nearest neighbours within segments (pytorch3d.ops.knn_points; render()'s post_process for all leaves) ----
 * q [Q,3] queries, q_seg int32 [Q] the segment of each query; p [M,3] the candidates in segment order with CSR offsets
 * p_off int64 [S+1] (segment s = rows [p_off[s], p_off[s+1]) of p); k_seg int32 [S] the K of each segment (device: no
 * host read).  A query sees only its own segment's candidates, itself included when it is one of them.  Squared
 * distance = (dx*dx + dy*dy) + dz*dz in float32, every operation rounded on its own (no FMA).  The K used for a query
 * is min(k_seg, segment size), and with a neighbour list also min(., k_max); a query whose segment is outside [0, S) or
 * whose K is 0 gets 0 in kth_dist / dist_sum / dist_sumsq and no list entries.  Outputs, each may be NULL (not all):
 *   kth_dist [Q]         the K-th smallest squared distance
 *   dist_sum, dist_sumsq double [Q]: sum and sum of squares of the K smallest squared distances, accumulated in fp64
 *   nn_dist [Q,k_max], nn_idx int64 [Q,k_max] (both or neither): the K nearest ordered by (distance, index), the index
 *                        relative to the segment's first row; entries K..k_max-1 of a row are not written.
 * One warp per query: a radix select of the K-th distance (three passes over the segment), then one collect pass.
 * With a neighbour list and k_max > 1024 the call takes Q * k_max * 8 bytes from the stream-ordered pool. */
int ogs_knn_segmented(int64_t Q, const float* q, const int32_t* q_seg, int32_t S, const float* p, const int64_t* p_off,
                      const int32_t* k_seg, int32_t k_max, float* kth_dist, double* dist_sum, double* dist_sumsq,
                      float* nn_dist, int64_t* nn_idx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OGS_B200_H */
