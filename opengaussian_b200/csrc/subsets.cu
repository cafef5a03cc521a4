// subsets.cu -- the two kernels that turn one binning of a frame into per-subset tile lists
// (ogs_raster_forward_subsets; render()'s no-grad cluster / leaf passes, reference
// gaussian_renderer/__init__.py:174-236,245-356).
//
// A subset pass of the reference gathers its rows in increasing index order, preprocesses them (per Gaussian,
// deterministic) and sorts them stably by depth, then stably by tile.  So each tile's list of a subset is exactly
// the full frame's list of that tile restricted to the subset, in the same order.  The entry point therefore runs ONE
// preprocess and ONE binning over the Gaussians that belong to some subset, then
//   subset_exclude_kernel   gives every Gaussian outside [0, S) the culled depth key (the first depth-sort pass drops
//                           it: no tiles_touched or record of it is read downstream, see binning.cu / radix.cu),
//   subset_partition_kernel stably partitions each tile's list by subset id,
// and the blend runs over the grid (tiles x S) on the (subset, tile) segments.
#include "common.cuh"

namespace ogs {

__global__ void subset_exclude_kernel(int P, int S, const int32_t* __restrict__ subset, uint32_t* __restrict__ depth_keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int32_t k = subset[i];
    if (k < 0 || k >= S) depth_keys[i] = 0xFFFFFFFFu;
}

int launch_subset_exclude(int P, int S, const int32_t* subset, uint32_t* depth_keys, cudaStream_t s) {
    if (P <= 0) return 0;
    subset_exclude_kernel<<<(P + 255) / 256, 256, 0, s>>>(P, S, subset, depth_keys);
    return 0;
}

// One CTA per tile.  Counts the tile's entries per subset (shared-memory histogram of S words), turns the counts into
// the segment bounds [ranges.x + exclusive prefix, + count) -- written to sub_ranges[s][tile] -- and scatters the
// entries to their segments in list order: warp 0 walks the list 32 entries at a time; lanes with the same subset
// find each other with __match_any_sync and take consecutive slots in lane order, so every segment keeps the order
// of the tile list (ties in depth stay in index order, as in a pass over the subset alone).
#define PART_THREADS 128
__global__ void __launch_bounds__(PART_THREADS) subset_partition_kernel(int tiles, int S, const uint2* __restrict__ ranges,
                                                                        const uint32_t* __restrict__ point_list,
                                                                        const int32_t* __restrict__ subset,
                                                                        uint32_t* __restrict__ out_list,
                                                                        uint2* __restrict__ sub_ranges) {
    extern __shared__ uint32_t s_cnt[];          // [S]: counts, then the next free slot of each segment
    __shared__ uint32_t s_warp[PART_THREADS / 32];
    const int t = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint2 r = ranges[t];
    for (int k = tid; k < S; k += PART_THREADS) s_cnt[k] = 0u;
    __syncthreads();
    for (uint32_t e = r.x + tid; e < r.y; e += PART_THREADS) atomicAdd(&s_cnt[subset[point_list[e]]], 1u);
    __syncthreads();

    // exclusive scan over the S counts: thread tid owns the contiguous block [lo, hi)
    const int per = (S + PART_THREADS - 1) / PART_THREADS;
    const int lo = min(S, tid * per), hi = min(S, lo + per);
    uint32_t sum = 0;
    for (int k = lo; k < hi; k++) sum += s_cnt[k];
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t run = r.x + incl - sum;
    for (int w = 0; w < warp; w++) run += s_warp[w];
    for (int k = lo; k < hi; k++) {
        const uint32_t c = s_cnt[k];
        sub_ranges[(size_t)k * tiles + t] = make_uint2(run, run + c);
        s_cnt[k] = run;
        run += c;
    }
    __syncthreads();

    if (warp != 0) return;
    const unsigned lt = (1u << lane) - 1u;
    for (uint32_t base = r.x; base < r.y; base += 32) {
        const uint32_t e = base + lane;
        const bool valid = e < r.y;
        uint32_t g = 0;
        int32_t k = -1;
        if (valid) { g = point_list[e]; k = subset[g]; }
        const unsigned peers = __match_any_sync(0xffffffffu, k);
        const uint32_t rank = __popc(peers & lt);
        uint32_t pos = 0;
        if (valid) {
            pos = s_cnt[k];
            out_list[pos + rank] = g;
        }
        __syncwarp();
        if (valid && rank == 0) s_cnt[k] = pos + __popc(peers);
        __syncwarp();
    }
}

int launch_subset_partition(int tiles, int S, const uint2* ranges, const uint32_t* point_list, const int32_t* subset,
                            uint32_t* out_list, uint2* sub_ranges, cudaStream_t s) {
    subset_partition_kernel<<<tiles, PART_THREADS, (size_t)S * sizeof(uint32_t), s>>>(tiles, S, ranges, point_list, subset,
                                                                                      out_list, sub_ranges);
    return 0;
}

}  // namespace ogs
