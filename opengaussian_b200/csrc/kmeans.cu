// kmeans.cu -- codebook assign / centroid-sum / finalize / straight-through gather kernels.
//
// Replaces the PyTorch ops of scene/kmeans_quantize.py: torch.cdist + argmin (:38-55,:181-182,
// :200-201,:223-224,:237-238), one-hot @ feat centroid sums and counts (:82-87,:183-187,:202-205),
// centres = sums / counts (:208-214), gather + straight-through (:273-275).
//
// Arithmetic contract (shared with oracle/kmeans_oracle.c so that ids are bit-exact) -- the matmul
// form that torch.cdist itself uses for these sizes (||x||^2 is constant per point and dropped):
//   cn_j     = fold_d fmaf(c_jd, c_jd, acc), acc0 = 0, d ascending            (once per centre)
//   s_j      = fold_d fmaf(x_d, c_jd, acc),  acc0 = 0, d ascending
//   score_j  = fmaf(-2, s_j, cn_j)           ( = ||x - c_j||^2 - ||x||^2 )
//   id = lowest index of the minimum score (strict '<' scan) -- torch.argmin's tie rule.
// The contraction is D <= 16 deep: FMA cores, not tensor cores (BASELINE.json north_star).  One FMA
// per (point, centre, dimension): the FP32 pipe is the bound at k = 64 (packed FFMA2 occupies it
// for two cycles, so the direct (x-c)^2 form -- a subtract and an FMA -- would cost twice as much).
//
// Throughput: a thread owns FOUR points, held as two packed pairs; per (pair, centre, dimension)
// the work is one FFMA2 -- bit-identical to the scalar fmaf of the contract -- and one centre row
// ([c_0..c_D-1, cn], padded to float4s, broadcast LDS.128) is reused by all four points.
//
// Fusion: the centroid sums are accumulated in the SAME pass that assigns.  Each warp owns a
// private [k][D+1] accumulator in shared memory; lanes with equal ids (peer groups from one ballot per
// id bit) are summed by pointer jumping over shuffles and only the group's lowest lane updates the
// group's row, so every update is a plain LDS/FADD/STS (no shared or global atomics) and the result is
// deterministic.  Block partials go to a [grid][k][D+1] scratch
// that a second tiny kernel reduces in fixed order.
// HBM-bound at the fine level (k <= 10), FP32-bound at the coarse level (k = 64, D = 9).
#include <string.h>

#include "common.cuh"
#include "peer.cuh"

namespace ogs {

#ifndef KM_THREADS
#define KM_THREADS 256
#endif
#define KM_WARPS (KM_THREADS / 32)
#define KM_MAX_D 16
#ifndef KM_PPT
#define KM_PPT 4                              // points per thread (packed pairs)
#endif
#define KM_CTA_POINTS (KM_THREADS * KM_PPT)   // 1024
// Tile buffers in shared memory.  A thread copies its four points into registers before it scores them, so the tile
// buffer is free again as soon as every thread has done that: ONE buffer, refilled by the next tile's bulk copy while
// the current tile is scored, hides the copy just as well as two -- and at k = 64, D = 9 it takes the CTA from 95 KB to
// 59 KB of shared memory, i.e. from two to three CTAs (24 warps) per SM.  The kernel is bound by fixed-latency
// dependencies (ncu: `wait` 1.8 and `short_scoreboard` 1.2 stall cycles per issue at 4 warps per scheduler), so the
// extra warps are what it needs.
#ifndef KM_NBUF
#define KM_NBUF 1
#endif
#define KM_MAX_PER_SM 3                       // 80 registers x 256 threads: three CTAs fill the register file
static inline int km_ctas_per_sm(size_t smem) {
    int n = (int)((size_t)226 * 1024 / (smem + 1024));
    return n < 1 ? 1 : (n > KM_MAX_PER_SM ? KM_MAX_PER_SM : n);
}
#define KM_GROUP 16                           // CTAs per first-level group of the fused reduction

// ---- TMA bulk copy (global -> shared, completion on an mbarrier) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}

// Optional tail of the assign kernel: the LAST CTA to finish (atomic ticket) sums the per-CTA partials in CTA order,
// all-reduces the [k][D+1] vector over the peers' memory (peer.cuh) when the points are sharded over GPUs, and applies
// the reference's centre update -- so that one Lloyd iteration (scene/kmeans_quantize.py:180-214) is ONE launch:
//   counts_state[j] += count_j + eps_add;  centre_j = sum_j / counts_state[j];  counts_state[j] = 0 where > 0.1
// for j < k_out (rows at or beyond k have no members: sum 0 -> centre 0, as the reference's leaf mode rewrites them).
struct KmTail {
    int mode;                    // 0: off (partials are reduced by kmeans_reduce_partials_kernel)
    unsigned int* ticket;        // zero at launch; the last CTA resets it
    int has_peer;
    PeerDev peer;
    float* counts_state;         // [k_out]
    float eps_add;
    float* centers_out;          // [k_out][D]
    int k_out;
};

// Persistent CTAs walk 1024-point tiles.  A tile's rows (a: [1024][Da], b: [1024][Db], contiguous in
// global memory) are brought into shared memory by ONE cp.async.bulk per array, double-buffered on
// two mbarriers, so the next tile streams in while the current one is scored; the ragged last tile
// (or unaligned inputs) is staged by plain cooperative loads.
template <int D>
__global__ void __launch_bounds__(KM_THREADS) kmeans_assign_kernel(
    int64_t N, const float* __restrict__ a, int Da, const float* __restrict__ b, int Db, float scale_b,
    const float* __restrict__ centers, int k, const int64_t* __restrict__ select_ids, int64_t selected,
    int64_t id_offset, int64_t* __restrict__ ids_out, float* __restrict__ partials /* [grid][k][D+1] or NULL */,
    int bulk_ok, KmTail tail) {
    constexpr int DP = (D + 1 + 3) & ~3;      // centre row [c_0..c_D-1, ||c||^2] padded to whole float4s
    constexpr int ROW = D + 1;
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t s_bar[2];
    const int tile_floats = KM_CTA_POINTS * D;            // a rows then b rows of one tile
    float* s_pts = smem;                                  // [KM_NBUF][tile_floats]
    float* s_c = smem + KM_NBUF * (size_t)tile_floats;    // [k][DP]
    float* s_acc = s_c + (size_t)k * DP;                  // [KM_WARPS][k][D+1] (only when partials)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int j = threadIdx.x; j < k; j += KM_THREADS) {
        float cn = 0.f;
#pragma unroll
        for (int d = 0; d < D; d++) {
            const float c = centers[j * D + d];
            s_c[j * DP + d] = c;
            cn = __fmaf_rn(c, c, cn);
        }
        s_c[j * DP + D] = cn;
#pragma unroll
        for (int d = D + 1; d < DP; d++) s_c[j * DP + d] = 0.f;
    }
    if (partials)
        for (int e = threadIdx.x; e < KM_WARPS * k * ROW; e += KM_THREADS) s_acc[e] = 0.f;
    if (threadIdx.x == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    float* my_acc = s_acc + (size_t)warp * k * ROW;
    int id_bits = 0;
    while ((1 << id_bits) < k) id_bits++;

    const int64_t n_tiles = (N + KM_CTA_POINTS - 1) / KM_CTA_POINTS;
    // leaf mode (select_ids): only ~1/k1 of the points take part -- read their rows straight from global
    // memory instead of streaming every tile through shared memory
    const bool staged = select_ids == nullptr;
    auto tile_is_bulk = [&](int64_t t) { return staged && bulk_ok && (t + 1) * KM_CTA_POINTS <= N; };
    auto issue = [&](int64_t t, int buf) {   // one thread: arm the barrier and start both bulk copies
        float* dst = s_pts + (size_t)buf * tile_floats;
        const uint32_t ba = (uint32_t)(KM_CTA_POINTS * Da * sizeof(float)), bb = (uint32_t)(KM_CTA_POINTS * Db * sizeof(float));
        mbar_expect_tx(&s_bar[buf], ba + bb);
        bulk_g2s(dst, a + t * KM_CTA_POINTS * Da, ba, &s_bar[buf]);
        if (Db > 0) bulk_g2s(dst + KM_CTA_POINTS * Da, b + t * KM_CTA_POINTS * Db, bb, &s_bar[buf]);
    };
    uint32_t phases = 0u;   // bit b: parity the next wait on barrier b expects
    int buf = 0;
    if (threadIdx.x == 0 && (int64_t)blockIdx.x < n_tiles && tile_is_bulk(blockIdx.x)) issue(blockIdx.x, 0);

    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, buf ^= (KM_NBUF - 1)) {
        const int64_t tn = t + gridDim.x;
        if (KM_NBUF == 2 && threadIdx.x == 0 && tn < n_tiles && tile_is_bulk(tn)) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // buffer was last read through the generic proxy
            issue(tn, buf ^ 1);
        }
        const float* pa = s_pts + (size_t)buf * tile_floats;
        const float* pb = pa + KM_CTA_POINTS * Da;
        const int64_t tile_start = t * KM_CTA_POINTS;
        if (tile_is_bulk(t)) {
            mbar_wait(&s_bar[buf], (phases >> buf) & 1u);
            phases ^= 1u << buf;
        } else if (staged) {
            const int64_t rem = N - tile_start < KM_CTA_POINTS ? N - tile_start : KM_CTA_POINTS;
            float* wa = s_pts + (size_t)buf * tile_floats;
            for (int64_t e = threadIdx.x; e < rem * Da; e += KM_THREADS) wa[e] = __ldg(a + tile_start * Da + e);
            for (int64_t e = threadIdx.x; e < rem * Db; e += KM_THREADS) wa[KM_CTA_POINTS * Da + e] = __ldg(b + tile_start * Db + e);
            __syncthreads();
        }
        // warp w owns 128 consecutive points of the tile; slot q of lane l is local point 128 w + 32 q + l
        const int lbase = warp * (32 * KM_PPT) + lane;
        const int64_t base = tile_start + lbase;
        bool active[KM_PPT];
        float2 X[KM_PPT / 2][D];
#pragma unroll
        for (int q = 0; q < KM_PPT; q++) {
            const int64_t i = base + 32 * q;
            active[q] = i < N;
            if (active[q] && select_ids) active[q] = (select_ids[i] == selected);
            const int li = lbase + 32 * q;
#pragma unroll
            for (int d = 0; d < D; d++) {
                float v = 0.f;
                if (active[q]) {
                    if (staged) v = (d < Da) ? pa[li * Da + d] : __fmul_rn(pb[li * Db + (d - Da)], scale_b);
                    else v = (d < Da) ? __ldg(a + i * Da + d) : __fmul_rn(__ldg(b + i * Db + (d - Da)), scale_b);
                }
                if (q & 1) X[q >> 1][d].y = v; else X[q >> 1][d].x = v;
            }
        }
        if (KM_NBUF == 1 && staged) {
            __syncthreads();             // every thread holds its points in registers: the buffer can take the next tile
            if (threadIdx.x == 0 && tn < n_tiles && tile_is_bulk(tn)) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue(tn, 0);
            }
        }
        float2 best[KM_PPT / 2];
        int best_j[KM_PPT];
#pragma unroll
        for (int p = 0; p < KM_PPT / 2; p++) { best[p] = s2(INFINITY); best_j[2 * p] = best_j[2 * p + 1] = 0; }
#pragma unroll 4
        for (int j = 0; j < k; j++) {
            float c[DP];
#pragma unroll
            for (int q4 = 0; q4 < DP / 4; q4++) {
                const float4 tt = reinterpret_cast<const float4*>(s_c + j * DP)[q4];
                c[4 * q4] = tt.x; c[4 * q4 + 1] = tt.y; c[4 * q4 + 2] = tt.z; c[4 * q4 + 3] = tt.w;
            }
#pragma unroll
            for (int p = 0; p < KM_PPT / 2; p++) {
                float2 acc = s2(0.f);
#pragma unroll
                for (int d = 0; d < D; d++) acc = __ffma2_rn(X[p][d], s2(c[d]), acc);
                acc = __ffma2_rn(s2(-2.0f), acc, s2(c[D]));
                if (acc.x < best[p].x) { best[p].x = acc.x; best_j[2 * p] = j; }
                if (acc.y < best[p].y) { best[p].y = acc.y; best_j[2 * p + 1] = j; }
            }
        }
#pragma unroll
        for (int q = 0; q < KM_PPT; q++)
            if (active[q]) ids_out[base + 32 * q] = id_offset + best_j[q];
        if (partials) {
            // conflict-free, atomic-free accumulate
#pragma unroll
            for (int q = 0; q < KM_PPT; q++) {
                unsigned peers = __ballot_sync(0xffffffffu, active[q]);
                if (!active[q]) peers = ~peers;
                for (int bb = 0; bb < id_bits; bb++) {
                    const bool bit = (best_j[q] >> bb) & 1;
                    const unsigned m = __ballot_sync(0xffffffffu, bit);
                    peers &= bit ? m : ~m;
                }
                // Segmented sum by pointer jumping: every lane links to the next higher lane with the same id;
                // after ceil(log2(multiplicity)) rounds of  v += v[next]; next = next[next]  the lowest lane of
                // each group holds the group's sums and is the only one to touch the group's row -- plain
                // LDS/FADD/STS, no conflicts, a fixed summation order, and the cost grows with log2 of the
                // multiplicity (spatially coherent data puts whole warps into one cluster).
                const unsigned above = peers & ~((2u << lane) - 1u);
                int nxt = (active[q] && above) ? __ffs(above) - 1 : -1;
                const bool leader = active[q] && (peers & ((1u << lane) - 1u)) == 0u;
                const int mult = __reduce_max_sync(0xffffffffu, active[q] ? __popc(peers) : 0);
                float v[D];
#pragma unroll
                for (int d = 0; d < D; d++) v[d] = active[q] ? ((q & 1) ? X[q >> 1][d].y : X[q >> 1][d].x) : 0.f;
                for (int span = 1; span < mult; span <<= 1) {
                    const int src = nxt >= 0 ? nxt : lane;
#pragma unroll
                    for (int d = 0; d < D; d++) {
                        const float o = __shfl_sync(0xffffffffu, v[d], src);
                        if (nxt >= 0) v[d] += o;
                    }
                    const int n2 = __shfl_sync(0xffffffffu, nxt, src);
                    nxt = nxt >= 0 ? n2 : -1;
                }
                if (leader) {
                    float* row = my_acc + best_j[q] * ROW;
#pragma unroll
                    for (int d = 0; d < D; d++) row[d] += v[d];
                    row[D] += (float)__popc(peers);
                }
                __syncwarp();
            }
        }
        if (KM_NBUF == 2 && staged) __syncthreads();   // everyone is done with s_pts[buf] before it is refilled two tiles from now
    }
    if (partials) {
        __syncthreads();
        float* out = partials + (size_t)blockIdx.x * k * ROW;
        for (int e = threadIdx.x; e < k * ROW; e += KM_THREADS) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < KM_WARPS; w++) s += s_acc[(size_t)w * k * ROW + e];
            out[e] = s;
        }
    }
    if (tail.mode && partials) {
        // Two-level "last arriver" reduction, deterministic (fixed CTA order inside a group, fixed group order):
        // the last CTA of each group of KM_GROUP CTAs sums the group's partial tables, the last group to finish sums
        // the group tables -- the reduction runs on ~gridDim/KM_GROUP SMs instead of one.
        __shared__ int s_last;
        const int n_groups = (gridDim.x + KM_GROUP - 1) / KM_GROUP;
        const int grp = blockIdx.x / KM_GROUP;
        const int gsize = min(KM_GROUP, (int)gridDim.x - grp * KM_GROUP);
        float* gpart = partials + (size_t)gridDim.x * k * ROW;           // [n_groups][k][ROW]
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(tail.ticket + 1 + grp, 1u) == (unsigned)gsize - 1u) ? 1 : 0;
        __syncthreads();
        if (!s_last) return;
        __threadfence();
        for (int e = threadIdx.x; e < k * ROW; e += KM_THREADS) {
            float s = 0.f;
            for (int c = 0; c < gsize; c++) s += __ldcg(partials + (size_t)(grp * KM_GROUP + c) * k * ROW + e);
            gpart[(size_t)grp * k * ROW + e] = s;
        }
        if (threadIdx.x == 0) tail.ticket[1 + grp] = 0u;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(tail.ticket, 1u) == (unsigned)n_groups - 1u) ? 1 : 0;
        __syncthreads();
        if (!s_last) return;
        __threadfence();
        float* vec = s_acc;                                  // [k][ROW]: the per-warp accumulators are done with
        for (int e = threadIdx.x; e < k * ROW; e += KM_THREADS) {
            float s = 0.f;
            for (int g2 = 0; g2 < n_groups; g2++) s += __ldcg(gpart + (size_t)g2 * k * ROW + e);
            vec[e] = s;
        }
        __syncthreads();
        bool ok = true;
        if (tail.has_peer) ok = peer_allreduce_cta<float>(tail.peer, vec, k * ROW);
        if (ok) {
            for (int e = threadIdx.x; e < tail.k_out * D; e += KM_THREADS) {
                const int j = e / D, d = e - j * D;
                const float cnt = __fadd_rn(tail.counts_state[j], __fadd_rn(j < k ? vec[j * ROW + D] : 0.f, tail.eps_add));
                tail.centers_out[e] = __fdiv_rn(j < k ? vec[j * ROW + d] : 0.f, cnt);
            }
            __syncthreads();
            for (int j = threadIdx.x; j < tail.k_out; j += KM_THREADS) {
                const float cnt = __fadd_rn(tail.counts_state[j], __fadd_rn(j < k ? vec[j * ROW + D] : 0.f, tail.eps_add));
                tail.counts_state[j] = cnt > 0.1f ? 0.f : cnt;
            }
        }
        if (threadIdx.x == 0) *tail.ticket = 0u;
    }
}

__global__ void kmeans_reduce_partials_kernel(int nblocks, int k, int D, const float* __restrict__ partials,
                                              float* __restrict__ sums, float* __restrict__ counts) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int ROW = D + 1;
    if (e >= k * ROW) return;
    float s = 0.f;
    for (int bk = 0; bk < nblocks; bk++) s += partials[(size_t)bk * k * ROW + e];
    const int j = e / ROW, d = e - j * ROW;
    if (d < D) { if (sums) sums[j * D + d] += s; }
    else if (counts) counts[j] += s;
}

// The dynamic-shared-memory attribute belongs to the KERNEL (per device): ONE cache per instantiation, shared by every
// launcher of that kernel, and only ever raised -- two launchers with private caches would lower each other's setting.
template <int D>
static int ensure_assign_smem(size_t smem) {
    static std::atomic<size_t> attr[OGS_MAX_DEVICES];        // per device: largest size the attribute was raised to
    std::atomic<size_t>& at = attr[current_device()];
    if (smem > 48 * 1024 && smem > at.load(std::memory_order_relaxed)) {
        OGS_CUDA(cudaFuncSetAttribute(kmeans_assign_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        at.store(smem, std::memory_order_relaxed);
    }
    return 0;
}

template <int D>
static int launch_assign_d(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b,
                           const float* centers, int k, const int64_t* select_ids, int64_t selected,
                           int64_t id_offset, int64_t* ids_out, float* sums, float* counts, cudaStream_t s) {
    const bool fuse = (sums != nullptr) || (counts != nullptr);
    size_t smem = (size_t)KM_NBUF * KM_CTA_POINTS * D * sizeof(float) + (size_t)k * ((D + 1 + 3) & ~3) * sizeof(float);
    if (fuse) smem += (size_t)KM_WARPS * k * (D + 1) * sizeof(float);
    if (smem > 220 * 1024) { set_error("kmeans_assign: k=%d D=%d needs %zu B shared memory", k, D, smem); return -5; }
    { const int rc_attr = ensure_assign_smem<D>(smem); if (rc_attr) return rc_attr; }
    // bulk copies need 16-byte aligned sources and sizes: tile strides are multiples of 4096 bytes
    const int bulk_ok = (((uintptr_t)a & 15) == 0 && (Db == 0 || ((uintptr_t)b & 15) == 0)) ? 1 : 0;
    int64_t want = (N + KM_CTA_POINTS - 1) / KM_CTA_POINTS;
    const int per_sm = km_ctas_per_sm(smem);
    int grid = (int)(want < (int64_t)OGS_NUM_SMS * per_sm ? want : (int64_t)OGS_NUM_SMS * per_sm);
    if (grid < 1) grid = 1;
    float* partials = nullptr;
    if (fuse) OGS_CUDA(cudaMallocAsync((void**)&partials, (size_t)grid * k * (D + 1) * sizeof(float), s));
    KmTail tail;
    memset(&tail, 0, sizeof tail);
    kmeans_assign_kernel<D><<<grid, KM_THREADS, smem, s>>>(N, a, Da, b, Db, scale_b, centers, k, select_ids, selected,
                                                           id_offset, ids_out, partials, bulk_ok, tail);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && fuse) {
        const int tot = k * (D + 1);
        kmeans_reduce_partials_kernel<<<(tot + 127) / 128, 128, 0, s>>>(grid, k, D, partials, sums, counts);
        e = cudaGetLastError();
    }
    if (partials) cudaFreeAsync(partials, s);
    if (e != cudaSuccess) return cuda_fail(e, "kmeans_assign");
    return 0;
}

int launch_kmeans_assign(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b,
                         const float* centers, int k, const int64_t* select_ids, int64_t selected, int64_t id_offset,
                         int64_t* ids_out, float* sums, float* counts, cudaStream_t s) {
    const int D = Da + Db;
#define OGS_KM_CASE(DD) case DD: return launch_assign_d<DD>(N, a, Da, b, Db, scale_b, centers, k, select_ids, selected, id_offset, ids_out, sums, counts, s);
    switch (D) {
        OGS_KM_CASE(1) OGS_KM_CASE(2) OGS_KM_CASE(3) OGS_KM_CASE(4) OGS_KM_CASE(5) OGS_KM_CASE(6) OGS_KM_CASE(7)
        OGS_KM_CASE(8) OGS_KM_CASE(9) OGS_KM_CASE(10) OGS_KM_CASE(11) OGS_KM_CASE(12) OGS_KM_CASE(13)
        OGS_KM_CASE(14) OGS_KM_CASE(15) OGS_KM_CASE(16)
    }
#undef OGS_KM_CASE
    set_error("kmeans_assign: unsupported point dimension %d (1..16)", D);
    return -5;
}

// ---- one Lloyd iteration in one launch (assign + centroid sums + [peer all-reduce] + centre update) ----
// workspace (caller-owned, zero-initialised once): [tickets: 256 B][partials: grid_max * k * (D+1) floats][group tables]
size_t kmeans_lloyd_workspace_bytes(int k, int D) {
    const size_t grid_max = (size_t)OGS_NUM_SMS * KM_MAX_PER_SM;
    return 256 + (grid_max + (grid_max + KM_GROUP - 1) / KM_GROUP) * k * (D + 1) * sizeof(float);
}

template <int D>
static int launch_lloyd_d(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b, float* centers, int k,
                          int k_out, const int64_t* select_ids, int64_t selected, int64_t id_offset, int64_t* ids_out,
                          float* counts_state, float eps_add, const ogs_peer_comm* comm, void* workspace, cudaStream_t s) {
    size_t smem = (size_t)KM_NBUF * KM_CTA_POINTS * D * sizeof(float) + (size_t)k * ((D + 1 + 3) & ~3) * sizeof(float);
    smem += (size_t)KM_WARPS * k * (D + 1) * sizeof(float);
    if (smem > 220 * 1024) { set_error("kmeans_lloyd_pass: k=%d D=%d needs %zu B shared memory", k, D, smem); return -5; }
    if (comm && (size_t)k * (D + 1) * sizeof(float) > peer_comm_slot_bytes(comm)) {
        set_error("kmeans_lloyd_pass: the communicator's slots are too small for k=%d D=%d", k, D);
        return -1;
    }
    { const int rc_attr = ensure_assign_smem<D>(smem); if (rc_attr) return rc_attr; }
    const int bulk_ok = (((uintptr_t)a & 15) == 0 && (Db == 0 || ((uintptr_t)b & 15) == 0)) ? 1 : 0;
    int64_t want = (N + KM_CTA_POINTS - 1) / KM_CTA_POINTS;
    const int per_sm = km_ctas_per_sm(smem);
    int grid = (int)(want < (int64_t)OGS_NUM_SMS * per_sm ? want : (int64_t)OGS_NUM_SMS * per_sm);
    if (grid < 1) grid = 1;                          // an empty shard still takes part in the collective
    KmTail tail;
    memset(&tail, 0, sizeof tail);
    tail.mode = 1;
    tail.ticket = (unsigned int*)workspace;
    tail.has_peer = comm ? 1 : 0;
    if (comm) tail.peer = *peer_comm_dev(comm);
    tail.counts_state = counts_state; tail.eps_add = eps_add; tail.centers_out = centers; tail.k_out = k_out;
    float* partials = (float*)((char*)workspace + 256);
    kmeans_assign_kernel<D><<<grid, KM_THREADS, smem, s>>>(N, a, Da, b, Db, scale_b, centers, k, select_ids, selected,
                                                           id_offset, ids_out, partials, bulk_ok, tail);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "kmeans_lloyd_pass");
    return 0;
}

int launch_kmeans_lloyd_pass(int64_t N, const float* a, int Da, const float* b, int Db, float scale_b, float* centers, int k,
                             int k_out, const int64_t* select_ids, int64_t selected, int64_t id_offset, int64_t* ids_out,
                             float* counts_state, float eps_add, const ogs_peer_comm* comm, void* workspace, cudaStream_t s) {
    const int D = Da + Db;
#define OGS_KL_CASE(DD) case DD: return launch_lloyd_d<DD>(N, a, Da, b, Db, scale_b, centers, k, k_out, select_ids, selected, id_offset, ids_out, counts_state, eps_add, comm, workspace, s);
    switch (D) {
        OGS_KL_CASE(1) OGS_KL_CASE(2) OGS_KL_CASE(3) OGS_KL_CASE(4) OGS_KL_CASE(5) OGS_KL_CASE(6) OGS_KL_CASE(7)
        OGS_KL_CASE(8) OGS_KL_CASE(9) OGS_KL_CASE(10) OGS_KL_CASE(11) OGS_KL_CASE(12) OGS_KL_CASE(13)
        OGS_KL_CASE(14) OGS_KL_CASE(15) OGS_KL_CASE(16)
    }
#undef OGS_KL_CASE
    set_error("kmeans_lloyd_pass: unsupported point dimension %d (1..16)", D);
    return -5;
}

__global__ void kmeans_gather_st_kernel(int64_t N, const float* __restrict__ feat, int Dout,
                                        const float* __restrict__ centers, int Dc, const int64_t* __restrict__ ids,
                                        float* __restrict__ out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N * Dout) return;
    const int64_t i = e / Dout;
    const int d = (int)(e - i * Dout);
    const float f = feat[e];
    out[e] = __fadd_rn(__fsub_rn(f, f), __ldg(centers + ids[i] * Dc + d));
}

int launch_kmeans_gather_st(int64_t N, const float* feat, int Dout, const float* centers, int Dc, const int64_t* ids,
                            float* out, cudaStream_t s) {
    const int64_t tot = N * Dout;
    if (tot <= 0) return 0;
    kmeans_gather_st_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(N, feat, Dout, centers, Dc, ids, out);
    return 0;
}

}  // namespace ogs
