// knn.cu -- exact k-nearest-neighbour selection within segments (ogs_knn_segmented).
//
// One warp per query.  The K-th smallest squared distance t is found by a radix select over the float bits (squared
// distances are >= 0, so their bit patterns order like the values): three passes over the query's segment, each
// building a warp-private shared-memory histogram of the next 11 / 10 / 10 bits of the candidates that share the bits
// fixed so far, and a warp scan that picks the bucket holding rank K.  After the third pass t is exact and the number of
// candidates strictly below it is known, so a collect pass can produce the sums (the ties at t contribute (K - c) * t
// whichever of them is taken) and the neighbour list (the candidates below t, then the lowest-index ties at t), which a
// rank sort orders by (distance, index).  No per-query top-K buffer; any K <= segment size.
//
// Distances are recomputed from the coordinates in every pass (12 bytes per candidate; a segment's candidates are read
// by the consecutive queries of that segment, so they stay in L1 / L2).  The squared distance is
// ((dx*dx + dy*dy) + dz*dz) with every operation rounded on its own (the unit is built with --fmad=false as well), the
// direct form pytorch3d's knn_points uses.
#include "common.cuh"

namespace ogs {

#define KNN_WARPS 4
#define KNN_BINS 2048                     // first pass: bits 30..20; then 19..10 and 9..0
#define KNN_SMEM_PAIRS (KNN_BINS / 2)     // (distance, index) pairs a warp's histogram space holds for the sort

static __device__ __forceinline__ float knn_sqdist(float qx, float qy, float qz, const float* __restrict__ p, int64_t j) {
    const float dx = __fsub_rn(qx, __ldg(p + 3 * j));
    const float dy = __fsub_rn(qy, __ldg(p + 3 * j + 1));
    const float dz = __fsub_rn(qz, __ldg(p + 3 * j + 2));
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

struct KnnArgs {
    int64_t Q;
    const float* q;
    const int32_t* q_seg;
    int32_t S;
    const float* p;
    const int64_t* p_off;
    const int32_t* k_seg;
    int32_t k_max;
    float* kth;
    double* sum;
    double* sumsq;
    float* nn_dist;
    int64_t* nn_idx;
    float* tmp_dist;      // [Q, k_max] when k_max > KNN_SMEM_PAIRS and a neighbour list is wanted, else NULL
    int32_t* tmp_idx;
};

__global__ void __launch_bounds__(KNN_WARPS * 32) knn_select_kernel(KnnArgs a) {
    __shared__ uint32_t s_hist[KNN_WARPS][KNN_BINS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t qi = (int64_t)blockIdx.x * KNN_WARPS + warp;
    if (qi >= a.Q) return;                // whole warps leave; nothing below synchronises the block
    const bool want_nn = a.nn_dist != nullptr;
    const int s = a.q_seg[qi];
    int64_t base = 0, n = 0;
    int k = 0;
    if (s >= 0 && s < a.S) {
        base = a.p_off[s];
        n = a.p_off[s + 1] - base;
        k = a.k_seg[s];
    }
    if (want_nn && k > a.k_max) k = a.k_max;
    if ((int64_t)k > n) k = (int)n;
    if (k <= 0) {
        if (lane == 0) {
            if (a.kth) a.kth[qi] = 0.f;
            if (a.sum) a.sum[qi] = 0.0;
            if (a.sumsq) a.sumsq[qi] = 0.0;
        }
        return;
    }
    const float qx = a.q[3 * qi], qy = a.q[3 * qi + 1], qz = a.q[3 * qi + 2];
    const float* __restrict__ p = a.p + 3 * base;
    uint32_t* hist = s_hist[warp];

    // ---- radix select: prefix/pmask = the bits of t fixed so far, kk = rank of t among the candidates sharing them ----
    uint32_t prefix = 0, pmask = 0;
    int kk = k;
#pragma unroll 1
    for (int pass = 0; pass < 3; pass++) {
        const int shift = pass == 0 ? 20 : (pass == 1 ? 10 : 0);
        const int nb = pass == 0 ? 2048 : 1024;
        for (int b = lane; b < nb; b += 32) hist[b] = 0;
        __syncwarp();
        for (int64_t j = lane; j < n; j += 32) {
            const uint32_t u = __float_as_uint(knn_sqdist(qx, qy, qz, p, j));
            if ((u & pmask) == prefix) atomicAdd(&hist[(u >> shift) & (nb - 1)], 1u);
        }
        __syncwarp();
        const int per = nb >> 5;          // consecutive buckets owned by this lane
        uint32_t c = 0;
        for (int b = 0; b < per; b++) c += hist[lane * per + b];
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const uint32_t excl = incl - c;
        const unsigned owner = __ballot_sync(0xffffffffu, excl < (uint32_t)kk && (uint32_t)kk <= incl);
        const int src = __ffs(owner) - 1;
        uint32_t bucket = 0, below = 0;
        if (lane == src) {
            uint32_t run = excl;
            for (int b = 0; b < per; b++) {
                const uint32_t h = hist[lane * per + b];
                if (run + h >= (uint32_t)kk) { bucket = lane * per + b; break; }
                run += h;
            }
            below = run;
        }
        bucket = __shfl_sync(0xffffffffu, bucket, src);
        below = __shfl_sync(0xffffffffu, below, src);
        prefix |= bucket << shift;
        pmask |= (uint32_t)(nb - 1) << shift;
        kk -= (int)below;
        __syncwarp();                     // the histogram is reused (next pass, or the sort below)
    }
    const float t = __uint_as_float(prefix);
    const int n_less = k - kk;            // candidates with distance < t; kk of the ties at t complete the K

    if (lane == 0 && a.kth) a.kth[qi] = t;
    const bool want_sums = a.sum != nullptr || a.sumsq != nullptr;
    if (!want_sums && !want_nn) return;

    // ---- collect: sums in fp64 (fixed lane assignment and reduction order: reproducible), neighbour list by index ----
    float* cd = want_nn ? (a.tmp_dist ? a.tmp_dist + qi * a.k_max : reinterpret_cast<float*>(hist)) : nullptr;
    int32_t* ci = want_nn ? (a.tmp_idx ? a.tmp_idx + qi * a.k_max : reinterpret_cast<int32_t*>(hist) + KNN_SMEM_PAIRS)
                          : nullptr;
    double s1 = 0.0, s2 = 0.0;
    int n_lt = 0, n_eq = 0;
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int64_t j0 = 0; j0 < n; j0 += 32) {
        const int64_t j = j0 + lane;
        const float d = j < n ? knn_sqdist(qx, qy, qz, p, j) : 0.f;
        const bool lt = j < n && d < t;
        if (lt) {
            s1 += (double)d;
            s2 += (double)d * (double)d;
        }
        if (want_nn) {
            const bool eq = j < n && d == t;
            const unsigned bl = __ballot_sync(0xffffffffu, lt), be = __ballot_sync(0xffffffffu, eq);
            if (lt) { const int slot = n_lt + __popc(bl & lt_mask); cd[slot] = d; ci[slot] = (int32_t)j; }
            if (eq) {
                const int r = n_eq + __popc(be & lt_mask);
                if (r < kk) { cd[n_less + r] = d; ci[n_less + r] = (int32_t)j; }
            }
            n_lt += __popc(bl);
            n_eq += __popc(be);
        }
    }
    if (want_sums) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (lane == 0) {
            const double td = (double)t;
            if (a.sum) a.sum[qi] = s1 + (double)kk * td;
            if (a.sumsq) a.sumsq[qi] = s2 + (double)kk * td * td;
        }
    }
    if (!want_nn) return;
    __syncwarp();                         // orders the list writes before the reads below (shared or global)

    // ---- rank sort by (distance, index): all lanes read the same entry j (a broadcast) ----
    float* od = a.nn_dist + qi * a.k_max;
    int64_t* oi = a.nn_idx + qi * a.k_max;
    for (int i0 = 0; i0 < k; i0 += 32) {
        const int i = i0 + lane;
        const float di = i < k ? cd[i] : 0.f;
        const int32_t ii = i < k ? ci[i] : 0;
        int rank = 0;
        for (int j = 0; j < k; j++) {
            const float dj = cd[j];
            const int32_t ij = ci[j];
            rank += (dj < di) | ((dj == di) & (ij < ii));
        }
        if (i < k) { od[rank] = di; oi[rank] = ii; }
    }
}

int launch_knn_segmented(int64_t Q, const float* q, const int32_t* q_seg, int32_t S, const float* p, const int64_t* p_off,
                         const int32_t* k_seg, int32_t k_max, float* kth, double* sum, double* sumsq, float* nn_dist,
                         int64_t* nn_idx, cudaStream_t s) {
    KnnArgs a{Q, q, q_seg, S, p, p_off, k_seg, k_max, kth, sum, sumsq, nn_dist, nn_idx, nullptr, nullptr};
    AsyncScratch tmp(s);
    if (nn_dist && k_max > KNN_SMEM_PAIRS) {
        OGS_CUDA(tmp.alloc((size_t)Q * k_max * 8));
        a.tmp_dist = (float*)tmp.p;
        a.tmp_idx = (int32_t*)((char*)tmp.p + (size_t)Q * k_max * 4);
    }
    const int64_t blocks = (Q + KNN_WARPS - 1) / KNN_WARPS;
    knn_select_kernel<<<(unsigned)blocks, KNN_WARPS * 32, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "knn_select_kernel");
    return 0;
}

}  // namespace ogs
