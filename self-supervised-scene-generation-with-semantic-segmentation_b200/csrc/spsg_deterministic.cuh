// spsg_deterministic.cuh -- SPSG_FLAG_DETERMINISTIC: canonical voxel -> pixel tables and loss sums in an order fixed by
// pixel position.  Launched only with the flag; the default path never reaches these kernels.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// canonical tables: row r keeps the min(num[r], P) smallest pixel indices registered to it, ascending
// ---------------------------------------------------------------------------------------------

constexpr int kCanonWarps = 8;
constexpr int kCanonSortMax = 64;  // rows of up to this many registered pixels are sorted in place by one warp (2 per lane)

struct CanonArgs {
    const int32_t *list_count;
    const int2 *list;        // (voxel, image) per (voxel, view) row that received a pixel (the forward's work list)
    const int32_t *num;      // mapping3dto2d_num
    int32_t *map;            // mapping3dto2d
    const int32_t *hits;     // per-pixel hit voxel of every image (-1 = miss)
    int max_pixels, views;
    long long num_locs;
    unsigned image_pixels;   // W * H
    long long total_pixels;  // images * W * H
};

// Rows whose table the forward could not hold completely (num > P), or that are longer than one warp sorts, are rebuilt
// from the per-pixel hit records instead of sorted.
__device__ __forceinline__ bool canon_rebuild(int cnt, int max_pixels) { return cnt > max_pixels || cnt > kCanonSortMax; }

// One warp per listed row: sort it in place (rank of each entry = number of smaller entries; the pixel indices of a row are
// distinct), or fill it with INT_MAX for canon_insert_kernel.
__global__ void __launch_bounds__(kCanonWarps * 32) canon_rows_kernel(const CanonArgs a) {
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int count = *a.list_count;
    for (int item = blockIdx.x * kCanonWarps + (threadIdx.x >> 5); item < count; item += gridDim.x * kCanonWarps) {
        const int2 e = a.list[item];
        const size_t row = (size_t)(e.y % a.views) * (size_t)a.num_locs + (size_t)e.x;
        const int cnt = a.num[row];
        int32_t *prow = a.map + row * a.max_pixels;
        if (canon_rebuild(cnt, a.max_pixels)) {
            for (int s = lane; s < a.max_pixels; s += 32) prow[s] = INT_MAX;
            continue;
        }
        const int v0 = lane < cnt ? prow[lane] : INT_MAX, v1 = lane + 32 < cnt ? prow[lane + 32] : INT_MAX;
        int r0 = 0, r1 = 0;
        for (int j = 0; j < 32; j++) {
            const int u0 = __shfl_sync(kFull, v0, j), u1 = __shfl_sync(kFull, v1, j);
            r0 += (u0 < v0) + (u1 < v0);
            r1 += (u0 < v1) + (u1 < v1);
        }
        if (lane < cnt) prow[r0] = v0;  // every lane has read its entries: the shuffles above synchronise the warp
        if (lane + 32 < cnt) prow[r1] = v1;
    }
}

// One thread per pixel of a rebuilt row: insert its index with a cascade of atomicMin over slots 0..P-1, carrying the larger
// value onward.  Slot s receives every inserted value except the s smallest, in whatever interleaving, so it ends up with
// the (s+1)-th smallest: the outcome does not depend on which pixel arrives first.  Slot values only ever decrease, so a
// slot already below the carried value (in any, possibly stale, read) would hand it straight back: skip its atomic.
__global__ void __launch_bounds__(256) canon_insert_kernel(const CanonArgs a) {
    for (long long g = (long long)blockIdx.x * 256 + threadIdx.x; g < a.total_pixels; g += (long long)gridDim.x * 256) {
        const int hit = __ldg(a.hits + g);
        if (hit < 0) continue;
        const unsigned img = (unsigned)(g / a.image_pixels);
        const size_t row = (size_t)(img % (unsigned)a.views) * (size_t)a.num_locs + (size_t)hit;
        if (!canon_rebuild(__ldg(a.num + row), a.max_pixels)) continue;
        int v = (int)(g - (long long)img * a.image_pixels);
        int32_t *prow = a.map + row * a.max_pixels;
        for (int s = 0; s < a.max_pixels; s++) {
            if (v > __ldcg(prow + s)) continue;
            const int old = atomicMin(prow + s, v);
            if (old == INT_MAX) break;  // the slot was free: nothing left to carry
            v = max(old, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// loss sums in pixel order: block b sums pixels [b * kDetLossPix, (b + 1) * kDetLossPix) in a fixed order into its own
// partial; the block that finishes last adds the partials in block order and finalises like the default path
// ---------------------------------------------------------------------------------------------

constexpr int kDetLossThreads = 256;
static_assert(kDetLossPix % kDetLossThreads == 0, "whole pixel rounds per block");

// a.loss.accum: kLossSlots * 8 doubles of scratch for the final stage; a.loss.done: a zeroed int32; partials: 8 doubles
// per block
__global__ void __launch_bounds__(kDetLossThreads) losses2d_det_kernel(const Losses2DArgs a, double *__restrict__ partials) {
    __shared__ float s_warp[kDetLossThreads / 32][6];
    __shared__ int s_last;
    float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    const long long p0 = (long long)blockIdx.x * kDetLossPix;
#pragma unroll 1
    for (int k = 0; k < kDetLossPix / kDetLossThreads; k++) {
        const long long p = p0 + k * kDetLossThreads + threadIdx.x;
        if (p < a.num_pixels) loss_terms_pixel(a, p, acc);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const float t = warp_sum(acc[k]);
        if (lane == 0) s_warp[warp][k] = t;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double s = 0.0;
        for (int w = 0; w < kDetLossThreads / 32; w++) s += (double)s_warp[w][threadIdx.x];
        partials[(size_t)blockIdx.x * 8 + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(a.loss.done, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x < kLossSlots) {
        // slot t = blocks t, t + kLossSlots, ... in block order; finalize_loss_warp then adds the slots in a fixed tree
        double t[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (unsigned b = threadIdx.x; b < gridDim.x; b += kLossSlots)
#pragma unroll
            for (int k = 0; k < 6; k++) t[k] += __ldcg(partials + (size_t)b * 8 + k);
#pragma unroll
        for (int k = 0; k < 6; k++) a.loss.accum[threadIdx.x * 8 + k] = t[k];
        __threadfence();
    }
    __syncthreads();
    if (warp == 0)
        finalize_loss_warp(a.loss.accum, a.loss.loss_out, a.loss.w_depth, a.loss.w_color, a.loss.w_sem,
                           a.loss.target_depth != nullptr, a.loss.target_color != nullptr, a.loss.target_label != nullptr,
                           lane);
}
