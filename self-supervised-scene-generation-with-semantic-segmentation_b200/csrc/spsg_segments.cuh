// spsg_segments.cuh -- SPSG_FLAG_ALL_PIXELS: the backward's voxel -> pixel segments, built from the forward's per-pixel hit
// records instead of the fixed mapping3dto2d table.  Launched only with the flag; the default path never reaches these
// kernels.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// Every (voxel, view) row r the forward listed gets a segment of num[r] int32 slots in seg_pix, and every hit pixel of the
// batch writes its in-image index into the segment of its row.  seg_end[r] serves as the scatter's cursor: the allocation
// stores the segment's start, the scatter advances it by one per pixel, so that it ends at start + num[r] and the start is
// seg_end[r] - num[r] -- no second per-row array.  The sums do not depend on where a segment sits, so the allocation is
// one warp-aggregated atomicAdd; with SPSG_FLAG_DETERMINISTIC the entries of each segment are then sorted ascending:
//   * rows of <= kSegWarpSort pixels: one warp, the rank sort of canon_rows_kernel;
//   * rows of <= kSegSmemSort pixels: one CTA, a bitonic sort in shared memory;
//   * longer rows: one CTA compacts the row's image's hit records in raster order (at most W*H / kSegSmemSort such rows per
//     image, so that pass reads at most (W*H)^2 / kSegSmemSort hit records per image).
// ---------------------------------------------------------------------------------------------

constexpr int kSegSmemSort = 4096;
constexpr int kSegThreads = 512;

struct SegArgs {
    const int32_t *list_count;
    const int2 *list;        // (voxel, image) per (voxel, view) row that received a pixel (the forward's work list)
    const int32_t *num;      // mapping3dto2d_num
    const int32_t *hits;     // per-pixel hit voxel of every image (-1 = miss)
    int32_t *seg_end;        // [F*N]
    int32_t *seg_pix;        // [images * W * H]
    int32_t *counters;       // [0] segment allocator, [1] long rows; zeroed before seg_alloc_kernel
    int32_t *long_items;     // work-list items of rows longer than kSegWarpSort, or NULL (no sorting)
    int views;
    long long num_locs;
    unsigned image_pixels;   // W * H
    long long total_pixels;  // images * W * H
};

__device__ __forceinline__ size_t seg_row(const SegArgs &a, int2 e) {
    return (size_t)(e.y % a.views) * (size_t)a.num_locs + (size_t)e.x;
}

// One lane per listed row: segment starts from one atomicAdd per warp (warp-inclusive scan of the counts); with sorting,
// the rows a warp cannot sort are listed for seg_sort_long_kernel.
__global__ void __launch_bounds__(256) seg_alloc_kernel(const SegArgs a) {
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int count = *a.list_count;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    for (int base = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; base < count; base += warps * 32) {
        const int item = base + lane;
        size_t row = 0;
        int cnt = 0;
        if (item < count) {
            row = seg_row(a, a.list[item]);
            cnt = max(a.num[row], 0);
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += t;
        }
        int start = 0;
        if (lane == 31) start = atomicAdd(a.counters, incl);
        start = __shfl_sync(kFull, start, 31) + incl - cnt;
        if (item < count) a.seg_end[row] = start;
        if (a.long_items) {
            const bool is_long = item < count && cnt > kSegWarpSort;
            const unsigned m = __ballot_sync(kFull, is_long);
            int lb = 0;
            if (m && lane == 0) lb = atomicAdd(a.counters + 1, __popc(m));
            lb = __shfl_sync(kFull, lb, 0);
            if (is_long) a.long_items[lb + __popc(m & ((1u << lane) - 1u))] = item;
        }
    }
}

// One thread per pixel: the hit pixels of one row within a warp take consecutive slots from a single atomicAdd on the row's
// cursor (as the forward registers them).
__global__ void __launch_bounds__(256) seg_scatter_kernel(const SegArgs a) {
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long g0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); g0 < a.total_pixels; g0 += stride) {
        const long long g = g0 + lane;
        const int hit = g < a.total_pixels ? __ldg(a.hits + g) : -1;
        const unsigned img = (unsigned)(g / a.image_pixels);
        const int row = hit >= 0 ? (int)((img % (unsigned)a.views) * a.num_locs + hit) : -1;  // F*N < 2^31 (check_params)
        const unsigned peers = __match_any_sync(kFull, row);
        if (hit >= 0) {
            const int leader = __ffs(peers) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(a.seg_end + row, __popc(peers));
            base = __shfl_sync(peers, base, leader);
            a.seg_pix[base + __popc(peers & ((1u << lane) - 1u))] = (int)(g - (long long)img * a.image_pixels);
        }
    }
}

// SPSG_FLAG_DETERMINISTIC: one warp per listed row of at most kSegWarpSort pixels, sorted in place (rank of each entry =
// number of smaller entries; a row's pixel indices are distinct).
__global__ void __launch_bounds__(256) seg_sort_warp_kernel(const SegArgs a) {
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int count = *a.list_count;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    for (int item = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); item < count; item += warps) {
        const size_t row = seg_row(a, a.list[item]);
        const int cnt = a.num[row];
        if (cnt > kSegWarpSort) continue;
        int32_t *seg = a.seg_pix + (a.seg_end[row] - cnt);
        const int v0 = lane < cnt ? seg[lane] : INT_MAX, v1 = lane + 32 < cnt ? seg[lane + 32] : INT_MAX;
        int r0 = 0, r1 = 0;
        for (int j = 0; j < 32; j++) {
            const int u0 = __shfl_sync(kFull, v0, j), u1 = __shfl_sync(kFull, v1, j);
            r0 += (u0 < v0) + (u1 < v0);
            r1 += (u0 < v1) + (u1 < v1);
        }
        if (lane < cnt) seg[r0] = v0;  // every lane has read its entries: the shuffles above synchronise the warp
        if (lane + 32 < cnt) seg[r1] = v1;
    }
}

// SPSG_FLAG_DETERMINISTIC: one CTA per row longer than kSegWarpSort.  Up to kSegSmemSort entries: bitonic sort in shared
// memory (padded with INT_MAX to a power of two).  Longer: the row's pixels are exactly the pixels of its image whose hit
// record is its voxel, so the CTA rewrites the segment by compacting that image's records in raster order.
__global__ void __launch_bounds__(kSegThreads) seg_sort_long_kernel(const SegArgs a) {
    __shared__ int s[kSegSmemSort];
    __shared__ int s_warp[kSegThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int count = a.counters[1];
    for (int k = blockIdx.x; k < count; k += gridDim.x) {
        const int2 e = a.list[a.long_items[k]];
        const size_t row = seg_row(a, e);
        const int cnt = a.num[row];
        int32_t *seg = a.seg_pix + (a.seg_end[row] - cnt);
        if (cnt <= kSegSmemSort) {
            int n2 = kSegWarpSort * 2;
            while (n2 < cnt) n2 <<= 1;
            for (int i = tid; i < n2; i += kSegThreads) s[i] = i < cnt ? seg[i] : INT_MAX;
            __syncthreads();
            for (int len = 2; len <= n2; len <<= 1) {
                for (int j = len >> 1; j > 0; j >>= 1) {
                    for (int i = tid; i < n2; i += kSegThreads) {
                        const int p = i ^ j;
                        if (p > i) {
                            const int x = s[i], y = s[p];
                            if ((x > y) == ((i & len) == 0)) { s[i] = y; s[p] = x; }
                        }
                    }
                    __syncthreads();
                }
            }
            for (int i = tid; i < cnt; i += kSegThreads) seg[i] = s[i];
        } else {
            const int32_t *h = a.hits + (size_t)e.y * a.image_pixels;
            int written = 0;  // entries of earlier rounds (uniform across the CTA)
            for (unsigned p0 = 0; p0 < a.image_pixels; p0 += kSegThreads) {
                const unsigned p = p0 + tid;
                const bool mine = p < a.image_pixels && __ldg(h + p) == e.x;
                const unsigned m = __ballot_sync(0xffffffffu, mine);
                if (lane == 0) s_warp[warp] = __popc(m);
                __syncthreads();
                int before = 0, total = 0;
                for (int w = 0; w < kSegThreads / 32; w++) {
                    const int c = s_warp[w];
                    before += w < warp ? c : 0;
                    total += c;
                }
                if (mine) seg[written + before + __popc(m & ((1u << lane) - 1u))] = (int)p;
                written += total;
                __syncthreads();
            }
        }
        __syncthreads();
    }
}
