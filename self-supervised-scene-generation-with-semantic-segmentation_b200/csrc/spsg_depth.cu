// spsg_depth.cu -- sm_100a kernels + C ABI for the depth-frame utilities of the training step: the reference's second
// CUDA extension, torch/utils/depth_utils (depth_utils_cuda_kernel.cu, cited as dkernel.cu:<line>), which turns the
// sensor depth frame into target normals and fills its holes in place (Depth2Normals, depth_utils.py:66-100).
// SURVEY.md section 8(f) rank 3.
//
// Same arithmetic as the reference, expression by expression (float / double mix of the two Gaussians included), so that
// the results can be compared bit for bit with the compiled reference extension.  What changes is the shape of the work:
//   * depth -> camera space -> normals is one kernel (the camera-space image is still written: callers can read it);
//   * the median hole fill selects the reference's order statistic by a warp-wide radix select instead of a 121-element
//     bubble sort in local memory, and only for hole pixels;
//   * the fill iterations terminate on the device: every fill pass counts the holes it leaves, so the whole pipeline is
//     enqueued without a host round trip per iteration (the reference synchronises on `(depth == 0).any()` up to 21
//     times, depth_utils.py:86-92);
//   * the fill rounds and the normals are ONE cooperative launch (fill_rounds_normals_kernel): passes of a grid-resident
//     kernel separated by grid barriers, and the fill loop simply ends when a round leaves no hole (the launch-per-pass
//     form, with passes that return at once, remains for devices without cooperative launch).
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <mutex>

#include "spsg_internal.h"
#include "spsg_raycast.h"

namespace {

constexpr int kFillRadius = 5;  // STRUCTURE_SIZE, dkernel.cu:88
constexpr int kFillDiameter = 2 * kFillRadius + 1;
constexpr int kFillCells = kFillDiameter * kFillDiameter;

__device__ __forceinline__ bool depth_valid(float d) { return d != -CUDART_INF_F && d != 0.0f; }

constexpr int kTableRadius = 8;  // spatial Gaussian table: windows up to 17x17 (the training step uses 9x9)
constexpr int kTableDiameter = 2 * kTableRadius + 1;

// gaussD (dkernel.cu:16-19) of every window offset, once per CTA: the expression of the per-tap form below, so the
// values are the same floats.
__device__ __forceinline__ void spatial_table_fill(float *table, float sigmaD, int radius) {
    if (radius > kTableRadius) return;
    for (int e = threadIdx.x; e < kTableDiameter * kTableDiameter; e += blockDim.x) {
        const int dx = e / kTableDiameter - kTableRadius, dy = e % kTableDiameter - kTableRadius;
        table[e] = exp(-((dx * dx + dy * dy) / (2.0f * sigmaD * sigmaD)));
    }
}

// bilateral_filter_floatmap_kernel (dkernel.cu:41-86) for the 32x8-pixel tile (bx, by) of frame bz; also counts the holes
// of the input (zero pixels) into *holes.
__device__ __forceinline__ void bilateral_tile(const float *__restrict__ in, float *__restrict__ out, int width, int height,
                                               float sigmaD, float sigmaR, int32_t *holes, int bx, int by, int bz,
                                               const float *table) {
    const int x = bx * 32 + (threadIdx.x & 31), y = by * 8 + (threadIdx.x >> 5);
    const float *img = in + (size_t)bz * width * height;
    const bool inside = x < width && y < height;
    float result = 0.0f;
    bool hole = false;
    if (inside) {
        const int radius = (int)ceil(2.0 * sigmaD);  // dkernel.cu:56
        const bool tabled = radius <= kTableRadius;
        const float center = img[y * width + x];
        hole = center == 0.0f;
        if (depth_valid(center)) {
            float sum = 0.0f, sum_weight = 0.0f;
            for (int m = x - radius; m <= x + radius; m++)
                for (int n = y - radius; n <= y + radius; n++)
                    if (m >= 0 && n >= 0 && m < width && n < height) {
                        const float cur = img[n * width + m];
                        if (depth_valid(cur)) {
                            const int dx = m - x, dy = n - y;
                            const float dist = cur - center;
                            // gaussD in float, gaussR through double, exactly as written at dkernel.cu:16-29
                            const float gd = tabled ? table[(dx + kTableRadius) * kTableDiameter + dy + kTableRadius]
                                                    : (float)exp(-((dx * dx + dy * dy) / (2.0f * sigmaD * sigmaD)));
                            const float gr = exp(-(dist * dist) / (2.0 * sigmaR * sigmaR));
                            const float weight = gd * gr;
                            sum_weight += weight;
                            sum += weight * cur;
                        }
                    }
            if (sum_weight > 0.0f) result = sum / sum_weight;
        }
        out[(size_t)bz * width * height + y * width + x] = result;
    }
    if (holes) {
        const unsigned m = __ballot_sync(0xffffffffu, hole);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(holes, __popc(m));
    }
}

__global__ void __launch_bounds__(256) bilateral_kernel(const float *__restrict__ in, float *__restrict__ out, int width,
                                                        int height, float sigmaD, float sigmaR, int32_t *holes) {
    __shared__ float s_table[kTableDiameter * kTableDiameter];
    spatial_table_fill(s_table, sigmaD, (int)ceil(2.0 * sigmaD));
    __syncthreads();
    bilateral_tile(in, out, width, height, sigmaD, sigmaR, holes, blockIdx.x, blockIdx.y, blockIdx.z, s_table);
}

// median_fill_depthmap_kernel (dkernel.cu:89-140).  Valid pixels are copied.  A hole takes the order statistic the
// reference reads out of its sorted 11x11 window: the ((n+1)/2)-th smallest (0-based) of the n valid values, each
// quantised to millimetres as (int)(1000 d + 0.5f).  (For n < 2 the reference indexes past its array; here: 0.)
// The reference bubble-sorts 121 values per hole in one thread; here a warp (32 pixels of a row) handles its holes one
// after the other TOGETHER: the lanes hold the window (4 values each) and find the wanted order statistic by a radix
// select over the bits the window's values differ in -- per bit four votes and a count; a window whose depths span less
// than a metre resolves in ten rounds, ~200 warp instructions per hole instead of ~15 000 steps in the thread that owns
// it.
__device__ __forceinline__ void median_fill_tile(const float *__restrict__ in, float *__restrict__ out, int width, int height,
                                                 int32_t *holes_out, int bx, int by, int bz) {
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = bx * 32 + lane, y = by * 8 + warp;
    const float *img = in + (size_t)bz * width * height;
    const bool inside = x < width && y < height;
    const float cur = inside ? img[y * width + x] : 1.0f;
    float result = cur;
    unsigned todo = __ballot_sync(kFull, inside && !depth_valid(cur));
    while (todo) {
        const int h = __ffs(todo) - 1;  // the hole lane served now: pixel (hx, y)
        todo &= todo - 1;
        const int hx = bx * 32 + h;
        unsigned key[4];  // quantised depth, sign bit flipped: unsigned order == the reference's int order
        bool alive[4];
        int n = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int e = lane + 32 * r;  // window element (row i, column j), row-major like the reference
            int q = 0;
            bool valid = false;
            if (e < kFillCells) {
                const int xx = hx + e % kFillDiameter - kFillRadius, yy = y + e / kFillDiameter - kFillRadius;
                if (xx >= 0 && xx < width && yy >= 0 && yy < height) {
                    const float d = img[yy * width + xx];
                    valid = depth_valid(d);
                    if (valid) q = (int)(1000 * d + 0.5f);
                }
            }
            // (a valid depth can quantise to a non-positive value only if it is below 0.5 mm or negative, -1 included;
            // such entries stay in the ranking, exactly as in the reference's array: an entry counts by its depth's
            // validity, not by its value)
            alive[r] = valid;
            key[r] = (unsigned)q ^ 0x80000000u;
            n += __popc(__ballot_sync(kFull, alive[r]));
        }
        int val = 0;
        if (n >= 2) {
            int k = (n + 1) / 2;  // rank among the valid values, ascending
            // bits on which all valid values agree need no vote
            unsigned mine = 0;
            bool have = false;
#pragma unroll
            for (int r = 3; r >= 0; r--)
                if (alive[r]) { mine = key[r]; have = true; }
            const unsigned who = __ballot_sync(kFull, have);
            const unsigned ref = __shfl_sync(kFull, mine, __ffs(who) - 1);
            unsigned diff = 0;
#pragma unroll
            for (int r = 0; r < 4; r++) diff |= alive[r] ? key[r] ^ ref : 0u;
            diff = __reduce_or_sync(kFull, diff);
            const int top = 32 - __clz(diff);  // bits [0, top) differ somewhere
            unsigned prefix = top >= 32 ? 0u : ref & ~((1u << top) - 1u);
            for (int bit = top - 1; bit >= 0; bit--) {
                int zeros = 0;
#pragma unroll
                for (int r = 0; r < 4; r++) zeros += __popc(__ballot_sync(kFull, alive[r] && !((key[r] >> bit) & 1u)));
                const bool one = k >= zeros;  // the wanted value has this bit set
                if (one) { k -= zeros; prefix |= 1u << bit; }
#pragma unroll
                for (int r = 0; r < 4; r++) alive[r] = alive[r] && (((key[r] >> bit) & 1u) != 0u) == one;
            }
            val = (int)(prefix ^ 0x80000000u);
        }
        if (lane == h) result = val <= 0 ? 0.0f : 0.001f * (float)val;
    }
    bool hole = false;
    if (inside) {
        out[(size_t)bz * width * height + y * width + x] = result;
        hole = result == 0.0f;
    }
    if (holes_out) {
        const unsigned m = __ballot_sync(kFull, hole);
        if (lane == 0 && m) atomicAdd(holes_out, __popc(m));
    }
}

// `gate` (may be NULL): the pass does nothing when *gate == 0.  `holes_out` (may be NULL): counts the zeros written.
__global__ void __launch_bounds__(256) median_fill_kernel(const float *__restrict__ in, float *__restrict__ out, int width,
                                                          int height, const int32_t *gate, int32_t *holes_out) {
    if (gate && *gate == 0) return;
    median_fill_tile(in, out, width, height, holes_out, blockIdx.x, blockIdx.y, blockIdx.z);
}

__device__ __forceinline__ float3 normal_from_points(float3 cc, float3 pc, float3 cp, float3 mc, float3 cm) {
    float3 out = make_float3(0.0f, 0.0f, 0.0f);
    const float ninf = -CUDART_INF_F;
    if ((cc.x != 0 || pc.x != 0 || cp.x != 0 || mc.x != 0 || cm.x != 0) &&
        (cc.x != ninf && pc.x != ninf && cp.x != ninf && mc.x != ninf && cm.x != ninf)) {
        const float ax = __fadd_rn(pc.x, -mc.x), ay = __fadd_rn(pc.y, -mc.y), az = __fadd_rn(pc.z, -mc.z);
        const float bx = __fadd_rn(cp.x, -cm.x), by = __fadd_rn(cp.y, -cm.y), bz = __fadd_rn(cp.z, -cm.z);
        // cross (cutil_math.h:1318), length (:1189) and n / -l (:904) with the contraction of the reference's sm_100
        // SASS: first product of each difference fused, second plain; squares summed x, then y, then z
        const float nx = __fmaf_rn(ay, bz, -__fmul_rn(az, by)), ny = __fmaf_rn(az, bx, -__fmul_rn(ax, bz)),
                    nz = __fmaf_rn(ax, by, -__fmul_rn(ay, bx));
        const float l = __fsqrt_rn(__fmaf_rn(nz, nz, __fmaf_rn(ny, ny, __fmul_rn(nx, nx))));
        if (l > 0.0f) out = make_float3(__fdiv_rn(nx, -l), __fdiv_rn(ny, -l), __fdiv_rn(nz, -l));
    }
    return out;
}

// kinectDepthToSkeleton (dkernel.cu:35-39) of one pixel; zero depth gives (0,0,0) (:158-168)
__device__ __forceinline__ float3 camera_point(const float *img, const float4 k, int width, unsigned x, unsigned y) {
    const float depth = img[y * width + x];
    if (depth == 0.0f) return make_float3(0.0f, 0.0f, 0.0f);
    const float px = __fdiv_rn(__fadd_rn((float)x, -k.z), k.x), py = __fdiv_rn(__fadd_rn((float)y, -k.w), k.y);
    return make_float3(__fmul_rn(depth, px), __fmul_rn(depth, py), depth);
}

// convert_depth_to_cameraspace_kernel (dkernel.cu:142-170) + compute_normals_kernel (:172-211) in one pass: the four
// neighbours' camera-space points are recomputed from the depth image instead of read back from the camspace image.
__device__ __forceinline__ void camspace_normals_tile(const float *__restrict__ depth, const float *__restrict__ intr,
                                                      float *__restrict__ camspace, float *__restrict__ normals, int width,
                                                      int height, int bx, int by, int b) {
    const unsigned x = bx * 32 + (threadIdx.x & 31), y = by * 8 + (threadIdx.x >> 5);
    if (x >= (unsigned)width || y >= (unsigned)height) return;
    const float *img = depth + (size_t)b * width * height;
    const float4 k = *reinterpret_cast<const float4 *>(intr + (size_t)b * 4);  // fx, fy, mx, my
    const size_t o = ((size_t)b * height * width + (size_t)y * width + x) * 3;
    const float3 cc = camera_point(img, k, width, x, y);
    if (camspace) { camspace[o] = cc.x; camspace[o + 1] = cc.y; camspace[o + 2] = cc.z; }
    if (!normals) return;
    float3 out = make_float3(0.0f, 0.0f, 0.0f);
    if (x > 0 && x < (unsigned)width - 1 && y > 0 && y < (unsigned)height - 1) {
        const float3 pc = camera_point(img, k, width, x, y + 1), cp = camera_point(img, k, width, x + 1, y);
        const float3 mc = camera_point(img, k, width, x, y - 1), cm = camera_point(img, k, width, x - 1, y);
        out = normal_from_points(cc, pc, cp, mc, cm);
    }
    normals[o] = out.x; normals[o + 1] = out.y; normals[o + 2] = out.z;
}

__global__ void __launch_bounds__(256) camspace_normals_kernel(const float *__restrict__ depth, const float *__restrict__ intr,
                                                               float *__restrict__ camspace, float *__restrict__ normals,
                                                               int width, int height) {
    camspace_normals_tile(depth, intr, camspace, normals, width, height, blockIdx.x, blockIdx.y, blockIdx.z);
}

// The fill rounds and the normals of Depth2Normals.forward (depth_utils.py:86-95) as one grid-resident launch: passes over
// 32x8-pixel tiles dealt round-robin to the CTAs, a grid barrier where a pass reads what the previous one wrote, and a
// loop that ends when a round leaves no hole.  (The bilateral filter in front stays a launch of its own: it is bound by
// double-precision throughput and wants every tile in flight at its own, higher occupancy.)
__global__ void __launch_bounds__(256) fill_rounds_normals_kernel(float *depth, const float *__restrict__ intr, float *filtered,
                                                                  float *camspace, float *normals, int32_t *hole_counts,
                                                                  int width, int height, int batch, int rounds) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    const int gx = (width + 31) / 32, gy = (height + 7) / 8, tiles = gx * gy * batch;
    auto for_tiles = [&](auto &&body) {
        for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
            const int bz = t / (gx * gy), r = t - bz * gx * gy;
            body(r % gx, r / gx, bz);
        }
    };
    for (int r = 0; r < rounds; r++) {
        // hole_counts[r] is final: its adds happened before the previous barrier (or in the bilateral launch)
        if (*reinterpret_cast<volatile int32_t *>(hole_counts + r) == 0) break;
        for_tiles([&](int bx, int by, int bz) { median_fill_tile(filtered, depth, width, height, hole_counts + r + 1, bx, by, bz); });
        grid.sync();
        for_tiles([&](int bx, int by, int bz) { median_fill_tile(depth, filtered, width, height, nullptr, bx, by, bz); });
        grid.sync();
    }
    for_tiles([&](int bx, int by, int bz) { camspace_normals_tile(depth, intr, camspace, normals, width, height, bx, by, bz); });
}

// compute_normals_kernel (dkernel.cu:172-211) on a camera-space image given by the caller
__global__ void __launch_bounds__(256) normals_from_camspace_kernel(const float *__restrict__ cam, float *__restrict__ normals,
                                                                    int width, int height) {
    const unsigned x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= (unsigned)width || y >= (unsigned)height) return;
    const float *img = cam + (size_t)blockIdx.z * width * height * 3;
    auto at = [&](unsigned xx, unsigned yy) {
        const float *p = img + ((size_t)yy * width + xx) * 3;
        return make_float3(p[0], p[1], p[2]);
    };
    float3 out = make_float3(0.0f, 0.0f, 0.0f);
    if (x > 0 && x < (unsigned)width - 1 && y > 0 && y < (unsigned)height - 1)
        out = normal_from_points(at(x, y), at(x, y + 1), at(x + 1, y), at(x, y - 1), at(x - 1, y));
    float *o = normals + ((size_t)blockIdx.z * width * height + (size_t)y * width + x) * 3;
    o[0] = out.x; o[1] = out.y; o[2] = out.z;
}

int check_image(const void *a, const void *b, int batch, int height, int width) {
    if (!a || !b) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL image pointer");
    if (batch <= 0 || height <= 0 || width <= 0) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad image size");
    return SPSG_OK;
}

dim3 image_grid(int batch, int height, int width) { return dim3((width + 31) / 32, (height + 7) / 8, batch); }

}  // namespace

extern "C" {

int spsg_depth_bilateral_filter(const float *depth, float *filtered, int32_t batch, int32_t height, int32_t width,
                                float sigma_d, float sigma_r, void *stream) {
    if (int rc = check_image(depth, filtered, batch, height, width)) return rc;
    bilateral_kernel<<<image_grid(batch, height, width), 256, 0, (cudaStream_t)stream>>>(depth, filtered, width, height, sigma_d,
                                                                                      sigma_r, nullptr);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_depth_median_fill(const float *in, float *out, int32_t batch, int32_t height, int32_t width, void *stream) {
    if (int rc = check_image(in, out, batch, height, width)) return rc;
    if (in == out) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "median fill cannot run in place");
    median_fill_kernel<<<image_grid(batch, height, width), 256, 0, (cudaStream_t)stream>>>(in, out, width, height, nullptr, nullptr);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_depth_to_cameraspace(const float *depth, const float *intrinsics, float *camspace, int32_t batch, int32_t height,
                              int32_t width, void *stream) {
    if (int rc = check_image(depth, camspace, batch, height, width)) return rc;
    if (!intrinsics || (reinterpret_cast<uintptr_t>(intrinsics) & 15u)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "intrinsics must be non-NULL and 16-byte aligned");
    camspace_normals_kernel<<<image_grid(batch, height, width), 256, 0, (cudaStream_t)stream>>>(depth, intrinsics, camspace,
                                                                                             nullptr, width, height);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_depth_compute_normals(const float *camspace, float *normals, int32_t batch, int32_t height, int32_t width,
                               void *stream) {
    if (int rc = check_image(camspace, normals, batch, height, width)) return rc;
    normals_from_camspace_kernel<<<image_grid(batch, height, width), 256, 0, (cudaStream_t)stream>>>(camspace, normals, width, height);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_depth_to_normals(float *depth, const float *intrinsics, float *filtered, float *camspace, float *normals,
                          int32_t *hole_counts, int32_t batch, int32_t height, int32_t width, float sigma_d, float sigma_r,
                          int32_t max_fill_iters, void *stream) {
    if (int rc = check_image(depth, filtered, batch, height, width)) return rc;
    if (!normals || !hole_counts) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL output pointer");
    if (!intrinsics || (reinterpret_cast<uintptr_t>(intrinsics) & 15u)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "intrinsics must be non-NULL and 16-byte aligned");
    if (max_fill_iters < 0 || max_fill_iters > 2 * (SPSG_DEPTH_MAX_FILL_ROUNDS)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "max_fill_iters out of range");
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid = image_grid(batch, height, width);
    const int rounds = max_fill_iters / 2;  // depth_utils.py:88
    // hole_counts[0] = zeros of the input frame, hole_counts[r] = zeros left in `depth` after fill round r
    SPSG_CUDA_TRY(cudaMemsetAsync(hole_counts, 0, sizeof(int32_t) * (SPSG_DEPTH_MAX_FILL_ROUNDS + 1), st));
    bilateral_kernel<<<grid, 256, 0, st>>>(depth, filtered, width, height, sigma_d, sigma_r, hole_counts);  // depth_utils.py:85
    SPSG_CUDA_TRY(cudaGetLastError());
    {
        // fill rounds + normals: one cooperative launch when the device has them, with as many CTAs as are resident at
        // once or, if the tiles need several turns, the count that gives every CTA the same number of turns
        static std::mutex mu;
        static int cached_room[64] = {0};  // resident CTAs of the kernel per device; -1 = no cooperative launch
        int dev = 0;
        SPSG_CUDA_TRY(cudaGetDevice(&dev));
        int resident = 0;
        {
            std::lock_guard<std::mutex> lk(mu);
            if (dev < 0 || dev >= 64 || cached_room[dev] == 0) {
                int coop = 0, per_sm = 0;
                SPSG_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
                SPSG_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fill_rounds_normals_kernel, 256, 0));
                resident = (coop && per_sm > 0) ? spsg_internal_sm_count() * per_sm : -1;
                if (dev >= 0 && dev < 64) cached_room[dev] = resident;
            } else {
                resident = cached_room[dev];
            }
        }
        if (resident > 0 && !getenv("SPSG_DEPTH_NO_COOPERATIVE")) {
            const long long tiles = (long long)grid.x * grid.y * grid.z, room = resident;
            const long long turns = (tiles + room - 1) / room;
            const int ctas = (int)((tiles + turns - 1) / turns);
            void *args[] = {&depth, &intrinsics, &filtered, &camspace, &normals, &hole_counts, &width, &height, &batch,
                            const_cast<int *>(&rounds)};
            SPSG_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)fill_rounds_normals_kernel, dim3(ctas), dim3(256), args, 0, st));
            return SPSG_OK;
        }
    }
    for (int r = 0; r < rounds; r++) {
        // one call of median_fill_depthmap(filt, depth, 2) (depth_utils.py:55-59,90): depth <- fill(filtered), filtered <- fill(depth);
        // both passes return immediately once the previous round left no hole
        median_fill_kernel<<<grid, 256, 0, st>>>(filtered, depth, width, height, hole_counts + r, hole_counts + r + 1);
        median_fill_kernel<<<grid, 256, 0, st>>>(depth, filtered, width, height, hole_counts + r, nullptr);
        SPSG_CUDA_TRY(cudaGetLastError());
    }
    camspace_normals_kernel<<<grid, 256, 0, st>>>(depth, intrinsics, camspace, normals, width, height);  // :94-95
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

}  // extern "C"
