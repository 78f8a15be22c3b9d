// spsg_sparsify.cu -- sm_100a kernels + C ABI for the producer glue between the generator's dense heads and the
// raycaster (SURVEY.md section 8(f) rank 1; reference torch/train.py:494-509):
//
//     locs = torch.nonzero((torch.abs(output_sdf.detach()[:, 0]) < truncation) [& ~empty[:, 0]])      train.py:495-497
//     locs = torch.cat([locs[:, 1:], locs[:, :1]], 1)                                                  train.py:498
//     vals = head[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]]            (sdf, colour, semantics)  :499-508
//
// The reference spends a nonzero (two library kernels + a host sync), a cat and one five-index advanced-indexing gather
// per head (each with an index_put backward).  Here: one ordered stream compaction (count + scan + write, rows in
// torch.nonzero's lexicographic (b,z,y,x) order, already in the raycaster's (z,y,x,b) column order) and one fused gather
// over all heads; the backward is one scatter into zero-filled dense gradients.  Results are identical (integer rows;
// values are copies).
//
// The heads may also be bfloat16 (a generator run under autocast) and NDHWC or channel slices (a generator in
// channels_last_3d): the compaction has bfloat16 twins of its count and write passes, and the *_strided gather /
// scatter pair reads and writes each head in its own dtype and strides, with float payloads on the sparse side.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "spsg_internal.h"
#include "spsg_raycast.h"

namespace {

constexpr int kTileThreads = 256;
constexpr int kCellsPerThread = 8;
constexpr int kTileCells = kTileThreads * kCellsPerThread;  // 2048 consecutive cells per CTA

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline long long num_tiles(long long cells) { return (cells + kTileCells - 1) / kTileCells; }

// scratch = int64 offsets[tiles + 1] (exclusive; the last entry is the total) after int32 counts[tiles]
struct Scratch {
    int32_t *counts;
    long long *offsets;
};
Scratch carve(void *scratch, long long tiles) {
    Scratch s;
    s.offsets = reinterpret_cast<long long *>(scratch);
    s.counts = reinterpret_cast<int32_t *>(reinterpret_cast<uint8_t *>(scratch) + align_up((size_t)(tiles + 1) * 8, 256));
    return s;
}

// The SDF head's element types: float, or bfloat16 (raw bits; widening is exact, a shift by 16).
__device__ __forceinline__ void load_cells8(const float *p, float (&v)[kCellsPerThread]) {
    const float4 a = __ldg(reinterpret_cast<const float4 *>(p));
    const float4 b = __ldg(reinterpret_cast<const float4 *>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load_cells8(const uint16_t *p, float (&v)[kCellsPerThread]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p));  // one 16-byte load: 8 cells
    const unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        v[2 * k] = __uint_as_float(w[k] << 16);
        v[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
    }
}
__device__ __forceinline__ float load_cell(const float *p) { return __ldg(p); }
__device__ __forceinline__ float load_cell(const uint16_t *p) { return __uint_as_float((unsigned)__ldg(p) << 16); }

// bit k of the result: cell (first + k) passes |sdf| < truncation (NaN fails, like torch) and is not marked empty;
// v[k] = the cell's SDF value widened to float (NaN beyond the end of the grid)
template <typename T>
__device__ __forceinline__ unsigned thread_cells(const T *__restrict__ sdf, const uint8_t *__restrict__ empty,
                                                 long long first, long long cells, float truncation,
                                                 float (&v)[kCellsPerThread]) {
    unsigned m = 0u;
    if (first + kCellsPerThread <= cells) {  // (sdf is 16-byte aligned and first is a multiple of 8)
        load_cells8(sdf + first, v);
#pragma unroll
        for (int k = 0; k < 8; k++) m |= (fabsf(v[k]) < truncation ? 1u : 0u) << k;
        if (empty && m) {
            const uint2 e = __ldg(reinterpret_cast<const uint2 *>(empty + first));
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const unsigned byte = ((k < 4 ? e.x : e.y) >> (8 * (k & 3))) & 0xffu;
                if (byte) m &= ~(1u << k);
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < kCellsPerThread; k++) {
            v[k] = __int_as_float(0x7fffffff);
            if (first + k < cells) {
                v[k] = load_cell(sdf + first + k);
                if (fabsf(v[k]) < truncation && !(empty && empty[first + k])) m |= 1u << k;
            }
        }
    }
    return m;
}

template <typename T>
__device__ __forceinline__ unsigned thread_mask(const T *__restrict__ sdf, const uint8_t *__restrict__ empty,
                                                long long first, long long cells, float truncation) {
    float v[kCellsPerThread];
    return thread_cells(sdf, empty, first, cells, truncation, v);
}

template <typename T>
__global__ void __launch_bounds__(kTileThreads) sparsify_count_kernel(const T *__restrict__ sdf,
                                                                      const uint8_t *__restrict__ empty, long long cells,
                                                                      float truncation, int32_t *__restrict__ counts) {
    __shared__ int s_warp[kTileThreads / 32];
    const long long first = ((long long)blockIdx.x * kTileThreads + threadIdx.x) * kCellsPerThread;
    int n = first < cells ? __popc(thread_mask(sdf, empty, first, cells, truncation)) : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
#pragma unroll
        for (int w = 0; w < kTileThreads / 32; w++) t += s_warp[w];
        counts[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts by one CTA (the tiles of a training batch number a few thousand)
__global__ void __launch_bounds__(1024) sparsify_scan_kernel(const int32_t *__restrict__ counts, long long tiles,
                                                             long long *__restrict__ offsets, long long *total_out) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long base = 0; base < tiles; base += 1024) {
        const long long i = base + threadIdx.x;
        const long long v = i < tiles ? (long long)counts[i] : 0;
        long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            long long w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            s_warp[lane] = w;  // inclusive over warps
        }
        __syncthreads();
        const long long before = s_carry + (warp > 0 ? s_warp[warp - 1] : 0) + inc - v;
        if (i < tiles) offsets[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        offsets[tiles] = s_carry;
        if (total_out) *total_out = s_carry;
    }
}

// kIndexed: the same pass also writes, for EVERY cell, what the raycaster's fill + index passes derive from `locs`
// (kernel.cu:346-362, 515 and the dense SDF brick of this implementation): index[cell] = row of the cell or -1,
// brick[cell] = its SDF or NaN (absent) -- two coalesced 32-byte stores per thread instead of a 32-byte read and two
// scattered 4-byte writes per row in a later launch.  (T = uint16_t: a bfloat16 head; the brick gets the widened value,
// which is what the gather hands the raycaster as vals_sdf.)
template <typename T, bool kIndexed>
__global__ void __launch_bounds__(kTileThreads) sparsify_write_kernel(const T *__restrict__ sdf,
                                                                      const uint8_t *__restrict__ empty, long long cells,
                                                                      int dimz, int dimy, int dimx, float truncation,
                                                                      const long long *__restrict__ offsets,
                                                                      longlong4 *__restrict__ locs, long long num_locs,
                                                                      int32_t *__restrict__ index, float *__restrict__ brick) {
    __shared__ int s_warp[kTileThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long first = ((long long)blockIdx.x * kTileThreads + threadIdx.x) * kCellsPerThread;
    float v[kCellsPerThread];
    const unsigned m = first < cells ? thread_cells(sdf, empty, first, cells, truncation, v) : 0u;
    const int n = __popc(m);
    int inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    int before = inc - n;
    for (int w = 0; w < warp; w++) before += s_warp[w];
    if (!kIndexed && !m) return;
    if (first >= cells) return;
    long long pos = offsets[blockIdx.x] + before;
    // (b, z, y, x) of the thread's first cell, then x runs with carries
    const long long plane = (long long)dimy * dimx;
    long long rest = first;
    const long long bz = rest / plane;
    rest -= bz * plane;
    long long b = bz / dimz, z = bz - b * dimz, y = rest / dimx, x = rest - y * dimx;
    int row[kCellsPerThread];
#pragma unroll
    for (int k = 0; k < kCellsPerThread; k++) {
        row[k] = -1;
        if ((m >> k) & 1u) {
            if (pos < num_locs) {
                locs[pos] = make_longlong4(z, y, x, b);  // train.py:498 column order
                row[k] = (int)pos;
            }
            pos++;
        }
        if (++x == dimx) {
            x = 0;
            if (++y == dimy) {
                y = 0;
                if (++z == dimz) { z = 0; b++; }
            }
        }
    }
    if (kIndexed) {
        const float absent = __int_as_float(0xffffffff);  // the brick's "no voxel here" (what the forward's fill writes)
        if (first + kCellsPerThread <= cells) {  // (index and brick are 16-byte aligned, first is a multiple of 8)
            int4 *ip = reinterpret_cast<int4 *>(index + first);
            float4 *bp = reinterpret_cast<float4 *>(brick + first);
            ip[0] = make_int4(row[0], row[1], row[2], row[3]);
            ip[1] = make_int4(row[4], row[5], row[6], row[7]);
            bp[0] = make_float4(row[0] < 0 ? absent : v[0], row[1] < 0 ? absent : v[1], row[2] < 0 ? absent : v[2],
                                row[3] < 0 ? absent : v[3]);
            bp[1] = make_float4(row[4] < 0 ? absent : v[4], row[5] < 0 ? absent : v[5], row[6] < 0 ? absent : v[6],
                                row[7] < 0 ? absent : v[7]);
        } else {
#pragma unroll
            for (int k = 0; k < kCellsPerThread; k++)
                if (first + k < cells) {
                    index[first + k] = row[k];
                    brick[first + k] = row[k] < 0 ? absent : v[k];
                }
        }
    }
}

constexpr int kMaxPayloads = 4;
struct PayloadArgs {
    float *dense[kMaxPayloads];
    float *sparse[kMaxPayloads];
    int channels[kMaxPayloads];
    int count;
};

// head[b, :, z, y, x] <-> vals[i, :] for the voxel rows of `locs`; kScatter writes the dense side (backward).
// A warp takes 32 consecutive voxels; their values go through shared memory so that the sparse side is read / written as
// one contiguous run of 32 * C floats and the dense side as 32 (mostly adjacent) cells per channel.
template <bool kScatter>
__global__ void __launch_bounds__(256) dense_payload_kernel(const PayloadArgs a, const longlong4 *__restrict__ locs,
                                                            long long num_locs, int dimz, int dimy, int dimx) {
    __shared__ float s_vals[8][32 * 16 + 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *s = s_vals[warp];
    const long long warps = (long long)gridDim.x * 8;
    const long long vol = (long long)dimz * dimy * dimx;
    for (long long base = ((long long)blockIdx.x * 8 + warp) * 32; base < num_locs; base += warps * 32) {
        const long long i = base + lane;
        const int n = (int)min((long long)32, num_locs - base);
        long long cell = 0, b = 0;
        if (lane < n) {
            const longlong4 l = locs[i];  // (z, y, x, b)
            cell = (l.x * dimy + l.y) * dimx + l.z;
            b = l.w;
        }
        for (int p = 0; p < a.count; p++) {
            const int C = a.channels[p];
            float *dense = a.dense[p] + b * C * vol + cell;
            float *sparse = a.sparse[p] + base * C;
            for (int c0 = 0; c0 < C; c0 += 16) {
                const int cc = min(16, C - c0);
                __syncwarp();
                if (!kScatter) {
                    if (lane < n)
                        for (int c = 0; c < cc; c++) s[lane * cc + c] = __ldg(dense + (long long)(c0 + c) * vol);
                    __syncwarp();
                    for (int e = lane; e < n * cc; e += 32) {
                        const int v = e / cc, c = e - v * cc;
                        sparse[(long long)v * C + c0 + c] = s[e];
                    }
                } else {
                    for (int e = lane; e < n * cc; e += 32) {
                        const int v = e / cc, c = e - v * cc;
                        s[e] = __ldg(sparse + (long long)v * C + c0 + c);
                    }
                    __syncwarp();
                    if (lane < n)
                        for (int c = 0; c < cc; c++) dense[(long long)(c0 + c) * vol] = s[lane * cc + c];
                }
            }
        }
    }
}

struct HeadArgs {
    void *dense[kMaxPayloads];
    float *sparse[kMaxPayloads];
    long long stride[kMaxPayloads][5];  // elements, (b, c, z, y, x)
    int channels[kMaxPayloads];
    int bf16[kMaxPayloads];
    int count;
};

__device__ __forceinline__ float load_elem(const void *p, long long o, bool bf16) {
    return bf16 ? __uint_as_float((unsigned)__ldg(static_cast<const uint16_t *>(p) + o) << 16)
                : __ldg(static_cast<const float *>(p) + o);
}

// The gradient of head[idx].float() with respect to a head of either dtype: the row's gradient rounded to the head's
// dtype (round-to-nearest-even, what the backward of .float() does) and added to the zero-filled dense gradient
// (index_put with accumulate): 0 + g, so -0 becomes +0, exactly as autograd of the literal expression gives it.  (A
// float32 NaN is stored as it comes, as the accumulation leaves it; a bfloat16 NaN is the conversion's.)
__device__ __forceinline__ void store_elem(void *p, long long o, float g, bool bf16) {
    if (bf16) {
        const float r = __bfloat162float(__float2bfloat16_rn(g));
        static_cast<__nv_bfloat16 *>(p)[o] = __float2bfloat16_rn(0.0f + r);
    } else {
        static_cast<float *>(p)[o] = g == 0.0f ? 0.0f : g;
    }
}

// As dense_payload_kernel, for heads of any element strides and of dtype float or bfloat16; the sparse side is float.
// A warp takes 32 consecutive voxels.  Heads whose channels are adjacent (stride 1: NDHWC, or a channel slice of it)
// are moved voxel by voxel: lane e of a pass handles channel e % C of voxel e / C, so both sides are contiguous runs of
// the warp's (mostly adjacent) voxels -- C * 2 or C * 4 bytes each on the dense side, one run of 32 * C floats on the
// sparse side.  Other heads (channels a volume apart) go channel by channel through shared memory, as in
// dense_payload_kernel.
template <bool kScatter>
__global__ void __launch_bounds__(256) strided_payload_kernel(const HeadArgs a, const longlong4 *__restrict__ locs,
                                                              long long num_locs) {
    __shared__ float s_vals[8][32 * 16 + 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *s = s_vals[warp];
    const long long warps = (long long)gridDim.x * 8;
    for (long long base = ((long long)blockIdx.x * 8 + warp) * 32; base < num_locs; base += warps * 32) {
        const int n = (int)min((long long)32, num_locs - base);
        longlong4 l = make_longlong4(0, 0, 0, 0);  // (z, y, x, b)
        if (lane < n) l = locs[base + lane];
        for (int p = 0; p < a.count; p++) {
            const long long *st = a.stride[p];
            const long long off = l.w * st[0] + l.x * st[2] + l.y * st[3] + l.z * st[4];
            const int C = a.channels[p];
            const bool bf = a.bf16[p] != 0;
            void *dense = a.dense[p];
            float *sparse = a.sparse[p] + base * C;
            if (st[1] == 1 || C == 1) {
                const int total = n * C;
                for (int e0 = 0; e0 < total; e0 += 32) {
                    const int e = e0 + lane;
                    const int v = min(e / C, 31), c = e - v * C;
                    const long long o = __shfl_sync(0xffffffffu, off, v) + c;
                    if (e < total) {
                        if (!kScatter) sparse[e] = load_elem(dense, o, bf);
                        else store_elem(dense, o, __ldg(sparse + e), bf);
                    }
                }
            } else {
                const long long sc = st[1];
                for (int c0 = 0; c0 < C; c0 += 16) {
                    const int cc = min(16, C - c0);
                    __syncwarp();
                    if (!kScatter) {
                        if (lane < n)
                            for (int c = 0; c < cc; c++) s[lane * cc + c] = load_elem(dense, off + (c0 + c) * sc, bf);
                        __syncwarp();
                        for (int e = lane; e < n * cc; e += 32) {
                            const int v = e / cc, c = e - v * cc;
                            sparse[(long long)v * C + c0 + c] = s[e];
                        }
                    } else {
                        for (int e = lane; e < n * cc; e += 32) {
                            const int v = e / cc, c = e - v * cc;
                            s[e] = __ldg(sparse + (long long)v * C + c0 + c);
                        }
                        __syncwarp();
                        if (lane < n)
                            for (int c = 0; c < cc; c++) store_elem(dense, off + (c0 + c) * sc, s[lane * cc + c], bf);
                    }
                }
            }
        }
    }
}

int check_grid(int num_chunks, int dimz, int dimy, int dimx) {
    if (num_chunks <= 0 || dimz <= 0 || dimy <= 0 || dimx <= 0)
        return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad grid sizes");
    return SPSG_OK;
}

int launch_payload(bool scatter, const spsg_dense_payload *payloads, int count, const int64_t *locs, int64_t num_locs,
                   int num_chunks, int dimz, int dimy, int dimx, cudaStream_t st) {
    if (int rc = check_grid(num_chunks, dimz, dimy, dimx)) return rc;
    if (count < 0 || count > kMaxPayloads) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "at most 4 payloads per call");
    if (num_locs < 0 || (num_locs > 0 && !locs)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad locs");
    if (reinterpret_cast<uintptr_t>(locs) & 15u) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "locs must be 16-byte aligned");
    PayloadArgs a = {};
    a.count = count;
    const size_t cells = (size_t)num_chunks * dimz * dimy * dimx;
    for (int p = 0; p < count; p++) {
        if (!payloads[p].dense || (num_locs > 0 && !payloads[p].sparse) || payloads[p].channels <= 0)
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad payload");
        a.dense[p] = payloads[p].dense;
        a.sparse[p] = payloads[p].sparse;
        a.channels[p] = payloads[p].channels;
        if (scatter)  // the dense gradient is zero everywhere else (index_put backward of the reference's gather)
            SPSG_CUDA_TRY(cudaMemsetAsync(payloads[p].dense, 0, cells * payloads[p].channels * sizeof(float), st));
    }
    if (num_locs == 0 || count == 0) return SPSG_OK;
    const unsigned grid = (unsigned)std::min<long long>((num_locs + 255) / 256, (long long)spsg_internal_sm_count() * 16);
    if (scatter) dense_payload_kernel<true><<<grid, 256, 0, st>>>(a, reinterpret_cast<const longlong4 *>(locs), num_locs, dimz, dimy, dimx);
    else dense_payload_kernel<false><<<grid, 256, 0, st>>>(a, reinterpret_cast<const longlong4 *>(locs), num_locs, dimz, dimy, dimx);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

// the head's strides are a permutation of a packed layout of its B * C * Dz * Dy * Dx elements (dimensions of size 1
// may carry any stride)
bool packed(const int64_t *stride, const long long *size) {
    int order[5] = {0, 1, 2, 3, 4};
    std::sort(order, order + 5, [&](int i, int j) {
        return size[i] == 1 ? false : size[j] == 1 ? true : stride[i] < stride[j];
    });
    long long expect = 1;
    for (int k = 0; k < 5 && size[order[k]] != 1; k++) {
        if (stride[order[k]] != expect) return false;
        expect *= size[order[k]];
    }
    return true;
}

int launch_strided(bool scatter, const spsg_dense_head *heads, int count, const int64_t *locs, int64_t num_locs,
                   int num_chunks, int dimz, int dimy, int dimx, cudaStream_t st) {
    if (int rc = check_grid(num_chunks, dimz, dimy, dimx)) return rc;
    if (count < 0 || count > kMaxPayloads) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "at most 4 heads per call");
    if (count > 0 && !heads) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL heads");
    if (num_locs < 0 || (num_locs > 0 && !locs)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad locs");
    if (reinterpret_cast<uintptr_t>(locs) & 15u) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "locs must be 16-byte aligned");
    HeadArgs a = {};
    a.count = count;
    for (int p = 0; p < count; p++) {
        const spsg_dense_head &h = heads[p];
        if (!h.dense || (num_locs > 0 && !h.sparse))
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL dense / sparse pointer of a head");
        if (h.channels <= 0) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "non-positive channels");
        if (h.dtype != SPSG_DTYPE_F32 && h.dtype != SPSG_DTYPE_BF16)
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "unknown head dtype");
        const size_t esize = h.dtype == SPSG_DTYPE_BF16 ? 2 : 4;
        if (reinterpret_cast<uintptr_t>(h.dense) & (esize - 1))
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "dense head not aligned to its element size");
        const long long size[5] = {num_chunks, h.channels, dimz, dimy, dimx};
        long long last = 0;  // offset of the head's last element
        for (int d = 0; d < 5; d++) {
            if (h.strides[d] < 0) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "negative head stride");
            if (h.strides[d] > 0 && (size[d] - 1) > (INT64_MAX - last) / h.strides[d])
                return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "head strides overflow");
            last += (size[d] - 1) * h.strides[d];
        }
        if (last >= h.extent) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "head strides leave the head's extent");
        if (scatter && !packed(h.strides, size))
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "the scatter's dense gradient must be packed");
        a.dense[p] = h.dense;
        a.sparse[p] = h.sparse;
        for (int d = 0; d < 5; d++) a.stride[p][d] = h.strides[d];
        a.channels[p] = h.channels;
        a.bf16[p] = h.dtype == SPSG_DTYPE_BF16;
    }
    if (scatter)
        for (int p = 0; p < count; p++) {
            const size_t elems = (size_t)num_chunks * heads[p].channels * dimz * dimy * dimx;
            SPSG_CUDA_TRY(cudaMemsetAsync(heads[p].dense, 0, elems * (heads[p].dtype == SPSG_DTYPE_BF16 ? 2 : 4), st));
        }
    if (num_locs == 0 || count == 0) return SPSG_OK;
    const unsigned grid = (unsigned)std::min<long long>((num_locs + 255) / 256, (long long)spsg_internal_sm_count() * 16);
    if (scatter) strided_payload_kernel<true><<<grid, 256, 0, st>>>(a, reinterpret_cast<const longlong4 *>(locs), num_locs);
    else strided_payload_kernel<false><<<grid, 256, 0, st>>>(a, reinterpret_cast<const longlong4 *>(locs), num_locs);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

// torch compares a bfloat16 tensor with a Python scalar in bfloat16: the scalar is rounded (double -> float -> bfloat16,
// nearest-even) before |sdf| < truncation is evaluated.  A truncation bfloat16 cannot represent that rounds down
// excludes the cells equal to the rounded value.
float bf16_truncation(float t) { return __bfloat162float(__float2bfloat16_rn(t)); }

template <typename T>
int sparsify_count_impl(const T *sdf, const uint8_t *empty, int64_t cells, float truncation, void *scratch,
                               size_t scratch_bytes, int64_t *total_out, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!sdf || cells <= 0) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad sdf / cells");
    if ((reinterpret_cast<uintptr_t>(sdf) & 15u) || (empty && (reinterpret_cast<uintptr_t>(empty) & 7u)))
        return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "sdf must be 16-byte and empty 8-byte aligned");
    if (!scratch || scratch_bytes < spsg_sparsify_scratch_bytes(cells) || (reinterpret_cast<uintptr_t>(scratch) & 255u))
        return spsg_internal_fail(SPSG_ERR_WORKSPACE_TOO_SMALL, "sparsify scratch too small or not 256-byte aligned");
    const long long tiles = num_tiles(cells);
    const Scratch s = carve(scratch, tiles);
    sparsify_count_kernel<T><<<(unsigned)tiles, kTileThreads, 0, st>>>(sdf, empty, cells, truncation, s.counts);
    SPSG_CUDA_TRY(cudaGetLastError());
    sparsify_scan_kernel<<<1, 1024, 0, st>>>(s.counts, tiles, s.offsets, reinterpret_cast<long long *>(total_out));
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

template <typename T>
int sparsify_locs_impl(const T *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz, int32_t dimy,
                              int32_t dimx, float truncation, const void *scratch, int64_t *locs, int64_t num_locs,
                              int32_t *index, float *brick, bool indexed, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (int rc = check_grid(num_chunks, dimz, dimy, dimx)) return rc;
    if (!sdf || !scratch) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL sdf / scratch");
    if (num_locs < 0 || (num_locs > 0 && !locs)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad locs");
    if (reinterpret_cast<uintptr_t>(locs) & 15u) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "locs must be 16-byte aligned");
    if (indexed) {
        if (!index || !brick) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "NULL index / brick");
        if ((reinterpret_cast<uintptr_t>(index) & 15u) || (reinterpret_cast<uintptr_t>(brick) & 15u))
            return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "index and brick must be 16-byte aligned");
        if (num_locs >= (1ll << 31)) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "num_locs exceeds 32-bit indexing");
    } else if (num_locs == 0) {
        return SPSG_OK;
    }
    const long long cells = (long long)num_chunks * dimz * dimy * dimx;
    const long long tiles = num_tiles(cells);
    const Scratch s = carve(const_cast<void *>(scratch), tiles);
    if (indexed)
        sparsify_write_kernel<T, true><<<(unsigned)tiles, kTileThreads, 0, st>>>(sdf, empty, cells, dimz, dimy, dimx, truncation, s.offsets,
                                                                                 reinterpret_cast<longlong4 *>(locs), num_locs, index, brick);
    else
        sparsify_write_kernel<T, false><<<(unsigned)tiles, kTileThreads, 0, st>>>(sdf, empty, cells, dimz, dimy, dimx, truncation, s.offsets,
                                                                                  reinterpret_cast<longlong4 *>(locs), num_locs, nullptr, nullptr);
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

}  // namespace

extern "C" {

SPSG_API size_t spsg_sparsify_scratch_bytes(int64_t cells) {
    if (cells <= 0) return 0;
    const long long tiles = num_tiles(cells);
    return align_up((size_t)(tiles + 1) * 8, 256) + align_up((size_t)tiles * 4, 256);
}

SPSG_API int spsg_sparsify_count(const float *sdf, const uint8_t *empty, int64_t cells, float truncation, void *scratch,
                                 size_t scratch_bytes, int64_t *total_out, void *stream) {
    return sparsify_count_impl(sdf, empty, cells, truncation, scratch, scratch_bytes, total_out, stream);
}

SPSG_API int spsg_sparsify_count_bf16(const uint16_t *sdf, const uint8_t *empty, int64_t cells, float truncation,
                                      void *scratch, size_t scratch_bytes, int64_t *total_out, void *stream) {
    return sparsify_count_impl(sdf, empty, cells, bf16_truncation(truncation), scratch, scratch_bytes, total_out, stream);
}

SPSG_API int spsg_sparsify_locs(const float *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz, int32_t dimy,
                                int32_t dimx, float truncation, const void *scratch, int64_t *locs, int64_t num_locs,
                                void *stream) {
    return sparsify_locs_impl(sdf, empty, num_chunks, dimz, dimy, dimx, truncation, scratch, locs, num_locs, nullptr, nullptr,
                              false, stream);
}

SPSG_API int spsg_sparsify_locs_indexed(const float *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                        int32_t dimy, int32_t dimx, float truncation, const void *scratch, int64_t *locs,
                                        int64_t num_locs, int32_t *sparse_mapping, void *raycast_workspace, void *stream) {
    // the dense SDF brick is the first num_chunks * Dz * Dy * Dx floats of the raycast workspace (Layout::dense_off == 0)
    return sparsify_locs_impl(sdf, empty, num_chunks, dimz, dimy, dimx, truncation, scratch, locs, num_locs, sparse_mapping,
                              static_cast<float *>(raycast_workspace), true, stream);
}

SPSG_API int spsg_sparsify_locs_bf16(const uint16_t *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                     int32_t dimy, int32_t dimx, float truncation, const void *scratch, int64_t *locs,
                                     int64_t num_locs, void *stream) {
    return sparsify_locs_impl(sdf, empty, num_chunks, dimz, dimy, dimx, bf16_truncation(truncation), scratch, locs, num_locs,
                              nullptr, nullptr, false, stream);
}

SPSG_API int spsg_sparsify_locs_indexed_bf16(const uint16_t *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                             int32_t dimy, int32_t dimx, float truncation, const void *scratch,
                                             int64_t *locs, int64_t num_locs, int32_t *sparse_mapping,
                                             void *raycast_workspace, void *stream) {
    return sparsify_locs_impl(sdf, empty, num_chunks, dimz, dimy, dimx, bf16_truncation(truncation), scratch, locs, num_locs,
                              sparse_mapping, static_cast<float *>(raycast_workspace), true, stream);
}

SPSG_API int spsg_dense_gather(const spsg_dense_payload *payloads, int32_t count, const int64_t *locs, int64_t num_locs,
                               int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream) {
    return launch_payload(false, payloads, count, locs, num_locs, num_chunks, dimz, dimy, dimx, static_cast<cudaStream_t>(stream));
}

SPSG_API int spsg_dense_scatter(const spsg_dense_payload *payloads, int32_t count, const int64_t *locs, int64_t num_locs,
                                int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream) {
    return launch_payload(true, payloads, count, locs, num_locs, num_chunks, dimz, dimy, dimx, static_cast<cudaStream_t>(stream));
}

SPSG_API int spsg_dense_gather_strided(const spsg_dense_head *heads, int32_t count, const int64_t *locs, int64_t num_locs,
                                       int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream) {
    return launch_strided(false, heads, count, locs, num_locs, num_chunks, dimz, dimy, dimx, static_cast<cudaStream_t>(stream));
}

SPSG_API int spsg_dense_scatter_strided(const spsg_dense_head *heads, int32_t count, const int64_t *locs, int64_t num_locs,
                                        int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream) {
    return launch_strided(true, heads, count, locs, num_locs, num_chunks, dimz, dimy, dimx, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
