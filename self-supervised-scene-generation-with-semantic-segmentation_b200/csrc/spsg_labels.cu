// spsg_labels.cu -- the 2D label maps of the training step (reference torch/train.py:614-616 target2d_label and
// :749-752 pred2d_label; SURVEY.md section 8 row a13):
//
//     cat = torch.cat((raycast_semantic, torch.ones(raycast_semantic.shape[:-1] + (1,))), dim=-1)
//     _, label = torch.max(cat, dim=-1, keepdim=True);  label = label.to(torch.uint8)
//
// i.e. per pixel the first index of the maximum of its 14 rendered values if that maximum is >= 1 (a tie with the
// appended 1 goes to the earlier index), else 14 (miss: -inf everywhere; unlabeled target voxel: all zeros).  torch.max
// treats NaN as the maximum; so does this kernel.  One pass over the rendering instead of cat + max + cast (three
// kernels and a 15-channel temporary), optionally with the per-class pixel histogram in the same pass.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "spsg_internal.h"
#include "spsg_raycast.h"

namespace {

constexpr int kClasses = 14;
constexpr int kMaxClasses = 64;  // spsg_labels_from_render_classes

__global__ void __launch_bounds__(256) labels_kernel(const float *__restrict__ semantic, long long num_pixels,
                                                     uint8_t *__restrict__ labels, unsigned long long *__restrict__ hist) {
    __shared__ unsigned s_hist[kClasses + 1];
    if (hist && threadIdx.x <= kClasses) s_hist[threadIdx.x] = 0u;
    if (hist) __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < num_pixels; i += stride) {
        const float2 *p = reinterpret_cast<const float2 *>(semantic + i * kClasses);
        float v[kClasses];
#pragma unroll
        for (int k = 0; k < kClasses / 2; k++) {
            const float2 t = __ldg(p + k);
            v[2 * k] = t.x; v[2 * k + 1] = t.y;
        }
        float best = v[0];
        int arg = 0;
#pragma unroll
        for (int k = 1; k < kClasses; k++)
            if (best == best && (v[k] > best || v[k] != v[k])) { best = v[k]; arg = k; }  // first maximum; NaN wins
        const int label = (best != best || best >= 1.0f) ? arg : kClasses;
        labels[i] = (uint8_t)label;
        if (hist) atomicAdd(&s_hist[label], 1u);
    }
    if (hist) {
        __syncthreads();
        if (threadIdx.x <= kClasses && s_hist[threadIdx.x]) atomicAdd(hist + threadIdx.x, (unsigned long long)s_hist[threadIdx.x]);
    }
}

// labels_kernel over C channels per pixel (label C = miss or unlabeled, hist of C + 1 bins): the same first-maximum scan,
// the values read one at a time
__global__ void __launch_bounds__(256) labels_classes_kernel(const float *__restrict__ semantic, int C, long long num_pixels,
                                                             uint8_t *__restrict__ labels, unsigned long long *__restrict__ hist) {
    __shared__ unsigned s_hist[kMaxClasses + 1];
    if (hist && threadIdx.x <= C) s_hist[threadIdx.x] = 0u;
    if (hist) __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < num_pixels; i += stride) {
        const float *p = semantic + i * C;
        float best = __ldg(p);
        int arg = 0;
#pragma unroll 1
        for (int k = 1; k < C; k++) {
            const float v = __ldg(p + k);
            if (best == best && (v > best || v != v)) { best = v; arg = k; }  // first maximum; NaN wins
        }
        const int label = (best != best || best >= 1.0f) ? arg : C;
        labels[i] = (uint8_t)label;
        if (hist) atomicAdd(&s_hist[label], 1u);
    }
    if (hist) {
        __syncthreads();
        if (threadIdx.x <= C && s_hist[threadIdx.x]) atomicAdd(hist + threadIdx.x, (unsigned long long)s_hist[threadIdx.x]);
    }
}

}  // namespace

extern "C" SPSG_API int spsg_labels_from_render_classes(const float *semantic, int32_t num_classes, int64_t num_pixels,
                                                        uint8_t *labels, int64_t *hist, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (num_classes < 1 || num_classes > kMaxClasses)
        return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "num_classes must be in 1..64");
    if (num_pixels < 0 || (num_pixels > 0 && (!semantic || !labels)))
        return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad semantic / labels / num_pixels");
    if (reinterpret_cast<uintptr_t>(semantic) & 3u) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "semantic must be 4-byte aligned");
    if (hist) SPSG_CUDA_TRY(cudaMemsetAsync(hist, 0, (num_classes + 1) * sizeof(int64_t), st));
    if (num_pixels == 0) return SPSG_OK;
    const unsigned grid = (unsigned)std::min<long long>((num_pixels + 255) / 256, (long long)spsg_internal_sm_count() * 8);
    labels_classes_kernel<<<grid, 256, 0, st>>>(semantic, num_classes, num_pixels, labels,
                                                 reinterpret_cast<unsigned long long *>(hist));
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

extern "C" SPSG_API int spsg_labels_from_render(const float *semantic, int64_t num_pixels, uint8_t *labels,
                                                int64_t *hist, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (num_pixels < 0 || (num_pixels > 0 && (!semantic || !labels)))
        return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "bad semantic / labels / num_pixels");
    if (reinterpret_cast<uintptr_t>(semantic) & 7u) return spsg_internal_fail(SPSG_ERR_INVALID_ARGUMENT, "semantic must be 8-byte aligned");
    if (hist) SPSG_CUDA_TRY(cudaMemsetAsync(hist, 0, (kClasses + 1) * sizeof(int64_t), st));
    if (num_pixels == 0) return SPSG_OK;
    const unsigned grid = (unsigned)std::min<long long>((num_pixels + 255) / 256, (long long)spsg_internal_sm_count() * 8);
    labels_kernel<<<grid, 256, 0, st>>>(semantic, num_pixels, labels, reinterpret_cast<unsigned long long *>(hist));
    SPSG_CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}
