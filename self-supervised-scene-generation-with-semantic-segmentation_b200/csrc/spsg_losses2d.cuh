// spsg_losses2d.cuh -- the 2D losses as stand-alone image-space kernels.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// the 2D losses as stand-alone image-space ops (the reference's own boundary: loss.compute_2dcolor_loss and the
// inline expressions of train.py:635-638, 744-746 applied to rendered images)
// ---------------------------------------------------------------------------------------------

struct Losses2DArgs {
    const float *image_color, *image_depth, *image_semantic;
    LossArgs loss;
    long long num_pixels;
};

// one thread per pixel: the same six sums the fused forward accumulates in its epilogue
// kGenericSem: C = a.loss.sem_channels logits per pixel (spsg_losses2d_forward_classes), label C = ignore
template <bool kGenericSem = false>
__global__ void __launch_bounds__(256) losses2d_forward_kernel(const Losses2DArgs a) {
    const float ninf = -CUDART_INF_F;
    float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    const LossArgs &L = a.loss;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < a.num_pixels; p += (long long)gridDim.x * blockDim.x) {
        if (L.target_depth) {  // train.py:635-638
            const float r = __ldg(a.image_depth + p), t = __ldg(L.target_depth + p);
            if (r != ninf && t != 0.0f) { acc[0] += fabsf(__fmul_rn(r, L.voxelsize) - t); acc[1] += 1.0f; }
        }
        if (L.target_color) {  // loss.py:246-257 (valid is per element)
            const float w = L.weight_color ? __ldg(L.weight_color + p) : 1.0f;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const float c = __ldg(a.image_color + p * 3 + k);
                if (c != ninf) {
                    acc[2] += fabsf(__fadd_rn(__fmul_rn(c, w), -__fmul_rn(__ldg(L.target_color + p * 3 + k), w)));
                    acc[3] += 1.0f;
                }
            }
        }
        if (kGenericSem && L.target_label) {  // the same over C logits
            const int y = L.target_label[p], C = a.loss.sem_channels;
            const float *l = a.image_semantic + p * C;
            if (y < C && __ldg(l) != ninf) {
                const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                acc[4] += w * ce_nll<false>(l, C, y);
                acc[5] += w;
            }
        } else if (L.target_label) {  // train.py:744-746
            const int y = L.target_label[p];
            if (y < 14) {
                float l[14];
                const float2 *s2 = reinterpret_cast<const float2 *>(a.image_semantic + p * 14);
#pragma unroll
                for (int k = 0; k < 7; k++) {
                    const float2 t2 = __ldg(s2 + k);
                    l[2 * k] = t2.x; l[2 * k + 1] = t2.y;
                }
                if (l[0] != ninf) {
                    float m = l[0];
#pragma unroll
                    for (int k = 1; k < 14; k++) m = fmaxf(m, l[k]);
                    float sum = 0.0f, ly = 0.0f;
#pragma unroll
                    for (int k = 0; k < 14; k++) {
                        sum += expf(l[k] - m);
                        if (k == y) ly = l[k];
                    }
                    const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                    acc[4] += w * (logf(sum) + m - ly);
                    acc[5] += w;
                }
            }
        }
    }
    const int lane = threadIdx.x & 31;
    float mine = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const float t = warp_sum(acc[k]);
        if (lane == k) mine = t;
    }
    const unsigned slot = (blockIdx.x * 8u + (threadIdx.x >> 5)) % kLossSlots;
    if (lane < 6 && mine != 0.0f) atomicAdd(L.accum + slot * 8 + lane, (double)mine);
}

// pixel p's share of the six sums, added onto acc: the body of losses2d_forward_kernel's loop, for the deterministic
// variant (spsg_deterministic.cuh).  (Kept apart so that losses2d_forward_kernel compiles exactly as before.)
template <bool kGenericSem>
__device__ __forceinline__ void loss_terms_pixel(const Losses2DArgs &a, long long p, float (&acc)[6]) {
    const float ninf = -CUDART_INF_F;
    const LossArgs &L = a.loss;
    if (L.target_depth) {  // train.py:635-638
        const float r = __ldg(a.image_depth + p), t = __ldg(L.target_depth + p);
        if (r != ninf && t != 0.0f) { acc[0] += fabsf(__fmul_rn(r, L.voxelsize) - t); acc[1] += 1.0f; }
    }
    if (L.target_color) {  // loss.py:246-257 (valid is per element)
        const float w = L.weight_color ? __ldg(L.weight_color + p) : 1.0f;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const float c = __ldg(a.image_color + p * 3 + k);
            if (c != ninf) {
                acc[2] += fabsf(__fadd_rn(__fmul_rn(c, w), -__fmul_rn(__ldg(L.target_color + p * 3 + k), w)));
                acc[3] += 1.0f;
            }
        }
    }
    if (kGenericSem && L.target_label) {  // the same over C logits
        const int y = L.target_label[p], C = a.loss.sem_channels;
        const float *l = a.image_semantic + p * C;
        if (y < C && __ldg(l) != ninf) {
            const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
            acc[4] += w * ce_nll<false>(l, C, y);
            acc[5] += w;
        }
    } else if (L.target_label) {  // train.py:744-746
        const int y = L.target_label[p];
        if (y < 14) {
            float l[14];
            const float2 *s2 = reinterpret_cast<const float2 *>(a.image_semantic + p * 14);
#pragma unroll
            for (int k = 0; k < 7; k++) {
                const float2 t2 = __ldg(s2 + k);
                l[2 * k] = t2.x; l[2 * k + 1] = t2.y;
            }
            if (l[0] != ninf) {
                float m = l[0];
#pragma unroll
                for (int k = 1; k < 14; k++) m = fmaxf(m, l[k]);
                float sum = 0.0f, ly = 0.0f;
#pragma unroll
                for (int k = 0; k < 14; k++) {
                    sum += expf(l[k] - m);
                    if (k == y) ly = l[k];
                }
                const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                acc[4] += w * (logf(sum) + m - ly);
                acc[5] += w;
            }
        }
    }
}

// gradient images of the weighted total w.r.t. the renderings (zero where a pixel is not part of a term)
// kGenericSem: C = a.loss.sem_channels; each thread's row of C + 7 gradients is built in dynamic shared memory
template <bool kGenericSem = false>
__global__ void __launch_bounds__(256) losses2d_backward_kernel(const BackwardArgs a, long long num_pixels, float *d_color,
                                                               float *d_depth, float *d_semantic) {
    const FusedCoef fc = fused_coef(a);
    if constexpr (kGenericSem) {
        extern __shared__ float s_rows[];
        const int C = a.loss.sem_channels;
        float *g = s_rows + (size_t)threadIdx.x * (C + 7);
        for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < num_pixels; p += (long long)gridDim.x * blockDim.x) {
            pixel_grads_fused_sem(a, fc, C, (unsigned)p, g);
            if (d_semantic)
                for (int k = 0; k < C; k++) d_semantic[p * C + k] = g[k];
            if (d_color) { d_color[p * 3] = g[C]; d_color[p * 3 + 1] = g[C + 1]; d_color[p * 3 + 2] = g[C + 2]; }
            if (d_depth) d_depth[p] = g[C + 3];
        }
    } else {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < num_pixels; p += (long long)gridDim.x * blockDim.x) {
        float g[21];
        pixel_grads_fused(a, fc, (unsigned)p, g);
        if (d_semantic) {
#pragma unroll
            for (int k = 0; k < 7; k++) reinterpret_cast<float2 *>(d_semantic + p * 14)[k] = make_float2(g[2 * k], g[2 * k + 1]);
        }
        if (d_color) { d_color[p * 3] = g[14]; d_color[p * 3 + 1] = g[15]; d_color[p * 3 + 2] = g[16]; }
        if (d_depth) d_depth[p] = g[17];
    }
    }
}
