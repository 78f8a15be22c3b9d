// spsg_backward.cuh -- the backward: gradient-row clearing and the per-(voxel, view) gather, plain or fused with the 2D losses.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------

struct BackwardArgs {
    const float *grad_color, *grad_depth, *grad_normal, *grad_semantic;  // plain variant
    const float *image_color, *image_depth, *image_semantic;             // fused-loss variant
    LossArgs loss;
    const float *loss_out;
    float w_depth, w_color, w_sem;
    const float *grad_scale;  // device scalar or NULL (= 1)
    const int32_t *mapping3dto2d, *mapping3dto2d_num;
    float *d_color, *d_depth, *d_normal, *d_semantic;
    const int32_t *list_count;
    const int2 *list;
    int width, height;
    int views, max_pixels;
    long long num_locs;
    int zero_blocks;  // leading CTAs of the launch that clear gradient rows instead of gathering
    // fused variant with upstream images (kUpstream): d objective / d rendering added to the recomputed loss gradients;
    // NULL plane = 0.  (Last in the struct: the other variants' parameter offsets stay where they were.)
    const float *up_color, *up_depth, *up_normal, *up_semantic;
};

// SPSG_FLAG_ALL_PIXELS (the gather's kSegments): row r's pixels are pix[end[r] - num[r], end[r]) (spsg_segments.cuh).  A
// kernel parameter of its own, after BackwardArgs, so that the struct -- and every kernel that takes it -- keeps its layout.
struct SegRows {
    const int32_t *end, *pix;
};

// Clears the 21 gradient slots of voxels [0, N) (replaces the 4 whole-buffer memsets of kernel.cu:557-560): a warp
// takes 32 consecutive voxels, so every store instruction writes one contiguous run of the AoS arrays.
// kSkipHit (one view per chunk): rows of voxels that received pixels are left to the gather, which overwrites them.
// kViewNormals (SPSG_FLAG_VIEW_NORMALS): d_normal holds F rows per voxel, all cleared.
template <bool kSkipHit, bool kViewNormals = false>
__device__ __forceinline__ void zero_rows(const BackwardArgs &a, long long first_warp, long long num_warps) {
    const int lane = threadIdx.x & 31;
    for (long long base = first_warp * 32; base < a.num_locs; base += num_warps * 32) {
        const long long i = base + lane;
        const bool keep = kSkipHit && i < a.num_locs && __ldg(a.mapping3dto2d_num + i) > 0;
        const unsigned kept = __ballot_sync(0xffffffffu, keep);
        const int n = (int)min((long long)32, a.num_locs - base);
        float2 *s = reinterpret_cast<float2 *>(a.d_semantic + (size_t)base * 14);
        for (int e = lane; e < n * 7; e += 32)
            if (!((kept >> (e / 7)) & 1u)) s[e] = make_float2(0.0f, 0.0f);
        float *c = a.d_color + (size_t)base * 3, *nm = a.d_normal + (size_t)base * 3;
        for (int e = lane; e < n * 3; e += 32)
            if (!((kept >> (e / 3)) & 1u)) {
                c[e] = 0.0f;
                if (!kViewNormals) nm[e] = 0.0f;
            }
        if (kViewNormals) {
            float *nv = a.d_normal + (size_t)base * 3 * a.views;
            for (int e = lane; e < n * 3 * a.views; e += 32) nv[e] = 0.0f;
        }
        if (lane < n && !keep) a.d_depth[i] = 0.0f;
    }
}

__global__ void __launch_bounds__(256) backward_zero_kernel(const BackwardArgs a) {
    zero_rows<false>(a, ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ((long long)gridDim.x * blockDim.x) >> 5);
}

__global__ void __launch_bounds__(256) backward_zero_view_normals_kernel(const BackwardArgs a) {
    zero_rows<false, true>(a, ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ((long long)gridDim.x * blockDim.x) >> 5);
}

// zero_rows with C = a.loss.sem_channels semantic slots per voxel (kGenericSem launches)
template <bool kSkipHit, bool kViewNormals = false>
__device__ __forceinline__ void zero_rows_sem(const BackwardArgs &a, long long first_warp, long long num_warps) {
    const int lane = threadIdx.x & 31, C = a.loss.sem_channels;
    for (long long base = first_warp * 32; base < a.num_locs; base += num_warps * 32) {
        const long long i = base + lane;
        const bool keep = kSkipHit && i < a.num_locs && __ldg(a.mapping3dto2d_num + i) > 0;
        const unsigned kept = __ballot_sync(0xffffffffu, keep);
        const int n = (int)min((long long)32, a.num_locs - base);
        float *s = a.d_semantic + (size_t)base * C;
        for (int e = lane; e < n * C; e += 32)
            if (!((kept >> (e / C)) & 1u)) s[e] = 0.0f;
        float *c = a.d_color + (size_t)base * 3, *nm = a.d_normal + (size_t)base * 3;
        for (int e = lane; e < n * 3; e += 32)
            if (!((kept >> (e / 3)) & 1u)) {
                c[e] = 0.0f;
                if (!kViewNormals) nm[e] = 0.0f;
            }
        if (kViewNormals) {
            float *nv = a.d_normal + (size_t)base * 3 * a.views;
            for (int e = lane; e < n * 3 * a.views; e += 32) nv[e] = 0.0f;
        }
        if (lane < n && !keep) a.d_depth[i] = 0.0f;
    }
}

template <bool kViewNormals>
__global__ void __launch_bounds__(256) backward_zero_sem_kernel(const BackwardArgs a) {
    zero_rows_sem<false, kViewNormals>(a, ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5,
                                       ((long long)gridDim.x * blockDim.x) >> 5);
}

// Upstream gradient of one pixel, all 21 channels (g[0..13] semantic, [14..16] colour, [17] depth->sdf, [18..20] normal).
// Plain variant: read from the four gradient images.  Fused variant (pixel_grads_fused): recomputed from the rendering and
// the targets of the 2D losses.
// per-term factors of the fused variant: weight * upstream scale / normaliser (loss_out[4..6]), hoisted out of the pixels
struct FusedCoef { float sem, col, dep; };

__device__ __forceinline__ FusedCoef fused_coef(const BackwardArgs &a) {
    FusedCoef c;
    const float scale = a.grad_scale ? __ldg(a.grad_scale) : 1.0f;
    c.dep = a.w_depth * a.loss.voxelsize * scale / a.loss_out[4];
    c.col = a.w_color * scale / a.loss_out[5];
    c.sem = a.w_sem * scale / a.loss_out[6];
    return c;
}

__device__ __forceinline__ void pixel_grads(const BackwardArgs &a, unsigned gpix, float (&g)[21]) {
    {
        const float2 *s2 = reinterpret_cast<const float2 *>(a.grad_semantic + (size_t)gpix * 14);
#pragma unroll
        for (int k = 0; k < 7; k++) {
            const float2 t = __ldg(s2 + k);
            g[2 * k] = t.x; g[2 * k + 1] = t.y;
        }
        const float *c = a.grad_color + (size_t)gpix * 3, *n = a.grad_normal + (size_t)gpix * 3;
        g[14] = __ldg(c); g[15] = __ldg(c + 1); g[16] = __ldg(c + 2);
        g[17] = __ldg(a.grad_depth + gpix);
        g[18] = __ldg(n); g[19] = __ldg(n + 1); g[20] = __ldg(n + 2);
    }
}

// Fused variant: the pixel's 21 upstream gradients recomputed from the rendering and the 2D losses' targets, written
// into `t` term by term (the gradient images of losses2d_backward_kernel; the gather splits it, see FusedItem).
__device__ __forceinline__ void pixel_grads_fused(const BackwardArgs &a, const FusedCoef &fc, unsigned gpix, float *__restrict__ t) {
    const LossArgs &L = a.loss;
    // semantic: w[y] * (softmax - onehot) / sum_w   (d/dlogits of F.cross_entropy(..., weight), train.py:745)
    const int y = L.target_label ? (int)L.target_label[gpix] : 14;
    bool sem_done = false;
    if (y < 14) {
        float l[14];
        const float2 *s2 = reinterpret_cast<const float2 *>(a.image_semantic + (size_t)gpix * 14);
#pragma unroll
        for (int k = 0; k < 7; k++) {
            const float2 v = __ldg(s2 + k);
            l[2 * k] = v.x; l[2 * k + 1] = v.y;
        }
        if (l[0] != -CUDART_INF_F) {  // valid = (label < 14) & (logit0 != -inf), train.py:744
            float m = l[0];
#pragma unroll
            for (int k = 1; k < 14; k++) m = fmaxf(m, l[k]);
            float sum = 0.0f;
#pragma unroll
            for (int k = 0; k < 14; k++) {
                l[k] = __expf(l[k] - m);  // arguments <= 0; 2^-21 relative error, far inside the gradients' 1e-3 bar
                sum += l[k];
            }
            const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
            const float f = fc.sem * w, fs = f * __frcp_rn(sum);
#pragma unroll
            for (int k = 0; k < 14; k++) t[k] = l[k] * fs - (k == y ? f : 0.0f);
            sem_done = true;
        }
    }
    if (!sem_done) {
#pragma unroll
        for (int k = 0; k < 14; k++) t[k] = 0.0f;
    }
    float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
    if (L.target_color) {  // d/dc mean|c*w - t*w|  (loss.py:246-257)
        const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
        const float *c = a.image_color + (size_t)gpix * 3, *tc = L.target_color + (size_t)gpix * 3;
        const float c0 = __ldg(c), c1 = __ldg(c + 1), c2 = __ldg(c + 2);
        const float d0 = __fadd_rn(__fmul_rn(c0, w), -__fmul_rn(__ldg(tc), w));
        const float d1 = __fadd_rn(__fmul_rn(c1, w), -__fmul_rn(__ldg(tc + 1), w));
        const float d2 = __fadd_rn(__fmul_rn(c2, w), -__fmul_rn(__ldg(tc + 2), w));
        const float f = fc.col * w;
        if (c0 != -CUDART_INF_F) g0 = f * (float)((d0 > 0.0f) - (d0 < 0.0f));  // valid = != -inf
        if (c1 != -CUDART_INF_F) g1 = f * (float)((d1 > 0.0f) - (d1 < 0.0f));
        if (c2 != -CUDART_INF_F) g2 = f * (float)((d2 > 0.0f) - (d2 < 0.0f));
    }
    t[14] = g0; t[15] = g1; t[16] = g2;
    float gd = 0.0f;
    if (L.target_depth) {  // d/ddepth mean|depth*voxelsize - t|  (train.py:635-638)
        const float td = __ldg(L.target_depth + gpix);
        const float r = __ldg(a.image_depth + gpix);
        if (td != 0.0f && r != -CUDART_INF_F) {
            const float d = __fmul_rn(r, L.voxelsize) - td;
            gd = fc.dep * (float)((d > 0.0f) - (d < 0.0f));
        }
    }
    t[17] = gd; t[18] = 0.0f; t[19] = 0.0f; t[20] = 0.0f;
}

// The gather's fused variant splits pixel_grads_fused into what is shared by all pixels of a (voxel, view) item and what
// is not.  The forward fills every pixel it registers to row (view, voxel) with plain copies of that voxel's 14 logits and
// 3 colours, so the item's logits and colour are read once, from its first registered pixel, and the softmax is formed
// once per item (fused_item: lane c < 14 loads logit c, e_c = exp(l_c - max) goes to shared memory, every lane holds
// 1 / sum_k e_k).  Each pixel then reads only its label, class weight, targets and rendered depth (fused_pixel_grads).
// Every term is rounded as pixel_grads_fused rounds it: the sum in k order, t_k = fma(e_k, f * rcp(sum), -[k == y] f).
struct FusedItem {
    float rs;          // __frcp_rn(sum_k e_k)
    bool sem;          // label targets given and logit 0 != -inf (train.py:744)
    float c0, c1, c2;  // the item's rendered colour
};

template <int G>
__device__ __forceinline__ FusedItem fused_item(const BackwardArgs &a, unsigned gpix0, int hl, unsigned hmask,
                                                float *__restrict__ e) {
    FusedItem it = {0.0f, false, 0.0f, 0.0f, 0.0f};
    if (a.loss.target_label) {
        // lanes >= 14 carry NaN, which fmaxf drops; the max does not depend on the order it is taken in
        const float l = hl < 14 ? __ldg(a.image_semantic + (size_t)gpix0 * 14 + hl) : CUDART_NAN_F;
        it.sem = __shfl_sync(hmask, l, 0, G) != -CUDART_INF_F;
        if (it.sem) {
            float m = l;
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(hmask, m, o, G));
            const float ec = __expf(l - m);
            if (hl < 14) e[hl] = ec;
            float sum = 0.0f;  // k order, as pixel_grads_fused adds them
#pragma unroll
            for (int k = 0; k < 14; k++) sum += __shfl_sync(hmask, ec, k, G);
            it.rs = __frcp_rn(sum);
        }
    }
    if (a.loss.target_color) {
        const float *c = a.image_color + (size_t)gpix0 * 3;
        it.c0 = __ldg(c); it.c1 = __ldg(c + 1); it.c2 = __ldg(c + 2);
    }
    __syncwarp(hmask);
    return it;
}

// One registered pixel of a fused item: its 21 gradients, as pixel_grads_fused, from the item's terms (e: the e_k that
// fused_item stored) and the pixel's own targets and depth.
__device__ __forceinline__ void fused_pixel_grads(const BackwardArgs &a, const FusedCoef &fc, const FusedItem &it,
                                                  const float *__restrict__ e, unsigned gpix, float *__restrict__ t) {
    const LossArgs &L = a.loss;
    const int y = it.sem ? (int)L.target_label[gpix] : 14;
    if (y < 14) {
        const float f = __fmul_rn(fc.sem, L.class_weight ? __ldg(L.class_weight + y) : 1.0f), fs = __fmul_rn(f, it.rs);
#pragma unroll
        for (int k = 0; k < 14; k++) t[k] = __fmaf_rn(e[k], fs, -(k == y ? f : 0.0f));
    } else {
#pragma unroll
        for (int k = 0; k < 14; k++) t[k] = 0.0f;
    }
    float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
    if (L.target_color) {  // d/dc mean|c*w - t*w|  (loss.py:246-257)
        const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
        const float *tc = L.target_color + (size_t)gpix * 3;
        const float d0 = __fadd_rn(__fmul_rn(it.c0, w), -__fmul_rn(__ldg(tc), w));
        const float d1 = __fadd_rn(__fmul_rn(it.c1, w), -__fmul_rn(__ldg(tc + 1), w));
        const float d2 = __fadd_rn(__fmul_rn(it.c2, w), -__fmul_rn(__ldg(tc + 2), w));
        const float fw = fc.col * w;
        if (it.c0 != -CUDART_INF_F) g0 = fw * (float)((d0 > 0.0f) - (d0 < 0.0f));  // valid = != -inf
        if (it.c1 != -CUDART_INF_F) g1 = fw * (float)((d1 > 0.0f) - (d1 < 0.0f));
        if (it.c2 != -CUDART_INF_F) g2 = fw * (float)((d2 > 0.0f) - (d2 < 0.0f));
    }
    t[14] = g0; t[15] = g1; t[16] = g2;
    float gd = 0.0f;
    if (L.target_depth) {  // d/ddepth mean|depth*voxelsize - t|  (train.py:635-638)
        const float td = __ldg(L.target_depth + gpix);
        const float r = __ldg(a.image_depth + gpix);
        if (td != 0.0f && r != -CUDART_INF_F) {
            const float d = __fmul_rn(r, L.voxelsize) - td;
            gd = fc.dep * (float)((d > 0.0f) - (d < 0.0f));
        }
    }
    t[17] = gd; t[18] = 0.0f; t[19] = 0.0f; t[20] = 0.0f;
}

// kUpstream: the caller's gradient images of the same pixel added, in fp32, onto the row fused_pixel_grads just wrote
// (read-modify-write of shared memory rather than 21 more live registers).  Which planes are present is the same for the
// whole launch, so the branches do not diverge.  Not scaled by grad_scale: that is d objective / d loss_out[3] only.
__device__ __forceinline__ void add_upstream_grads(const BackwardArgs &a, unsigned gpix, float *__restrict__ t) {
    if (a.up_semantic) {
        const float2 *s2 = reinterpret_cast<const float2 *>(a.up_semantic + (size_t)gpix * 14);
#pragma unroll
        for (int k = 0; k < 7; k++) {
            const float2 v = __ldg(s2 + k);
            t[2 * k] += v.x; t[2 * k + 1] += v.y;
        }
    }
    if (a.up_color) {
        const float *c = a.up_color + (size_t)gpix * 3;
        t[14] += __ldg(c); t[15] += __ldg(c + 1); t[16] += __ldg(c + 2);
    }
    if (a.up_depth) t[17] += __ldg(a.up_depth + gpix);
    if (a.up_normal) {
        const float *n = a.up_normal + (size_t)gpix * 3;
        t[18] += __ldg(n); t[19] += __ldg(n + 1); t[20] += __ldg(n + 2);
    }
}

// ---- C-generic twins of the four per-pixel helpers above (kGenericSem).  A pixel's row has R = C + 7 channels: [0, C)
// semantic, [C, C+3) colour, C+3 depth->sdf, [C+4, C+7) normal -- at C = 14 exactly the 21-channel layout.  Every term is
// rounded as its 14-channel counterpart rounds it.
__device__ __forceinline__ void pixel_grads_sem(const BackwardArgs &a, int C, unsigned gpix, float *__restrict__ t) {
    const float *s = a.grad_semantic + (size_t)gpix * C;
#pragma unroll 1
    for (int k = 0; k < C; k++) t[k] = __ldg(s + k);
    const float *c = a.grad_color + (size_t)gpix * 3, *n = a.grad_normal + (size_t)gpix * 3;
    t[C] = __ldg(c); t[C + 1] = __ldg(c + 1); t[C + 2] = __ldg(c + 2);
    t[C + 3] = __ldg(a.grad_depth + gpix);
    t[C + 4] = __ldg(n); t[C + 5] = __ldg(n + 1); t[C + 6] = __ldg(n + 2);
}

// pixel_grads_fused over C logits (the stand-alone backward's gradient images)
__device__ __forceinline__ void pixel_grads_fused_sem(const BackwardArgs &a, const FusedCoef &fc, int C, unsigned gpix,
                                                      float *__restrict__ t) {
    const LossArgs &L = a.loss;
    const int y = L.target_label ? (int)L.target_label[gpix] : C;
    const float *l = a.image_semantic + (size_t)gpix * C;
    if (y < C && __ldg(l) != -CUDART_INF_F) {  // valid = (label < C) & (logit0 != -inf)
        float m = __ldg(l);
#pragma unroll 1
        for (int k = 1; k < C; k++) m = fmaxf(m, __ldg(l + k));
        float sum = 0.0f;
#pragma unroll 1
        for (int k = 0; k < C; k++) {
            const float e = __expf(__ldg(l + k) - m);
            t[k] = e;
            sum += e;
        }
        const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
        const float f = fc.sem * w, fs = f * __frcp_rn(sum);
#pragma unroll 1
        for (int k = 0; k < C; k++) t[k] = t[k] * fs - (k == y ? f : 0.0f);
    } else {
#pragma unroll 1
        for (int k = 0; k < C; k++) t[k] = 0.0f;
    }
    float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
    if (L.target_color) {
        const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
        const float *c = a.image_color + (size_t)gpix * 3, *tc = L.target_color + (size_t)gpix * 3;
        const float c0 = __ldg(c), c1 = __ldg(c + 1), c2 = __ldg(c + 2);
        const float d0 = __fadd_rn(__fmul_rn(c0, w), -__fmul_rn(__ldg(tc), w));
        const float d1 = __fadd_rn(__fmul_rn(c1, w), -__fmul_rn(__ldg(tc + 1), w));
        const float d2 = __fadd_rn(__fmul_rn(c2, w), -__fmul_rn(__ldg(tc + 2), w));
        const float f = fc.col * w;
        if (c0 != -CUDART_INF_F) g0 = f * (float)((d0 > 0.0f) - (d0 < 0.0f));
        if (c1 != -CUDART_INF_F) g1 = f * (float)((d1 > 0.0f) - (d1 < 0.0f));
        if (c2 != -CUDART_INF_F) g2 = f * (float)((d2 > 0.0f) - (d2 < 0.0f));
    }
    t[C] = g0; t[C + 1] = g1; t[C + 2] = g2;
    float gd = 0.0f;
    if (L.target_depth) {
        const float td = __ldg(L.target_depth + gpix);
        const float r = __ldg(a.image_depth + gpix);
        if (td != 0.0f && r != -CUDART_INF_F) {
            const float d = __fmul_rn(r, L.voxelsize) - td;
            gd = fc.dep * (float)((d > 0.0f) - (d < 0.0f));
        }
    }
    t[C + 3] = gd; t[C + 4] = 0.0f; t[C + 5] = 0.0f; t[C + 6] = 0.0f;
}

// fused_item over C logits: lane c of the group loads logits c, c + G, ...; e_k goes to e[k], the sum is taken in k order
// from there (what the 14-channel shuffles add, in the same order)
template <int G>
__device__ __forceinline__ FusedItem fused_item_sem(const BackwardArgs &a, int C, unsigned gpix0, int hl, unsigned hmask,
                                                    float *__restrict__ e) {
    FusedItem it = {0.0f, false, 0.0f, 0.0f, 0.0f};
    if (a.loss.target_label) {
        const float *l = a.image_semantic + (size_t)gpix0 * C;
        float m = CUDART_NAN_F;  // fmaxf drops it: lanes without a channel do not take part
        for (int k = hl; k < C; k += G) m = fmaxf(m, __ldg(l + k));
        it.sem = __ldg(l) != -CUDART_INF_F;
        if (it.sem) {
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(hmask, m, o, G));
            for (int k = hl; k < C; k += G) e[k] = __expf(__ldg(l + k) - m);
            __syncwarp(hmask);
            float sum = 0.0f;
            for (int k = 0; k < C; k++) sum += e[k];
            it.rs = __frcp_rn(sum);
        }
    }
    if (a.loss.target_color) {
        const float *c = a.image_color + (size_t)gpix0 * 3;
        it.c0 = __ldg(c); it.c1 = __ldg(c + 1); it.c2 = __ldg(c + 2);
    }
    __syncwarp(hmask);
    return it;
}

// fused_pixel_grads over C logits
__device__ __forceinline__ void fused_pixel_grads_sem(const BackwardArgs &a, const FusedCoef &fc, const FusedItem &it, int C,
                                                      const float *__restrict__ e, unsigned gpix, float *__restrict__ t) {
    const LossArgs &L = a.loss;
    const int y = it.sem ? (int)L.target_label[gpix] : C;
    if (y < C) {
        const float f = __fmul_rn(fc.sem, L.class_weight ? __ldg(L.class_weight + y) : 1.0f), fs = __fmul_rn(f, it.rs);
#pragma unroll 1
        for (int k = 0; k < C; k++) t[k] = __fmaf_rn(e[k], fs, -(k == y ? f : 0.0f));
    } else {
#pragma unroll 1
        for (int k = 0; k < C; k++) t[k] = 0.0f;
    }
    float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
    if (L.target_color) {
        const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
        const float *tc = L.target_color + (size_t)gpix * 3;
        const float d0 = __fadd_rn(__fmul_rn(it.c0, w), -__fmul_rn(__ldg(tc), w));
        const float d1 = __fadd_rn(__fmul_rn(it.c1, w), -__fmul_rn(__ldg(tc + 1), w));
        const float d2 = __fadd_rn(__fmul_rn(it.c2, w), -__fmul_rn(__ldg(tc + 2), w));
        const float fw = fc.col * w;
        if (it.c0 != -CUDART_INF_F) g0 = fw * (float)((d0 > 0.0f) - (d0 < 0.0f));
        if (it.c1 != -CUDART_INF_F) g1 = fw * (float)((d1 > 0.0f) - (d1 < 0.0f));
        if (it.c2 != -CUDART_INF_F) g2 = fw * (float)((d2 > 0.0f) - (d2 < 0.0f));
    }
    t[C] = g0; t[C + 1] = g1; t[C + 2] = g2;
    float gd = 0.0f;
    if (L.target_depth) {
        const float td = __ldg(L.target_depth + gpix);
        const float r = __ldg(a.image_depth + gpix);
        if (td != 0.0f && r != -CUDART_INF_F) {
            const float d = __fmul_rn(r, L.voxelsize) - td;
            gd = fc.dep * (float)((d > 0.0f) - (d < 0.0f));
        }
    }
    t[C + 3] = gd; t[C + 4] = 0.0f; t[C + 5] = 0.0f; t[C + 6] = 0.0f;
}

__device__ __forceinline__ void add_upstream_grads_sem(const BackwardArgs &a, int C, unsigned gpix, float *__restrict__ t) {
    if (a.up_semantic) {
        const float *s = a.up_semantic + (size_t)gpix * C;
#pragma unroll 1
        for (int k = 0; k < C; k++) t[k] += __ldg(s + k);
    }
    if (a.up_color) {
        const float *c = a.up_color + (size_t)gpix * 3;
        t[C] += __ldg(c); t[C + 1] += __ldg(c + 1); t[C + 2] += __ldg(c + 2);
    }
    if (a.up_depth) t[C + 3] += __ldg(a.up_depth + gpix);
    if (a.up_normal) {
        const float *n = a.up_normal + (size_t)gpix * 3;
        t[C + 4] += __ldg(n); t[C + 5] += __ldg(n + 1); t[C + 6] += __ldg(n + 2);
    }
}

// The gather (kernel.cu:391-419 turned inside out).  Work items are the (voxel, view) pairs the forward listed; one
// warp per item.  Lane k fetches the k-th registered pixel id (one coalesced load) and that pixel's 21 upstream
// gradients (independent 8- and 4-byte loads; the fused variant reads only its targets and depth, see FusedItem), parks
// them in shared memory, and lane c then adds column c in registration order (kernel.cu:398-418: mean = sum / count),
// accumulating in double precision: the registration order
// depends on which warp's atomic reached a voxel first, and a double sum rounded once gives the same fp32 mean for every
// order (up to an exact tie).  With one view per chunk the result is written with plain stores, no float atomics; with several
// views see kViews in the loop.
constexpr int kGatherWarps = 8;
#ifndef SPSG_GATHER_GROUP
#define SPSG_GATHER_GROUP 16
#endif
constexpr int kGatherGroup = SPSG_GATHER_GROUP;  // lanes per (voxel, view) item

// kViews: 0 = one view per chunk; 1 = several, per-view means added with float atomics (fast); 2 = several, deterministic
// kUpstream (needs kFused): each pixel's row is the recomputed loss gradient plus the caller's upstream gradient images
// kViewNormals (needs kViews != 0, SPSG_FLAG_VIEW_NORMALS): the normal channels of item (voxel, view) are that view's mean,
// stored to row (voxel, view) of the (N,F,3) d_normal; the other channels are gathered as without it
// kSegments (SPSG_FLAG_ALL_PIXELS): a row's pixels are its segment of seg_pix, all num[row] of them (no cap), instead of
// the first min(num, max_pixels) entries of its mapping3dto2d row
// kGenericSem (C = a.loss.sem_channels != 14, or SPSG_FLAG_GENERIC_SEMANTIC): rows of R = C + 7 channels, staged in dynamic
// shared memory (kGatherWarps * 32 / G * G * R floats: 21.5 KB at C = 14, 72.7 KB at C = 64), the per-pixel helpers'
// *_sem twins; lane c of a group sums channels c, c + G, ... as without it
template <bool kFused, bool kUpstream, int kViews, bool kViewNormals, bool kSegments = false, bool kGenericSem = false>
#ifndef SPSG_GATHER_MIN_BLOCKS
#define SPSG_GATHER_MIN_BLOCKS 8  // 32 registers: full occupancy hides the dependent gathers (the fused variants spill 24-92 B and are still faster)
#endif
// kSegments: the row's segment start is one more dependent load; at 8 CTAs per SM (32 registers) that variant spills more
// than the table variant of the same instantiation, at 5 (48 registers) less than it
__global__ void __launch_bounds__(kGatherWarps * 32, kSegments ? 5 : SPSG_GATHER_MIN_BLOCKS) backward_gather_kernel(const BackwardArgs a,
                                                                                                    const SegRows seg) {
    static_assert(kFused || !kUpstream, "upstream images are added to the fused variant's recomputed gradients");
    static_assert(kViews != 0 || !kViewNormals, "per-view normal rows need several views per chunk");
    if ((int)blockIdx.x < a.zero_blocks) {
        if (kGenericSem) {
            zero_rows_sem<true>(a, ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ((long long)a.zero_blocks * blockDim.x) >> 5);
            return;
        }
        zero_rows<true>(a, ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ((long long)a.zero_blocks * blockDim.x) >> 5);
        return;
    }
    // kGatherGroup lanes per item, 32 / kGatherGroup items in flight per warp: the groups work on different items
    constexpr int G = kGatherGroup, kPerWarp = 32 / G;
    constexpr int kSlots = ((kGenericSem ? kMaxSemanticChannels + 7 : 21) + G - 1) / G;
    static_assert(!kFused || G >= 14, "the fused variant's softmax takes one lane per semantic channel");
    __shared__ float s_g[kGenericSem ? 1 : kGatherWarps * kPerWarp][kGenericSem ? 1 : G * 21];
    extern __shared__ float s_dyn[];  // kGenericSem: the groups' rows of R floats
    constexpr int kE = kGenericSem ? kMaxSemanticChannels : 16;
    __shared__ __align__(16) float s_e[kFused ? kGatherWarps * kPerWarp : 1][kE];  // fused: the item's e_k (FusedItem)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hl = lane & (G - 1), half = lane / G;
    const unsigned hmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (G * half);
    const int C = kGenericSem ? a.loss.sem_channels : 14, R = kGenericSem ? C + 7 : 21;
    float *tile = kGenericSem ? s_dyn + (size_t)(warp * kPerWarp + half) * G * R : s_g[warp * kPerWarp + half];
    const int groups_total = (int)(gridDim.x - a.zero_blocks) * kGatherWarps * kPerWarp;
    const int count = *a.list_count;
    const unsigned P = (unsigned)(a.width * a.height);
    int item = (((int)blockIdx.x - a.zero_blocks) * kGatherWarps + warp) * kPerWarp + half;
    int2 e = item < count ? a.list[item] : make_int2(0, 0);
    FusedCoef fc = {0.0f, 0.0f, 0.0f};
    if (kFused) fc = fused_coef(a);
    // (Tried: a two-deep software pipeline that also fetches the next item's pixel count and first pixel ids ahead of time.
    // Slower -- fused 161 -> 223 us, plain 105 -> 112 us on C3: it doubles the registers and halves the occupancy that
    // hides these dependent loads in the first place.)
    while (item < count) {
        const int idx = e.x, img = e.y;
        const int next_item = item + groups_total;
        if (next_item < count) e = a.list[next_item];  // prefetch the next pair
        // One view per chunk: the item is the voxel, its mean is written with plain stores.  Several views: the forward listed
        // one item per (voxel, view) that received pixels.  kViews == 1: every item adds its view's mean with float atomics
        // onto rows the forward (or the zero kernel) cleared.  kViews == 2 (SPSG_FLAG_DETERMINISTIC_GRADS): the item of the
        // voxel's LOWEST such view does the whole voxel -- the per-view means added in view order (what F reference calls
        // accumulated by autograd give), plain stores -- and the others step aside: nothing depends on the order in which
        // items run, gradients are bit-reproducible, at the price of longer dependent chains (gather +30 % on C3).
        const int view0 = kViews ? img % a.views : 0, image0 = img - view0;
        bool owner = true;
        if (kViews == 2)
            for (int f = 0; f < view0; f++)
                if (__ldg(a.mapping3dto2d_num + (size_t)f * a.num_locs + idx) > 0) owner = false;
        if (owner) {
            float tot[kSlots];
#pragma unroll
            for (int j = 0; j < kSlots; j++) tot[j] = 0.0f;
            for (int view = view0; view < (kViews == 2 ? a.views : view0 + 1); view++) {
                const size_t row = (size_t)view * a.num_locs + idx;
                const int32_t *prow = kSegments ? seg.pix : a.mapping3dto2d + row * a.max_pixels;
                const int num = max(__ldg(a.mapping3dto2d_num + row), 0);
                const int cnt = kSegments ? num : min(num, a.max_pixels);  // kernel.cu:392-393
                if (cnt == 0) continue;
                if (kSegments) prow += __ldg(seg.end + row) - cnt;
                const unsigned pixbase = (unsigned)(image0 + view) * P;  // global pixel index < 2^32 / 14 (check_params)
                const float inv = __frcp_rn((float)cnt);
                FusedItem it;
                if (kFused && kGenericSem)
                    it = fused_item_sem<G>(a, C, pixbase + (unsigned)__ldg(prow), hl, hmask, s_e[warp * kPerWarp + half]);
                else if (kFused)
                    it = fused_item<G>(a, pixbase + (unsigned)__ldg(prow), hl, hmask, s_e[warp * kPerWarp + half]);
                double acc[kSlots];  // channels hl + G j; double: the sum does not depend on the pixel order to fp32 precision
#pragma unroll
                for (int j = 0; j < kSlots; j++) acc[j] = 0.0;
                for (int k0 = 0; k0 < cnt; k0 += G) {
                    const int m = min(G, cnt - k0);
                    if (hl < m) {
                        const unsigned gpix = pixbase + (unsigned)__ldg(prow + k0 + hl);
                        if (kGenericSem) {
                            if (kFused) {
                                fused_pixel_grads_sem(a, fc, it, C, s_e[warp * kPerWarp + half], gpix, tile + hl * R);
                                if (kUpstream) add_upstream_grads_sem(a, C, gpix, tile + hl * R);
                            } else {
                                pixel_grads_sem(a, C, gpix, tile + hl * R);
                            }
                        } else if (kFused) {
                            fused_pixel_grads(a, fc, it, s_e[warp * kPerWarp + half], gpix, tile + hl * 21);
                            if (kUpstream) add_upstream_grads(a, gpix, tile + hl * 21);
                        } else {
                            float g[21];
                            pixel_grads(a, gpix, g);
#pragma unroll
                            for (int c = 0; c < 21; c++) tile[hl * 21 + c] = g[c];
                        }
                    }
                    __syncwarp(hmask);
                    for (int r = 0; r < m; r++) {
#pragma unroll
                        for (int j = 0; j < kSlots; j++)
                            if (hl + G * j < R) acc[j] += (double)tile[r * R + hl + G * j];
                    }
                    __syncwarp(hmask);
                }
#pragma unroll
                for (int j = 0; j < kSlots; j++) {
                    const float mean = (float)(acc[j] * (double)inv);  // mean = sum / count (kernel.cu:398-418)
                    const int c = hl + G * j;
                    if (kViewNormals && c >= R - 3 && c < R) a.d_normal[((size_t)idx * a.views + view) * 3 + (c - (R - 3))] = mean;
                    else tot[j] += mean;
                }
            }
            // channel c -> destination: 0-13 semantic, 14-16 colour, 17 depth->sdf, 18-20 normal (generic: C, C+3, C+4)
#pragma unroll
            for (int j = 0; j < kSlots; j++) {
                const int c = hl + G * j;
                if (c < (kViewNormals ? R - 3 : R)) {
                    float *d = c < C ? a.d_semantic + (size_t)idx * C + c
                             : c < C + 3 ? a.d_color + (size_t)idx * 3 + (c - C)
                             : c == C + 3 ? a.d_depth + idx : a.d_normal + (size_t)idx * 3 + (c - (C + 4));
                    if (kViews == 1) atomicAdd(d, tot[j]);
                    else *d = tot[j];
                }
            }
        }
        item = next_item;
    }
}
