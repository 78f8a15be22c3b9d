// spsg_raycast.cu -- hand-written sm_100a kernels + C ABI of the SPSG-semantic raycaster.
//
// Functional contract: reference torch/utils/raycast_rgbd/raycast_rgbd_cuda_kernel.cu (cited per function
// as kernel.cu:<line>) evaluated with the exact fp32 operation order of its sm_100 SASS (SURVEY.md
// section 3.5; re-derived from `cuobjdump -sass oracle/_ref/*.so`).  Every rounding that can change a hit
// mask is spelled with __f*_rn intrinsics so nvcc can neither contract nor re-associate it.
//
// Design (not a port): see DESIGN.md.  In short
//   * the march replays the reference's `ray += inc` running sum bit-exactly but jumps over samples whose
//     outcome is known without evaluating them: samples outside the grid, samples inside an aligned 4/8/16/32-
//     voxel region without any valid sample cell ("empty"), and samples inside a region whose valid cells all
//     have 8 strictly positive (or all strictly negative) corners ("sign-uniform": no crossing can start there);
//     jumps use a closed form of the fp32 recurrence that is exact inside one binade;
//   * one byte per 4^3 block (region kind + size, staged in shared memory) and one byte per cell (class of the
//     cell's 8 corners) answer "does this sample need arithmetic"; SDF values come from a dense fp32 brick
//     (NaN = absent voxel), so a sample that does need arithmetic costs 8 independent loads, not 16 dependent ones;
//   * the regula-falsi refinement is deferred until every lane of the warp has found its crossing;
//   * rendered pixels are staged in shared memory and written with coalesced 128-bit stores;
//   * the forward appends every (voxel, view) pair that received a pixel to a list, so the backward is one launch:
//     a per-voxel gather over that list (no float atomics for one view per chunk, no 524288-block
//     launch, no 164 MB memsets), optionally fused with the 2D losses.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "spsg_raycast.h"

namespace {

// the device side, in dependency order
#include "spsg_common.cuh"
#include "spsg_fp32.cuh"
#include "spsg_prep.cuh"
#include "spsg_forward.cuh"
#include "spsg_backward.cuh"
#include "spsg_losses2d.cuh"
#include "spsg_occ.cuh"
#include "spsg_normals.cuh"

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------

int check_params(const spsg_raycast_params *p) {
    if (!p) return fail(SPSG_ERR_INVALID_ARGUMENT, "params is NULL");
    if (p->width <= 0 || p->height <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "width/height must be positive");
    if (p->dimx <= 0 || p->dimy <= 0 || p->dimz <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "dims must be positive");
    if (p->num_chunks <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "num_chunks must be positive");
    if (p->views_per_chunk <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "views_per_chunk must be >= 1");
    if (p->num_locs < 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "num_locs must be >= 0");
    if ((long long)p->num_chunks * p->dimx * p->dimy * p->dimz >= (1ll << 31))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "dense grid exceeds 32-bit indexing (reference limit, SURVEY 3.5)");
    if ((long long)p->num_chunks * p->views_per_chunk * p->width * p->height * 14 >= (1ll << 32))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "image batch exceeds 32-bit indexing (reference limit, SURVEY 3.5)");
    if ((long long)p->num_locs * p->views_per_chunk >= (1ll << 31))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "num_locs * views_per_chunk exceeds 32-bit indexing");
    return SPSG_OK;
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cached[dev] = sms > 0 ? sms : 148;
    }
    return cached[dev];
}

LossArgs make_loss_args(const spsg_loss_targets *t, double *accum) {
    LossArgs L;
    memset(&L, 0, sizeof(L));
    if (t) {
        L.target_depth = t->target_depth; L.target_color = t->target_color; L.weight_color = t->weight_color;
        L.target_label = t->target_label; L.class_weight = t->class_weight; L.voxelsize = t->voxelsize;
    }
    L.accum = accum;
    L.loss_out = nullptr; L.done = nullptr;
    if (t) { L.w_depth = t->weight_depth; L.w_color = t->weight_color_loss; L.w_sem = t->weight_semantic; }
    return L;
}

int launch_forward(const spsg_raycast_params *p, bool build_index, int32_t *sparse_mapping, const int64_t *locs,
                   const float *vals_sdf, const float *vals_color, const float *vals_normal,
                   const float *vals_semantic, const float *view_matrix, const float *intrinsics, float *image_color,
                   float *image_depth, float *image_normal, float *image_semantic, int32_t *mapping3dto2d,
                   int32_t *mapping3dto2d_num, const spsg_loss_targets *targets, float *loss_out,
                   const spsg_grad_buffers *clear_grads, void *workspace, size_t workspace_bytes, cudaStream_t st) {
    if (int rc = check_params(p)) return rc;
    if (p->max_pixels_per_voxel <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "max_pixels_per_voxel must be positive");
    if (!sparse_mapping || !view_matrix || !intrinsics || !image_color || !image_depth || !image_normal ||
        !image_semantic || !mapping3dto2d || !mapping3dto2d_num)
        return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL tensor pointer");
    if (p->num_locs > 0 && (!locs || !vals_sdf || !vals_color || !vals_normal || !vals_semantic))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL voxel tensor pointer");
    if (!aligned16(view_matrix) || !aligned16(intrinsics))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "view_matrix / intrinsics must be 16-byte aligned");
    const bool packed = (p->flags & SPSG_FLAG_PACKED_LOCS) != 0;
    if (p->num_locs > 0 && ((reinterpret_cast<uintptr_t>(vals_semantic) & 7u) || (reinterpret_cast<uintptr_t>(locs) & (packed ? 3u : 15u))))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "vals_semantic must be 8-byte and locs 16-byte (packed: 4-byte) aligned");
    if (packed && !build_index) return fail(SPSG_ERR_INVALID_ARGUMENT, "packed locs need an entry point that builds the index");
    if (packed && (unsigned long long)p->num_chunks * p->dimz * p->dimy * p->dimx >= 0xffffffffull)
        return fail(SPSG_ERR_INVALID_ARGUMENT, "packed locs need fewer than 2^32 - 1 cells");
    if (reinterpret_cast<uintptr_t>(sparse_mapping) & 3u) return fail(SPSG_ERR_INVALID_ARGUMENT, "sparse_mapping must be 4-byte aligned");
    if (targets && !loss_out) return fail(SPSG_ERR_INVALID_ARGUMENT, "loss_out is NULL");
    const Layout L = make_layout(p);
    if (!workspace || workspace_bytes < L.total) return fail(SPSG_ERR_WORKSPACE_TOO_SMALL, "workspace too small");
    if (reinterpret_cast<uintptr_t>(workspace) & 255u) return fail(SPSG_ERR_INVALID_ARGUMENT, "workspace must be 256-byte aligned");
    uint8_t *ws = (uint8_t *)workspace;
    float *dense = (float *)(ws + L.dense_off);
    uint2 *vbits = (uint2 *)(ws + L.vbit_off);
    uint8_t *bmap = ws + L.bmap_off, *marks = ws + L.marks_off;
    double *accum = (double *)(ws + L.loss_off);
    const size_t cells = (size_t)p->num_chunks * p->dimz * p->dimy * p->dimx;
    const int sms = sm_count();
    const bool prebuilt = (p->flags & SPSG_FLAG_INDEX_PREBUILT) && p->num_locs > 0;

    {
        // sparse_mapping := -1 (kernel.cu:515), dense brick := NaN (0xffffffff: every voxel absent), block marks / list
        // counter / loss accumulators := 0 -- one launch
        FillArgs f;
        memset(&f, 0, sizeof(f));
        f.ptr[0] = build_index ? (uint32_t *)sparse_mapping : nullptr; f.words[0] = cells; f.value[0] = 0xffffffffu;
        f.ptr[1] = (uint32_t *)dense; f.words[1] = L.dense_bytes / 4; f.value[1] = 0xffffffffu;
        if (prebuilt) {
            // index and brick were written together with locs (spsg_sparsify_locs_indexed): what is left of the two
            // passes is the reset of the voxel -> pixel counters, rows [0, F * N)
            f.ptr[0] = (uint32_t *)mapping3dto2d_num; f.words[0] = (size_t)p->views_per_chunk * p->num_locs; f.value[0] = 0u;
            f.ptr[1] = nullptr; f.words[1] = 0;
        }
        f.ptr[2] = (uint32_t *)(ws + L.zero_off); f.words[2] = L.zero_bytes / 4; f.value[2] = 0u;
        if (clear_grads && p->num_locs > 0 &&
            (!clear_grads->d_color || !clear_grads->d_depth || !clear_grads->d_normal || !clear_grads->d_semantic))
            return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL gradient pointer in clear_grads");
        const size_t vecs = ((prebuilt ? f.words[0] : cells * (build_index ? 2 : 1)) + L.zero_bytes / 4) / 4;
        const unsigned blocks = (unsigned)std::min<size_t>((vecs + 1023) / 1024 + 1, (size_t)sms * 8);
        fill_kernel<<<blocks, 256, 0, st>>>(f);
        CUDA_TRY(cudaGetLastError());
    }
    if (p->num_locs > 0 && !prebuilt) {
        const unsigned blocks = (unsigned)((p->num_locs + 255) / 256);
        if (packed)
            index_packed_kernel<<<blocks, 256, 0, st>>>((const uint32_t *)locs, p->num_locs, sparse_mapping, vals_sdf, dense,
                                                        mapping3dto2d_num, p->views_per_chunk, (unsigned long long)cells);
        else if (build_index)
            index_kernel<true><<<blocks, 256, 0, st>>>((const longlong4 *)locs, p->num_locs, sparse_mapping, vals_sdf,
                                                       dense, mapping3dto2d_num, p->views_per_chunk, p->dimz, p->dimy,
                                                       p->dimx, p->num_chunks);
        else
            index_kernel<false><<<blocks, 256, 0, st>>>((const longlong4 *)locs, p->num_locs, sparse_mapping, vals_sdf,
                                                        dense, mapping3dto2d_num, p->views_per_chunk, p->dimz, p->dimy,
                                                        p->dimx, p->num_chunks);
        CUDA_TRY(cudaGetLastError());
    }
    ForwardArgs a;
    memset(&a, 0, sizeof(a));
    // shared-memory residency of one chunk's maps: class bit planes + block map
    const size_t map_bytes = L.vpc * sizeof(uint2) + L.bpc;
    // One chunk: the maps are TMA-staged in shared memory (the launch is one wave, latency-bound: the staging overlaps the
    // first tile's set-up and every look-up stays on the SM).  Several chunks: the maps are read through L1 instead, which is
    // as fast per look-up (C3: 538 vs 534 us with the same scheduling) and frees the CTAs from their chunks -- one global
    // tile counter, no chunk-switch barriers, no tail behind them (C3 forward 483 -> 455 us).  Flags force either path.
    a.maps_in_smem = kFwdSmemFixed + map_bytes <= kFwdSmemMax && !(p->flags & SPSG_FLAG_GLOBAL_MAPS) &&
                     (p->num_chunks == 1 || (p->flags & SPSG_FLAG_SMEM_MAPS));
    {
        const dim3 cgrid((unsigned)((L.nby * L.wpr + 3) / 4), (unsigned)L.nbz, (unsigned)p->num_chunks);
        cell_class_kernel<<<cgrid, 128, 0, st>>>(dense, vbits, L.vpc, marks, p->dimz, p->dimy, p->dimx, L.wpr, L.nby, L.nbx, L.bpc,
                                                 bmap, (int32_t *)(ws + L.arrive_off), L.nbz);
        CUDA_TRY(cudaGetLastError());
    }
    a.sparse_mapping = sparse_mapping;
    a.vals_sdf = vals_sdf; a.vals_color = vals_color; a.vals_normal = vals_normal; a.vals_semantic = vals_semantic;
    a.view_matrix = view_matrix; a.intrinsics = intrinsics;
    a.image_color = image_color; a.image_depth = image_depth; a.image_normal = image_normal;
    a.image_semantic = image_semantic;
    a.mapping3dto2d = mapping3dto2d; a.mapping3dto2d_num = mapping3dto2d_num;
    a.dense = dense; a.vbits = vbits; a.bmap = bmap; a.vpc = L.vpc; a.bpc = L.bpc; a.wpr = L.wpr;
    a.tile_counter = (int32_t *)(ws + L.tiles_off);
    a.num_chunks = p->num_chunks;
    a.list_count = (int32_t *)(ws + L.head_off);
    a.list = (int2 *)(ws + L.list_off);
    a.hits = (p->flags & SPSG_FLAG_RECORD_HITS) ? (int32_t *)(ws + L.hits_off) : nullptr;
    a.width = p->width; a.height = p->height;
    a.depth_min = p->depth_min; a.depth_max = p->depth_max; a.thresh = p->thresh_sample_dist; a.inc = p->ray_increment;
    a.dimx = p->dimx; a.dimy = p->dimy; a.dimz = p->dimz;
    {
        const bool maps = !(p->flags & SPSG_FLAG_NO_BRICK_SKIP) && std::max(p->dimx, std::max(p->dimy, p->dimz)) <= kMaxFastDim;
        a.vx = maps ? p->dimx - 1 : 0; a.vy = maps ? p->dimy - 1 : 0; a.vz = maps ? p->dimz - 1 : 0;
    }
    a.nbx = L.nbx; a.nby = L.nby; a.nbz = L.nbz;
    a.views = p->views_per_chunk; a.max_pixels = p->max_pixels_per_voxel;
    a.num_locs = p->num_locs;
    a.flags = p->flags;
    a.vec_ok = (p->width % 4 == 0) && aligned16(image_color) && aligned16(image_depth) && aligned16(image_normal) &&
               aligned16(image_semantic);
    {
        int k = 0;
        while ((1 << k) < std::max(p->dimx, std::max(p->dimy, p->dimz))) k++;
        a.guard = std::min(kFracGuard, std::max(ldexpf(1.0f, k - 21), ldexpf(1.0f, -18)));  // 8 ulp of the largest coordinate
    }
    a.loss = make_loss_args(targets, accum);
    a.loss.loss_out = loss_out;
    a.loss.done = (int32_t *)(ws + L.head_off) + 16;  // in the per-call zeroed header, next to the list counter
    if (clear_grads && p->num_locs > 0) {  // rows [0, N) of the backward's outputs (kernel.cu:557-560), cleared by the forward's warps
        a.clear = *clear_grads;
        a.clear_rows = p->num_locs;
    }
    // persistent: one CTA per SM (fewer when there is less than one tile per warp)
    const long long tiles_x = (p->width + kWarpW - 1) / kWarpW, tiles_y = (p->height + kWarpH - 1) / kWarpH;
    const long long all_tiles = ((tiles_x + 1) / 2) * ((tiles_y + 1) / 2) * 4 * p->views_per_chunk * p->num_chunks;
    const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(sms, all_tiles));
    // CTA size: 24 warps when every warp gets about one tile (latency-bound), 28 when there are many tiles per SM
    const bool large = all_tiles >= (long long)sms * 4 * kFwdWarpsLarge;
    // one normal per (voxel, view); with one view per chunk that is the shared-normals kernel
    const bool view_normals = (p->flags & SPSG_FLAG_VIEW_NORMALS) && p->views_per_chunk > 1;
    const int warps = large ? kFwdWarpsLarge : kFwdWarps;
    const size_t dyn = fwd_smem_fixed(warps) + (a.maps_in_smem ? map_bytes : 0);
    {
        static std::mutex mu;
        static bool configured[64] = {false};
        int dev = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lk(mu);
        if (dev < 0 || dev >= 64 || !configured[dev]) {
#define SPSG_SET_SMEM(L, M, W, VN) CUDA_TRY(cudaFuncSetAttribute(raycast_forward_kernel<L, M, W, VN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmemMax))
#define SPSG_SET_SMEM_ALL(VN)                                                                                   \
    SPSG_SET_SMEM(true, true, kFwdWarps, VN); SPSG_SET_SMEM(false, true, kFwdWarps, VN);                         \
    SPSG_SET_SMEM(true, false, kFwdWarps, VN); SPSG_SET_SMEM(false, false, kFwdWarps, VN);                       \
    SPSG_SET_SMEM(true, true, kFwdWarpsLarge, VN); SPSG_SET_SMEM(false, true, kFwdWarpsLarge, VN);               \
    SPSG_SET_SMEM(true, false, kFwdWarpsLarge, VN); SPSG_SET_SMEM(false, false, kFwdWarpsLarge, VN)
            SPSG_SET_SMEM_ALL(false);
            SPSG_SET_SMEM_ALL(true);
#undef SPSG_SET_SMEM_ALL
#undef SPSG_SET_SMEM
            if (dev >= 0 && dev < 64) configured[dev] = true;
        }
    }
    {
        ScopedKernelTimer timer(0, st);
#define SPSG_LAUNCH_VN(L, M, VN)                                                                                  \
    do {                                                                                                          \
        if (large) raycast_forward_kernel<L, M, kFwdWarpsLarge, VN><<<grid, kFwdWarpsLarge * 32, dyn, st>>>(a);  \
        else raycast_forward_kernel<L, M, kFwdWarps, VN><<<grid, kFwdWarps * 32, dyn, st>>>(a);                  \
    } while (0)
#define SPSG_LAUNCH(L, M)                                                                                         \
    do {                                                                                                          \
        if (view_normals) SPSG_LAUNCH_VN(L, M, true); else SPSG_LAUNCH_VN(L, M, false);                           \
    } while (0)
        if (targets) {
            if (a.maps_in_smem) SPSG_LAUNCH(true, true); else SPSG_LAUNCH(true, false);
        } else {
            if (a.maps_in_smem) SPSG_LAUNCH(false, true); else SPSG_LAUNCH(false, false);
        }
#undef SPSG_LAUNCH
#undef SPSG_LAUNCH_VN
    }
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int launch_backward(const spsg_raycast_params *p, bool fused, const float *g_or_img_color, const float *g_or_img_depth,
                    const float *grad_normal, const float *g_or_img_semantic, const spsg_loss_targets *targets,
                    const float *loss_out, const float *grad_scale, const int32_t *sparse_mapping,
                    const int32_t *mapping3dto2d, const int32_t *mapping3dto2d_num, float *d_color, float *d_depth,
                    float *d_normal, float *d_semantic, void *workspace, size_t workspace_bytes, cudaStream_t st,
                    const spsg_upstream_grads *upstream = nullptr) {
    if (int rc = check_params(p)) return rc;
    if (!g_or_img_color || !g_or_img_depth || !g_or_img_semantic || (!fused && !grad_normal) || !sparse_mapping ||
        !mapping3dto2d || !mapping3dto2d_num)
        return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL tensor pointer");
    if (fused && (!targets || !loss_out)) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL loss targets");
    // upstream images (fused only): any plane may be NULL; none at all is exactly the fused backward without them
    const bool up = fused && upstream &&
                    (upstream->grad_color || upstream->grad_depth || upstream->grad_normal || upstream->grad_semantic);
    if (up && (reinterpret_cast<uintptr_t>(upstream->grad_semantic) & 7u))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "upstream grad_semantic must be 8-byte aligned");
    if (p->max_pixels_per_voxel <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "max_pixels_per_voxel must be positive");
    if (p->num_locs == 0) return SPSG_OK;
    if (!d_color || !d_depth || !d_normal || !d_semantic) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL gradient pointer");
    if (reinterpret_cast<uintptr_t>(d_semantic) & 7u) return fail(SPSG_ERR_INVALID_ARGUMENT, "d_semantic must be 8-byte aligned");
    const Layout L = make_layout(p);
    if (!workspace || workspace_bytes < L.total) return fail(SPSG_ERR_WORKSPACE_TOO_SMALL, "workspace too small");
    uint8_t *ws = (uint8_t *)workspace;
    BackwardArgs a;
    memset(&a, 0, sizeof(a));
    if (fused) {
        a.image_color = g_or_img_color; a.image_depth = g_or_img_depth; a.image_semantic = g_or_img_semantic;
        a.loss = make_loss_args(targets, nullptr);
        a.loss_out = loss_out;
        a.w_depth = targets->weight_depth; a.w_color = targets->weight_color_loss; a.w_sem = targets->weight_semantic;
        a.grad_scale = grad_scale;
        if (up) {
            a.up_color = upstream->grad_color; a.up_depth = upstream->grad_depth; a.up_normal = upstream->grad_normal;
            a.up_semantic = upstream->grad_semantic;
        }
    } else {
        a.grad_color = g_or_img_color; a.grad_depth = g_or_img_depth; a.grad_normal = grad_normal;
        a.grad_semantic = g_or_img_semantic;
    }
    a.mapping3dto2d = mapping3dto2d; a.mapping3dto2d_num = mapping3dto2d_num;
    a.d_color = d_color; a.d_depth = d_depth; a.d_normal = d_normal; a.d_semantic = d_semantic;
    a.list_count = (const int32_t *)(ws + L.head_off);
    a.list = (const int2 *)(ws + L.list_off);
    a.width = p->width; a.height = p->height;
    a.views = p->views_per_chunk; a.max_pixels = p->max_pixels_per_voxel;
    a.num_locs = p->num_locs;
    const int sms = sm_count();
    // half a warp per listed (voxel, view) pair; the list length is only known on the device: size for its bound N * F
    const long long max_items = p->num_locs * p->views_per_chunk;
    const unsigned gather_blocks = (unsigned)std::max<long long>(1, std::min<long long>((max_items + (32 / kGatherGroup) * kGatherWarps - 1) / ((32 / kGatherGroup) * kGatherWarps), (long long)sms * 8));
    const unsigned zero_blocks = (unsigned)std::min<long long>((p->num_locs + 255) / 256, (long long)sms * 4);
    const bool cleared = (p->flags & SPSG_FLAG_GRADS_CLEARED) != 0;  // the forward's fill pass cleared rows [0, N)
    const bool multi = p->views_per_chunk > 1, exact = (p->flags & SPSG_FLAG_DETERMINISTIC_GRADS) != 0;
    const bool view_normals = multi && (p->flags & SPSG_FLAG_VIEW_NORMALS);  // d_normal (N,F,3), one row per view
#define SPSG_GATHER(FUSED, UP, VIEWS, VN, BLOCKS) backward_gather_kernel<FUSED, UP, VIEWS, VN><<<(BLOCKS), kGatherWarps * 32, 0, st>>>(a)
#define SPSG_GATHER_VIEWS(VIEWS, VN, BLOCKS)                                                                      \
    do {                                                                                                          \
        if (up) SPSG_GATHER(true, true, VIEWS, VN, BLOCKS);                                                       \
        else if (fused) SPSG_GATHER(true, false, VIEWS, VN, BLOCKS);                                              \
        else SPSG_GATHER(false, false, VIEWS, VN, BLOCKS);                                                        \
    } while (0)
#define SPSG_GATHER_ANY(BLOCKS)                                                                                   \
    do {                                                                                                          \
        if (!multi) SPSG_GATHER_VIEWS(0, false, BLOCKS);                                                          \
        else if (view_normals && !exact) SPSG_GATHER_VIEWS(1, true, BLOCKS);                                      \
        else if (view_normals) SPSG_GATHER_VIEWS(2, true, BLOCKS);                                                \
        else if (!exact) SPSG_GATHER_VIEWS(1, false, BLOCKS);                                                     \
        else SPSG_GATHER_VIEWS(2, false, BLOCKS);                                                                 \
    } while (0)
    if (cleared) {
        a.zero_blocks = 0;
        ScopedKernelTimer timer(1, st);
        SPSG_GATHER_ANY(gather_blocks);
    } else if (!multi) {
        // one launch: leading CTAs clear the rows of voxels nothing hit, the rest gather (plain stores)
        a.zero_blocks = (int)zero_blocks;
        ScopedKernelTimer timer(1, st);
        SPSG_GATHER_ANY(zero_blocks + gather_blocks);
    } else {
        a.zero_blocks = 0;
        if (view_normals) backward_zero_view_normals_kernel<<<zero_blocks, 256, 0, st>>>(a);
        else backward_zero_kernel<<<zero_blocks, 256, 0, st>>>(a);
        CUDA_TRY(cudaGetLastError());
        ScopedKernelTimer timer(1, st);
        SPSG_GATHER_ANY(gather_blocks);
    }
#undef SPSG_GATHER_ANY
#undef SPSG_GATHER_VIEWS
#undef SPSG_GATHER
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

}  // namespace

// error plumbing for the other translation units of the library (csrc/spsg_internal.h)
int spsg_internal_fail(int code, const char *msg) { return fail(code, msg); }
int spsg_internal_fail_cuda(cudaError_t e, const char *where) { return fail_cuda(e, where); }
int spsg_internal_sm_count() { return sm_count(); }

extern "C" {

#ifdef SPSG_STATS
SPSG_API int spsg_debug_tile_stats(int *out) {
    return cudaMemcpyFromSymbol(out, g_tile_stats, sizeof(int) * 131072 * 8) == cudaSuccess ? SPSG_OK : SPSG_ERR_CUDA;
}

SPSG_API int spsg_debug_stats(unsigned long long *out, int reset) {
    if (cudaMemcpyFromSymbol(out, g_stats, sizeof(unsigned long long) * 48) != cudaSuccess) return SPSG_ERR_CUDA;
    if (reset) {
        unsigned long long z[48] = {0};
        cudaMemcpyToSymbol(g_stats, z, sizeof(z));
    }
    return SPSG_OK;
}
#endif

const char *spsg_version(void) { return "spsg_raycast_b200 0.3 (sm_100a)"; }
const char *spsg_last_error(void) { return g_err; }

void spsg_timing_enable(int on) {
    std::lock_guard<std::mutex> lk(g_timing_mu);
    g_timing = on != 0;
}

int spsg_timing_read(int which, double *total_ms, int *launches) {
    if (which < 0 || which > 1 || !total_ms || !launches) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad timing query");
    std::vector<EventPair> evs;
    {
        std::lock_guard<std::mutex> lk(g_timing_mu);
        evs.swap(g_ev[which]);
    }
    *total_ms = 0.0;
    *launches = 0;
    for (EventPair &e : evs) {
        float ms = 0.0f;
        if (cudaEventSynchronize(e.b) == cudaSuccess && cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) {
            *total_ms += ms;
            *launches += 1;
        }
        cudaEventDestroy(e.a);
        cudaEventDestroy(e.b);
    }
    return SPSG_OK;
}

size_t spsg_workspace_bytes(const spsg_raycast_params *p) {
    if (check_params(p)) return 0;
    return make_layout(p).total;
}

int spsg_build_index(const int64_t *locs, int64_t num_locs, int32_t *sparse_mapping, int32_t num_chunks, int32_t dimz,
                     int32_t dimy, int32_t dimx, void *stream) {
    if (!sparse_mapping || (num_locs > 0 && !locs)) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL tensor pointer");
    if (num_chunks <= 0 || dimz <= 0 || dimy <= 0 || dimx <= 0 || num_locs < 0)
        return fail(SPSG_ERR_INVALID_ARGUMENT, "bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t cells = (size_t)num_chunks * dimz * dimy * dimx;
    CUDA_TRY(cudaMemsetAsync(sparse_mapping, 0xff, cells * sizeof(int32_t), st));
    if (num_locs > 0) {
        index_kernel<true><<<(unsigned)((num_locs + 255) / 256), 256, 0, st>>>(
            (const longlong4 *)locs, num_locs, sparse_mapping, nullptr, nullptr, nullptr, 0, dimz, dimy, dimx, num_chunks);
        CUDA_TRY(cudaGetLastError());
    }
    return SPSG_OK;
}

int spsg_raycast_forward(const spsg_raycast_params *p, const int32_t *sparse_mapping, const int64_t *locs,
                         const float *vals_sdf, const float *vals_color, const float *vals_normal,
                         const float *vals_semantic, const float *view_matrix, const float *intrinsics,
                         float *image_color, float *image_depth, float *image_normal, float *image_semantic,
                         int32_t *mapping3dto2d, int32_t *mapping3dto2d_num, void *workspace, size_t workspace_bytes,
                         void *stream) {
    return launch_forward(p, false, const_cast<int32_t *>(sparse_mapping), locs, vals_sdf, vals_color, vals_normal,
                          vals_semantic, view_matrix, intrinsics, image_color, image_depth, image_normal,
                          image_semantic, mapping3dto2d, mapping3dto2d_num, nullptr, nullptr, nullptr, workspace,
                          workspace_bytes, (cudaStream_t)stream);
}

int spsg_raycast_forward_indexed(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                                 const float *vals_sdf, const float *vals_color, const float *vals_normal,
                                 const float *vals_semantic, const float *view_matrix, const float *intrinsics,
                                 float *image_color, float *image_depth, float *image_normal, float *image_semantic,
                                 int32_t *mapping3dto2d, int32_t *mapping3dto2d_num,
                                 const spsg_grad_buffers *clear_grads, void *workspace, size_t workspace_bytes,
                                 void *stream) {
    return launch_forward(p, true, sparse_mapping, locs, vals_sdf, vals_color, vals_normal, vals_semantic, view_matrix,
                          intrinsics, image_color, image_depth, image_normal, image_semantic, mapping3dto2d,
                          mapping3dto2d_num, nullptr, nullptr, clear_grads, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

int spsg_raycast_backward(const spsg_raycast_params *p, const float *grad_color, const float *grad_depth,
                          const float *grad_normal, const float *grad_semantic, const int32_t *sparse_mapping,
                          const int32_t *mapping3dto2d, const int32_t *mapping3dto2d_num, float *d_color,
                          float *d_depth, float *d_normal, float *d_semantic, void *workspace, size_t workspace_bytes,
                          void *stream) {
    return launch_backward(p, false, grad_color, grad_depth, grad_normal, grad_semantic, nullptr, nullptr, nullptr,
                           sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color, d_depth, d_normal, d_semantic,
                           workspace, workspace_bytes, (cudaStream_t)stream);
}

int spsg_raycast_occ(const spsg_raycast_params *p, const uint8_t *occ3d, uint8_t *occ2d, const float *view_matrix,
                     const float *intrinsics, void *stream) {
    if (int rc = check_params(p)) return rc;
    if (!occ3d || !occ2d || !view_matrix || !intrinsics) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL tensor pointer");
    if (!aligned16(view_matrix) || !aligned16(intrinsics))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "view_matrix / intrinsics must be 16-byte aligned");
    OccArgs a;
    a.occ3d = occ3d; a.occ2d = occ2d; a.view_matrix = view_matrix; a.intrinsics = intrinsics;
    a.width = p->width; a.height = p->height;
    a.depth_min = p->depth_min; a.depth_max = p->depth_max; a.inc = p->ray_increment;
    a.dimx = p->dimx; a.dimy = p->dimy; a.dimz = p->dimz;
    a.flags = p->flags;
    const dim3 grid((p->width + kTileW - 1) / kTileW, (p->height + kTileH - 1) / kTileH, p->num_chunks);
    raycast_occ_kernel<<<grid, kTilePix, 0, (cudaStream_t)stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_raycast_forward_loss(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                              const float *vals_sdf, const float *vals_color, const float *vals_normal,
                              const float *vals_semantic, const float *view_matrix, const float *intrinsics,
                              float *image_color, float *image_depth, float *image_normal, float *image_semantic,
                              int32_t *mapping3dto2d, int32_t *mapping3dto2d_num, const spsg_loss_targets *t,
                              float *loss_out, const spsg_grad_buffers *clear_grads, void *workspace,
                              size_t workspace_bytes, void *stream) {
    if (!t) return fail(SPSG_ERR_INVALID_ARGUMENT, "loss targets are NULL");
    return launch_forward(p, true, sparse_mapping, locs, vals_sdf, vals_color, vals_normal, vals_semantic, view_matrix,
                          intrinsics, image_color, image_depth, image_normal, image_semantic, mapping3dto2d,
                          mapping3dto2d_num, t, loss_out, clear_grads, workspace, workspace_bytes, (cudaStream_t)stream);
}

int spsg_raycast_backward_loss(const spsg_raycast_params *p, const float *image_color, const float *image_depth,
                               const float *image_semantic, const spsg_loss_targets *t, const float *loss_out,
                               const float *grad_scale, const int32_t *sparse_mapping, const int32_t *mapping3dto2d,
                               const int32_t *mapping3dto2d_num, float *d_color, float *d_depth, float *d_normal,
                               float *d_semantic, void *workspace, size_t workspace_bytes, void *stream) {
    return launch_backward(p, true, image_color, image_depth, nullptr, image_semantic, t, loss_out, grad_scale,
                           sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color, d_depth, d_normal, d_semantic,
                           workspace, workspace_bytes, (cudaStream_t)stream);
}

int spsg_raycast_backward_loss_upstream(const spsg_raycast_params *p, const float *image_color, const float *image_depth,
                                        const float *image_semantic, const spsg_loss_targets *t, const float *loss_out,
                                        const float *grad_scale, const spsg_upstream_grads *upstream,
                                        const int32_t *sparse_mapping, const int32_t *mapping3dto2d,
                                        const int32_t *mapping3dto2d_num, float *d_color, float *d_depth, float *d_normal,
                                        float *d_semantic, void *workspace, size_t workspace_bytes, void *stream) {
    return launch_backward(p, true, image_color, image_depth, nullptr, image_semantic, t, loss_out, grad_scale,
                           sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color, d_depth, d_normal, d_semantic,
                           workspace, workspace_bytes, (cudaStream_t)stream, upstream);
}

static int normals_check(const int64_t *locs, int64_t n, const float *sdf, const int32_t *index, int32_t num_chunks,
                         int32_t dimz, int32_t dimy, int32_t dimx) {
    if (n < 0 || num_chunks <= 0 || dimz <= 0 || dimy <= 0 || dimx <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad sizes");
    if ((long long)num_chunks * dimz * dimy * dimx >= (1ll << 31)) return fail(SPSG_ERR_INVALID_ARGUMENT, "dense grid exceeds 32-bit indexing");
    if (!index || (n > 0 && (!locs || !sdf))) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL tensor pointer");
    if (reinterpret_cast<uintptr_t>(locs) & 15u) return fail(SPSG_ERR_INVALID_ARGUMENT, "locs must be 16-byte aligned");
    return SPSG_OK;
}

int spsg_normals_forward(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                         int32_t *index, int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, float *normals,
                         void *stream) {
    if (int rc = normals_check(locs, num_locs, vals_sdf, index, num_chunks, dimz, dimy, dimx)) return rc;
    if (num_locs > 0 && !normals) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL output pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = spsg_build_index(locs, num_locs, index, num_chunks, dimz, dimy, dimx, stream)) return rc;
    if (num_locs == 0) return SPSG_OK;
    NormalsArgs a;
    memset(&a, 0, sizeof(a));
    a.locs = (const longlong4 *)locs; a.sdf = vals_sdf; a.transform = transform; a.index = index; a.out = normals;
    a.n = num_locs; a.dimx = dimx; a.dimy = dimy; a.dimz = dimz;
    normals_forward_kernel<<<(unsigned)((num_locs + 255) / 256), 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_normals_backward(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                          const int32_t *index, int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx,
                          const float *grad_normals, float *scratch_u, float *d_sdf, void *stream) {
    if (int rc = normals_check(locs, num_locs, vals_sdf, index, num_chunks, dimz, dimy, dimx)) return rc;
    if (num_locs == 0) return SPSG_OK;
    if (!grad_normals || !scratch_u || !d_sdf) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL gradient pointer");
    cudaStream_t st = (cudaStream_t)stream;
    NormalsArgs a;
    memset(&a, 0, sizeof(a));
    a.locs = (const longlong4 *)locs; a.sdf = vals_sdf; a.transform = transform; a.index = index;
    a.grad_out = grad_normals; a.out = scratch_u; a.d_sdf = d_sdf;
    a.n = num_locs; a.dimx = dimx; a.dimy = dimy; a.dimz = dimz;
    const unsigned blocks = (unsigned)((num_locs + 255) / 256);
    normals_backward_u_kernel<<<blocks, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    normals_backward_gather_kernel<<<blocks, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

static int normals_views_check(const float *transform, int32_t views_per_chunk) {
    if (views_per_chunk <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "views_per_chunk must be >= 1");
    if (views_per_chunk > 1 && !transform) return fail(SPSG_ERR_INVALID_ARGUMENT, "per-view normals need a (B*F,4,4) transform");
    return SPSG_OK;
}

int spsg_normals_forward_views(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                               int32_t views_per_chunk, int32_t *index, int32_t num_chunks, int32_t dimz, int32_t dimy,
                               int32_t dimx, float *normals, void *stream) {
    if (int rc = normals_views_check(transform, views_per_chunk)) return rc;
    if (views_per_chunk == 1)
        return spsg_normals_forward(locs, num_locs, vals_sdf, transform, index, num_chunks, dimz, dimy, dimx, normals, stream);
    if (int rc = normals_check(locs, num_locs, vals_sdf, index, num_chunks, dimz, dimy, dimx)) return rc;
    if ((long long)num_chunks * views_per_chunk >= (1ll << 31)) return fail(SPSG_ERR_INVALID_ARGUMENT, "too many images");
    if (num_locs > 0 && !normals) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL output pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = spsg_build_index(locs, num_locs, index, num_chunks, dimz, dimy, dimx, stream)) return rc;
    if (num_locs == 0) return SPSG_OK;
    NormalsArgs a;
    memset(&a, 0, sizeof(a));
    a.locs = (const longlong4 *)locs; a.sdf = vals_sdf; a.transform = transform; a.index = index; a.out = normals;
    a.n = num_locs; a.dimx = dimx; a.dimy = dimy; a.dimz = dimz;
    normals_forward_views_kernel<<<(unsigned)((num_locs + 255) / 256), 256, 0, st>>>(a, views_per_chunk);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_normals_backward_views(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                                int32_t views_per_chunk, const int32_t *index, int32_t num_chunks, int32_t dimz,
                                int32_t dimy, int32_t dimx, const float *grad_normals, float *scratch_u, float *d_sdf,
                                void *stream) {
    if (int rc = normals_views_check(transform, views_per_chunk)) return rc;
    if (views_per_chunk == 1)
        return spsg_normals_backward(locs, num_locs, vals_sdf, transform, index, num_chunks, dimz, dimy, dimx, grad_normals,
                                     scratch_u, d_sdf, stream);
    if (int rc = normals_check(locs, num_locs, vals_sdf, index, num_chunks, dimz, dimy, dimx)) return rc;
    if ((long long)num_chunks * views_per_chunk >= (1ll << 31)) return fail(SPSG_ERR_INVALID_ARGUMENT, "too many images");
    if (num_locs == 0) return SPSG_OK;
    if (!grad_normals || !scratch_u || !d_sdf) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL gradient pointer");
    cudaStream_t st = (cudaStream_t)stream;
    NormalsArgs a;
    memset(&a, 0, sizeof(a));
    a.locs = (const longlong4 *)locs; a.sdf = vals_sdf; a.transform = transform; a.index = index;
    a.grad_out = grad_normals; a.out = scratch_u; a.d_sdf = d_sdf;
    a.n = num_locs; a.dimx = dimx; a.dimy = dimy; a.dimz = dimz;
    const unsigned blocks = (unsigned)((num_locs + 255) / 256);
    normals_backward_u_views_kernel<<<blocks, 256, 0, st>>>(a, views_per_chunk);
    CUDA_TRY(cudaGetLastError());
    normals_backward_gather_kernel<<<blocks, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_losses2d_forward(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                          const float *image_semantic, int64_t num_pixels, float *loss_out, void *scratch,
                          size_t scratch_bytes, void *stream) {
    if (!t || !loss_out) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL loss targets / loss_out");
    if (num_pixels < 0 || num_pixels * 14 >= (1ll << 32)) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad pixel count");
    if ((t->target_depth && !image_depth) || (t->target_color && !image_color) || (t->target_label && !image_semantic))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "a target is set but its rendering is NULL");
    if (image_semantic && (reinterpret_cast<uintptr_t>(image_semantic) & 7u)) return fail(SPSG_ERR_INVALID_ARGUMENT, "image_semantic must be 8-byte aligned");
    const size_t need = (size_t)kLossSlots * 8 * sizeof(double);
    if (!scratch || scratch_bytes < need || (reinterpret_cast<uintptr_t>(scratch) & 7u)) return fail(SPSG_ERR_WORKSPACE_TOO_SMALL, "scratch too small");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(scratch, 0, need, st));
    Losses2DArgs a;
    memset(&a, 0, sizeof(a));
    a.image_color = image_color; a.image_depth = image_depth; a.image_semantic = image_semantic;
    a.loss = make_loss_args(t, (double *)scratch);
    a.num_pixels = num_pixels;
    if (num_pixels > 0) {
        const unsigned blocks = (unsigned)std::min<long long>((num_pixels + 255) / 256, (long long)sm_count() * 8);
        losses2d_forward_kernel<<<blocks, 256, 0, st>>>(a);
        CUDA_TRY(cudaGetLastError());
    }
    finalize_loss_kernel<<<1, 32, 0, st>>>((const double *)scratch, loss_out, t->weight_depth, t->weight_color_loss,
                                           t->weight_semantic, t->target_depth != nullptr, t->target_color != nullptr,
                                           t->target_label != nullptr);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

int spsg_losses2d_backward(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                           const float *image_semantic, int64_t num_pixels, const float *loss_out,
                           const float *grad_scale, float *d_color, float *d_depth, float *d_semantic, void *stream) {
    if (!t || !loss_out) return fail(SPSG_ERR_INVALID_ARGUMENT, "NULL loss targets / loss_out");
    if (num_pixels < 0 || num_pixels * 14 >= (1ll << 32)) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad pixel count");
    if ((t->target_depth && !image_depth) || (t->target_color && !image_color) || (t->target_label && !image_semantic))
        return fail(SPSG_ERR_INVALID_ARGUMENT, "a target is set but its rendering is NULL");
    if (d_semantic && (reinterpret_cast<uintptr_t>(d_semantic) & 7u)) return fail(SPSG_ERR_INVALID_ARGUMENT, "d_semantic must be 8-byte aligned");
    if (num_pixels == 0) return SPSG_OK;
    BackwardArgs a;
    memset(&a, 0, sizeof(a));
    a.image_color = image_color; a.image_depth = image_depth; a.image_semantic = image_semantic;
    a.loss = make_loss_args(t, nullptr);
    a.loss_out = loss_out;
    a.w_depth = t->weight_depth; a.w_color = t->weight_color_loss; a.w_sem = t->weight_semantic;
    a.grad_scale = grad_scale;
    const unsigned blocks = (unsigned)std::min<long long>((num_pixels + 255) / 256, (long long)sm_count() * 8);
    losses2d_backward_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a, num_pixels, d_color, d_depth, d_semantic);
    CUDA_TRY(cudaGetLastError());
    return SPSG_OK;
}

}  // extern "C"

// ---- host side of a host-fed call (no CUDA in here)
extern "C" SPSG_API int spsg_pack_locs_host(const int64_t *locs, int64_t num_locs, int32_t num_chunks, int32_t dimz,
                                            int32_t dimy, int32_t dimx, uint32_t *cells_out, int32_t threads) {
    if (num_locs < 0 || (num_locs > 0 && (!locs || !cells_out))) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad locs / output");
    if (num_chunks <= 0 || dimz <= 0 || dimy <= 0 || dimx <= 0) return fail(SPSG_ERR_INVALID_ARGUMENT, "bad grid sizes");
    if ((unsigned long long)num_chunks * dimz * dimy * dimx >= 0xffffffffull)
        return fail(SPSG_ERR_INVALID_ARGUMENT, "packed locs need fewer than 2^32 - 1 cells");
    const int t = std::max(1, std::min(threads, 64));
    const long long dz = dimz, dy = dimy, dx = dimx, nb = num_chunks;
#pragma omp parallel for num_threads(t) schedule(static)
    for (long long i = 0; i < (long long)num_locs; i++) {
        const long long z = locs[4 * i], y = locs[4 * i + 1], x = locs[4 * i + 2], b = locs[4 * i + 3];
        const bool in = (unsigned long long)z < (unsigned long long)dz && (unsigned long long)y < (unsigned long long)dy &&
                        (unsigned long long)x < (unsigned long long)dx && (unsigned long long)b < (unsigned long long)nb;
        cells_out[i] = in ? (uint32_t)(((b * dz + z) * dy + y) * dx + x) : 0xffffffffu;
    }
    return SPSG_OK;
}
