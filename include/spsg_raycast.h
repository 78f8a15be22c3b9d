/*
 * spsg_raycast.h -- C ABI of the B200-native SPSG-semantic raycaster (libspsg_raycast.so).
 *
 * This is the drop-in boundary for the reference's native extension module `raycast_rgbd_cuda`
 * (reference: torch/utils/raycast_rgbd/raycast_rgbd_cuda.cpp:155-160).  Plain device pointers, sizes
 * and a cudaStream_t (as void*): no ATen / torch types.  All tensors are caller-owned, contiguous,
 * and live on the device that is current for the calling thread; nothing is allocated or retained
 * by the library.  Every call is asynchronous on `stream` and re-entrant per (device, stream).
 *
 * Error convention: 0 == SPSG_OK, otherwise an SPSG_ERR_* code; spsg_last_error() returns a
 * thread-local message.  (The reference prints and exit(-1)s on CUDA errors,
 * cutil_inline_runtime.h:284-292; this library never exits the process.)
 *
 * Layouts (identical to the reference, SURVEY.md section 8(b)):
 *   locs            int64 (N,4) rows (z,y,x,chunk)          sparse_mapping  int32 (B,Dz,Dy,Dx), -1 = absent
 *   vals_sdf        f32 (N,1)    vals_color f32 (N,3)       vals_normal f32 (N,3)   vals_semantic f32 (N,14)
 *   view_matrix     f32 (I,4,4) row-major camera->grid      intrinsics  f32 (I,4) = fx,fy,mx,my
 *   image_color     f32 (I,H,W,3)   image_depth f32 (I,H,W)   image_normal f32 (I,H,W,3)
 *   image_semantic  f32 (I,H,W,14)                           miss == -inf in every channel
 *   mapping3dto2d   int32 (R,max_pixels_per_voxel)           mapping3dto2d_num int32 (R),  R >= F*N
 *                   (mapping3dto2d: NULL allowed with SPSG_FLAG_ALL_PIXELS)
 *   d_color (N,3)   d_depth (N,1)   d_normal (N,3)   d_semantic (N,14)
 * with I = num_chunks * views_per_chunk images; image i renders chunk i / views_per_chunk
 * (reference style.py:9-16); views_per_chunk == 1 is exactly the reference.
 *
 * Semantic class count C (spsg_raycast_params.semantic_channels; 0 means 14, the reference's float14): every "14" of the
 * layouts above and of the loss structs below is C -- vals_semantic (N,C), image_semantic (I,H,W,C), d_semantic (N,C),
 * grad_semantic / upstream grad_semantic (I,H,W,C), class_weight (C), and target_label == C means ignore.  A miss is -inf in
 * all C channels.  C = 1..64; anything else is SPSG_ERR_INVALID_ARGUMENT.  Nothing but the semantic channels depends on C:
 * the colour, depth and normal renderings, mapping3dto2d(_num), the backward's work list and the SPSG_FLAG_DETERMINISTIC
 * tables are bit-identical to those of the C = 14 call on the same voxels, and each semantic pixel is a copy of its hit
 * voxel's row.  The cross-entropy (fused and stand-alone) is valid where label < C and logit 0 != -inf and equals
 * sum w[y] * nll / sum w[y] over C logits, with the 14-channel path's arithmetic in the same order.  C != 14 runs
 * C-generic kernels (SPSG_FLAG_GENERIC_SEMANTIC forces them at C = 14); C = 14 without that flag runs exactly the
 * 14-channel kernels.  spsg_workspace_bytes does not depend on C.  C composes with every flag.  A backward must be called
 * with the C of its forward (the library cannot tell: the workspace does not record it).
 */
#ifndef SPSG_RAYCAST_H_
#define SPSG_RAYCAST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SPSG_API __attribute__((visibility("default")))
#else
#define SPSG_API
#endif

#define SPSG_SEMANTIC_CHANNELS 14 /* float14, raycast_rgbd_cuda_kernel.cu:18-21 */
#define SPSG_GRAD_CHANNELS 21     /* colour 3 + depth 1 + normal 3 + semantic 14 */
#define SPSG_MAX_SEMANTIC_CHANNELS 64 /* largest spsg_raycast_params.semantic_channels */

enum {
    SPSG_OK = 0,
    SPSG_ERR_INVALID_ARGUMENT = 1,
    SPSG_ERR_CUDA = 2,
    SPSG_ERR_WORKSPACE_TOO_SMALL = 3
};

/* spsg_raycast_params.flags */
enum {
    SPSG_FLAG_NO_CLIP = 1u << 0,       /* debug: march every sample like the reference (no ray/box clip)   */
    SPSG_FLAG_NO_BRICK_SKIP = 1u << 1, /* debug: no empty-block skipping                                    */
    SPSG_FLAG_RECORD_HITS = 1u << 2,   /* also write the per-pixel hit voxel index into the workspace       */
    SPSG_FLAG_GRADS_CLEARED = 1u << 3, /* backward only: rows [0,N) of d_* were cleared by the matching forward */
    SPSG_FLAG_SMEM_MAPS = 1u << 5,     /* debug: march maps staged in shared memory (TMA) even for several chunks          */
    SPSG_FLAG_GLOBAL_MAPS = 1u << 6,   /* debug: march maps read through L1 + one global tile counter even for one chunk   */
    SPSG_FLAG_PACKED_LOCS = 1u << 8,   /* forward (entry points that build the index): `locs` points to num_locs uint32 linear
                                          cell indices, the output of spsg_pack_locs_host, instead of int64 (z,y,x,b) rows      */
    SPSG_FLAG_INDEX_PREBUILT = 1u << 7, /* forward: sparse_mapping and the workspace's dense SDF brick already hold exactly
                                          these locs / vals_sdf (written by spsg_sparsify_locs_indexed): skip the -1 / NaN
                                          fill and the index pass (only mapping3dto2d_num is reset)                          */
    SPSG_FLAG_DETERMINISTIC_GRADS = 1u << 4, /* backward, several views per chunk: add a voxel's per-view means in view order
                                               without float atomics (bit-reproducible; the gather takes ~30 % longer) */
    SPSG_FLAG_DETERMINISTIC = 1u << 10, /* forward and backward: results that depend on nothing but the inputs.  Renderings and
                                           mapping3dto2d_num are those of the flag off, bit for bit.  Each row r of
                                           mapping3dto2d holds the min(num[r], P) SMALLEST pixel indices registered to it, in
                                           ascending order (with num[r] > P a canonical subset: the reference keeps an
                                           arbitrary P).  The loss block of spsg_raycast_forward_loss is summed in an order
                                           fixed by pixel position.  The backward gathers the canonical tables; with several
                                           views the flag implies SPSG_FLAG_DETERMINISTIC_GRADS.  No float atomics.  Pass it
                                           to the forward and to its backward alike: spsg_workspace_bytes grows by the loss
                                           partials (8 doubles per 4096 pixels of the batch) and always records the per-pixel
                                           hits the tables are rebuilt from. */
    SPSG_FLAG_VIEW_NORMALS = 1u << 9,   /* forward and backward, several views per chunk: one normal per (voxel, view).
                                           vals_normal is (N,F,3) voxel-major: row (v, f) is voxel v's normal as image
                                           chunk(v)*F + f sees it, and that image's normal rendering reads it (a row of
                                           zeros renders -inf, per row).  d_normal is (N,F,3): row (v, f) is the mean of
                                           grad_normal over view f's pixels registered to v -- not summed over views.  The
                                           forward's clear_grads->d_normal must hold N*F rows.  Colour, depth and semantic
                                           are unchanged.  With views_per_chunk == 1 the flag changes nothing.  Pass it
                                           to the forward and to its backward alike. */
    SPSG_FLAG_ALL_PIXELS = 1u << 11,    /* forward and backward: the gradient of row (v, f) is the mean over EVERY pixel of view f
                                           whose hit voxel is v, not over the first max_pixels_per_voxel of them:
                                               d_x[v] = sum_f (1 / num[f*N + v]) * sum over S(v, f) of grad_x[pixel]
                                           with num = mapping3dto2d_num = |S(v, f)|.  No table is written or read:
                                           mapping3dto2d may be NULL on every forward and backward entry point and
                                           max_pixels_per_voxel is ignored.  Renderings, mapping3dto2d_num and loss_out are
                                           those of the flag off, bit for bit.  The backward builds one segment of pixel
                                           indices per (voxel, view) row from the forward's per-pixel hit records, then
                                           gathers it.  Without SPSG_FLAG_DETERMINISTIC each row is summed in double in any
                                           order and rounded once; with it every segment is summed in ascending pixel
                                           order, the views' means are added in view order and no kernel uses float
                                           atomics.  Composes with VIEW_NORMALS, DETERMINISTIC_GRADS, GRADS_CLEARED,
                                           PACKED_LOCS, INDEX_PREBUILT and the fused losses.  Pass it to the forward and to
                                           its backward alike; spsg_workspace_bytes grows as stated there. */
    SPSG_FLAG_GENERIC_SEMANTIC = 1u << 12 /* debug: run the C-generic semantic kernels (forward epilogue, gather, loss sums)
                                           even at C = 14, where the 14-channel kernels run otherwise.  Results are those of
                                           the 14-channel kernels; under SPSG_FLAG_DETERMINISTIC bit for bit (renderings,
                                           tables, loss_out, gradients).  For tests and timing of the two paths. */
};

/* Replaces the reference's `opts` CPU tensor [W,H,depth_min,depth_max,thresh,ray_inc,Dx,Dy,Dz]
 * (raycast_rgbd.py:24-25, raycast_rgbd_cuda_kernel.cu:443-456) plus the sizes it read off tensors
 * (:471 max pixels, :490 batch). */
typedef struct spsg_raycast_params {
    int32_t width, height;
    float depth_min, depth_max, thresh_sample_dist, ray_increment;
    int32_t dimx, dimy, dimz;
    int32_t num_chunks;           /* B = sparse_mapping.size(0)                        */
    int32_t views_per_chunk;      /* F >= 1; images = B*F                              */
    int32_t max_pixels_per_voxel; /* mapping3dto2d.size(1)                             */
    int64_t num_locs;             /* N = locs.size(0)                                  */
    uint32_t flags;               /* SPSG_FLAG_*                                       */
    uint32_t semantic_channels;   /* C, semantic classes per voxel / pixel: 1..64, 0 = 14 (see the top of this file) */
} spsg_raycast_params;

/* Fused 2D losses (reference: depth L1 train.py:635-638, colour L1 loss.py:246-257,
 * 2D semantic cross-entropy train.py:744-746).  Targets are per image, same pixel layout as the
 * renderings.  Any target pointer may be NULL to switch that term off. */
typedef struct spsg_loss_targets {
    const float *target_depth;    /* (I,H,W) metres; 0 = hole (ignored)                               */
    const float *target_color;    /* (I,H,W,3) already permuted to channels-last                      */
    const float *weight_color;    /* (I,H,W) optional per-pixel colour weight or NULL (loss.py:250-253) */
    const uint8_t *target_label;  /* (I,H,W) class id, 14 (C) = ignore (train.py:614-616)             */
    const float *class_weight;    /* (14) / (C) cross-entropy class weights (train.py:118-119) or NULL = 1 */
    float voxelsize;              /* depth scale applied to the rendering (train.py:635)              */
    float weight_depth, weight_color_loss, weight_semantic; /* loss = sum_k weight_k * loss_k         */
} spsg_loss_targets;

/* Optional argument of the indexed / fused forwards: the gradient buffers the matching backward will write.  When
 * given, the forward also clears their rows [0, N) (16-byte stores by the raycast kernel's own warps), and the
 * backward -- called with SPSG_FLAG_GRADS_CLEARED -- is a single gather launch that only touches voxels that received
 * pixels.  Pass NULL when no backward will follow (the backward then clears the rows itself, like the reference's
 * memsets at raycast_rgbd_cuda_kernel.cu:557-560). */
typedef struct spsg_grad_buffers {
    float *d_color;    /* (>=N,3)  */
    float *d_depth;    /* (>=N,1)  */
    float *d_normal;   /* (>=N,3)  */
    float *d_semantic; /* (>=N,14) */
} spsg_grad_buffers;

/* Number of floats in the loss block written by spsg_raycast_forward_loss:
 * out[0]=depth L1  out[1]=colour L1  out[2]=semantic CE  out[3]=weight_depth*out[0]+weight_color_loss*out[1]+
 * weight_semantic*out[2]   out[4]=#valid depth pixels  out[5]=#valid colour elements  out[6]=sum of w[label]
 * (the normalisers spsg_raycast_backward_loss needs)  out[7]=reserved.  An empty valid set gives NaN, like torch. */
#define SPSG_LOSS_OUT_FLOATS 8

SPSG_API const char *spsg_version(void);
SPSG_API const char *spsg_last_error(void);

/* Measurement aid for bench.py's roofline leg: while enabled, every raycast forward kernel (which = 0) and backward
 * gather kernel (which = 1) is bracketed by CUDA events on its launch stream; spsg_timing_read waits for the
 * recorded launches, returns their summed device time and count, and clears the record.  Do not enable during
 * stream capture. */
SPSG_API void spsg_timing_enable(int on);
SPSG_API int spsg_timing_read(int which, double *total_ms, int *launches);

/* Scratch shared by forward and backward of one call pair: dense SDF brick (4*B*Dz*Dy*Dx bytes), skip-level map,
 * hit-voxel list, loss accumulators, optional per-pixel hit records.  Must be 256-byte aligned.
 * SPSG_FLAG_ALL_PIXELS adds, with R = F*N rows, X = B*F*W*H pixels and A(b) = b rounded up to a multiple of 256:
 *     256 + A(4*R) + A(4*X)                        (counters, per-row segment ends, one int32 per rendered pixel)
 *     + A(4*(floor(X / 65) + 1))                   (with SPSG_FLAG_DETERMINISTIC: the rows longer than 64 pixels) */
SPSG_API size_t spsg_workspace_bytes(const spsg_raycast_params *p);

/* == raycast_rgbd_cuda.construct_dense_sparse_mapping (raycast_rgbd_cuda.cpp:93-100,
 *    raycast_rgbd_cuda_kernel.cu:346-362, 506-533): sparse_mapping := -1, then [chunk,z,y,x] := row. */
SPSG_API int spsg_build_index(const int64_t *locs, int64_t num_locs, int32_t *sparse_mapping, int32_t num_chunks,
                              int32_t dimz, int32_t dimy, int32_t dimx, void *stream);

/* == raycast_rgbd_cuda.forward (raycast_rgbd_cuda.cpp:57-91, raycast_rgbd_cuda_kernel.cu:265-297,
 *    426-503).  sparse_mapping must already hold the index of `locs`.  Differences from the reference,
 *    none observable through its Python API: mapping3dto2d is not pre-filled with -1 (only entries
 *    [row][< num[row]] are defined) and only the first F*N counters of mapping3dto2d_num are reset. */
SPSG_API int spsg_raycast_forward(const spsg_raycast_params *p, const int32_t *sparse_mapping, const int64_t *locs,
                                  const float *vals_sdf, const float *vals_color, const float *vals_normal,
                                  const float *vals_semantic, const float *view_matrix, const float *intrinsics,
                                  float *image_color, float *image_depth, float *image_normal,
                                  float *image_semantic, int32_t *mapping3dto2d, int32_t *mapping3dto2d_num,
                                  void *workspace, size_t workspace_bytes, void *stream);

/* spsg_build_index + spsg_raycast_forward in one call (what RayCastRGBDFunction.forward does back
 * to back, raycast_rgbd.py:23-28), sharing one pass over `locs`. */
SPSG_API int spsg_raycast_forward_indexed(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                                          const float *vals_sdf, const float *vals_color, const float *vals_normal,
                                          const float *vals_semantic, const float *view_matrix,
                                          const float *intrinsics, float *image_color, float *image_depth,
                                          float *image_normal, float *image_semantic, int32_t *mapping3dto2d,
                                          int32_t *mapping3dto2d_num, const spsg_grad_buffers *clear_grads,
                                          void *workspace, size_t workspace_bytes, void *stream);

/* Label render: the march of spsg_raycast_forward_indexed (same hit voxel per pixel, bit for bit), with one uint8 label per
 *    voxel as its only payload and one uint8 label per pixel as its only output -- what label maps of a one-hot render
 *    (argmax of cat(render, ones), train.py:590-616) give, without the C-wide semantic image:
 *        image_label[pixel] = hit voxel v ? min(voxel_labels[v], C) : C          C = p->semantic_channels (0 = 14)
 *    voxel_labels: (N) uint8; a label above C renders as C.  image_label: (I,H,W) uint8.  hist: C + 1 device int64, cleared
 *    and then the number of pixels per label (integer atomics: deterministic), or NULL.  Index routes as in
 *    spsg_raycast_forward_indexed (int64 rows, SPSG_FLAG_PACKED_LOCS, SPSG_FLAG_INDEX_PREBUILT); SPSG_FLAG_NO_CLIP,
 *    NO_BRICK_SKIP, SMEM_MAPS and GLOBAL_MAPS act as in the forward; every other flag is ignored.  Nothing else is
 *    written: no float image, no mapping3dto2d(_num), no work list, no hit records, no gradient rows -- so no backward may
 *    follow it on this workspace.  Needs no more workspace than spsg_workspace_bytes(p); 256-byte aligned. */
SPSG_API int spsg_raycast_labels(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                                 const float *vals_sdf, const uint8_t *voxel_labels,
                                 const float *view_matrix, const float *intrinsics,
                                 uint8_t *image_label, int64_t *hist,
                                 void *workspace, size_t workspace_bytes, void *stream);

/* Eval render: the march of spsg_raycast_labels (same hit voxel per pixel) with an epilogue for evaluation without a
 *    backward.  One call gives, for the prediction (vals_color (N,3), vals_semantic (N,C) logits, pred_labels (N) uint8 --
 *    the voxels' predicted labels, e.g. spsg_labels_from_render_classes of the logits; a label above C counts as C):
 *      loss_out     SPSG_LOSS_OUT_FLOATS floats, the loss block of spsg_raycast_forward_loss for the same inputs and targets
 *                   (same per-pixel arithmetic and per-warp partials as its C-generic epilogue; the partials are added in
 *                   double in an order fixed by tile position, so the result is bit-reproducible in every mode, and the
 *                   normalisers out[4..6] equal the fused forward's).  t: as there; any target may be NULL.
 *      image_label  (I,H,W) uint8: hit voxel v ? min(pred_labels[v], C) : C, or NULL.
 *      confusion    (C+1)^2 device uint64, cleared and then confusion[min(target_label, C) * (C + 1) + label] = number of
 *                   pixels (integer atomics: deterministic), or NULL.  Needs t->target_label.
 *    vals_color may be NULL without t->target_color, vals_semantic without t->target_label.  No normals are read; nothing else
 *    is written: no float image, no mapping3dto2d(_num), no work list, no hit records, no gradient rows -- so no backward
 *    may follow it on this workspace.  Index routes and flags as in spsg_raycast_labels (every flag but the march's debug
 *    switches and the index routes is ignored, SPSG_FLAG_DETERMINISTIC included: the result does not depend on it).  Needs
 *    no more workspace than spsg_workspace_bytes(p), and scratch_bytes >= spsg_raycast_eval_scratch_bytes(p); both
 *    256-byte aligned.  Every argument is checked before anything is enqueued. */
SPSG_API int spsg_raycast_eval(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                               const float *vals_sdf, const float *vals_color, const float *vals_semantic,
                               const uint8_t *pred_labels, const float *view_matrix, const float *intrinsics,
                               const spsg_loss_targets *t, float *loss_out, uint8_t *image_label, uint64_t *confusion,
                               void *scratch, size_t scratch_bytes, void *workspace, size_t workspace_bytes, void *stream);

/* Scratch of spsg_raycast_eval (8 floats per 8x4-pixel warp tile of the batch, plus a few KB); 0 for invalid params. */
SPSG_API size_t spsg_raycast_eval_scratch_bytes(const spsg_raycast_params *p);

/* == raycast_rgbd_cuda.backward (raycast_rgbd_cuda.cpp:102-140, raycast_rgbd_cuda_kernel.cu:365-423,
 *    535-586): d_x[v] = sum over views of mean over the first min(num, max_pixels) pixels registered to
 *    voxel v of grad_x[pixel].  Rows [0, N) of every d_* are fully written (zeros where nothing hit);
 *    rows >= N are left untouched (the reference zero-fills the whole buffer, Python only ever
 *    returns [:N], raycast_rgbd.py:42).  Per-voxel sums are accumulated in double precision and rounded once.  With one view
 *    per chunk (the reference's case) results are written with plain stores, no float atomics.  They are bit-identical from
 *    run to run only when no row got more than max_pixels_per_voxel pixels: which pixels an overflowing row keeps depends on
 *    which warp of the forward reached it first.  With several views per chunk the per-view means are added with float
 *    atomics (last-bit differences between runs, like the reference's own atomics) unless SPSG_FLAG_DETERMINISTIC_GRADS is
 *    set, which adds them in view order with plain stores.  With SPSG_FLAG_DETERMINISTIC (forward and backward) gradients
 *    are always bit-identical from run to run. */
SPSG_API int spsg_raycast_backward(const spsg_raycast_params *p, const float *grad_color, const float *grad_depth,
                                   const float *grad_normal, const float *grad_semantic,
                                   const int32_t *sparse_mapping, const int32_t *mapping3dto2d,
                                   const int32_t *mapping3dto2d_num, float *d_color, float *d_depth,
                                   float *d_normal, float *d_semantic, void *workspace, size_t workspace_bytes,
                                   void *stream);

/* == raycast_rgbd_cuda.raycast_occ (raycast_rgbd_cuda.cpp:142-153, raycast_rgbd_cuda_kernel.cu:300-344,
 *    589-623).  occ3d u8 (B,1,Dz,Dy,Dx), occ2d u8 (B,1,H,W); uses width,height,depth_min,depth_max,
 *    ray_increment,dim*,num_chunks of `p`. */
SPSG_API int spsg_raycast_occ(const spsg_raycast_params *p, const uint8_t *occ3d, uint8_t *occ2d,
                              const float *view_matrix, const float *intrinsics, void *stream);

/* Fused forward + 2D losses: renders like spsg_raycast_forward_indexed and writes the three loss terms of `t`,
 * their weighted total and their normalisers into loss_out (SPSG_LOSS_OUT_FLOATS device floats). */
SPSG_API int spsg_raycast_forward_loss(const spsg_raycast_params *p, int32_t *sparse_mapping, const int64_t *locs,
                                       const float *vals_sdf, const float *vals_color, const float *vals_normal,
                                       const float *vals_semantic, const float *view_matrix,
                                       const float *intrinsics, float *image_color, float *image_depth,
                                       float *image_normal, float *image_semantic, int32_t *mapping3dto2d,
                                       int32_t *mapping3dto2d_num, const spsg_loss_targets *t, float *loss_out,
                                       const spsg_grad_buffers *clear_grads, void *workspace, size_t workspace_bytes,
                                       void *stream);

/* Fused backward of the 2D losses through the raycast: the upstream gradient images are never
 * materialised; each registered pixel's gradient is recomputed from (rendering, target, loss_out).
 * grad_scale: device scalar multiplying everything (d objective / d out[3]); NULL means 1.
 * The renderings must be those the matching spsg_raycast_forward_loss wrote, unmodified: the forward fills every pixel
 * registered to a voxel with that voxel's colour and logits, so the backward reads them once per (voxel, view), from one
 * of its pixels, and reads only the depth and the targets per pixel. */
SPSG_API int spsg_raycast_backward_loss(const spsg_raycast_params *p, const float *image_color,
                                        const float *image_depth, const float *image_semantic,
                                        const spsg_loss_targets *t, const float *loss_out, const float *grad_scale,
                                        const int32_t *sparse_mapping, const int32_t *mapping3dto2d,
                                        const int32_t *mapping3dto2d_num, float *d_color, float *d_depth,
                                        float *d_normal, float *d_semantic, void *workspace, size_t workspace_bytes,
                                        void *stream);

/* Gradients of an objective with respect to the four renderings of a fused forward, from terms the library does not
 * compute itself (a patch-GAN discriminator or a style loss on the rendered colour and normals). */
typedef struct spsg_upstream_grads {   /* d objective / d rendering, same layouts as the images; NULL plane = 0 */
    const float *grad_color;    /* (I,H,W,3)  */
    const float *grad_depth;    /* (I,H,W)    */
    const float *grad_normal;   /* (I,H,W,3)  */
    const float *grad_semantic; /* (I,H,W,14), 8-byte aligned */
} spsg_upstream_grads;

/* spsg_raycast_backward_loss that also gathers caller-supplied upstream gradient images, in the same launch:
 *     d_x[v] = sum over views of mean over the pixels registered to voxel v of
 *              (recomputed 2D-loss gradient * grad_scale + upstream gradient)
 * Upstream gradients are not multiplied by grad_scale.  Gradients at pixels that hit nothing are ignored, as in
 * spsg_raycast_backward.  Loss targets switched off (NULL target pointers) give exactly spsg_raycast_backward of the
 * upstream images; upstream NULL, or all four planes NULL, gives exactly spsg_raycast_backward_loss.  The renderings must be
 * those of the matching spsg_raycast_forward_loss, unmodified (see spsg_raycast_backward_loss). */
SPSG_API int spsg_raycast_backward_loss_upstream(const spsg_raycast_params *p, const float *image_color,
                                                 const float *image_depth, const float *image_semantic,
                                                 const spsg_loss_targets *t, const float *loss_out,
                                                 const float *grad_scale, const spsg_upstream_grads *upstream,
                                                 const int32_t *sparse_mapping, const int32_t *mapping3dto2d,
                                                 const int32_t *mapping3dto2d_num, float *d_color, float *d_depth,
                                                 float *d_normal, float *d_semantic, void *workspace,
                                                 size_t workspace_bytes, void *stream);

/* == loss.compute_normals_sparse (reference torch/loss.py:285-306, with compute_normals_dense :261-267): per-voxel
 *    normals of the sparse SDF, the producer of the raycaster's vals_normals (train.py:542).  normals[i] =
 *    -normalize(R_chunk * central_difference(sdf at voxel i), eps 1e-5); absent neighbours count as 0, voxels on the
 *    volume border get 0.  transform: (B,4,4) row-major (its upper-left 3x3 is R) or NULL.  `index` is caller-owned
 *    scratch of B*Dz*Dy*Dx int32 (the voxel index, same content as sparse_mapping); the forward fills it, the
 *    backward reads it.  One fill + one scatter + one gather launch; no dense volumes, no per-chunk host loop. */
SPSG_API int spsg_normals_forward(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                                  int32_t *index, int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx,
                                  float *normals, void *stream);

/* Gradient of the above w.r.t. vals_sdf: d_sdf (N,1) is fully written.  scratch_u: N*3 floats of caller-owned
 *    scratch.  Two gather launches, deterministic (no atomics). */
SPSG_API int spsg_normals_backward(const int64_t *locs, int64_t num_locs, const float *vals_sdf, const float *transform,
                                   const int32_t *index, int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx,
                                   const float *grad_normals, float *scratch_u, float *d_sdf, void *stream);

/* Per-view normals for renders with several views per chunk (SPSG_FLAG_VIEW_NORMALS): the central difference g is
 *    computed once per voxel, then normals[(i*F + f)*3 ..] = -normalize(R_{b*F+f} * g), b = chunk of voxel i, with the
 *    arithmetic of spsg_normals_forward.  normals: (N,F,3); transform: (B*F,4,4), the inverse view matrices of the
 *    render's images in image order, required when F > 1.  views_per_chunk == 1 is exactly spsg_normals_forward.
 *    views_per_chunk <= 0, or a NULL transform with F > 1, is SPSG_ERR_INVALID_ARGUMENT. */
SPSG_API int spsg_normals_forward_views(const int64_t *locs, int64_t num_locs, const float *vals_sdf,
                                        const float *transform, int32_t views_per_chunk, int32_t *index,
                                        int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, float *normals,
                                        void *stream);

/* Gradient of spsg_normals_forward_views w.r.t. vals_sdf.  grad_normals: (N,F,3).  Pass 1 writes u = dL/dg (N,3) into
 *    scratch_u, the per-view terms of spsg_normals_backward summed in view order; pass 2 is spsg_normals_backward's
 *    neighbour gather.  views_per_chunk == 1 is exactly spsg_normals_backward; same argument checks as the forward. */
SPSG_API int spsg_normals_backward_views(const int64_t *locs, int64_t num_locs, const float *vals_sdf,
                                         const float *transform, int32_t views_per_chunk, const int32_t *index,
                                         int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx,
                                         const float *grad_normals, float *scratch_u, float *d_sdf, void *stream);

/* The 2D losses as stand-alone image-space ops, i.e. at the boundary the reference applies them: to rendered images
 *    (depth L1 train.py:635-638, colour L1 loss.compute_2dcolor_loss loss.py:246-257, 2D semantic CE train.py:744-746).
 *    Same terms, targets struct and loss_out block as spsg_raycast_forward_loss; a rendering pointer may be NULL when its
 *    target is NULL.  scratch: >= 4096 bytes, 8-byte aligned.  One pass over the pixels + finalize. */
SPSG_API int spsg_losses2d_forward(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                                   const float *image_semantic, int64_t num_pixels, float *loss_out, void *scratch,
                                   size_t scratch_bytes, void *stream);

/* spsg_losses2d_forward with the sums in an order fixed by pixel position (SPSG_FLAG_DETERMINISTIC): bit-identical
 *    loss_out from run to run, whatever the device's SM count.  scratch: spsg_losses2d_deterministic_scratch_bytes(num_pixels)
 *    bytes, 8-byte aligned. */
SPSG_API size_t spsg_losses2d_deterministic_scratch_bytes(int64_t num_pixels);
SPSG_API int spsg_losses2d_forward_deterministic(const spsg_loss_targets *t, const float *image_color,
                                                 const float *image_depth, const float *image_semantic, int64_t num_pixels,
                                                 float *loss_out, void *scratch, size_t scratch_bytes, void *stream);

/* Gradient images of grad_scale * loss_out[3] w.r.t. the renderings (one thread per pixel, no atomics: deterministic): d_color (P,3), d_depth (P), d_semantic (P,14), any
 *    of them NULL to skip; pixels outside a term's valid set get 0. */
SPSG_API int spsg_losses2d_backward(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                                    const float *image_semantic, int64_t num_pixels, const float *loss_out,
                                    const float *grad_scale, float *d_color, float *d_depth, float *d_semantic,
                                    void *stream);

/* The three stand-alone 2D-loss calls above with C = num_classes logits per pixel (1..64): image_semantic and d_semantic
 *    (P,C), class_weight (C), target_label C = ignore; no alignment beyond 4 bytes.  These always run the C-generic kernels,
 *    also at C = 14, where they give the results of the 14-channel calls (the deterministic forward bit for bit). */
SPSG_API int spsg_losses2d_forward_classes(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                                           const float *image_semantic, int32_t num_classes, int64_t num_pixels,
                                           float *loss_out, void *scratch, size_t scratch_bytes, void *stream);
SPSG_API int spsg_losses2d_forward_deterministic_classes(const spsg_loss_targets *t, const float *image_color,
                                                         const float *image_depth, const float *image_semantic,
                                                         int32_t num_classes, int64_t num_pixels, float *loss_out,
                                                         void *scratch, size_t scratch_bytes, void *stream);
SPSG_API int spsg_losses2d_backward_classes(const spsg_loss_targets *t, const float *image_color, const float *image_depth,
                                            const float *image_semantic, int32_t num_classes, int64_t num_pixels,
                                            const float *loss_out, const float *grad_scale, float *d_color,
                                            float *d_depth, float *d_semantic, void *stream);

/* ---- host side of a host-fed call.  The reference hands its voxel rows to the GPU as int64 (z,y,x,b) -- 32 bytes per voxel, 28
 *      of them zero -- (raycast_rgbd.py:22-28; data_util.py builds them from the chunk file's uint32 triples).  This packs them,
 *      on the host, into what the index pass derives from them anyway: one uint32 linear cell index ((b*Dz+z)*Dy+y)*Dx+x per
 *      row (0xffffffff for a row outside the grid, which the device skips like the int64 path does), to be written straight
 *      into the pinned staging buffer and passed as `locs` with SPSG_FLAG_PACKED_LOCS: 4 instead of 32 bytes per voxel over
 *      PCIe.  Plain host pointers, `threads` OpenMP threads (clamped to 1..64), no CUDA call.  Needs B*Dz*Dy*Dx < 2^32 - 1. */
SPSG_API int spsg_pack_locs_host(const int64_t *locs, int64_t num_locs, int32_t num_chunks, int32_t dimz, int32_t dimy,
                                 int32_t dimx, uint32_t *cells_out, int32_t threads);

/* ---- depth-frame utilities: the reference's second extension on the training step, torch/utils/depth_utils
 *      (depth_utils_cuda.cpp:80-85, depth_utils_cuda_kernel.cu; Python depth_utils.py:46-100).  Images are (B,1,H,W)
 *      f32 depth in metres (0 = hole), camera space / normals (B,H,W,3), intrinsics (B,4) = fx,fy,mx,my. ---- */
#define SPSG_DEPTH_MAX_FILL_ROUNDS 64

/* == depth_utils_cuda.bilateral_filter_floatmap (depth_utils_cuda_kernel.cu:41-86, 215-243) */
SPSG_API int spsg_depth_bilateral_filter(const float *depth, float *filtered, int32_t batch, int32_t height, int32_t width,
                                         float sigma_d, float sigma_r, void *stream);

/* == depth_utils_cuda.median_fill_depthmap(out, in) (depth_utils_cuda_kernel.cu:89-140, 245-268): 11x11 median fill of
 *    hole pixels, everything else copied.  Not in place. */
SPSG_API int spsg_depth_median_fill(const float *in, float *out, int32_t batch, int32_t height, int32_t width, void *stream);

/* == depth_utils_cuda.convert_depth_to_cameraspace (depth_utils_cuda_kernel.cu:142-170, 296-323) */
SPSG_API int spsg_depth_to_cameraspace(const float *depth, const float *intrinsics, float *camspace, int32_t batch,
                                       int32_t height, int32_t width, void *stream);

/* == depth_utils_cuda.compute_normals (depth_utils_cuda_kernel.cu:172-211, 270-294): camera space (B,H,W,3) -> normals */
SPSG_API int spsg_depth_compute_normals(const float *camspace, float *normals, int32_t batch, int32_t height,
                                        int32_t width, void *stream);

/* == Depth2Normals.forward (depth_utils.py:84-100) enqueued in one go: bilateral filter into `filtered`, up to
 *    max_fill_iters/2 rounds of { depth <- fill(filtered); filtered <- fill(depth) } that modify `depth` IN PLACE like the
 *    reference and stop on the device as soon as a round leaves no hole, then camera space (may be NULL) + normals
 *    (depth_utils_cuda_kernel.cu:172-211) from the filled depth.  hole_counts: SPSG_DEPTH_MAX_FILL_ROUNDS + 1 device
 *    int32; [0] = holes of the input, [r] = holes left after round r (0 for rounds that did not run).  The caller reads
 *    hole_counts[max_fill_iters / 2] (one synchronisation) to decide whether the reference would have returned None.
 *    Two launches: the filter, then one cooperative grid-resident kernel for the fill rounds and the normals (devices without
 *    cooperative launch, or the environment variable SPSG_DEPTH_NO_COOPERATIVE, get one launch per pass; same results). */
SPSG_API int spsg_depth_to_normals(float *depth, const float *intrinsics, float *filtered, float *camspace, float *normals,
                                   int32_t *hole_counts, int32_t batch, int32_t height, int32_t width, float sigma_d,
                                   float sigma_r, int32_t max_fill_iters, void *stream);

/* == Producer glue of the training step (reference torch/train.py:494-509): which voxels of the generator's dense SDF
 *    head enter the raycaster, in which order, and their payloads.  Replaces
 *        locs = torch.nonzero((torch.abs(output_sdf.detach()[:, 0]) < truncation) [& ~empty[:, 0]])   train.py:495-497
 *        locs = torch.cat([locs[:, 1:], locs[:, :1]], 1)                                               train.py:498
 *        vals = head[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]]   for every head              train.py:499-508
 *    and the index_put backward of those gathers.  Rows come out in torch.nonzero's order (lexicographic in b, z, y, x)
 *    with columns (z, y, x, b), i.e. exactly the `locs` the raycaster takes.
 *
 *    1. spsg_sparsify_count  -> *total_out (device int64) = N; the caller reads it back (the one host synchronisation the
 *       reference's nonzero has too) and allocates locs (N,4) int64 and the value tensors;
 *    2. spsg_sparsify_locs   -> locs, using the offsets step 1 left in `scratch`;
 *    3. spsg_dense_gather    -> sparse[i, c] = dense[b_i, c, z_i, y_i, x_i] for up to 4 heads in one launch;
 *       spsg_dense_scatter   -> the backward: dense := 0, then dense[b_i, c, z_i, y_i, x_i] = sparse[i, c].
 *    sdf: (B,Dz,Dy,Dx) float32, 16-byte aligned (channel 0 of a contiguous (B,1,Dz,Dy,Dx) head); empty: same shape,
 *    one byte per cell (torch.bool), 8-byte aligned, or NULL; cells = B*Dz*Dy*Dx; scratch: caller-owned,
 *    spsg_sparsify_scratch_bytes(cells) bytes, 256-byte aligned.  |sdf| < truncation is false for NaN, like torch. */
typedef struct spsg_dense_payload {
    float *dense;      /* (B, channels, Dz, Dy, Dx) contiguous; read by gather, written by scatter */
    float *sparse;     /* (N, channels) contiguous; written by gather, read by scatter */
    int32_t channels;
    int32_t reserved;
} spsg_dense_payload;
SPSG_API size_t spsg_sparsify_scratch_bytes(int64_t cells);
SPSG_API int spsg_sparsify_count(const float *sdf, const uint8_t *empty, int64_t cells, float truncation, void *scratch,
                                 size_t scratch_bytes, int64_t *total_out, void *stream);
SPSG_API int spsg_sparsify_locs(const float *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz, int32_t dimy,
                                int32_t dimx, float truncation, const void *scratch, int64_t *locs, int64_t num_locs,
                                void *stream);
/* Step 2 feeding the raycaster directly (SURVEY.md section 8(f) rank 1): as spsg_sparsify_locs, and in the same pass, for EVERY
 * cell of the grid, what construct_dense_sparse_mapping (raycast_rgbd_cuda_kernel.cu:346-362, 506-533) and this
 * implementation's dense-brick pass would derive from those rows afterwards: sparse_mapping[cell] = row of the cell or -1,
 * and the dense SDF brick at the start of `raycast_workspace` (its first B*Dz*Dy*Dx floats; the workspace of the forward
 * that will render these rows, at least spsg_raycast_workspace_bytes() of that call) = the cell's SDF or "absent".  A
 * forward over exactly these rows, with vals_sdf = the gathered head values, may then be called with
 * SPSG_FLAG_INDEX_PREBUILT.  sparse_mapping: (B,Dz,Dy,Dx) int32; it and the workspace 16-byte aligned; num_locs < 2^31. */
SPSG_API int spsg_sparsify_locs_indexed(const float *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                        int32_t dimy, int32_t dimx, float truncation, const void *scratch, int64_t *locs,
                                        int64_t num_locs, int32_t *sparse_mapping, void *raycast_workspace, void *stream);
SPSG_API int spsg_dense_gather(const spsg_dense_payload *payloads, int32_t count, const int64_t *locs, int64_t num_locs,
                               int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream);
SPSG_API int spsg_dense_scatter(const spsg_dense_payload *payloads, int32_t count, const int64_t *locs, int64_t num_locs,
                                int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream);

/* == The same glue on heads as a generator in channels_last_3d and/or under bfloat16 autocast produces them.
 *
 *    Compaction of a bfloat16 SDF head: spsg_sparsify_count_bf16 / spsg_sparsify_locs_bf16 /
 *    spsg_sparsify_locs_indexed_bf16 take `sdf` as B*Dz*Dy*Dx bfloat16 values (raw bits; a (B,1,Dz,Dy,Dx) head is
 *    contiguous in NCDHW and NDHWC alike), 16-byte aligned, and are otherwise exactly their float32 counterparts.  The
 *    comparison is torch's for a bfloat16 tensor and a Python scalar: `truncation` is first rounded to bfloat16 (nearest
 *    even), then |sdf| < rounded truncation is evaluated (NaN fails).  The indexed variant writes the widened value into
 *    the float32 SDF brick, which equals the gathered vals_sdf below, so SPSG_FLAG_INDEX_PREBUILT holds as before.
 *
 *    Gather / scatter of strided heads: spsg_dense_gather_strided / spsg_dense_scatter_strided, up to 4 heads per call.
 *    Element (b, c, z, y, x) of a head is at dense + b*strides[0] + c*strides[1] + z*strides[2] + y*strides[3] +
 *    x*strides[4] (in elements of its dtype); NCDHW- and NDHWC-contiguous heads and channel slices of either are all
 *    expressible.  gather: sparse[i, c] = (float) dense[b_i, c, z_i, y_i, x_i], exact (bfloat16 widens exactly).
 *    scatter: the head's B*C*Dz*Dy*Dx elements are zeroed, then dense[b_i, c, z_i, y_i, x_i] = 0 + round(sparse[i, c]),
 *    rounded to the head's dtype to nearest even; each cell takes at most one row, so this is autograd of
 *    head[idx].float() bit for bit (including -0 -> +0).  The scatter's head must be packed: its strides a permutation of a
 *    contiguous layout (dimensions of size 1 excepted).
 *    SPSG_ERR_INVALID_ARGUMENT: NULL heads / dense / sparse (sparse may be NULL when num_locs == 0) / locs, an unknown
 *    dtype, channels or grid sizes <= 0, a negative stride, a head whose last element lies at or beyond `extent`, a dense
 *    pointer not aligned to its element size, a scatter head that is not packed, more than 4 heads. */
enum { SPSG_DTYPE_F32 = 0, SPSG_DTYPE_BF16 = 1 };
typedef struct spsg_dense_head {
    void *dense;         /* the head, SPSG_DTYPE_* elements; read by gather, written by scatter */
    float *sparse;       /* (N, channels) float32 contiguous; written by gather, read by scatter */
    int64_t strides[5];  /* (b, c, z, y, x), in elements, >= 0 */
    int64_t extent;      /* elements addressable from `dense` (the head's storage from `dense` on) */
    int32_t channels;
    int32_t dtype;       /* SPSG_DTYPE_F32 or SPSG_DTYPE_BF16 */
} spsg_dense_head;
SPSG_API int spsg_sparsify_count_bf16(const uint16_t *sdf, const uint8_t *empty, int64_t cells, float truncation,
                                      void *scratch, size_t scratch_bytes, int64_t *total_out, void *stream);
SPSG_API int spsg_sparsify_locs_bf16(const uint16_t *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                     int32_t dimy, int32_t dimx, float truncation, const void *scratch, int64_t *locs,
                                     int64_t num_locs, void *stream);
SPSG_API int spsg_sparsify_locs_indexed_bf16(const uint16_t *sdf, const uint8_t *empty, int32_t num_chunks, int32_t dimz,
                                             int32_t dimy, int32_t dimx, float truncation, const void *scratch,
                                             int64_t *locs, int64_t num_locs, int32_t *sparse_mapping,
                                             void *raycast_workspace, void *stream);
SPSG_API int spsg_dense_gather_strided(const spsg_dense_head *heads, int32_t count, const int64_t *locs, int64_t num_locs,
                                       int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream);
SPSG_API int spsg_dense_scatter_strided(const spsg_dense_head *heads, int32_t count, const int64_t *locs, int64_t num_locs,
                                        int32_t num_chunks, int32_t dimz, int32_t dimy, int32_t dimx, void *stream);

/* == 2D label maps (reference torch/train.py:614-616 target2d_label, :749-752 pred2d_label):
 *        label = argmax(cat(raycast_semantic, ones), -1).to(uint8)
 *    = first index of the pixel's maximum among its 14 rendered values if that maximum is >= 1, else 14 (miss or
 *    unlabeled); NaN counts as the maximum, like torch.max.  semantic: (P,14) float32, 8-byte aligned; labels: P bytes;
 *    hist: 15 device int64 (cleared, then the number of pixels per label) or NULL. */
SPSG_API int spsg_labels_from_render(const float *semantic, int64_t num_pixels, uint8_t *labels, int64_t *hist,
                                     void *stream);

/* spsg_labels_from_render over C = num_classes (1..64) channels: semantic (P,C), 4-byte aligned; label C = miss or
 *    unlabeled; hist: C + 1 device int64 or NULL. */
SPSG_API int spsg_labels_from_render_classes(const float *semantic, int32_t num_classes, int64_t num_pixels,
                                             uint8_t *labels, int64_t *hist, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SPSG_RAYCAST_H_ */
